"""ctypes binding of include/arp_b200.h.

This is the only place Python touches the native library. There is no CPU path: if the shared
library is missing or no sm_100 device is present, construction raises — it never falls back.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np
import torch

_PKG = Path(__file__).resolve().parent
_LIB_PATH = Path(os.environ.get("ARP_B200_LIB") or _PKG / "_lib" / "libarp_b200.so")   # env override: dev builds only

ARP_OK = 0
ARP_ERR_INVALID, ARP_ERR_CUDA, ARP_ERR_STATE, ARP_ERR_NO_DEVICE, ARP_ERR_UNKNOWN_KEY = -1, -2, -3, -4, -5
PRE_PIL_BICUBIC, PRE_BILINEAR = 0, 1
HEAD_CLIP, HEAD_ADAPTER, HEAD_ADAPTER_ENSEMBLE, HEAD_CLIP_GOAL, HEAD_ADAPTER_GOAL = 0, 1, 2, 3, 4
REDUCE_FIRST, REDUCE_MEAN = 0, 1
DT_F32, DT_BF16, DT_F16 = 0, 1, 2
ACT_NONE, ACT_QUICKGELU, ACT_RELU = 0, 1, 2
PREC_BF16, PREC_F32, PREC_F32RESID = 0, 1, 2   # PREC_BF16 = the 16-bit tensor-core path (name is historical)
PREC_16BIT = PREC_BF16
#: precision names of the Python entry points ("bf16" / "fp16" name the 16-bit path whatever the operand format)
PRECISIONS = {"16bit": PREC_16BIT, "bf16": PREC_16BIT, "fp16": PREC_16BIT, "fp32resid": PREC_F32RESID, "fp32": PREC_F32}
#: ArpInflateStatus: per-row result of the device zlib inflate (inflate_rows)
(ARP_INFLATE_OK, ARP_INFLATE_TRUNCATED, ARP_INFLATE_BAD_HEADER, ARP_INFLATE_BAD_BLOCK, ARP_INFLATE_BAD_CODE,
 ARP_INFLATE_DISTANCE_TOO_FAR, ARP_INFLATE_TOO_LONG, ARP_INFLATE_TOO_SHORT, ARP_INFLATE_BAD_ADLER) = range(9)
MAX_TEXT = 16            # texts of one instruction set (one text group)
MAX_TEXT_GROUPS = 16     # instruction sets of one set_text_groups call
MAX_TEXT_TOTAL = 64      # texts of all groups together

#: every symbol include/arp_b200.h declares (tests check the library exports exactly these)
EXPORTS = (
    "arp_create", "arp_destroy", "arp_last_error", "arp_abi_version", "arp_set_weight", "arp_missing_weights",
    "arp_set_text", "arp_label", "arp_label_host", "arp_compute_reward", "arp_encode_image", "arp_decode_only",
    "arp_scan_only", "arp_gemm_bf16", "arp_layernorm_bf16", "arp_attention", "arp_launch_count",
    "arp_profile_begin", "arp_profile_end", "arp_online_reward", "arp_preprocess_rtgs",
    "arp_quantile_f32", "arp_encode_taps_chw", "arp_operand_dtype", "arp_ln_gemm", "arp_resid_gemm_stats", "arp_label_file", "arp_wants_weight",
    "arp_set_text_groups", "arp_text_groups", "arp_embedding_dim", "arp_embed_host", "arp_embed_file",
    "arp_label_embeddings", "arp_tower_dim", "arp_embed_tower_host", "arp_embed_tower_file", "arp_label_tower",
    "arp_label_zfile", "arp_embed_zfile", "arp_embed_tower_zfile", "arp_inflate_rows",
    "arp_label_zchunks", "arp_embed_zchunks", "arp_embed_tower_zchunks", "arp_gather_frames", "arp_cls_attention",
)
PROFILE_CLASSES = ("gemm", "attention", "layernorm", "decode", "head", "scan", "other")


class ArpProfileStats(C.Structure):
    _fields_ = [("launches", C.c_int64), ("total_ms", C.c_double), ("flops", C.c_double), ("bytes", C.c_double)]


class ArpConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "struct_size", "device", "patch", "width", "layers", "heads", "embed_dim", "in_h", "in_w", "use_crop",
        "preprocess", "head", "reduce", "max_batch", "precision")]


class ArpChunkLayout(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("ndim", C.c_int32), ("shape", C.c_int64 * 5), ("chunk", C.c_int64 * 5)]


#: device scratch bound of one max_batch batch's inflated chunks (ARP_ZCHUNK_SCRATCH_BYTES)
ZCHUNK_SCRATCH_BYTES = 4 << 30
#: largest compressed chunk the compressed-chunk calls take (ARP_ZCHUNK_MAX_COMPRESSED_BYTES)
ZCHUNK_MAX_COMPRESSED_BYTES = 64 << 20


def chunk_layout(shape, chunks) -> ArpChunkLayout:
    """ArpChunkLayout of a uint8 dataset `shape` ([T, F, H, W, 3] or [T, H, W, 3]) stored in chunks of shape `chunks`"""
    assert len(shape) == len(chunks) and len(shape) in (4, 5), (shape, chunks)
    pad = (0,) * (5 - len(shape))
    return ArpChunkLayout(C.sizeof(ArpChunkLayout), len(shape), (C.c_int64 * 5)(*shape, *pad),
                          (C.c_int64 * 5)(*chunks, *pad))


class ArpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"arp_b200 error {code}: {msg}")
        self.code = code


_lib = None


def precision_enum(name: str) -> int:
    """The PREC_* value of a precision name; ValueError naming the valid ones otherwise."""
    if name not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {name!r}")
    return PRECISIONS[name]


def lib_path() -> Path:
    return _LIB_PATH


def load_library() -> C.CDLL:
    """dlopen the in-tree library and declare its prototypes. Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise FileNotFoundError(
            f"{_LIB_PATH} not built — run `python -m arp_b200.build` (or __graft_entry__.build()). "
            "arp_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(os.fspath(_LIB_PATH))
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    lib.arp_create.argtypes = [C.POINTER(ArpConfig), C.POINTER(vp)]
    lib.arp_destroy.argtypes = [vp]
    lib.arp_destroy.restype = None
    lib.arp_last_error.argtypes = [vp]
    lib.arp_last_error.restype = C.c_char_p
    lib.arp_abi_version.argtypes = []
    lib.arp_operand_dtype.argtypes = []
    lib.arp_set_weight.argtypes = [vp, C.c_char_p, vp, i32, C.POINTER(i64), i32, vp]
    lib.arp_missing_weights.argtypes = [vp, C.c_char_p, i64]
    lib.arp_set_text.argtypes = [vp, vp, i32, i32, f32, vp]
    lib.arp_set_text_groups.argtypes = [vp, vp, i32, i32, vp, i32, f32, vp]
    lib.arp_text_groups.argtypes = [vp]
    lib.arp_label.argtypes = [vp, vp, i64, i64, vp, i32, i32, vp, vp, vp, vp, vp]
    lib.arp_label_host.argtypes = [vp, vp, i64, i64, vp, i32, i32, vp, vp, vp, vp]
    lib.arp_label_file.argtypes = [vp, i32, i64, i64, i64, vp, i32, i32, vp, vp, vp, vp]
    lib.arp_wants_weight.argtypes = [vp, C.c_char_p]
    lib.arp_embedding_dim.argtypes = [vp]
    lib.arp_embed_host.argtypes = [vp, vp, i64, i64, vp]
    lib.arp_embed_file.argtypes = [vp, i32, i64, i64, i64, vp]
    lib.arp_label_embeddings.argtypes = [vp, vp, i64, vp, i32, i32, vp, vp, vp, vp, vp]
    lib.arp_tower_dim.argtypes = [vp]
    lib.arp_embed_tower_host.argtypes = [vp, vp, i64, i64, vp]
    lib.arp_embed_tower_file.argtypes = [vp, i32, i64, i64, i64, vp]
    lib.arp_label_tower.argtypes = [vp, vp, i64, vp, i32, i32, vp, vp, vp, vp, vp]
    lib.arp_label_zfile.argtypes = [vp, i32, vp, vp, i64, i64, vp, i32, i32, vp, vp, vp, vp]
    lib.arp_embed_zfile.argtypes = [vp, i32, vp, vp, i64, i64, vp]
    lib.arp_embed_tower_zfile.argtypes = [vp, i32, vp, vp, i64, i64, vp]
    lib.arp_inflate_rows.argtypes = [vp, vp, vp, vp, i64, i64, vp, vp, vp]
    lay = C.POINTER(ArpChunkLayout)
    lib.arp_label_zchunks.argtypes = [vp, i32, lay, vp, vp, vp, i64, i64, i64, vp, i32, i32, vp, vp, vp, vp]
    lib.arp_embed_zchunks.argtypes = [vp, i32, lay, vp, vp, vp, i64, i64, i64, vp]
    lib.arp_embed_tower_zchunks.argtypes = [vp, i32, lay, vp, vp, vp, i64, i64, i64, vp]
    lib.arp_gather_frames.argtypes = [vp, lay, i64, i64, vp, vp, vp]
    lib.arp_compute_reward.argtypes = [vp, vp, i64, i64, vp, vp, vp]
    lib.arp_online_reward.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.arp_preprocess_rtgs.argtypes = [vp, vp, i64, vp, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.arp_quantile_f32.argtypes = [vp, vp, i64, i64, i64, vp, vp]
    lib.arp_encode_taps_chw.argtypes = [vp, vp, i64, vp, vp, vp]
    lib.arp_encode_image.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.arp_decode_only.argtypes = [vp, vp, i64, i64, vp, vp]
    lib.arp_scan_only.argtypes = [vp, vp, i64, vp, i32, i32, f32, vp, vp, vp, vp]
    lib.arp_gemm_bf16.argtypes = [vp, vp, vp, vp, i32, i64, i32, i32, vp, vp, i32, vp]
    lib.arp_ln_gemm.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]
    lib.arp_resid_gemm_stats.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]
    lib.arp_layernorm_bf16.argtypes = [vp, vp, vp, vp, vp, i64, vp]
    lib.arp_attention.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.arp_cls_attention.argtypes = [vp, vp, vp, vp, i32, i32, vp]
    lib.arp_launch_count.argtypes = [vp]
    lib.arp_launch_count.restype = i64
    lib.arp_profile_begin.argtypes = [vp]
    lib.arp_profile_end.argtypes = [vp, C.POINTER(ArpProfileStats), i32]
    for name in EXPORTS:
        if name not in ("arp_destroy", "arp_last_error", "arp_launch_count"):
            getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


_TORCH_DT = {torch.float32: DT_F32, torch.bfloat16: DT_BF16, torch.float16: DT_F16}


def operand_dtype() -> torch.dtype:
    """The 16-bit format the library's contractions run in (bf16 unless it was built with -DARP_OP_FP16=1)."""
    return {DT_BF16: torch.bfloat16, DT_F16: torch.float16}[load_library().arp_operand_dtype()]


def _ptr(t: "torch.Tensor | None"):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """One native handle on one GPU. Thin: argument checking + pointer plumbing only."""

    def __init__(self, *, device: int = 0, patch: int = 16, in_h: int = 64, in_w: int = 64, use_crop: bool = False,
                 preprocess: int = PRE_PIL_BICUBIC, head: int = HEAD_CLIP, reduce: int = REDUCE_FIRST,
                 max_batch: int = 256, layers: int = 12, width: int = 768, heads: int = 12, embed_dim: int = 512,
                 precision: int = PREC_BF16):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.cfg = ArpConfig(C.sizeof(ArpConfig), device, patch, width, layers, heads, embed_dim, in_h, in_w,
                             int(bool(use_crop)), preprocess, head, reduce, max_batch, precision)
        rc = self._lib.arp_create(C.byref(self.cfg), C.byref(self._h))
        if rc != ARP_OK:
            raise ArpError(rc, (self._lib.arp_last_error(None) or b"").decode())
        self.device = torch.device("cuda", device)
        self.tokens = (224 // patch) ** 2 + 1
        self.adapter = head in (HEAD_ADAPTER, HEAD_ADAPTER_ENSEMBLE, HEAD_ADAPTER_GOAL)
        self.goal = head in (HEAD_CLIP_GOAL, HEAD_ADAPTER_GOAL)
        self.feat_dim = (layers + 1) * embed_dim if self.adapter else embed_dim
        self.n_text = 0
        self._grouped = False            # set_text_groups was called last: outputs carry a leading group axis

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.arp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != ARP_OK:
            raise ArpError(rc, (self._lib.arp_last_error(self._h) or b"").decode())

    @property
    def launch_count(self) -> int:
        return int(self._lib.arp_launch_count(self._h))

    def profile_begin(self):
        self._check(self._lib.arp_profile_begin(self._h))

    def profile_end(self) -> dict:
        """{class: {launches, total_ms, flops, bytes}} of the launches since profile_begin (device-synchronising)."""
        arr = (ArpProfileStats * len(PROFILE_CLASSES))()
        self._check(self._lib.arp_profile_end(self._h, arr, len(PROFILE_CLASSES)))
        return {n: {"launches": int(a.launches), "total_ms": a.total_ms, "flops": a.flops, "bytes": a.bytes}
                for n, a in zip(PROFILE_CLASSES, arr)}

    # -- weights / text ---------------------------------------------------------------------------
    def set_weight(self, name: str, tensor: torch.Tensor, strict: bool = True) -> bool:
        t = tensor.detach()
        if t.dtype not in _TORCH_DT:
            t = t.float()
        t = t.to(self.device).contiguous()
        shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
        rc = self._lib.arp_set_weight(self._h, name.encode(), _ptr(t), _TORCH_DT[t.dtype], shape, t.dim(),
                                      _stream_ptr(self.device))
        if rc == ARP_ERR_UNKNOWN_KEY and not strict:
            return False
        self._check(rc)
        torch.cuda.current_stream(self.device).synchronize()  # `t` may be a temporary
        return True

    def load_state_dict(self, state_dict, strict: bool = False) -> list[str]:
        """Feed every tensor of a CLIP (or adapter) state_dict; returns the names still missing. Tensors whose storage
        (data pointer, shape, dtype, in-place version counter) is exactly what this handle uploaded last time are skipped:
        labeling the same model again — another instruction, another dataset — does not pay for the upload twice. Only the
        very same tensor OBJECTS count (pass the same state_dict again; the handle keeps them referenced until it is closed)."""
        seen = getattr(self, "_uploaded", None)
        if seen is None:
            seen = self._uploaded = {}
        for k, v in state_dict.items():
            if not torch.is_tensor(v):
                continue
            if not strict and not self._lib.arp_wants_weight(self._h, k.encode()):
                continue                      # text tower / bookkeeping entries: never copied to the device
            mark = (v.data_ptr(), tuple(v.shape), v.dtype, v._version, v.device)
            if k in seen and seen[k][0] == mark and seen[k][1] is v:
                continue
            if self.set_weight(k, v, strict=strict):
                seen[k] = (mark, v)           # the reference keeps the storage alive: its address cannot be recycled
        return self.missing_weights()

    def missing_weights(self) -> list[str]:
        buf = C.create_string_buffer(1 << 16)
        n = self._lib.arp_missing_weights(self._h, buf, len(buf))
        return [s for s in buf.value.decode().split("\n") if s] if n else []

    def set_text(self, text_emb: torch.Tensor, logit_scale_exp: float):
        t = text_emb.detach().to(self.device, torch.float32).contiguous()
        assert t.dim() == 2
        self._check(self._lib.arp_set_text(self._h, _ptr(t), t.shape[0], t.shape[1], float(logit_scale_exp),
                                           _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()
        self.n_text = t.shape[0]
        self._grouped = False

    def set_text_groups(self, embs: "list[torch.Tensor]", logit_scale_exp: float):
        """G instruction sets at once: embs[g] is group g's [n_g, dim] embedding, as set_text takes it. From now on label,
        label_host, label_file and compute_reward score every group in one encoder pass and return arrays with a leading
        group axis [G, ...] (also for G = 1); group g equals what the same call returns after set_text(embs[g]).
        set_text goes back to one group and the plain shapes."""
        rows = [e.detach().to(self.device, torch.float32) for e in embs]
        assert rows and all(r.dim() == 2 for r in rows)
        t = torch.cat(rows).contiguous()
        off = np.concatenate([[0], np.cumsum([r.shape[0] for r in rows])]).astype(np.int32)
        self._check(self._lib.arp_set_text_groups(self._h, _ptr(t), t.shape[0], t.shape[1], C.c_void_p(off.ctypes.data),
                                                  len(rows), float(logit_scale_exp), _stream_ptr(self.device)))
        torch.cuda.current_stream(self.device).synchronize()
        self.n_text = t.shape[0]
        self._grouped = True

    @property
    def n_groups(self) -> int:
        """G of the text currently set (1 after set_text)."""
        return int(self._lib.arp_text_groups(self._h))

    def _lead(self) -> tuple:
        """leading shape of the per-frame outputs: (G,) after set_text_groups, () after set_text"""
        return (self.n_groups,) if self._grouped else ()

    def _host_outputs(self, T: int, num_frames: int):
        lead = self._lead()
        return (np.empty(lead + (T,), np.float32), np.empty(lead + (T,), np.float32),
                np.empty(lead + (T, num_frames), np.float32), np.empty(lead + (T, num_frames), np.float32))

    # -- hot path ---------------------------------------------------------------------------------
    @staticmethod
    def _frames_view(ob: torch.Tensor):
        """ob: uint8 [T,F,H,W,3] (reference layout; the LAST stacked frame is scored) or [T,H,W,3]."""
        assert ob.dtype == torch.uint8 and ob.is_contiguous() and ob.dim() in (4, 5)
        T = ob.shape[0]
        frame = int(np.prod(ob.shape[-3:]))
        if ob.dim() == 5:
            F = ob.shape[1]
            return T, ob.data_ptr() + (F - 1) * frame, F * frame
        return T, ob.data_ptr(), frame

    def label(self, ob: torch.Tensor, ep_offsets: torch.Tensor, num_frames: int):
        """Device tensors in, device tensors out: (reward[T], rtg[T], reward_stacked[T,F], rtg_stacked[T,F]), each with a
        leading group axis [G, ...] after set_text_groups."""
        T, p, stride = self._frames_view(ob)
        off = ep_offsets.to(self.device, torch.int64).contiguous()
        n_eps = off.numel() - 1
        lead = self._lead()
        r = torch.empty(lead + (T,), device=self.device, dtype=torch.float32)
        g = torch.empty(lead + (T,), device=self.device, dtype=torch.float32)
        rs = torch.empty(lead + (T, num_frames), device=self.device, dtype=torch.float32)
        gs = torch.empty(lead + (T, num_frames), device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_label(self._h, C.c_void_p(p), T, stride, _ptr(off), n_eps, num_frames, _ptr(r),
                                        _ptr(g), _ptr(rs), _ptr(gs), _stream_ptr(self.device)))
        return r, g, rs, gs

    def label_host(self, ob: "np.ndarray | torch.Tensor", ep_offsets: np.ndarray, num_frames: int, out=None):
        """Host buffers in/out (numpy or CPU torch, ideally pinned). Blocks until the results are on the host. Shapes as for
        label (a leading group axis after set_text_groups); `out`, when given, must have them."""
        if isinstance(ob, np.ndarray):
            assert ob.dtype == np.uint8 and ob.flags.c_contiguous and ob.ndim in (4, 5)
            base, shape = ob.ctypes.data, ob.shape
        else:
            assert ob.device.type == "cpu" and ob.dtype == torch.uint8 and ob.is_contiguous()
            base, shape = ob.data_ptr(), tuple(ob.shape)
        T = shape[0]
        frame = int(np.prod(shape[-3:]))
        if len(shape) == 5:
            p, stride = base + (shape[1] - 1) * frame, shape[1] * frame
        else:
            p, stride = base, frame
        off = np.ascontiguousarray(ep_offsets, dtype=np.int64)
        if out is None:
            out = self._host_outputs(T, num_frames)

        def hp(a):
            return C.c_void_p(a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())

        self._check(self._lib.arp_label_host(self._h, C.c_void_p(p), T, stride, C.c_void_p(off.ctypes.data),
                                             off.size - 1, num_frames, hp(out[0]), hp(out[1]), hp(out[2]),
                                             hp(out[3])))
        return out

    def label_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int, ep_offsets: np.ndarray,
                   num_frames: int, out=None):
        """arp_label_file: like label_host, the scored frame of row t read from `fd` at file_offset + t*row_stride_bytes."""
        off = np.ascontiguousarray(ep_offsets, dtype=np.int64)
        if out is None:
            out = self._host_outputs(T, num_frames)
        hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
        self._check(self._lib.arp_label_file(self._h, int(fd), int(file_offset), int(T), int(row_stride_bytes),
                                             C.c_void_p(off.ctypes.data), off.size - 1, num_frames, hp(out[0]), hp(out[1]),
                                             hp(out[2]), hp(out[3])))
        return out

    # -- stored embeddings ------------------------------------------------------------------------
    @property
    def embedding_dim(self) -> int:
        """Width of the per-frame embedding: 512 for the clip heads, 13*512 for the adapter heads."""
        return int(self._lib.arp_embedding_dim(self._h))

    def _emb_out(self, T: int, out, dim: "int | None" = None):
        dim = self.embedding_dim if dim is None else dim
        if out is None:
            return torch.empty((T, dim), dtype=torch.float32, pin_memory=True).numpy()
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.shape == (T, dim), out.shape
        return out

    @staticmethod
    def _host_frames(ob: "np.ndarray | torch.Tensor"):
        """(T, pointer to row 0's scored frame, row stride) of host frames as label_host takes them"""
        if isinstance(ob, np.ndarray):
            assert ob.dtype == np.uint8 and ob.flags.c_contiguous and ob.ndim in (4, 5)
            base, shape = ob.ctypes.data, ob.shape
        else:
            assert ob.device.type == "cpu" and ob.dtype == torch.uint8 and ob.is_contiguous()
            base, shape = ob.data_ptr(), tuple(ob.shape)
        frame = int(np.prod(shape[-3:]))
        p, stride = (base + (shape[1] - 1) * frame, shape[1] * frame) if len(shape) == 5 else (base, frame)
        return shape[0], p, stride

    def embed_host(self, ob: "np.ndarray | torch.Tensor", out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_host: host frames as label_host takes them -> float32 [T, embedding_dim] host array (clip heads:
        encode_image before normalisation; adapter heads: the gated feature before normalisation). Without `out` each
        call allocates a new pinned array of T * embedding_dim * 4 bytes; pass `out` to reuse one across calls."""
        T, p, stride = self._host_frames(ob)
        out = self._emb_out(T, out)
        self._check(self._lib.arp_embed_host(self._h, C.c_void_p(p), T, stride, C.c_void_p(out.ctypes.data)))
        return out

    def embed_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int,
                   out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_file: the scored frame of row t read from `fd` at file_offset + t*row_stride_bytes."""
        out = self._emb_out(int(T), out)
        self._check(self._lib.arp_embed_file(self._h, int(fd), int(file_offset), int(T), int(row_stride_bytes),
                                             C.c_void_p(out.ctypes.data)))
        return out

    def _device_outputs(self, T: int, num_frames: int):
        lead = self._lead()
        return (torch.empty(lead + (T,), device=self.device, dtype=torch.float32),
                torch.empty(lead + (T,), device=self.device, dtype=torch.float32),
                torch.empty(lead + (T, num_frames), device=self.device, dtype=torch.float32),
                torch.empty(lead + (T, num_frames), device=self.device, dtype=torch.float32))

    def label_embeddings(self, emb: torch.Tensor, ep_offsets: torch.Tensor, num_frames: int):
        """arp_label_embeddings: stored embeddings [T, embedding_dim] in, label's outputs out (device tensors, a leading
        group axis after set_text_groups). Needs no image-side weights."""
        x = emb.to(self.device, torch.float32).contiguous()
        assert x.dim() == 2 and x.shape[1] == self.embedding_dim, (tuple(x.shape), self.embedding_dim)
        T = x.shape[0]
        off = ep_offsets.to(self.device, torch.int64).contiguous()
        r, g, rs, gs = self._device_outputs(T, num_frames)
        self._check(self._lib.arp_label_embeddings(self._h, _ptr(x), T, _ptr(off), off.numel() - 1, num_frames, _ptr(r),
                                                   _ptr(g), _ptr(rs), _ptr(gs), _stream_ptr(self.device)))
        return r, g, rs, gs

    # -- CLIP tower records -----------------------------------------------------------------------
    @property
    def tower_dim(self) -> int:
        """Width of the CLIP tower record: 12*768 + 512 = 9728 for the adapter heads, 0 for the clip heads."""
        return int(self._lib.arp_tower_dim(self._h))

    def embed_tower_host(self, ob: "np.ndarray | torch.Tensor", out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_tower_host (adapter heads): host frames as label_host takes them -> float32 [T, tower_dim] host array,
        the frozen CLIP tower's class-token taps and un-normalised feature per frame. Allocation as embed_host."""
        T, p, stride = self._host_frames(ob)
        out = self._emb_out(T, out, self.tower_dim)
        self._check(self._lib.arp_embed_tower_host(self._h, C.c_void_p(p), T, stride, C.c_void_p(out.ctypes.data)))
        return out

    def embed_tower_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int,
                         out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_tower_file: the scored frame of row t read from `fd` at file_offset + t*row_stride_bytes."""
        out = self._emb_out(int(T), out, self.tower_dim)
        self._check(self._lib.arp_embed_tower_file(self._h, int(fd), int(file_offset), int(T), int(row_stride_bytes),
                                                   C.c_void_p(out.ctypes.data)))
        return out

    def label_tower(self, rec: torch.Tensor, ep_offsets: torch.Tensor, num_frames: int):
        """arp_label_tower: tower records [T, tower_dim] in, label's outputs out (device tensors, a leading group axis after
        set_text_groups), computed with this handle's adapter. Needs only the image-adapter tensors."""
        x = rec.to(self.device, torch.float32).contiguous()
        assert x.dim() == 2 and x.shape[1] == self.tower_dim, (tuple(x.shape), self.tower_dim)
        T = x.shape[0]
        off = ep_offsets.to(self.device, torch.int64).contiguous()
        r, g, rs, gs = self._device_outputs(T, num_frames)
        self._check(self._lib.arp_label_tower(self._h, _ptr(x), T, _ptr(off), off.numel() - 1, num_frames, _ptr(r),
                                              _ptr(g), _ptr(rs), _ptr(gs), _stream_ptr(self.device)))
        return r, g, rs, gs

    # -- compressed rows (gzip-chunked HDF5) --------------------------------------------------------
    @staticmethod
    def _chunk_table(chunk_offsets, chunk_bytes):
        off = np.ascontiguousarray(chunk_offsets, dtype=np.int64)
        nb = np.ascontiguousarray(chunk_bytes, dtype=np.int64)
        assert off.ndim == 1 and off.shape == nb.shape, (off.shape, nb.shape)
        return off, nb, C.c_void_p(off.ctypes.data), C.c_void_p(nb.ctypes.data)

    def label_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int,
                    ep_offsets: np.ndarray, num_frames: int, out=None):
        """arp_label_zfile: label_file's outputs when row t is the zlib stream of chunk_bytes[t] bytes at file offset
        chunk_offsets[t] of `fd`, inflating to row_bytes = F*H*W*3 bytes (F stacked frames, the last one scored)."""
        off, nb, p_off, p_nb = self._chunk_table(chunk_offsets, chunk_bytes)
        ep = np.ascontiguousarray(ep_offsets, dtype=np.int64)
        T = off.size
        if out is None:
            out = self._host_outputs(T, num_frames)
        hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
        self._check(self._lib.arp_label_zfile(self._h, int(fd), p_off, p_nb, T, int(row_bytes), hp(ep), ep.size - 1,
                                              num_frames, hp(out[0]), hp(out[1]), hp(out[2]), hp(out[3])))
        return out

    def embed_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int,
                    out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_zfile: embed_file's result from compressed rows as label_zfile takes them."""
        off, nb, p_off, p_nb = self._chunk_table(chunk_offsets, chunk_bytes)
        out = self._emb_out(off.size, out)
        self._check(self._lib.arp_embed_zfile(self._h, int(fd), p_off, p_nb, off.size, int(row_bytes),
                                              C.c_void_p(out.ctypes.data)))
        return out

    def embed_tower_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int,
                          out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_tower_zfile: embed_tower_file's result from compressed rows as label_zfile takes them."""
        off, nb, p_off, p_nb = self._chunk_table(chunk_offsets, chunk_bytes)
        out = self._emb_out(off.size, out, self.tower_dim)
        self._check(self._lib.arp_embed_tower_zfile(self._h, int(fd), p_off, p_nb, off.size, int(row_bytes),
                                                    C.c_void_p(out.ctypes.data)))
        return out

    def inflate_rows(self, src: torch.Tensor, src_offsets: torch.Tensor, src_bytes: torch.Tensor, row_bytes: int):
        """arp_inflate_rows on device tensors: uint8 src (concatenated zlib streams), int64 offsets and sizes [n] ->
        (uint8 rows [n, row_bytes], int32 ArpInflateStatus [n]). Rows that fail are zero past where they stopped."""
        assert src.dtype == torch.uint8 and src.is_cuda and src.is_contiguous()
        so = src_offsets.to(self.device, torch.int64).contiguous()
        sb = src_bytes.to(self.device, torch.int64).contiguous()
        n = so.numel()
        assert sb.numel() == n
        out = torch.zeros((n, int(row_bytes)), device=self.device, dtype=torch.uint8)
        status = torch.full((n,), -1, device=self.device, dtype=torch.int32)
        self._check(self._lib.arp_inflate_rows(self._h, _ptr(src), _ptr(so), _ptr(sb), n, int(row_bytes), _ptr(out),
                                               _ptr(status), _stream_ptr(self.device)))
        return out, status

    # -- compressed chunks of any shape ------------------------------------------------------------
    @staticmethod
    def _zchunk_args(layout, origins, offsets, sizes):
        """(ArpChunkLayout, arrays kept alive, ctypes pointers to origins / offsets / sizes, n_chunks); layout is the
        dataset's (shape, chunks) and origins [n_chunks, ndim] the chunks' logical origins"""
        lay = chunk_layout(*layout)
        o = np.ascontiguousarray(origins, dtype=np.int64).reshape(-1, lay.ndim)
        off, nb, p_off, p_nb = Engine._chunk_table(offsets, sizes)
        assert o.shape[0] == off.size, (o.shape, off.shape)
        return lay, (o, off, nb), C.c_void_p(o.ctypes.data), p_off, p_nb, off.size

    def label_zchunks(self, fd: int, layout, origins: np.ndarray, offsets: np.ndarray, sizes: np.ndarray, row_lo: int,
                      T: int, ep_offsets: np.ndarray, num_frames: int, out=None):
        """arp_label_zchunks: label_file's outputs for dataset rows [row_lo, row_lo + T) (frame F-1 of each) of a gzip
        dataset stored in chunks of any shape: layout = (shape, chunks), chunk i is the zlib stream of sizes[i] bytes at
        file offset offsets[i] of `fd` with logical origin origins[i]. ep_offsets are relative to row_lo."""
        lay, keep, p_o, p_off, p_nb, n = self._zchunk_args(layout, origins, offsets, sizes)
        ep = np.ascontiguousarray(ep_offsets, dtype=np.int64)
        if out is None:
            out = self._host_outputs(int(T), num_frames)
        hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
        self._check(self._lib.arp_label_zchunks(self._h, int(fd), C.byref(lay), p_o, p_off, p_nb, n, int(row_lo), int(T),
                                                hp(ep), ep.size - 1, num_frames, hp(out[0]), hp(out[1]), hp(out[2]),
                                                hp(out[3])))
        return out

    def embed_zchunks(self, fd: int, layout, origins: np.ndarray, offsets: np.ndarray, sizes: np.ndarray, row_lo: int,
                      T: int, out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_zchunks: embed_file's result for the rows label_zchunks reads."""
        lay, keep, p_o, p_off, p_nb, n = self._zchunk_args(layout, origins, offsets, sizes)
        out = self._emb_out(int(T), out)
        self._check(self._lib.arp_embed_zchunks(self._h, int(fd), C.byref(lay), p_o, p_off, p_nb, n, int(row_lo), int(T),
                                                C.c_void_p(out.ctypes.data)))
        return out

    def embed_tower_zchunks(self, fd: int, layout, origins: np.ndarray, offsets: np.ndarray, sizes: np.ndarray,
                            row_lo: int, T: int, out: "np.ndarray | None" = None) -> np.ndarray:
        """arp_embed_tower_zchunks: embed_tower_file's result for the rows label_zchunks reads."""
        lay, keep, p_o, p_off, p_nb, n = self._zchunk_args(layout, origins, offsets, sizes)
        out = self._emb_out(int(T), out, self.tower_dim)
        self._check(self._lib.arp_embed_tower_zchunks(self._h, int(fd), C.byref(lay), p_o, p_off, p_nb, n, int(row_lo),
                                                      int(T), C.c_void_p(out.ctypes.data)))
        return out

    def gather_frames(self, layout, row0: int, n: int, chunks: torch.Tensor) -> torch.Tensor:
        """arp_gather_frames on device tensors: chunks (uint8, the batch's inflated chunks in (row-chunk, H-, W-,
        channel-chunk) order) -> frame F-1 of dataset rows [row0, row0 + n) as uint8 [n, H, W, 3]."""
        assert chunks.dtype == torch.uint8 and chunks.is_cuda and chunks.is_contiguous()
        lay = chunk_layout(*layout)
        shape = tuple(layout[0])
        out = torch.empty((int(n),) + tuple(shape[-3:]), device=self.device, dtype=torch.uint8)
        self._check(self._lib.arp_gather_frames(self._h, C.byref(lay), int(row0), int(n), _ptr(chunks), _ptr(out),
                                                _stream_ptr(self.device)))
        return out

    def compute_reward(self, ob: torch.Tensor, want_logits: bool = False):
        """reward [T] (or [G, T] after set_text_groups); logits [T, n_text] over the texts of all groups."""
        T, p, stride = self._frames_view(ob)
        r = torch.empty(self._lead() + (T,), device=self.device, dtype=torch.float32)
        lg = torch.empty(T, max(self.n_text, 1), device=self.device, dtype=torch.float32) if want_logits else None
        self._check(self._lib.arp_compute_reward(self._h, C.c_void_p(p), T, stride, _ptr(r), _ptr(lg),
                                                 _stream_ptr(self.device)))
        return (r, lg) if want_logits else r

    def online_reward(self, frames: np.ndarray, want_logits: bool = False, want_features: bool = False):
        """Latency mode: host uint8 [n,H,W,3] (or [H,W,3]) -> dict of host arrays (reward [n], logits [n,n_text],
        features [n,feat_dim]); one CUDA-graph launch per call."""
        f = np.ascontiguousarray(frames, dtype=np.uint8)
        if f.ndim == 3:
            f = f[None]
        assert f.ndim == 4 and f.shape[1:] == (self.cfg.in_h, self.cfg.in_w, 3), f.shape
        n = f.shape[0]
        out = {}
        r = lg = ft = None
        if not self.goal:
            r = out["reward"] = np.empty(n, np.float32)
            if want_logits:
                lg = out["logits"] = np.empty((n, self.n_text), np.float32)
        if want_features or self.goal:
            ft = out["features"] = np.empty((n, self.feat_dim), np.float32)
        p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)  # noqa: E731
        self._check(self._lib.arp_online_reward(self._h, p(f), n, p(r), p(lg), p(ft)))
        return out

    def preprocess_rtgs(self, reward: torch.Tensor, ep_offsets: torch.Tensor, num_frames: int, use_normalize: bool):
        """data_procgen.py:142-168 on the device: returns (rtg_stacked [T,F] device tensor, rtg [T],
        (reward_min, reward_max, rtg_min, rtg_max) as np.float32)."""
        r = reward.to(self.device, torch.float32).contiguous()
        off = ep_offsets.to(self.device, torch.int64).contiguous()
        T = r.numel()
        g = torch.zeros(T, device=self.device, dtype=torch.float32)
        gs = torch.zeros(T, num_frames, device=self.device, dtype=torch.float32)
        shifted = torch.empty(T, device=self.device, dtype=torch.float32) if use_normalize else None
        stats = np.zeros(4, np.float32)
        self._check(self._lib.arp_preprocess_rtgs(self._h, _ptr(r), T, _ptr(off), off.numel() - 1, num_frames,
                                                  int(bool(use_normalize)), _ptr(shifted), _ptr(g), _ptr(gs),
                                                  C.c_void_p(stats.ctypes.data), _stream_ptr(self.device)))
        return gs, g, stats

    def order_statistics(self, x: torch.Tensor, k_lo: int, k_hi: int) -> np.ndarray:
        """The k_lo-th and k_hi-th smallest values (0-based) of a device float32 tensor, exactly."""
        x = x.to(self.device, torch.float32).contiguous().view(-1)
        out = np.zeros(2, np.float32)
        self._check(self._lib.arp_quantile_f32(self._h, _ptr(x), x.numel(), int(k_lo), int(k_hi),
                                               C.c_void_p(out.ctypes.data), _stream_ptr(self.device)))
        return out

    def encode_taps(self, chw: torch.Tensor):
        """Frozen-CLIP features of preprocessed images: chw float32 [T,3,224,224] (device) ->
        (taps [T, layers*width] — class-token row of every block — , clip feature [T, embed_dim])."""
        x = chw.to(self.device, torch.float32).contiguous()
        assert x.dim() == 4 and tuple(x.shape[1:]) == (3, 224, 224), x.shape
        T = x.shape[0]
        taps = torch.empty(T, self.cfg.layers * self.cfg.width, device=self.device, dtype=torch.float32)
        feat = torch.empty(T, self.cfg.embed_dim, device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_encode_taps_chw(self._h, _ptr(x), T, _ptr(taps), _ptr(feat), _stream_ptr(self.device)))
        return taps, feat

    def encode_image(self, ob: torch.Tensor) -> torch.Tensor:
        T, p, stride = self._frames_view(ob)
        f = torch.empty(T, self.feat_dim, device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_encode_image(self._h, C.c_void_p(p), T, stride, _ptr(f), _stream_ptr(self.device)))
        return f

    # -- seams ------------------------------------------------------------------------------------
    def decode_only(self, ob: torch.Tensor) -> torch.Tensor:
        T, p, stride = self._frames_view(ob)
        out = torch.empty(T, 3, 224, 224, device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_decode_only(self._h, C.c_void_p(p), T, stride, _ptr(out), _stream_ptr(self.device)))
        return out

    def scan_only(self, reward: torch.Tensor, ep_offsets: torch.Tensor, num_frames: int, gamma: float = 1.0):
        r = reward.to(self.device, torch.float32).contiguous()
        off = ep_offsets.to(self.device, torch.int64).contiguous()
        T = r.numel()
        g = torch.empty(T, device=self.device, dtype=torch.float32)
        rs = torch.empty(T, num_frames, device=self.device, dtype=torch.float32)
        gs = torch.empty(T, num_frames, device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_scan_only(self._h, _ptr(r), T, _ptr(off), off.numel() - 1, num_frames, gamma,
                                            _ptr(g), _ptr(rs), _ptr(gs), _stream_ptr(self.device)))
        return g, rs, gs

    def gemm(self, a: torch.Tensor, w: torch.Tensor, bias=None, resid=None, act: int = ACT_NONE,
             out_dtype=None) -> torch.Tensor:
        """Test hook. a, w: 16-bit float tensors (converted to the library's operand format if they are in the other
        one); out_dtype None = operand format, or torch.float32; resid is converted to the output dtype (the residual
        stream is accumulated into in that format)."""
        op = operand_dtype()
        assert a.dtype in (torch.bfloat16, torch.float16) and w.dtype in (torch.bfloat16, torch.float16)
        a, w = a.to(op).contiguous(), w.to(op).contiguous()
        M, K = a.shape
        N = w.shape[0]
        out_dtype = op if out_dtype in (None, torch.bfloat16, torch.float16) else out_dtype
        out = torch.empty(M, N, device=self.device, dtype=out_dtype)
        if resid is not None:
            resid = resid.to(out_dtype).contiguous()
        self._check(self._lib.arp_gemm_bf16(self._h, _ptr(a), _ptr(w), _ptr(out),
                                            DT_F32 if out_dtype == torch.float32 else _TORCH_DT[op], M, N, K, _ptr(bias),
                                            _ptr(resid), act, _stream_ptr(self.device)))
        return out

    def resid_gemm_stats(self, a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, x: torch.Tensor):
        """Test hook: x (16-bit, updated IN PLACE) += a w^T + bias in the GEMM epilogue; returns stats [M,2] =
        (rstd, -mean*rstd) of the updated rows."""
        op = operand_dtype()
        assert x.dtype == op and x.is_contiguous() and x.device == self.device
        a, w = a.to(op).contiguous(), w.to(op).contiguous()
        bias = bias.to(self.device, torch.float32).contiguous()
        M, K = a.shape
        N = w.shape[0]
        stats = torch.empty(M, 2, device=self.device, dtype=torch.float32)
        self._check(self._lib.arp_resid_gemm_stats(self._h, _ptr(a), _ptr(w), _ptr(bias), _ptr(x), _ptr(stats), M, N, K,
                                                   _stream_ptr(self.device)))
        return stats

    def ln_gemm(self, x: torch.Tensor, gamma, beta, w: torch.Tensor, bias: torch.Tensor, act: int = ACT_NONE) -> torch.Tensor:
        """Test hook: act(LayerNorm(x) W^T + bias) with the LayerNorm folded into the GEMM (default-path ln_1/ln_2).
        x [M,768] 16-bit (converted to the operand format); gamma, beta, w [N,768], bias fp32."""
        op = operand_dtype()
        x = x.to(op).contiguous()
        f = lambda t: t.to(self.device, torch.float32).contiguous()  # noqa: E731
        gamma, beta, w, bias = f(gamma), f(beta), f(w), f(bias)
        M, N = x.shape[0], w.shape[0]
        out = torch.empty(M, N, device=self.device, dtype=op)
        self._check(self._lib.arp_ln_gemm(self._h, _ptr(x), _ptr(gamma), _ptr(beta), _ptr(w), _ptr(bias), _ptr(out),
                                          M, N, act, _stream_ptr(self.device)))
        return out

    def layernorm(self, x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor) -> torch.Tensor:
        assert x.dtype == torch.float32 and x.is_contiguous() and x.shape[-1] == 768
        y = torch.empty(x.shape, device=self.device, dtype=operand_dtype())
        self._check(self._lib.arp_layernorm_bf16(self._h, _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y),
                                                 x.numel() // 768, _stream_ptr(self.device)))
        return y

    def attention(self, qkv: torch.Tensor, B: int, tokens: int) -> torch.Tensor:
        assert qkv.dtype in (torch.bfloat16, torch.float16)
        qkv = qkv.to(operand_dtype()).contiguous()
        out = torch.empty(B * tokens, qkv.shape[-1] // 3, device=self.device, dtype=qkv.dtype)
        self._check(self._lib.arp_attention(self._h, _ptr(qkv), _ptr(out), B, tokens, _stream_ptr(self.device)))
        return out

    def cls_attention(self, q: torch.Tensor, qkv: torch.Tensor, B: int, tokens: int) -> torch.Tensor:
        """Test hook: the last block's class-token attention. q [B, W] (one query row per frame), qkv [B*tokens, 3W]
        (K and V of every token; the Q third is not read) -> [B, W], all in the operand format."""
        assert q.dtype in (torch.bfloat16, torch.float16) and qkv.dtype in (torch.bfloat16, torch.float16)
        q, qkv = q.to(operand_dtype()).contiguous(), qkv.to(operand_dtype()).contiguous()
        out = torch.empty(B, qkv.shape[-1] // 3, device=self.device, dtype=qkv.dtype)
        self._check(self._lib.arp_cls_attention(self._h, _ptr(q), _ptr(qkv), _ptr(out), B, tokens,
                                                _stream_ptr(self.device)))
        return out
