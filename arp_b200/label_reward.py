"""Drop-in for the reference's offline reward labeler, `arp_dt/label_reward.py`.

Same entry point, same arguments and defaults (label_reward.py:44-60), same CLI flags (:295-312), same
`model_type` names and checkpoint format, same output datasets
    f"{img_key}_{model_type}_reward[_{inst_type}]",  f"{img_key}_{model_type}_pos_rtg[_{inst_type}]"
as float32 [T, num_frames] (:257-289) — but every frame is scored by the native sm_100a library
(include/arp_b200.h) instead of a Python loop over PyTorch calls:

    reference (per episode, :265-271)                      here (per slab of many episodes)
    -------------------------------------------------      ----------------------------------------------
    g[img_key][traj, -1]  (host gather)                    strided host pointer -> cudaMemcpy2DAsync
    [preprocess(img) for img in imgs]  (PIL, 1 thread)     fused decode kernel (Pillow-exact)
    clip.tokenize + text tower, every episode              text embedding cached once per run
    model(images, text)                                    tcgen05 ViT + fused cosine head
    discount_cumsum / stack_outputs  (python loops)        per-episode scan + window stack kernel

There is no CPU fallback: without the built library and a B200 this module raises.

Keyword-only extensions (all optional; defaults reproduce the reference):
    clip_state_dict  CLIP weights (openai/CLIP state_dict keys). The reference downloads pretrained
                     weights inside clip.load (:126); offline, pass them here or set ARP_CLIP_CHECKPOINT.
    arch             "ViT-B/16" (what the reference hard-codes) or "ViT-B/32".
    reduce           "first" (reference behaviour, SURVEY.md Q1) or "mean" (envs/vl_reward.py semantics).
    max_batch        frames per device chunk.      slab_frames  frames per host slab.
    device           CUDA ordinal (default: LOCAL_RANK or 0).
    precision        "16bit" (default; "bf16"/"fp16" are accepted aliases): the tensor-core product path — 16-bit operands
                     in the library's operand format (fp16 by default, the reference's own CUDA format), 16-bit residual
                     stream, LayerNorm folded into the GEMMs. "fp32resid": same tensor-core kernels with an fp32 residual
                     stream and standalone LayerNorm (~2x closer to fp32, ~10 % slower). "fp32": verification path, every
                     weight, activation and contraction in fp32 (what the reference's CPU route computes; ~50x slower).
    distributed      shard episodes over torch.distributed ranks (default: on when a process group exists).
    tokenizer        None: openai/CLIP's clip.tokenize (label_reward.py:136) — if the package is missing the call REFUSES
                     unless ARP_ALLOW_STANDIN_TOKENIZER=1; "standin": the deterministic stand-in (random-init experiments
                     only); or a callable(list[str]) -> int tensor [n, 77].
    extra_instructions  {inst_type: text or list of texts}: more instruction sets labeled in the SAME pass over the frames
                     (one decode + encoder pass for all of them). Each writes its own dataset pair, named by its inst_type
                     with the reference's rule ("none" = no suffix), and equal bit for bit to a separate call with that
                     text and inst_type. Not for goal-conditioned model types (they take no text).
    embeddings       None (default): label from the frames. "save": run the image side once, store the per-frame
                     embeddings, and label from them (same reward / pos_rtg datasets, bit for bit, plus the embedding
                     dataset). "load": label from stored embeddings; no frame is read and no image-side weight is
                     uploaded. "save_tower" / "load_tower" (adapter model types): the same with the CLIP tower record,
                     which any adapter checkpoint fine-tuned from the same CLIP relabels. See label_reward().
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os

import numpy as np
import torch

from . import capi
from .instructions import get_clip_instruct, get_clip_special_instruct
from .sharding import gather_rows, partition_episodes
from .store import open_store
from .text_tower import adapter_text_embedding, clip_text_embedding
from .tokenizer import resolve as resolve_tokenizer
from .weights import load_checkpoint


def center_crop(image, crop_size):
    """label_reward.py:15-36 (imported by envs/vl_reward.py:6 and envs/rollout_procgen.py:14): [N,H,W,C] centre crop."""
    _, H, W, _ = image.shape
    ch, cw = crop_size
    top, left = int((H - ch) / 2), int((W - cw) / 2)
    return image[:, top:top + ch, left:left + cw, :]


def episode_index(g, done_key=None):
    """label_reward.py:71-87 — (len_data, num_frames, g_traj_idx)."""
    if done_key is None:
        for cand in ("done", "rewards", "is_terminal"):
            if g.get(cand):
                done_key = cand
                break
        else:
            raise ValueError
    try:
        len_data, num_frames = g[done_key].shape[:2]
        idx = list(np.nonzero(np.asarray(g[done_key][:, -1]))[0] + 1)
        idx.insert(0, 0)
    except Exception:  # noqa: BLE001 — the reference's bare `except:` fallback for the "time" layout (:84-87)
        len_data, num_frames = g["time"].shape[:2]
        idx = list(np.where(np.asarray(g["time"][:, -1, 0]) == 1.0)[0])
        idx.append(len(g["time"]))
    return int(len_data), int(num_frames), [int(i) for i in idx]


def _head_for(model_type: str) -> tuple[int, int]:
    """model_type -> (ArpHead, ArpPreprocess), following the dispatch at label_reward.py:123-230."""
    if model_type == "clip":
        return capi.HEAD_CLIP, capi.PRE_PIL_BICUBIC
    if model_type == "clip_goal_conditioned":
        return capi.HEAD_CLIP_GOAL, capi.PRE_PIL_BICUBIC
    if model_type.startswith("clip_"):
        # Only "clip_ft" constructs a model in the reference (:166-173); other clip_* names crash there
        # (SURVEY.md Q3). They are served by the same CLIPMultiscaleAdapter weights.
        if "_goal_conditioned" in model_type:
            return capi.HEAD_ADAPTER_GOAL, capi.PRE_BILINEAR
        if "ensemble" in model_type:
            return capi.HEAD_ADAPTER_ENSEMBLE, capi.PRE_BILINEAR
        return capi.HEAD_ADAPTER, capi.PRE_BILINEAR
    raise ValueError(f"unsupported model_type {model_type!r}: the labeler only defines clip* reward models")


def _texts(text) -> list:
    return list(text) if isinstance(text, (list, tuple)) else [text]


def _text_groups(model_type: str, text, extra_instructions) -> list[list]:
    """The instruction sets of one labeling pass: `text`, then the values of extra_instructions in order. ValueError for
    sets one pass cannot label: a goal-conditioned head (it takes no text), more sets or texts than the library holds."""
    groups = [_texts(text)] + [_texts(t) for t in (extra_instructions or {}).values()]
    if extra_instructions:
        head, _ = _head_for(model_type)
        if head in (capi.HEAD_CLIP_GOAL, capi.HEAD_ADAPTER_GOAL):
            raise ValueError(f"extra_instructions: {model_type!r} is goal-conditioned and takes no instruction")
        if len(groups) > capi.MAX_TEXT_GROUPS:
            raise ValueError(f"extra_instructions: {len(groups)} instruction sets, at most {capi.MAX_TEXT_GROUPS}")
        for g in groups:
            if not 1 <= len(g) <= capi.MAX_TEXT:
                raise ValueError(f"extra_instructions: an instruction set has {len(g)} texts, must be 1..{capi.MAX_TEXT}")
        if sum(len(g) for g in groups) > capi.MAX_TEXT_TOTAL:
            raise ValueError(f"extra_instructions: {sum(len(g) for g in groups)} texts in all, at most "
                             f"{capi.MAX_TEXT_TOTAL}")
    return groups


def _target_keys(model_type: str, inst_type: str, extra_instructions) -> list[str]:
    """[reward, pos_rtg] key pair of every instruction set, in group order (label_reward.py:257-259: inst_type "none"
    adds no suffix). ValueError when two sets would write the same datasets."""
    keys = []
    for it in [inst_type, *(extra_instructions or {})]:
        pair = [f"{model_type}_reward", f"{model_type}_pos_rtg"]
        keys += pair if it == "none" else [f"{x}_{it}" for x in pair]
    if len(set(keys)) != len(keys):
        raise ValueError(f"extra_instructions: two instruction sets would write the same datasets ({keys})")
    return keys


def embedding_family(model_type: str) -> str:
    """"clip" (clip, clip_goal_conditioned: the 512-wide encode_image) or "clip_adapter" (every adapter model type: the
    13*512-wide gated adapter feature). One stored embedding serves every model type of its family."""
    head, _ = _head_for(model_type)
    return "clip" if head in (capi.HEAD_CLIP, capi.HEAD_CLIP_GOAL) else "clip_adapter"


EMBEDDING_DIM = {"clip": 512, "clip_adapter": 13 * 512}


def embedding_key(img_key: str, model_type: str) -> str:
    """Dataset of the stored embeddings of img_key: f"{img_key}_clip_emb" or f"{img_key}_clip_adapter_emb"; its SHA-256
    provenance signature is the uint8 [32] dataset f"{key}_sig"."""
    return f"{img_key}_{embedding_family(model_type)}_emb"


#: the CLIP tower record of the adapter family: 12 class-token taps of 768 + the 512-wide CLIP feature (include/arp_b200.h)
TOWER_DIM = 12 * 768 + 512


def tower_key(img_key: str) -> str:
    """Dataset of the CLIP tower records of img_key, f"{img_key}_clip_tower_emb"; its signature is f"{key}_sig"."""
    return f"{img_key}_clip_tower_emb"


_IMAGE_ADAPTER_PREFIXES = ("image_intermediate_linear.", "image_adapter.", "image_residual_weight")


def _image_weights(state_dict: dict, adapter: bool) -> dict:
    """The image-side tensors Engine.load_state_dict uploads for a head of this family, by their library names ("visual.*"
    and, for the adapter heads, the image adapter; an adapter checkpoint's "clip_model." prefix removed)."""
    out = {}
    for k, v in state_dict.items():
        if not torch.is_tensor(v):
            continue
        name = k[len("clip_model."):] if k.startswith("clip_model.") else k
        if name.startswith("visual.") or (adapter and name.startswith(_IMAGE_ADAPTER_PREFIXES)):
            out[name] = v
    return out


SIGNATURE_SAMPLES = 4096


def embedding_signature(model_type: str, arch: str, frame_hw, use_crop: bool, precision: str,
                        state_dict: dict, *, tower: bool = False) -> np.ndarray:
    """uint8 [32]: SHA-256 over what decides a stored embedding's bits — the embedding family, arch, frame H x W,
    use_crop, the precision's pipeline, the library's operand format, and a digest of the image-side weights: every tensor
    Engine.load_state_dict uploads for the family, by name, shape and its values at <= 4096 fixed, evenly spaced flat
    indices (cheap on a 2 GB adapter checkpoint). This is a provenance check, not a guarantee: two checkpoints that differ
    only at unsampled indices get the same signature.
    tower=True: the signature of a CLIP tower record (family "clip_tower"): the same fields, but only the visual.*
    tensors (an adapter checkpoint's "clip_model.visual.*"), not the image adapter — the record does not depend on it."""
    family = "clip_tower" if tower else embedding_family(model_type)
    h = hashlib.sha256()
    h.update(json.dumps({"family": family, "arch": arch, "frame_hw": [int(x) for x in frame_hw],
                         "use_crop": bool(use_crop), "precision": capi.precision_enum(precision),
                         "operand_dtype": str(capi.operand_dtype())}, sort_keys=True).encode())
    for name, t in sorted(_image_weights(state_dict, family == "clip_adapter").items()):
        flat = t.detach().reshape(-1)
        n = flat.numel()
        k = min(n, SIGNATURE_SAMPLES)
        idx = torch.arange(k, dtype=torch.int64) * max(n - 1, 0) // max(k - 1, 1)
        h.update(json.dumps([name, list(t.shape)]).encode())
        h.update(flat[idx.to(flat.device)].float().cpu().numpy().astype("<f4").tobytes())
    return np.frombuffer(h.digest(), np.uint8).copy()


def _resolve_clip_weights(clip_state_dict, arch: str) -> dict:
    if clip_state_dict is not None:
        return clip_state_dict
    path = os.environ.get("ARP_CLIP_CHECKPOINT")
    if path:
        return load_checkpoint(path)
    try:  # the reference's own route, if the real package and its cached weights exist
        import clip  # type: ignore
        model, _ = clip.load(arch, device="cpu")
        return model.state_dict()
    except Exception as e:  # noqa: BLE001
        raise RuntimeError(
            "CLIP weights unavailable: pass clip_state_dict=..., set ARP_CLIP_CHECKPOINT to a state_dict file, "
            "or install openai/CLIP with its cached checkpoint (the reference downloads it in clip.load, "
            "label_reward.py:126)") from e


# One native handle is kept alive between label_reward() calls of a process (key = its whole configuration): creating it
# (4 GB of workspace, the pinned staging ring) and tearing it down cost ~0.25 s, a tenth of a 70k-frame labeling pass.
# Weights and the instruction embedding are uploaded again on every call. release_cached_engine() frees it.
_ENGINE_CACHE: dict = {}


def release_cached_engine():
    for e in _ENGINE_CACHE.values():
        e.close()
    _ENGINE_CACHE.clear()


def _model_state_dict(model_type: str, model_ckpt_dir, clip_state_dict, arch: str) -> dict:
    """The state_dict a labeler of model_type uploads: CLIP weights, or the adapter checkpoint with CLIP nested under
    "clip_model." (label_reward.py:165-176)."""
    head, _ = _head_for(model_type)
    if head in (capi.HEAD_ADAPTER, capi.HEAD_ADAPTER_ENSEMBLE, capi.HEAD_ADAPTER_GOAL):
        assert model_ckpt_dir is not None, "specify model_ckpt_dir"  # label_reward.py:174
        sd = load_checkpoint(model_ckpt_dir) if not isinstance(model_ckpt_dir, dict) else model_ckpt_dir
        if not any(k.startswith("clip_model.") for k in sd):
            # strict=False load in the reference (:176): CLIP tensors missing from the checkpoint keep
            # the values clip.load gave them.
            base = _resolve_clip_weights(clip_state_dict, arch)
            sd = {**{"clip_model." + k: v for k, v in base.items()}, **sd}
        return sd
    return _resolve_clip_weights(clip_state_dict, arch)


def _cached_engine(**cfg):
    key = tuple(sorted(cfg.items()))
    e = _ENGINE_CACHE.get(key)
    if e is None:
        release_cached_engine()                      # a single handle: workspaces of different configurations do not add up
        e = capi.Engine(**cfg)
        _ENGINE_CACHE[key] = e
    return e


class RewardLabeler:
    """Model + cached instruction embedding on one GPU; label() scores slabs of episodes.

    This is the object form of the closures `compute_reward` / `discount_cumsum` / `stack_outputs`
    that the reference builds inside label_reward() (:132-254)."""

    def __init__(self, model_type: str, text, frame_hw: tuple[int, int], *, model_ckpt_dir=None,
                 clip_state_dict=None, arch: str = "ViT-B/16", use_crop: bool = False, reduce: str = "first",
                 max_batch: int = 1024, device: int | None = None, precision: str = "16bit", tokenizer=None,
                 extra_instructions: dict | None = None, relabel_only: bool = False, tower_only: bool = False):
        """extra_instructions: {inst_type: text(s)} scored with `text` in one pass; label_slab / label_file /
        label_embeddings then return arrays with a leading group axis [1 + len(extra_instructions), ...], `text` first.
        relabel_only: the labeler only labels stored embeddings (label_embeddings); no image-side weight is uploaded.
        tower_only (adapter model types): the labeler only labels CLIP tower records (label_tower); of the image-side
        weights only the image adapter is uploaded."""
        head, pre = _head_for(model_type)
        prec = capi.precision_enum(precision)
        groups = _text_groups(model_type, text, extra_instructions)
        adapter = head in (capi.HEAD_ADAPTER, capi.HEAD_ADAPTER_ENSEMBLE, capi.HEAD_ADAPTER_GOAL)
        if adapter:
            assert model_ckpt_dir is not None, "specify model_ckpt_dir"  # label_reward.py:174
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        self.model_type, self.device_index = model_type, device
        patch = 32 if arch.endswith("/32") else 16
        self.engine = _cached_engine(device=device, patch=patch, in_h=int(frame_hw[0]), in_w=int(frame_hw[1]),
                                     use_crop=bool(use_crop), preprocess=pre, head=head,
                                     reduce=capi.REDUCE_MEAN if reduce == "mean" else capi.REDUCE_FIRST,
                                     max_batch=int(max_batch), precision=prec)
        dev = self.engine.device
        sd = _model_state_dict(model_type, model_ckpt_dir, clip_state_dict, arch)
        if tower_only:
            assert adapter, "tower records serve the adapter model types"
            self.engine.load_state_dict({k: v for k, v in sd.items() if k.startswith(_IMAGE_ADAPTER_PREFIXES)})
            missing = [k for k in self.engine.missing_weights() if k.startswith(_IMAGE_ADAPTER_PREFIXES)]
            if missing:
                raise RuntimeError(f"checkpoint lacks {len(missing)} image-adapter tensors, e.g. {missing[:3]}")
        elif not relabel_only:
            missing = self.engine.load_state_dict(sd, strict=False)
            if missing:
                raise RuntimeError(f"checkpoint lacks {len(missing)} tensors the {model_type} path needs, e.g. {missing[:3]}")
        self.goal = self.engine.goal
        if not self.goal:
            tokenize = resolve_tokenizer(tokenizer)
            tokens = [tokenize(g) for g in groups]
            # the instruction embeddings of the previous call are reused when the very same weight tensors (objects and
            # in-place version counters) and token ids come back — the cached handle keeps them referenced
            text_sd = {k: v for k, v in sd.items() if torch.is_tensor(v) and "visual." not in k}
            sig = ([t.tolist() for t in tokens], head, [(k, v._version) for k, v in text_sd.items()])
            cached = getattr(self.engine, "_text_cache", None)
            if cached is not None and cached[0] == sig and all(cached[1].get(k) is v for k, v in text_sd.items()):
                embs = cached[2]
            else:
                # the text tower runs once per group, so each group's rows are exactly those of a call with it alone
                if adapter:
                    embs = [adapter_text_embedding(sd, t, dev, ensemble=head == capi.HEAD_ADAPTER_ENSEMBLE) for t in tokens]
                else:
                    embs = [clip_text_embedding(sd, t, dev) for t in tokens]
                self.engine._text_cache = (sig, text_sd, embs)
            if extra_instructions:
                self.engine.set_text_groups([e for e, _ in embs], embs[0][1])
            else:
                self.engine.set_text(*embs[0])

    def label_slab(self, ob: np.ndarray, ep_offsets: np.ndarray, num_frames: int):
        """ob: host uint8 [T,F,H,W,3] (or [T,H,W,3]); ep_offsets: int64 [n+1] relative to the slab.
        Returns host (reward[T], rtg[T], reward_stacked[T,F], rtg_stacked[T,F]), each [G, ...] with extra_instructions."""
        return self.engine.label_host(ob, ep_offsets, num_frames)

    def label_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int, ep_offsets: np.ndarray, num_frames: int):
        """Same, the scored frame of row t read by the library from `fd` at file_offset + t*row_stride_bytes."""
        return self.engine.label_file(fd, file_offset, T, row_stride_bytes, ep_offsets, num_frames)

    @property
    def embedding_dim(self) -> int:
        return self.engine.embedding_dim

    def embed_slab(self, ob: np.ndarray) -> np.ndarray:
        """The image side of label_slab: float32 [T, embedding_dim] host array, one stored embedding per row."""
        return self.engine.embed_host(ob)

    def embed_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int) -> np.ndarray:
        """The image side of label_file."""
        return self.engine.embed_file(fd, file_offset, T, row_stride_bytes)

    def label_embeddings(self, emb: np.ndarray, ep_offsets: np.ndarray, num_frames: int):
        """label_slab's outputs (host arrays) from stored embeddings [T, embedding_dim] of the same rows."""
        dev = self.engine.device
        # a read-only memory map (a stored dataset) is copied once: torch does not wrap non-writable arrays
        out = self.engine.label_embeddings(torch.from_numpy(np.require(emb, np.float32, ["C", "W"])).to(dev),
                                           torch.from_numpy(np.asarray(ep_offsets, np.int64)), num_frames)
        return tuple(a.cpu().numpy() for a in out)

    @property
    def tower_dim(self) -> int:
        return self.engine.tower_dim

    def embed_tower_slab(self, ob: np.ndarray) -> np.ndarray:
        """The frozen-CLIP side of label_slab (adapter model types): float32 [T, tower_dim] host array of tower records."""
        return self.engine.embed_tower_host(ob)

    def embed_tower_file(self, fd: int, file_offset: int, T: int, row_stride_bytes: int) -> np.ndarray:
        """The frozen-CLIP side of label_file."""
        return self.engine.embed_tower_file(fd, file_offset, T, row_stride_bytes)

    def label_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int,
                    ep_offsets: np.ndarray, num_frames: int):
        """label_file's outputs when row t is the zlib stream of chunk_bytes[t] bytes at chunk_offsets[t] of `fd` (a gzip
        dataset chunked one row per chunk), inflated on the device."""
        return self.engine.label_zfile(fd, chunk_offsets, chunk_bytes, row_bytes, ep_offsets, num_frames)

    def embed_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int) -> np.ndarray:
        """The image side of label_zfile."""
        return self.engine.embed_zfile(fd, chunk_offsets, chunk_bytes, row_bytes)

    def embed_tower_zfile(self, fd: int, chunk_offsets: np.ndarray, chunk_bytes: np.ndarray, row_bytes: int) -> np.ndarray:
        """The frozen-CLIP side of label_zfile."""
        return self.engine.embed_tower_zfile(fd, chunk_offsets, chunk_bytes, row_bytes)

    def label_tower(self, rec: np.ndarray, ep_offsets: np.ndarray, num_frames: int):
        """label_slab's outputs (host arrays) from the CLIP tower records [T, tower_dim] of the same rows, with this
        labeler's adapter."""
        dev = self.engine.device
        out = self.engine.label_tower(torch.from_numpy(np.require(rec, np.float32, ["C", "W"])).to(dev),
                                      torch.from_numpy(np.asarray(ep_offsets, np.int64)), num_frames)
        return tuple(a.cpu().numpy() for a in out)

    def close(self, release: bool = False):
        """The native handle stays cached for the next call of this process unless release=True."""
        if release:
            release_cached_engine()


def _slabs(ep_offsets: np.ndarray, e_lo: int, e_hi: int, slab_frames: int):
    """Group whole episodes [e_lo, e_hi) into slabs of at most ~slab_frames frames (at least one episode)."""
    e = e_lo
    while e < e_hi:
        j = e + 1
        while j < e_hi and ep_offsets[j + 1] - ep_offsets[e] <= slab_frames:
            j += 1
        yield e, j
        e = j


SIDECAR_SUFFIX = "_last"   # "<img_key>_last": uint8 [T,H,W,3], the scored (last stacked) frame of every row


def write_destacked_sidecar(store, img_key: str = "ob", rows_per_pass: int = 4096) -> str:
    """SURVEY.md §8(f)3: the recorder stores every row as F stacked frames in gzip chunks (1,F,H,W,3)
    (data/PPG/trajectory_recorder.py:154-162), so scoring the LAST frame of a row inflates F times more bytes than it
    uses (label_reward.py:268). This writes the scored frames once as "<img_key>_last" [T,H,W,3]; label_reward() reads
    the sidecar when it exists. Returns the sidecar key."""
    ds = store[img_key]
    T = ds.shape[0]
    key = img_key + SIDECAR_SUFFIX
    if store.get(key) is not None:
        return key
    out = store.create_dataset(key, shape=(T,) + tuple(ds.shape[2:]), dtype=np.uint8, chunks=(1,) + tuple(ds.shape[2:]),
                               compression="gzip")
    for lo in range(0, T, rows_per_pass):
        hi = min(T, lo + rows_per_pass)
        out[lo:hi] = np.asarray(ds[lo:hi, -1])
    return key


def _rows_array(ds, lo: int, hi: int, sidecar=None) -> np.ndarray:
    """Rows [lo, hi) of an image dataset as a C-contiguous host array WITHOUT touching the frames that
    are not scored when the container allows it (memory-mapped store); h5py reads only `[:, -1]`; a de-stacked
    sidecar ([T,H,W,3], see write_destacked_sidecar) is read instead of the stacked dataset when present."""
    if sidecar is not None:
        arr = getattr(sidecar, "array", None)
        if arr is not None and arr.flags.c_contiguous:
            return arr[lo:hi]
        return np.ascontiguousarray(sidecar[lo:hi])
    arr = getattr(ds, "array", None)
    if arr is not None and arr.flags.c_contiguous:
        return arr[lo:hi]                       # strided pointer goes straight to arp_label_host
    return np.ascontiguousarray(ds[lo:hi, -1])  # label_reward.py:268 — last stacked frame only


def label_reward(
    env_name,
    distribution_mode,
    num_levels,
    start_level,
    text,
    base_path,
    data_path=None,
    image_keys="ob",
    num_demonstrations=500,
    num_frames=8,
    env_type=None,
    model_type="clip",
    model_ckpt_dir=None,
    use_crop=False,
    inst_type="none",
    *,
    clip_state_dict=None,
    arch="ViT-B/16",
    reduce="first",
    max_batch=1024,
    slab_frames=16384,
    device=None,
    distributed=None,
    precision="16bit",
    tokenizer=None,
    extra_instructions=None,
    embeddings=None,
):
    """embeddings (keyword-only):
        None    label from the frames (the reference's behaviour).
        "save"  embed the frames (the image side: decode, ViT, projection / adapter), label from the embeddings on the
                device, and write, next to the same reward / pos_rtg datasets as None (bit for bit), the float32
                [rows, dim] dataset embedding_key(img_key, model_type) over the labeled rows [off[0], off[n_eps]),
                uncompressed (assigned in place when it exists with that shape; ValueError when its shape differs), and
                its SHA-256 signature f"{key}_sig" (embedding_signature). dim = 512 for the clip family, 13*512 for the
                adapter family. Sharded, each rank embeds and labels its own episodes and the embeddings reach rank 0
                through a second gather: rank 0 then holds all of them, 4 * rows * dim bytes (the adapter family at
                73 k frames: 1.9 GB; at configs[4] size: 38 GB). With NCCL that gather lands in rank 0's DEVICE
                memory first (plus the padded all-gather buffer), then is copied to the host.
        "load"  label from the stored embeddings instead of the frames: the done key and the image dataset's shape are
                read, never its frames, and no image-side weight is uploaded. ValueError before any engine is created
                when the embedding dataset or its signature is missing, its row count or width differs, or the signature
                differs (another checkpoint, crop, frame size, arch or precision). Combines with extra_instructions, both
                reduce values and goal-conditioned model types; an embedding saved by one model type loads in any model
                type of its family (clip_ft -> clip_multiscale_ensemble, clip -> clip_goal_conditioned). Sharded, each
                rank reads its own rows.
        "save_tower" / "load_tower"  (adapter model types only) the same with the CLIP tower record instead of the gated
                adapter feature: the float32 [rows, TOWER_DIM] dataset tower_key(img_key) = f"{img_key}_clip_tower_emb"
                (the 12 class-token taps and the un-normalised CLIP feature of every row, 38 912 bytes per row) and its
                signature embedding_signature(..., tower=True), which covers the visual.* weights but not the image
                adapter. Fine-tuning freezes CLIP, so the records of one CLIP serve every adapter checkpoint trained from
                it: "load_tower" with a new model_ckpt_dir relabels with only that checkpoint's adapter GEMMs (0.468
                GFLOP per frame instead of the ViT's 35.1), uploads only its image-adapter tensors, and writes what
                embeddings=None with that checkpoint writes. Which to keep: "save" (26.6 KB per row) relabels new
                instructions of ONE checkpoint with a single head launch; "save_tower" (38.9 KB per row) survives
                re-fine-tuning the adapter. Refusals as for "load", and a clip-family model_type is refused (its
                512-wide embedding does not depend on a checkpoint of its own: use "save" / "load")."""
    if embeddings not in (None, "save", "load", "save_tower", "load_tower"):
        raise ValueError(f"embeddings must be None, 'save', 'load', 'save_tower' or 'load_tower', got {embeddings!r}")
    tower = embeddings in ("save_tower", "load_tower")
    stored = embeddings.split("_")[0] if embeddings else None     # "save" / "load" / None, records of either kind
    if tower and embedding_family(model_type) != "clip_adapter":
        raise ValueError(f"embeddings={embeddings!r}: tower records serve the adapter model types, not {model_type!r}; "
                         "the clip family's embeddings='save' / 'load' already serve any instruction")
    # instruction sets this pass cannot label are refused before the dataset is opened or an engine is built
    target_keys = _target_keys(model_type, inst_type, extra_instructions)
    _text_groups(model_type, text, extra_instructions)
    n_groups = len(target_keys) // 2
    image_keys = image_keys.split(", ")
    if data_path is None:
        dirname = (
            f"{env_name}_{distribution_mode}_level{start_level}to{num_levels}_num{num_demonstrations}_frame{num_frames}"
        )
        if env_type != "none":
            dirname += f"_{env_type}"
        data_path = os.path.join(base_path, dirname, "data.hdf5")

    import torch.distributed as dist
    if distributed is None:
        distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    rank = dist.get_rank() if distributed else 0
    world = dist.get_world_size() if distributed else 1

    import time
    _t = [("start", time.perf_counter())]
    _mark = lambda name: _t.append((name, time.perf_counter()))  # noqa: E731 — ARP_TIMING=1 prints the phase breakdown
    # Every rank READS through its own read-only handle; rank 0 reopens the container for writing only after all
    # readers have closed (HDF5 file locking refuses a writer next to readers, and a reader next to the writer).
    g = open_store(data_path, "r")
    labeler = None
    failure = None
    results = {}
    embs, sigs = {}, {}
    try:
        len_data, num_frames, g_traj_idx = episode_index(g)  # num_frames comes from the file (Q4)
        n_eps = len(g_traj_idx) - 1
        off = np.minimum(np.asarray(g_traj_idx, dtype=np.int64), len_data)  # min(idx[i+1], len_data) (:267)
        shards = partition_episodes(off, world)
        e_lo, e_hi = shards[rank]
        _mark("open + episode index")
        try:
            H, W = g[image_keys[0]].shape[-3:-1]
            if use_crop:
                print(f"image_size: {g[image_keys[0]].shape[-2]}")  # label_reward.py:104-105
            if embeddings is not None:
                # the weights are resolved once here: the signature needs them, and a refused load builds no engine
                sd = _model_state_dict(model_type, model_ckpt_dir, clip_state_dict, arch)
                model_ckpt_dir, clip_state_dict = (sd, None) if embedding_family(model_type) == "clip_adapter" else \
                    (model_ckpt_dir, sd)
                for img_key in image_keys:
                    sigs[img_key] = embedding_signature(model_type, arch, g[img_key].shape[-3:-1], use_crop, precision,
                                                        sd, tower=tower)
                    _check_stored_embeddings(g, img_key, model_type, off, n_eps, sigs[img_key], embeddings)
            labeler = RewardLabeler(model_type, text, (int(H), int(W)), model_ckpt_dir=model_ckpt_dir,
                                    clip_state_dict=clip_state_dict, arch=arch, use_crop=use_crop, reduce=reduce,
                                    max_batch=max_batch, device=device, precision=precision, tokenizer=tokenizer,
                                    extra_instructions=extra_instructions, relabel_only=embeddings == "load",
                                    tower_only=embeddings == "load_tower")
            _mark("engine + weights + text tower")
            for img_key in image_keys:
                if stored == "load":
                    key, first = _stored_key(img_key, model_type, tower), int(off[0])
                    emb = np.ascontiguousarray(g[key][int(off[e_lo]) - first:int(off[e_hi]) - first], np.float32)
                    results[img_key] = _label_embedding_rows(labeler, emb, off, e_lo, e_hi, num_frames, n_groups, tower)
                    continue
                ds = g[img_key]
                side = g.get(img_key + SIDECAR_SUFFIX)
                if side is not None and (side.shape[0] != ds.shape[0] or tuple(side.shape[1:]) != tuple(ds.shape[2:])):
                    side = None                      # stale or foreign sidecar: fall back to the stacked dataset
                if stored == "save":
                    embs[img_key] = _embed_rows(labeler, ds, side, off, e_lo, e_hi, slab_frames, tower)
                    results[img_key] = _label_embedding_rows(labeler, embs[img_key], off, e_lo, e_hi, num_frames,
                                                             n_groups, tower)
                else:
                    results[img_key] = _label_rows(labeler, ds, side, off, e_lo, e_hi, num_frames, slab_frames, n_groups)
            _mark("label (decode + encoder + head + scan, H2D / D2H)")
        except Exception as e:  # noqa: BLE001 — reported to every rank below, then re-raised
            failure = e
        if distributed:
            # a rank that failed must not leave the others waiting in the gather: agree on success first
            backend = dist.get_backend()
            cdev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
            flag = torch.tensor([0 if failure is None else 1], device=cdev)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            if int(flag) and failure is None:
                failure = RuntimeError("label_reward failed on another rank; nothing was written")
        if failure is not None:
            release_cached_engine()                  # do not keep a handle that may be in an error state
            raise failure
        if distributed:
            rows = [int(off[b] - off[a]) for a, b in shards]
            for img_key in image_keys:
                # [n, 2G, F] (reward, rtg of group 0, then of group 1, ...): the path's one collective
                both = torch.from_numpy(np.stack(results[img_key], axis=1)).to(cdev)
                full = gather_rows(both, rows, dst=0)
                if rank == 0:
                    full = full.cpu().numpy()
                    results[img_key] = [np.ascontiguousarray(full[:, k]) for k in range(full.shape[1])]
                if stored == "save":                 # the second gather: every rank's embeddings (records) to rank 0
                    full = gather_rows(torch.from_numpy(embs[img_key]).to(cdev), rows, dst=0)
                    embs[img_key] = full.cpu().numpy() if rank == 0 else None
    finally:
        if labeler is not None:
            labeler.close()
        g.close()
    _mark("gather + close")
    if distributed:
        dist.barrier()                                   # every reader has closed
    if rank == 0:
        g = open_store(data_path, "a")
        try:
            for img_key in image_keys:
                _write_labels(g, img_key, target_keys, results[img_key], off, n_eps, len_data, num_frames)
                if stored == "save" and n_eps > 0:
                    _write_embeddings(g, _stored_key(img_key, model_type, tower), embs[img_key], sigs[img_key],
                                      embeddings)
        finally:
            g.close()
    _mark("write labels")
    if distributed:
        dist.barrier()
    if os.environ.get("ARP_TIMING", "0") not in ("", "0") and rank == 0:
        print("[arp_b200] label_reward phases: " + ", ".join(f"{b[0]} {b[1] - a[1]:.3f} s" for a, b in zip(_t[:-1], _t[1:]))
              + f"; total {_t[-1][1] - _t[0][1]:.3f} s", flush=True)


def _empty_pairs(labeler, n_groups: int, num_frames: int):
    empty = np.zeros((n_groups, 0, num_frames), np.float64 if labeler.goal else np.float32)
    return _pairs(empty, empty)


def _pairs(rs, gs):
    """[G, rows, F] x 2 -> [reward_stacked, rtg_stacked] of each group in turn"""
    return [a for g in range(rs.shape[0]) for a in (rs[g], gs[g])]


def _finish(labeler, r, rs, gs, rel_off, num_frames):
    """[G, rows, F] whether or not the labeler returned a group axis (goal heads: the float64 scan of their rewards)"""
    if labeler.goal:
        rs, gs = _goal_float64(r, rel_off, num_frames)
    return (rs, gs) if rs.ndim == 3 else (rs[None], gs[None])


def _file_rows(labeler, src, method: str, lo_all: int):
    """(path, byte offset of row lo_all's scored frame, row stride) when the rows sit contiguously in a file and the
    labeler reads files itself (`method`), else None"""
    fsrc = src.file_source() if hasattr(src, "file_source") and hasattr(labeler, method) else None
    if fsrc is None:
        return None
    path, base = fsrc
    frame = int(np.prod(src.shape[-3:]))
    stride = frame * (src.shape[1] if len(src.shape) == 5 else 1)
    return path, base + lo_all * stride + (stride - frame), stride        # last stacked frame of row lo_all


def _zfile_rows(ds):
    """(path, chunk byte offsets [T], chunk sizes [T], row bytes) when every row of the image dataset `ds` is one plain
    zlib stream at a known place of its HDF5 file, else None: an h5py dataset (its low-level chunk index is read through
    DatasetID.get_num_chunks / get_chunk_info) of uint8 rows chunked (1, *shape[1:]), gzip and no other filter (no shuffle,
    fletcher32 or scale-offset), every row's chunk allocated and written with filter_mask 0. No HDF5 structure is parsed
    here: h5py says where each chunk is, and the library inflates it."""
    dsid = getattr(ds, "id", None)
    if dsid is None or not hasattr(dsid, "get_chunk_info") or getattr(getattr(ds, "file", None), "filename", None) is None:
        return None
    shape = tuple(ds.shape)
    if len(shape) not in (4, 5) or np.dtype(ds.dtype) != np.uint8 or tuple(ds.chunks or ()) != (1,) + shape[1:]:
        return None
    if ds.compression != "gzip" or ds.shuffle or ds.fletcher32 or getattr(ds, "scaleoffset", None) is not None:
        return None
    plist = getattr(dsid, "get_create_plist", None)
    if plist is not None and plist().get_nfilters() != 1:      # a filter h5py has no property for
        return None
    T = shape[0]
    n = dsid.get_num_chunks()
    if n != T:                                                   # an unallocated row
        return None
    offsets = np.full(T, -1, np.int64)
    sizes = np.zeros(T, np.int64)
    for i in range(n):
        info = dsid.get_chunk_info(i)
        t = int(info.chunk_offset[0])
        if info.filter_mask != 0 or info.byte_offset is None or not 0 <= t < T or offsets[t] >= 0:
            return None
        offsets[t], sizes[t] = int(info.byte_offset), int(info.size)
    return ds.file.filename, offsets, sizes, int(np.prod(shape[1:]))


def _read_slabs(ds, side, off, e_lo: int, e_hi: int, slab_frames: int):
    """(a, b, rows) of every non-empty slab of whole episodes [a, b), read on a thread one slab ahead of the consumer"""
    import threading
    slabs = [(a, b) for a, b in _slabs(off, e_lo, e_hi, slab_frames) if off[b] > off[a]]
    box = {}

    def read(i):
        a, b = slabs[i]
        try:
            box[i] = _rows_array(ds, int(off[a]), int(off[b]), side)
        except Exception as e:  # noqa: BLE001 — re-raised on the consumer side
            box[i] = e

    if not slabs:
        return
    th = threading.Thread(target=read, args=(0,))
    th.start()
    for i, (a, b) in enumerate(slabs):
        th.join()
        rows = box.pop(i)
        if isinstance(rows, Exception):
            raise rows
        if i + 1 < len(slabs):
            th = threading.Thread(target=read, args=(i + 1,))
            th.start()
        yield a, b, rows


def _label_rows(labeler, ds, side, off, e_lo: int, e_hi: int, num_frames: int, slab_frames: int, n_groups: int = 1):
    """[reward_stacked, rtg_stacked] of each of the n_groups instruction sets in turn (2 * n_groups arrays [rows, F]) for
    episodes [e_lo, e_hi). A memory-mapped container is handed to the library in ONE call (a strided pointer into the file
    mapping; the native stager overlaps page-cache reads, PCIe and compute). An h5py gzip dataset chunked one row per
    chunk (_zfile_rows) is handed over as its chunk table: the library reads the compressed rows and inflates them on the
    device. Any other container that has to be read through its API is read slab by slab on a reader thread, one slab
    ahead of the GPU."""
    lo_all, hi_all = int(off[e_lo]), int(off[e_hi])
    if hi_all <= lo_all:
        return _empty_pairs(labeler, n_groups, num_frames)
    src = side if side is not None else ds
    rel = off[e_lo:e_hi + 1] - lo_all
    zrows = _zfile_rows(ds) if side is None and hasattr(labeler, "label_zfile") else None
    if zrows is not None:
        # gzip rows, one per chunk: the library preads this shard's compressed chunks and inflates them on the device
        path, offsets, sizes, row_bytes = zrows
        fd = os.open(path, os.O_RDONLY)
        try:
            r, _, rs, gs = labeler.label_zfile(fd, offsets[lo_all:hi_all], sizes[lo_all:hi_all], row_bytes, rel,
                                               num_frames)
        finally:
            os.close(fd)
        return _pairs(*_finish(labeler, r, rs, gs, rel, num_frames))
    frows = _file_rows(labeler, src, "label_file", lo_all)
    if frows is not None:
        # rows contiguous in a file: the library preads the scored frame of every row itself (arp_label_file)
        path, first, stride = frows
        fd = os.open(path, os.O_RDONLY)
        try:
            r, _, rs, gs = labeler.label_file(fd, first, hi_all - lo_all, stride, rel, num_frames)
        finally:
            os.close(fd)
        return _pairs(*_finish(labeler, r, rs, gs, rel, num_frames))
    arr = getattr(src, "array", None)
    if arr is not None and arr.flags.c_contiguous:
        r, _, rs, gs = labeler.label_slab(arr[lo_all:hi_all], rel, num_frames)
        return _pairs(*_finish(labeler, r, rs, gs, rel, num_frames))

    parts_r, parts_g = [], []
    for a, b, rows in _read_slabs(ds, side, off, e_lo, e_hi, slab_frames):
        rel = off[a:b + 1] - off[a]
        r, _, rs, gs = labeler.label_slab(rows, rel, num_frames)
        rs, gs = _finish(labeler, r, rs, gs, rel, num_frames)
        parts_r.append(rs)
        parts_g.append(gs)
    if not parts_r:
        return _empty_pairs(labeler, n_groups, num_frames)
    return _pairs(np.concatenate(parts_r, axis=1), np.concatenate(parts_g, axis=1))


def _embed_rows(labeler, ds, side, off, e_lo: int, e_hi: int, slab_frames: int, tower: bool = False) -> np.ndarray:
    """float32 [rows, dim]: the stored embedding (tower: the CLIP tower record) of every row of episodes [e_lo, e_hi),
    read from the container as _label_rows reads it (same calls, same chunking of the encoder pass)."""
    embed_file, embed_slab = ("embed_tower_file", "embed_tower_slab") if tower else ("embed_file", "embed_slab")
    dim = labeler.tower_dim if tower else labeler.embedding_dim
    lo_all, hi_all = int(off[e_lo]), int(off[e_hi])
    if hi_all <= lo_all:
        return np.zeros((0, dim), np.float32)
    src = side if side is not None else ds
    embed_zfile = "embed_tower_zfile" if tower else "embed_zfile"
    zrows = _zfile_rows(ds) if side is None and hasattr(labeler, embed_zfile) else None
    if zrows is not None:
        path, offsets, sizes, row_bytes = zrows
        fd = os.open(path, os.O_RDONLY)
        try:
            return getattr(labeler, embed_zfile)(fd, offsets[lo_all:hi_all], sizes[lo_all:hi_all], row_bytes)
        finally:
            os.close(fd)
    frows = _file_rows(labeler, src, embed_file, lo_all)
    if frows is not None:
        path, first, stride = frows
        fd = os.open(path, os.O_RDONLY)
        try:
            return getattr(labeler, embed_file)(fd, first, hi_all - lo_all, stride)
        finally:
            os.close(fd)
    arr = getattr(src, "array", None)
    if arr is not None and arr.flags.c_contiguous:
        return getattr(labeler, embed_slab)(arr[lo_all:hi_all])
    parts = [getattr(labeler, embed_slab)(rows) for _, _, rows in _read_slabs(ds, side, off, e_lo, e_hi, slab_frames)]
    return np.concatenate(parts) if parts else np.zeros((0, dim), np.float32)


def _label_embedding_rows(labeler, emb: np.ndarray, off, e_lo: int, e_hi: int, num_frames: int, n_groups: int = 1,
                          tower: bool = False):
    """_label_rows' result from the stored embeddings (tower: CLIP tower records) of the same rows, labeled in one call
    on the device"""
    lo_all, hi_all = int(off[e_lo]), int(off[e_hi])
    if hi_all <= lo_all:
        return _empty_pairs(labeler, n_groups, num_frames)
    rel = off[e_lo:e_hi + 1] - lo_all
    label = labeler.label_tower if tower else labeler.label_embeddings
    r, _, rs, gs = label(emb, rel, num_frames)
    return _pairs(*_finish(labeler, r, rs, gs, rel, num_frames))


def _stored_key(img_key: str, model_type: str, tower: bool) -> str:
    return tower_key(img_key) if tower else embedding_key(img_key, model_type)


def _check_stored_embeddings(g, img_key, model_type, off, n_eps, sig, embeddings):
    """"load" / "load_tower": the embedding (tower record) dataset and its signature exist, cover the labeled rows and
    match `sig`. "save" / "save_tower": an existing dataset has the shape this pass writes. ValueError otherwise."""
    tower = embeddings in ("save_tower", "load_tower")
    key = _stored_key(img_key, model_type, tower)
    shape = (int(off[n_eps] - off[0]) if n_eps > 0 else 0,
             TOWER_DIM if tower else EMBEDDING_DIM[embedding_family(model_type)])
    ds = g.get(key)
    if embeddings in ("save", "save_tower"):
        if ds is not None and tuple(ds.shape) != shape:
            raise ValueError(f"embeddings={embeddings!r}: {key} exists with shape {tuple(ds.shape)}, this pass writes "
                             f"{shape}")
        return
    save = "save_tower" if tower else "save"
    if ds is None:
        raise ValueError(f"embeddings={embeddings!r}: no dataset {key}; label once with embeddings={save!r}")
    sds = g.get(key + "_sig")
    if sds is None:
        raise ValueError(f"embeddings={embeddings!r}: {key} has no signature dataset {key}_sig")
    if tuple(ds.shape) != shape:
        raise ValueError(f"embeddings={embeddings!r}: {key} has shape {tuple(ds.shape)}, the labeled rows need {shape}")
    stored = np.asarray(sds[:], np.uint8).reshape(-1)
    if not np.array_equal(stored, sig):
        what = "CLIP weights" if tower else "checkpoint"
        raise ValueError(f"embeddings={embeddings!r}: the signature of {key} differs: it was saved with another {what}, "
                         "crop, frame size, arch or precision")


def _write_embeddings(g, key, emb: np.ndarray, sig: np.ndarray, embeddings: str = "save"):
    """float32 [rows, dim] uncompressed (assigned in place when it exists with this shape) + the uint8 [32] signature"""
    for k, a in ((key, np.ascontiguousarray(emb, np.float32)), (key + "_sig", sig)):
        existing = g.get(k)
        if existing is None:
            g.create_dataset(k, data=a)
        elif tuple(existing.shape) != a.shape:
            raise ValueError(f"embeddings={embeddings!r}: {k} exists with shape {tuple(existing.shape)}, this pass "
                             f"writes {a.shape}")
        else:
            existing[...] = a


def _goal_float64(r: np.ndarray, ep_off: np.ndarray, num_frames: int):
    """Goal-conditioned rewards are a float64 array in the reference (np.array of .item() values,
    label_reward.py:160-162,193-195), so its discount_cumsum / stack_outputs run in float64 and the
    datasets are float64. The per-frame distances come from the GPU in fp32 (exactly what .item()
    widens); the O(T) float64 scan is done here, sequentially right-to-left like :252-253."""
    r64 = r.astype(np.float64)
    g64 = np.empty_like(r64)
    for lo, hi in zip(ep_off[:-1], ep_off[1:]):
        if hi > lo:
            g64[lo:hi] = np.cumsum(r64[lo:hi][::-1])[::-1]
    F = num_frames
    idx = np.arange(len(r64))
    start = np.repeat(ep_off[:-1], np.diff(ep_off))
    win = np.maximum(start[:, None], idx[:, None] - (F - 1 - np.arange(F))[None, :])
    return r64[win], g64[win]


def _write_labels(g, img_key, target_keys, data, off, n_eps, len_data, num_frames):
    """label_reward.py:260-289, for every (key, array) of target_keys and data (a reward / rtg pair per instruction
    set). `data` rows are the labeled rows [off[0], off[n_eps]) in order. When the key does not
    exist the reference creates the dataset from the first episode (gzip, chunks (1,F), maxshape (len_data,F)) and
    APPENDS every later episode (:273-286) — one dataset of off[n_eps]-off[0] rows, whatever off[0] is (it is non-zero
    only in the "time" layout, :84-87). When the key exists it assigns in place at the true row indices (:288-289)."""
    if n_eps <= 0:
        return
    first, last = int(off[0]), int(off[n_eps])
    for _key, arr in zip(target_keys, data):
        key = f"{img_key}_{_key}"
        arr = arr[:last - first]
        existing = g.get(key)
        if not existing:
            g.create_dataset(key, compression="gzip", chunks=(1, num_frames), maxshape=(len_data, num_frames), data=arr)
        else:
            existing[first:last] = arr


def main():
    parser = argparse.ArgumentParser(description="Process rollout training arguments.")
    parser.add_argument("--env_name", type=str, default="coinrun")
    parser.add_argument("--env_type", type=str, default="none")
    parser.add_argument("--num_levels", type=int, default=500)
    parser.add_argument("--start_level", type=int, default=0)
    parser.add_argument("--distribution_mode", type=str, default="hard")
    parser.add_argument("--image_keys", type=str, default="ob")
    parser.add_argument("--data_path", type=str, default=None)
    parser.add_argument("--base_path", type=str, default="./demonstrations")
    parser.add_argument("--num_demonstrations", type=int, default=500)
    parser.add_argument("--save_type", type=str, default="npy", choices=["npy", "hdf5"])  # parsed, unused (:306)
    parser.add_argument("--num_frames", type=int, default=8)
    parser.add_argument("--model_type", type=str, default="clip")
    parser.add_argument("--model_ckpt_dir", type=str, default=None)
    parser.add_argument("--use_crop", type=bool, default=False)  # any non-empty string is True, as in :311
    parser.add_argument("--inst_type", type=str, default="none")
    # extensions
    parser.add_argument("--arch", type=str, default="ViT-B/16")
    parser.add_argument("--reduce", type=str, default="first", choices=["first", "mean"])
    parser.add_argument("--max_batch", type=int, default=1024)
    parser.add_argument("--precision", type=str, default="16bit", choices=sorted(capi.PRECISIONS))
    parser.add_argument("--tokenizer", type=str, default=None, choices=["clip", "standin"])
    parser.add_argument("--extra_inst_types", type=str, default=None,
                        help="comma-separated inst_types labeled in the same pass as --inst_type, e.g. random1,misinfo")
    parser.add_argument("--embeddings", type=str, default=None, choices=["save", "load", "save_tower", "load_tower"],
                        help="save: also store per-frame image embeddings; load: label from stored embeddings, no frames; "
                             "save_tower / load_tower (adapter model types): the same with CLIP tower records, which "
                             "relabel with any adapter checkpoint fine-tuned from the same CLIP")
    args = parser.parse_args()

    env_name = f"{args.env_name}" if args.env_type == "none" else f"{args.env_name}_{args.env_type}"

    def instruction(inst_type):
        return get_clip_instruct(env_name) if inst_type == "none" else get_clip_special_instruct(env_name, inst_type)

    text = instruction(args.inst_type)
    print(f"[INFO] env_name: {env_name}\t instruction: {text}")
    extra = None
    if args.extra_inst_types:
        extra = {t: instruction(t) for t in (x.strip() for x in args.extra_inst_types.split(",")) if t}
        for t, x in extra.items():
            print(f"[INFO] inst_type {t}: {x}")

    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")

    label_reward(
        env_name=args.env_name, env_type=args.env_type, distribution_mode=args.distribution_mode,
        image_keys=args.image_keys, data_path=args.data_path, text=text, num_levels=args.num_levels,
        start_level=args.start_level, num_demonstrations=args.num_demonstrations, num_frames=args.num_frames,
        base_path=args.base_path, model_type=args.model_type, model_ckpt_dir=args.model_ckpt_dir,
        use_crop=args.use_crop, inst_type=args.inst_type, arch=args.arch, reduce=args.reduce,
        max_batch=args.max_batch, precision=args.precision, tokenizer=args.tokenizer, extra_instructions=extra,
        embeddings=args.embeddings,
    )


if __name__ == "__main__":
    main()
