"""Relabeling with another fine-tuned adapter from stored CLIP tower records.

CPU: the tower signature follows the visual.* weights, crop, frame size, precision and arch but not the image adapter;
every refusal of label_reward(embeddings="save_tower" / "load_tower") happens before an engine is built; with a stand-in
labeler, "save_tower" then "load_tower" (frames zeroed) writes the datasets of embeddings=None; the CLI passes the new
values through; a world-size-2 gloo "save_tower" writes what one process writes.
GPU (-m gpu): arp_label_tower(arp_embed_tower_*(frames)) is arp_label(frames) bit for bit for every adapter head, reduce
mode, ragged text groups and precision, and the three record entry points agree; an engine holding only adapter B's
tensors labels adapter A's records to the bits of the full checkpoint B on the frames; labels do not depend on where the
records are cut into calls or chunks; the launch count does not depend on G; the C ABI refuses bad arguments; the
drop-in relabels with a new checkpoint from the records with the frames zeroed."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_embeddings import EXTRA, GROUPS, TEXT, _EmbStubLabeler, _fake_clip_sd, _read, _stub_embed, _zero_frames
from test_sharding_gloo import _free_port, _make_store

TOWER_DIM = 12 * 768 + 512


def _fake_ckpt(clip_seed=0, adapter_seed=0):
    """an adapter checkpoint: CLIP under "clip_model." plus small image-adapter (and text-adapter) tensors"""
    g = torch.Generator().manual_seed(1000 + adapter_seed)
    sd = {"clip_model." + k: v for k, v in _fake_clip_sd(clip_seed).items()}
    sd.update({"image_intermediate_linear.weight": torch.randn(24, 36, generator=g),
               "image_adapter.layers.0.weight": torch.randn(8, 5, generator=g),
               "image_adapter.layers.3.bias": torch.randn(5, generator=g),
               "image_residual_weight": torch.randn(1, generator=g),
               "text_adapter.layers.0.weight": torch.randn(8, 5, generator=g)})
    return sd


# ------------------------------------------------------------------------------------------------
# CPU: stand-in labeler
# ------------------------------------------------------------------------------------------------
class _TowerStubLabeler(_EmbStubLabeler):
    """_EmbStubLabeler with the tower methods (test-only): the record is the scored frame tiled to TOWER_DIM floats, and
    label_tower scales its first 512 columns by a gain taken from the checkpoint's image adapter before the embedding
    stand-in labels them, so a new adapter changes the labels; label_slab is label_tower(embed_tower_slab(frames))."""
    tower_dim = TOWER_DIM

    def __init__(self, model_type, text, frame_hw, **kw):
        super().__init__(model_type, text, frame_hw, **kw)
        self.gain = np.float32(1.0 + float(kw["model_ckpt_dir"]["image_residual_weight"].reshape(-1)[0]) / 8)

    def embed_tower_slab(self, ob):
        return np.ascontiguousarray(np.tile(_stub_embed(ob), (1, TOWER_DIM // 512)))

    def label_tower(self, rec, ep_offsets, num_frames):
        return self.label_embeddings(np.asarray(rec)[:, :512] * self.gain, ep_offsets, num_frames)

    def label_slab(self, ob, ep_offsets, num_frames):
        return self.label_tower(self.embed_tower_slab(ob), ep_offsets, num_frames)


def _stub_label(path, embeddings, distributed=False, extra=EXTRA, ckpt=None):
    import arp_b200.label_reward as lr
    real = lr.RewardLabeler
    lr.RewardLabeler = _TowerStubLabeler
    try:
        lr.label_reward("coinrun", "hard", 500, 0, TEXT, ".", data_path=str(path), model_type="clip_ft", env_type="none",
                        slab_frames=16, distributed=distributed, extra_instructions=extra, embeddings=embeddings,
                        model_ckpt_dir=ckpt if ckpt is not None else _fake_ckpt())
    finally:
        lr.RewardLabeler = real


LABEL_KEYS = sorted(["ob_clip_ft_reward", "ob_clip_ft_pos_rtg", "ob_clip_ft_reward_random1", "ob_clip_ft_pos_rtg_random1",
                     "ob_clip_ft_reward_misinfo", "ob_clip_ft_pos_rtg_misinfo"])
TOWER_KEYS = ["ob_clip_tower_emb", "ob_clip_tower_emb_sig"]


def test_save_tower_then_load_tower_writes_the_datasets_of_frames(tmp_path, built_lib):
    plain, saved, plain_b = tmp_path / "plain", tmp_path / "saved", tmp_path / "plain_b"
    for p in (plain, saved, plain_b):
        _make_store(p)
    _stub_label(plain, None)
    _stub_label(saved, "save_tower")
    want, got = _read(plain), _read(saved)
    assert sorted(want) == LABEL_KEYS
    assert sorted(got) == sorted(LABEL_KEYS + TOWER_KEYS)
    for k in LABEL_KEYS:
        assert got[k].dtype == want[k].dtype == np.float32 and np.array_equal(got[k], want[k]), k
    rows = want["ob_clip_ft_reward"].shape[0]
    assert got["ob_clip_tower_emb"].shape == (rows, TOWER_DIM) and got["ob_clip_tower_emb"].dtype == np.float32
    assert got["ob_clip_tower_emb_sig"].shape == (32,) and got["ob_clip_tower_emb_sig"].dtype == np.uint8
    # "load_tower" reads no frame: zero them, drop the labels, relabel from the records
    _zero_frames(saved)
    for k in LABEL_KEYS:
        os.unlink(saved / f"{k}.npy")
    _stub_label(saved, "load_tower")
    again = _read(saved)
    for k in LABEL_KEYS:
        assert np.array_equal(again[k], want[k]), k
    # ... and with another adapter of the same CLIP it writes what embeddings=None writes with that adapter
    other = _fake_ckpt(adapter_seed=1)
    _stub_label(plain_b, None, ckpt=other)
    _stub_label(saved, "load_tower", ckpt=other)
    want_b, again_b = _read(plain_b), _read(saved)
    assert not np.array_equal(want_b["ob_clip_ft_reward"], want["ob_clip_ft_reward"])
    for k in LABEL_KEYS:
        assert np.array_equal(again_b[k], want_b[k]), k
    # the gated-embedding datasets of embeddings="save" are not written by the tower modes
    assert "ob_clip_adapter_emb" not in again_b


def _worker_save(rank, world, port, path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _stub_label(path, "save_tower", distributed=True)
    finally:
        dist.destroy_process_group()


def test_sharded_save_tower_gloo_equals_single_process(tmp_path, built_lib):
    single, multi = tmp_path / "single", tmp_path / "multi"
    _make_store(single)
    _make_store(multi)
    _stub_label(single, "save_tower")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker_save, args=(r, 2, port, multi)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    a, b = _read(single), _read(multi)
    assert sorted(a) == sorted(b) == sorted(LABEL_KEYS + TOWER_KEYS)
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


def _signature(**kw):
    from arp_b200.label_reward import embedding_signature
    args = dict(model_type="clip_ft", arch="ViT-B/16", frame_hw=(64, 64), use_crop=False, precision="16bit",
                state_dict=_fake_ckpt(), tower=True)
    args.update(kw)
    return embedding_signature(**args)


def test_tower_signature_follows_visual_weights_not_the_adapter(built_lib):
    from arp_b200.label_reward import SIGNATURE_SAMPLES
    base = _signature()
    assert base.dtype == np.uint8 and base.shape == (32,)
    assert np.array_equal(base, _signature())

    def changed(name, flat_index, delta=1.0):
        sd = _fake_ckpt()
        t = sd[name].reshape(-1)
        t[flat_index] += delta
        return _signature(state_dict=sd)

    n = _fake_ckpt()["clip_model.visual.proj"].numel()
    sampled = 1 * (n - 1) // (SIGNATURE_SAMPLES - 1)
    assert not np.array_equal(changed("clip_model.visual.proj", sampled), base)
    assert not np.array_equal(changed("clip_model.visual.conv1.weight", 7), base)
    assert not np.array_equal(_signature(use_crop=True), base)
    assert not np.array_equal(_signature(frame_hw=(256, 256)), base)
    assert not np.array_equal(_signature(precision="fp32resid"), base)
    assert not np.array_equal(_signature(precision="fp32"), base)
    assert not np.array_equal(_signature(arch="ViT-B/32"), base)
    # another family than the gated embedding of the same checkpoint
    assert not np.array_equal(_signature(tower=False), base)
    # what does not decide the record's bits: every image-adapter tensor, the text side, the adapter head variant
    for name in ("image_intermediate_linear.weight", "image_adapter.layers.0.weight", "image_adapter.layers.3.bias",
                 "image_residual_weight", "text_adapter.layers.0.weight", "clip_model.token_embedding.weight"):
        assert np.array_equal(changed(name, 0), base), name
    assert np.array_equal(_signature(state_dict=_fake_ckpt(adapter_seed=5)), base)
    assert np.array_equal(_signature(model_type="clip_multiscale_ensemble"), base)
    assert np.array_equal(_signature(model_type="clip_ft_goal_conditioned"), base)
    # the CLIP tensors are read from the checkpoint's "clip_model." prefix: a bare CLIP state_dict signs the same
    assert np.array_equal(_signature(state_dict=_fake_clip_sd()), base)
    # ... while the gated embedding's signature does follow the adapter
    assert not np.array_equal(_signature(tower=False, state_dict=_fake_ckpt(adapter_seed=5)), _signature(tower=False))


# ------------------------------------------------------------------------------------------------
# CPU: refusals before an engine exists
# ------------------------------------------------------------------------------------------------
def _no_engine(monkeypatch):
    import arp_b200.label_reward as lr
    from arp_b200 import capi

    def no_engine(**kw):
        raise AssertionError("an engine was built")
    monkeypatch.setattr(capi, "Engine", no_engine)
    # a refused call releases the process's cached engine: start from none, whatever earlier tests left there
    monkeypatch.setattr(lr, "_ENGINE_CACHE", {})


def _load(path, **kw):
    from arp_b200.label_reward import label_reward
    args = dict(data_path=str(path), model_type="clip_ft", env_type="none", model_ckpt_dir=_fake_ckpt(),
                embeddings="load_tower")
    args.update(kw)
    label_reward("coinrun", "hard", 500, 0, TEXT, ".", **args)


def test_refusals_happen_before_an_engine_is_built(tmp_path, monkeypatch, built_lib):
    path = tmp_path / "ds"
    _make_store(path)
    _stub_label(path, "save_tower", extra=None)
    good = _read(path)
    _no_engine(monkeypatch)
    for mode in ("save_tower", "load_tower"):                               # the clip family has no tower record
        for mt in ("clip", "clip_goal_conditioned"):
            with pytest.raises(ValueError, match="adapter model types"):
                _load(path, embeddings=mode, model_type=mt, model_ckpt_dir=None, clip_state_dict=_fake_clip_sd())
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, model_ckpt_dir=_fake_ckpt(clip_seed=1))                  # another CLIP
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, use_crop=True)
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, precision="fp32")
    with pytest.raises(AssertionError, match="an engine was built"):        # the stored records pass every check
        _load(path)
    with pytest.raises(AssertionError, match="an engine was built"):        # ... with another adapter of that CLIP
        _load(path, model_ckpt_dir=_fake_ckpt(adapter_seed=3))
    with pytest.raises(AssertionError, match="an engine was built"):        # ... and for every adapter model type
        _load(path, model_type="clip_multiscale_ensemble")
    with pytest.raises(AssertionError, match="an engine was built"):
        _load(path, model_type="clip_ft_goal_conditioned")
    with pytest.raises(ValueError, match="no dataset ob_clip_adapter_emb"):  # the gated embedding is a separate record
        _load(path, embeddings="load")

    def rewrite(key, arr):
        if arr is None:
            os.unlink(path / f"{key}.npy")
        else:
            np.save(path / f"{key}.npy", arr)

    rewrite("ob_clip_tower_emb", good["ob_clip_tower_emb"][:-1])            # a row short
    with pytest.raises(ValueError, match="shape"):
        _load(path)
    with pytest.raises(ValueError, match="exists with shape"):              # "save_tower" will not overwrite another shape
        _load(path, embeddings="save_tower")
    rewrite("ob_clip_tower_emb", good["ob_clip_tower_emb"][:, :-512])       # another width
    with pytest.raises(ValueError, match="shape"):
        _load(path)
    rewrite("ob_clip_tower_emb", good["ob_clip_tower_emb"])
    rewrite("ob_clip_tower_emb_sig", None)
    with pytest.raises(ValueError, match="no signature"):
        _load(path)
    rewrite("ob_clip_tower_emb", None)
    with pytest.raises(ValueError, match="no dataset ob_clip_tower_emb"):
        _load(path)


def test_cli_passes_tower_modes_through(monkeypatch):
    from arp_b200 import label_reward as lr
    seen = {}
    monkeypatch.setattr(lr, "label_reward", lambda **kw: seen.update(kw))
    for flag in ("save_tower", "load_tower"):
        monkeypatch.setattr(sys, "argv", ["label_reward", "--model_type", "clip_ft", "--model_ckpt_dir", "new.pt",
                                          "--embeddings", flag])
        lr.main()
        assert seen["embeddings"] == flag and seen["model_type"] == "clip_ft" and seen["model_ckpt_dir"] == "new.pt"


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


def _engine(capi, meta, model_type, reduce, precision, sd=None, max_batch=6, adapter_only=False):
    """sd=None: no weight; adapter_only: only the image-adapter tensors of sd (no visual.*)"""
    from arp_b200.label_reward import _IMAGE_ADAPTER_PREFIXES, _head_for
    head, pre = _head_for(model_type)
    size = meta["data"]["size"]
    e = capi.Engine(device=0, patch=32 if meta["arch"].endswith("/32") else 16, in_h=size, in_w=size,
                    use_crop=meta.get("use_crop", False), preprocess=pre, head=head,
                    reduce=capi.REDUCE_MEAN if reduce == "mean" else capi.REDUCE_FIRST, max_batch=max_batch,
                    precision=capi.precision_enum(precision))
    if sd is not None and adapter_only:
        e.load_state_dict({k: v for k, v in sd.items() if k.startswith(_IMAGE_ADAPTER_PREFIXES)})
        assert e.missing_weights() and all(k.startswith("visual.") for k in e.missing_weights())
    elif sd is not None:
        assert not e.load_state_dict(sd)
    return e


def _text(capi, e, sd, groups, grouped):
    from test_embeddings import _text as text
    text(capi, e, sd, groups, grouped)


def _inputs(golden):
    from test_embeddings import _inputs as inputs
    return inputs(golden)


def _records_three_ways(e, ob, path):
    T, S = ob.shape[:2]
    frame = int(np.prod(ob.shape[2:]))
    pinned = e.embed_tower_host(torch.from_numpy(ob).pin_memory())
    pageable = e.embed_tower_host(ob)
    fd = os.open(path, os.O_RDONLY)
    try:
        from_file = e.embed_tower_file(fd, (S - 1) * frame, T, S * frame)
    finally:
        os.close(fd)
    assert pinned.shape == (T, TOWER_DIM) and pinned.dtype == np.float32
    assert np.array_equal(pinned, pageable) and np.array_equal(pinned, from_file)
    return pinned


@pytest.mark.gpu
@pytest.mark.parametrize("golden,model_type,reduce,precision", [
    ("g6_clipft_b16_64", "clip_ft", "first", "16bit"),
    ("g6_clipft_b16_64", "clip_ft", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "first", "16bit"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_ft_goal_conditioned", "first", "16bit"),
    ("g7_clipft_b16_256_crop", "clip_ft", "first", "16bit"),
    ("g7_clipft_b16_256_crop", "clip_multiscale_ensemble", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_ft", "first", "fp32resid"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "mean", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft_goal_conditioned", "first", "fp32resid"),
    ("g7_clipft_b16_256_crop", "clip_ft", "mean", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft", "mean", "fp32"),
    ("g6_clipft_b16_64", "clip_ft", "first", "fp32"),
])
def test_labels_from_tower_records_equal_labels_from_frames(capi, tmp_path, golden, model_type, reduce, precision):
    meta, ob, off, clip_sd, adapter_sd = _inputs(golden)
    e = _engine(capi, meta, model_type, reduce, precision, adapter_sd)
    assert e.tower_dim == TOWER_DIM
    path = tmp_path / "ob.bin"
    ob.tofile(path)
    T, F = ob.shape[:2]
    rec = _records_three_ways(e, ob, path)
    if precision != "fp32":
        # the 16-bit paths store the operand-format taps widened: narrowing them back is exact
        taps = torch.from_numpy(rec[:, :12 * 768])
        assert torch.equal(taps.to(capi.operand_dtype()).float(), taps)
    rec_dev = torch.from_numpy(rec).cuda()
    ob_dev = torch.from_numpy(ob).cuda()
    off_t = torch.from_numpy(off)
    for grouped in ((False,) if e.goal else (False, True)):
        _text(capi, e, adapter_sd, GROUPS if grouped else GROUPS[:1], grouped)
        want = [t.cpu().numpy() for t in e.label(ob_dev, off_t, F)]
        got = [t.cpu().numpy() for t in e.label_tower(rec_dev, off_t, F)]
        lead = (len(GROUPS),) if grouped else ()
        assert [a.shape for a in got] == [lead + (T,), lead + (T,), lead + (T, F), lead + (T, F)]
        for i, (a, b) in enumerate(zip(got, want)):
            assert a.shape == b.shape and np.array_equal(a, b), (grouped, i)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type,precision", [("clip_ft", "16bit"), ("clip_multiscale_ensemble", "fp32resid"),
                                                  ("clip_ft_goal_conditioned", "16bit"), ("clip_ft", "fp32")])
def test_records_relabel_with_another_adapter_checkpoint(capi, model_type, precision):
    """Records written by an engine with adapter A, labeled by an engine that holds only adapter B's tensors (no visual.*),
    give the bits of an engine with the whole checkpoint B labeling the frames — and differ from A's labels."""
    from arp_b200.weights import random_adapter_state_dict
    meta, ob, off, clip_sd, sd_a = _inputs("g6_clipft_b16_64")
    sd_b = random_adapter_state_dict(meta["arch"], seed=11, device="cuda",
                                     clip_sd={k: v.cuda() for k, v in clip_sd.items()})
    eng_a = _engine(capi, meta, model_type, "mean", precision, sd_a)
    rec = torch.from_numpy(eng_a.embed_tower_host(ob)).cuda()
    ob_dev = torch.from_numpy(ob).cuda()
    off_t = torch.from_numpy(off)
    F = ob.shape[1]
    _text(capi, eng_a, sd_a, GROUPS[:1], False)
    labels_a = [t.cpu().numpy() for t in eng_a.label(ob_dev, off_t, F)]
    eng_a.close()
    full_b = _engine(capi, meta, model_type, "mean", precision, sd_b)
    bare_b = _engine(capi, meta, model_type, "mean", precision, sd_b, adapter_only=True)
    for e in (full_b, bare_b):
        _text(capi, e, sd_b, GROUPS[:1], False)
    want = [t.cpu().numpy() for t in full_b.label(ob_dev, off_t, F)]
    got = [t.cpu().numpy() for t in bare_b.label_tower(rec, off_t, F)]
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), i
    assert not np.array_equal(got[0], labels_a[0])
    assert bare_b.missing_weights()                                           # still no visual.* weight
    full_b.close()
    bare_b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32resid", "fp32"])
def test_labels_do_not_depend_on_how_records_are_cut(capi, precision):
    """Two calls on the records cut at an episode boundary, on an engine with another max_batch, give the bits of one
    call: the adapter GEMM rows do not depend on which rows share a chunk (the sharded "load_tower" relies on it)."""
    meta, ob, off, clip_sd, adapter_sd = _inputs("g6_clipft_b16_64")
    one = _engine(capi, meta, "clip_ft", "mean", precision, adapter_sd, max_batch=6)
    rec = torch.from_numpy(one.embed_tower_host(ob)).cuda()
    two = _engine(capi, meta, "clip_ft", "mean", precision, adapter_sd, max_batch=4, adapter_only=True)
    F = ob.shape[1]
    for grouped in (False, True):
        groups = GROUPS if grouped else GROUPS[:1]
        for e in (one, two):
            _text(capi, e, adapter_sd, groups, grouped)
        want = [t.cpu().numpy() for t in one.label_tower(rec, torch.from_numpy(off), F)]
        for k in range(1, len(off) - 1):                                      # every inner episode boundary
            cut = int(off[k])
            first = two.label_tower(rec[:cut], torch.from_numpy(off[:k + 1]), F)
            second = two.label_tower(rec[cut:], torch.from_numpy(off[k:] - cut), F)
            for i, (a, b) in enumerate(zip(first, second)):
                got = np.concatenate([a.cpu().numpy(), b.cpu().numpy()], axis=-2 if i >= 2 else -1)
                assert np.array_equal(got, want[i]), (grouped, k, i)
    one.close()
    two.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision,per_chunk", [("16bit", 6), ("fp32", 5)])
def test_launch_count_does_not_depend_on_groups(capi, precision, per_chunk):
    """Per max_batch chunk: one unpack + the adapter tail (16-bit: intermediate GEMM, f32_to_bf16, fc1, fc2, head; fp32:
    three SGEMMs, head); one scan per call, for G = 1 and G = 7."""
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from test_instruction_sets import COINRUN_TYPES
    meta, ob, off, clip_sd, adapter_sd = _inputs("g6_clipft_b16_64")
    full = _engine(capi, meta, "clip_ft", "first", precision, adapter_sd, max_batch=4)
    rec = torch.from_numpy(full.embed_tower_host(ob)).cuda()
    full.close()
    bare = _engine(capi, meta, "clip_ft", "first", precision, adapter_sd, max_batch=4, adapter_only=True)
    texts = [[get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t)]
             for t in COINRUN_TYPES]
    T, F = ob.shape[:2]
    chunks = -(-T // 4)
    for groups in (texts[:1], texts):
        _text(capi, bare, adapter_sd, groups, len(groups) > 1)
        l0 = bare.launch_count
        bare.label_tower(rec, torch.from_numpy(off), F)
        assert bare.launch_count - l0 == chunks * per_chunk + 1, len(groups)
    bare.close()


@pytest.mark.gpu
def test_c_abi_refusals(capi):
    import ctypes as C
    from arp_b200.weights import random_adapter_state_dict
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rec = torch.zeros(3, TOWER_DIM, device="cuda")
    off = torch.tensor([0, 3], dtype=torch.int64, device="cuda")
    out = torch.empty(3, 4, device="cuda")
    frames = np.zeros((2, 64, 64, 3), np.uint8)
    host = np.empty((2, TOWER_DIM), np.float32)

    clip = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4)
    lib = clip._lib
    assert lib.arp_tower_dim(clip._h) == 0 and lib.arp_tower_dim(None) == 0 and clip.tower_dim == 0
    clip.set_text(torch.nn.functional.normalize(torch.randn(1, 512), dim=1), 14.3)
    assert lib.arp_label_tower(clip._h, p(rec), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == \
        capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_host(clip._h, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_file(clip._h, 0, 0, 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    clip.close()

    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4, head=capi.HEAD_ADAPTER,
                    preprocess=capi.PRE_BILINEAR)
    h = e._h
    assert lib.arp_tower_dim(h) == TOWER_DIM and e.tower_dim == TOWER_DIM
    # a text head without text, then an adapter tensor missing
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_ERR_STATE
    e.set_text(torch.nn.functional.normalize(torch.randn(1, 13 * 512), dim=1), 14.3)
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_ERR_STATE
    sd = random_adapter_state_dict("ViT-B/32", seed=2, device="cuda")
    adapter = {k: v for k, v in sd.items() if k.startswith(("image_intermediate_linear.", "image_adapter.",
                                                            "image_residual_weight"))}
    e.load_state_dict({k: v for k, v in adapter.items() if k != "image_residual_weight"})
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_ERR_STATE
    e.load_state_dict(adapter)
    assert lib.arp_label_tower(None, p(rec), 3, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, None, 3, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, C.c_void_p(rec.data_ptr() + 4), 2, p(off), 1, 4, None, None, None, None, stream) == \
        capi.ARP_ERR_INVALID                                                 # not 16-byte aligned
    assert lib.arp_label_tower(h, p(rec), -1, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, p(rec), 3, None, 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, p(rec), 3, p(off), -1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 0, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 65, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_tower(h, p(rec), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_OK
    # the embed entry points need the whole checkpoint (the tower runs the ViT)
    assert lib.arp_embed_tower_host(h, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_STATE
    assert not e.load_state_dict(sd)
    assert lib.arp_embed_tower_host(None, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_host(h, hp(frames), 2, 64 * 64 * 3, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_host(h, None, 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_host(h, hp(frames), -1, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_file(h, -1, 0, 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_file(h, 0, 0, 2, 64 * 64 * 3, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_host(h, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_OK
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type", ["clip_ft", "clip_ft_goal_conditioned"])
def test_drop_in_relabels_a_new_checkpoint_from_tower_records(tmp_path, model_type):
    """label_reward(embeddings="save_tower") writes the bytes of embeddings=None; with the frames zeroed,
    embeddings="load_tower" with checkpoint B writes what embeddings=None with B writes, extra instruction sets included."""
    from arp_b200.label_reward import label_reward, tower_key
    from arp_b200.store import NpyStore
    from arp_b200.synth import make_dataset, write_dataset
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    sd = random_clip_state_dict("ViT-B/32", 0, "cpu")
    ckpt_a = random_adapter_state_dict("ViT-B/32", seed=1, device="cpu", clip_sd=sd)
    ckpt_b = random_adapter_state_dict("ViT-B/32", seed=2, device="cpu", clip_sd=sd)
    data = make_dataset(n_episodes=4, len_lo=3, len_hi=11, size=64, num_frames=4, seed=7, tail_rows=2)
    extra = None if "goal" in model_type else EXTRA

    def store(name):
        s = NpyStore(tmp_path / name, "w")
        write_dataset(s, data)
        s.close()
        return tmp_path / name

    def run(path, embeddings, ckpt):
        label_reward("coinrun", "hard", 500, 0, TEXT, str(tmp_path), data_path=str(path), model_type=model_type,
                     model_ckpt_dir=ckpt, arch="ViT-B/32", max_batch=8, env_type="none", reduce="mean",
                     tokenizer="standin", extra_instructions=extra, embeddings=embeddings)

    plain_a, plain_b, saved = store("plain_a"), store("plain_b"), store("saved")
    run(plain_a, None, ckpt_a)
    run(plain_b, None, ckpt_b)
    run(saved, "save_tower", ckpt_a)
    want_a, want_b, got = _read(plain_a), _read(plain_b), _read(saved)
    key = tower_key("ob")
    assert sorted(got) == sorted(list(want_a) + [key, key + "_sig"])
    assert got[key].shape == (want_a[sorted(want_a)[0]].shape[0], TOWER_DIM)
    for k in want_a:
        assert got[k].tobytes() == want_a[k].tobytes() and got[k].dtype == want_a[k].dtype, k
    _zero_frames(saved)
    for k in want_a:
        os.unlink(saved / f"{k}.npy")
    run(saved, "load_tower", ckpt_b)
    again = _read(saved)
    for k in want_b:
        assert again[k].tobytes() == want_b[k].tobytes(), k
    assert any(want_a[k].tobytes() != want_b[k].tobytes() for k in want_a)
