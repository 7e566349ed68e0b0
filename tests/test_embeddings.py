"""Relabeling from stored image embeddings.

CPU: every refusal of label_reward(embeddings=...) happens before an engine is built; the CLI passes --embeddings
through; with a stand-in labeler, "save" then "load" writes the datasets of embeddings=None, a world-size-2 gloo "save"
writes what one process writes (embeddings included), and the signature follows the image-side weights, crop and frame
size.
GPU (-m gpu): arp_label_embeddings(arp_embed_*(frames)) is arp_label(frames) bit for bit for every head, reduce mode,
ragged text groups and precision; the three embed entry points agree; an embedding serves every head of its family; the
relabel needs no image weights and makes two launches; the drop-in reproduces its outputs from embeddings with the frames
zeroed; the C ABI refuses bad arguments."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharding_gloo import _free_port, _make_store

TEXT = "the goal is to collect the coin."
EXTRA = {"random1": "His voice echoed through the empty hallway.",
         "misinfo": ["The agent must go to the far right of the level.", "The goal is to reach the saw."]}


def _fake_clip_sd(seed=0):
    """a few image-side tensors (one above the signature's 4096 samples) and one text-side tensor"""
    g = torch.Generator().manual_seed(seed)
    return {"visual.proj": torch.randn(768, 16, generator=g), "visual.conv1.weight": torch.randn(10, 3, 4, 4, generator=g),
            "visual.class_embedding": torch.randn(768, generator=g), "token_embedding.weight": torch.randn(20, 8, generator=g)}


# ------------------------------------------------------------------------------------------------
# CPU: stand-in labeler
# ------------------------------------------------------------------------------------------------
def _stub_embed(ob):
    ob = np.asarray(ob)
    last = ob[:, -1] if ob.ndim == 5 else ob
    flat = last.reshape(len(last), -1).astype(np.float32) / 255.0
    reps = -(-512 // flat.shape[1])
    return np.ascontiguousarray(np.tile(flat, (1, reps))[:, :512])


class _EmbStubLabeler:
    """Deterministic stand-in with the labeler's embedding methods (test-only; the product has no CPU path): the embedding
    is the scored frame tiled to 512 floats, group g's reward its mean scaled by a number derived from the group's texts,
    and label_slab is label_embeddings(embed_slab(frames))."""
    goal = False
    embedding_dim = 512

    class _Eng:
        device = torch.device("cpu")

    def __init__(self, model_type, text, frame_hw, **kw):
        from arp_b200.label_reward import _text_groups
        self.engine = self._Eng()
        self.groups = _text_groups(model_type, text, kw.get("extra_instructions"))
        self.grouped = bool(kw.get("extra_instructions"))

    def embed_slab(self, ob):
        return _stub_embed(ob)

    def label_embeddings(self, emb, ep_offsets, num_frames):
        base = np.asarray(emb, np.float64).mean(axis=1)
        r = np.stack([(base * (1 + sum(map(len, g)) / 97.0)).astype(np.float32) for g in self.groups])
        g = np.zeros_like(r)
        for lo, hi in zip(ep_offsets[:-1], ep_offsets[1:]):
            acc = np.zeros(len(r), np.float32)
            for t in range(hi - 1, lo - 1, -1):
                acc = (r[:, t] + acc).astype(np.float32)
                g[:, t] = acc
        idx = np.arange(r.shape[1])
        start = np.repeat(ep_offsets[:-1], np.diff(ep_offsets))
        win = np.maximum(start[:, None], idx[:, None] - (num_frames - 1 - np.arange(num_frames))[None, :])
        out = r, g, r[:, win], g[:, win]
        return out if self.grouped else tuple(a[0] for a in out)

    def label_slab(self, ob, ep_offsets, num_frames):
        return self.label_embeddings(self.embed_slab(ob), ep_offsets, num_frames)

    def close(self):
        pass


def _stub_label(path, embeddings, distributed=False, extra=EXTRA):
    import arp_b200.label_reward as lr
    real = lr.RewardLabeler
    lr.RewardLabeler = _EmbStubLabeler
    try:
        lr.label_reward("coinrun", "hard", 500, 0, TEXT, ".", data_path=str(path), model_type="clip", env_type="none",
                        slab_frames=16, distributed=distributed, extra_instructions=extra, embeddings=embeddings,
                        clip_state_dict=_fake_clip_sd())
    finally:
        lr.RewardLabeler = real


def _read(path):
    from arp_b200.store import NpyStore
    s = NpyStore(path, "r")
    out = {k: np.array(s[k][:]) for k in s.keys() if k.startswith("ob_")}
    s.close()
    return out


def _zero_frames(path):
    from arp_b200.store import NpyStore
    s = NpyStore(path, "a")
    s["ob"][...] = 0
    s.close()


LABEL_KEYS = sorted(["ob_clip_reward", "ob_clip_pos_rtg", "ob_clip_reward_random1", "ob_clip_pos_rtg_random1",
                     "ob_clip_reward_misinfo", "ob_clip_pos_rtg_misinfo"])


def test_save_then_load_writes_the_datasets_of_frames(tmp_path, built_lib):
    plain, saved = tmp_path / "plain", tmp_path / "saved"
    _make_store(plain)
    _make_store(saved)
    _stub_label(plain, None)
    _stub_label(saved, "save")
    want, got = _read(plain), _read(saved)
    assert sorted(want) == LABEL_KEYS
    assert sorted(got) == sorted(LABEL_KEYS + ["ob_clip_emb", "ob_clip_emb_sig"])
    for k in LABEL_KEYS:
        assert got[k].dtype == want[k].dtype == np.float32 and np.array_equal(got[k], want[k]), k
    rows = want["ob_clip_reward"].shape[0]
    assert got["ob_clip_emb"].shape == (rows, 512) and got["ob_clip_emb"].dtype == np.float32
    assert got["ob_clip_emb_sig"].shape == (32,) and got["ob_clip_emb_sig"].dtype == np.uint8
    # "load" reads no frame: zero them, drop the labels, relabel from the embeddings
    _zero_frames(saved)
    for k in LABEL_KEYS:
        os.unlink(saved / f"{k}.npy")
    _stub_label(saved, "load")
    again = _read(saved)
    for k in LABEL_KEYS:
        assert np.array_equal(again[k], want[k]), k
    # a second "save" on the (now zeroed) frames assigns the embedding dataset in place
    _stub_label(saved, "save")
    assert not np.array_equal(_read(saved)["ob_clip_emb"], got["ob_clip_emb"])


def _worker_save(rank, world, port, path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _stub_label(path, "save", distributed=True)
    finally:
        dist.destroy_process_group()


def test_sharded_save_gloo_equals_single_process(tmp_path, built_lib):
    single, multi = tmp_path / "single", tmp_path / "multi"
    _make_store(single)
    _make_store(multi)
    _stub_label(single, "save")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker_save, args=(r, 2, port, multi)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    a, b = _read(single), _read(multi)
    assert sorted(a) == sorted(b) == sorted(LABEL_KEYS + ["ob_clip_emb", "ob_clip_emb_sig"])
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


def _signature(**kw):
    from arp_b200.label_reward import embedding_signature
    args = dict(model_type="clip", arch="ViT-B/16", frame_hw=(64, 64), use_crop=False, precision="16bit",
                state_dict=_fake_clip_sd())
    args.update(kw)
    return embedding_signature(**args)


def test_signature_follows_image_side_weights_crop_and_frame_size(built_lib):
    from arp_b200.label_reward import SIGNATURE_SAMPLES
    base = _signature()
    assert base.dtype == np.uint8 and base.shape == (32,)
    assert np.array_equal(base, _signature())

    def changed(name, flat_index, delta=1.0):
        sd = _fake_clip_sd()
        t = sd[name].reshape(-1)
        t[flat_index] += delta
        return _signature(state_dict=sd)

    n = _fake_clip_sd()["visual.proj"].numel()                  # 12288 values: 4096 of them are sampled
    sampled = 1 * (n - 1) // (SIGNATURE_SAMPLES - 1)
    assert not np.array_equal(changed("visual.proj", sampled), base)
    assert not np.array_equal(changed("visual.conv1.weight", 7), base)       # small tensors: every value
    assert not np.array_equal(_signature(use_crop=True), base)
    assert not np.array_equal(_signature(frame_hw=(256, 256)), base)
    assert not np.array_equal(_signature(frame_hw=(64, 32)), base)
    assert not np.array_equal(_signature(precision="fp32resid"), base)
    assert not np.array_equal(_signature(arch="ViT-B/32"), base)
    assert not np.array_equal(_signature(model_type="clip_ft"), base)       # another family
    # what does not decide the embedding's bits: the text tower, the head of the family, a precision alias
    assert np.array_equal(changed("token_embedding.weight", 3), base)
    assert np.array_equal(_signature(model_type="clip_goal_conditioned"), base)
    assert np.array_equal(_signature(precision="fp16"), base)
    assert np.array_equal(_signature(model_type="clip_ft"), _signature(model_type="clip_multiscale_ensemble"))
    # a provenance check, not a guarantee: a value between two sampled indices is not covered
    assert np.array_equal(changed("visual.proj", 1), base)


# ------------------------------------------------------------------------------------------------
# CPU: refusals before an engine exists
# ------------------------------------------------------------------------------------------------
def _no_engine(monkeypatch):
    from arp_b200 import capi

    def no_engine(**kw):
        raise AssertionError("an engine was built")
    monkeypatch.setattr(capi, "Engine", no_engine)


def _load(path, **kw):
    from arp_b200.label_reward import label_reward
    args = dict(data_path=str(path), model_type="clip", env_type="none", clip_state_dict=_fake_clip_sd(),
                embeddings="load")
    args.update(kw)
    label_reward("coinrun", "hard", 500, 0, TEXT, ".", **args)


def test_refusals_happen_before_an_engine_is_built(tmp_path, monkeypatch, built_lib):
    path = tmp_path / "ds"
    _make_store(path)
    _stub_label(path, "save", extra=None)
    good = _read(path)
    _no_engine(monkeypatch)
    with pytest.raises(ValueError, match="embeddings must be"):
        _load(path, embeddings="reuse")
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, clip_state_dict=_fake_clip_sd(seed=1))                  # another checkpoint
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, use_crop=True)
    with pytest.raises(ValueError, match="signature .* differs"):
        _load(path, precision="fp32")
    with pytest.raises(ValueError, match="no dataset ob_clip_adapter_emb"):
        _load(path, model_type="clip_ft", model_ckpt_dir={"image_residual_weight": torch.zeros(1)})
    with pytest.raises(AssertionError, match="an engine was built"):        # the stored set passes every check
        _load(path)
    with pytest.raises(AssertionError, match="an engine was built"):        # ... for every head of its family
        _load(path, model_type="clip_goal_conditioned")

    def rewrite(key, arr):
        if arr is None:
            os.unlink(path / f"{key}.npy")
        else:
            np.save(path / f"{key}.npy", arr)

    rewrite("ob_clip_emb", good["ob_clip_emb"][:-1])                        # a row short
    with pytest.raises(ValueError, match="shape"):
        _load(path)
    with pytest.raises(ValueError, match="exists with shape"):              # "save" will not overwrite another shape
        _load(path, embeddings="save")
    rewrite("ob_clip_emb", good["ob_clip_emb"])
    rewrite("ob_clip_emb_sig", None)
    with pytest.raises(ValueError, match="no signature"):
        _load(path)
    rewrite("ob_clip_emb", None)
    with pytest.raises(ValueError, match="no dataset ob_clip_emb"):
        _load(path)


def test_cli_passes_embeddings_through(monkeypatch):
    from arp_b200 import label_reward as lr
    seen = {}
    monkeypatch.setattr(lr, "label_reward", lambda **kw: seen.update(kw))
    for flag in ("save", "load"):
        monkeypatch.setattr(sys, "argv", ["label_reward", "--embeddings", flag])
        lr.main()
        assert seen["embeddings"] == flag
    monkeypatch.setattr(sys, "argv", ["label_reward"])
    lr.main()
    assert seen["embeddings"] is None
    monkeypatch.setattr(sys, "argv", ["label_reward", "--embeddings", "reuse"])
    with pytest.raises(SystemExit):
        lr.main()


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
# ragged groups: 1, 3 and 16 texts
GROUPS = [["the goal is to collect the coin."],
          ["His voice echoed through the empty hallway.", "The agent must go to the far right of the level.",
           "The goal is to collect the red strawberry."],
          [f"instruction number {i}: navigate to object {i % 5} and avoid hazard {i % 3}." for i in range(16)]]


@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


def _engine(capi, meta, model_type, reduce, precision, sd, max_batch=6, load=True):
    from arp_b200.label_reward import _head_for
    head, pre = _head_for(model_type)
    size = meta["data"]["size"]
    e = capi.Engine(device=0, patch=32 if meta["arch"].endswith("/32") else 16, in_h=size, in_w=size, preprocess=pre,
                    head=head, reduce=capi.REDUCE_MEAN if reduce == "mean" else capi.REDUCE_FIRST, max_batch=max_batch,
                    precision=capi.precision_enum(precision))
    if load:
        assert not e.load_state_dict(sd)
    return e


def _text(capi, e, sd, groups, grouped):
    from arp_b200.text_tower import adapter_text_embedding, clip_text_embedding
    from arp_b200.tokenizer import tokenize
    if e.goal:
        return
    if e.adapter:
        embs = [adapter_text_embedding(sd, tokenize(g), e.device, ensemble=e.cfg.head == capi.HEAD_ADAPTER_ENSEMBLE)
                for g in groups]
    else:
        embs = [clip_text_embedding(sd, tokenize(g), e.device) for g in groups]
    if grouped:
        e.set_text_groups([x for x, _ in embs], embs[0][1])
    else:
        e.set_text(*embs[0])


def _inputs(golden):
    from _util import load_golden, rebuild_inputs
    from oracle import port
    meta, _ = load_golden(golden)
    data, clip_sd, adapter_sd = rebuild_inputs(meta)
    idx = port.episode_index(data["done"][:, -1])
    ob = np.ascontiguousarray(data["ob"][:idx[-1]])
    return meta, ob, np.asarray(idx, np.int64), clip_sd, adapter_sd


def _embed_three_ways(e, ob, path):
    T, S = ob.shape[:2]
    frame = int(np.prod(ob.shape[2:]))
    pinned = e.embed_host(torch.from_numpy(ob).pin_memory())
    pageable = e.embed_host(ob)
    fd = os.open(path, os.O_RDONLY)
    try:
        from_file = e.embed_file(fd, (S - 1) * frame, T, S * frame)
    finally:
        os.close(fd)
    assert pinned.shape == (T, e.embedding_dim) and pinned.dtype == np.float32
    assert np.array_equal(pinned, pageable) and np.array_equal(pinned, from_file)
    return pinned


@pytest.mark.gpu
@pytest.mark.parametrize("golden,model_type,reduce,precision", [
    ("g6_clipft_b16_64", "clip", "first", "16bit"),
    ("g6_clipft_b16_64", "clip", "mean", "16bit"),
    ("g2_clip_b16_256", "clip", "first", "16bit"),
    ("g2_clip_b16_256", "clip", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_ft", "first", "16bit"),
    ("g6_clipft_b16_64", "clip_ft", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "first", "16bit"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "mean", "16bit"),
    ("g6_clipft_b16_64", "clip_goal_conditioned", "first", "16bit"),
    ("g6_clipft_b16_64", "clip_ft_goal_conditioned", "first", "16bit"),
    ("g6_clipft_b16_64", "clip", "mean", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft", "first", "fp32resid"),
    ("g6_clipft_b16_64", "clip_multiscale_ensemble", "mean", "fp32resid"),
    ("g6_clipft_b16_64", "clip_goal_conditioned", "first", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft_goal_conditioned", "first", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft", "mean", "fp32"),
])
def test_labels_from_embeddings_equal_labels_from_frames(capi, tmp_path, golden, model_type, reduce, precision):
    meta, ob, off, clip_sd, adapter_sd = _inputs(golden)
    family_adapter = model_type not in ("clip", "clip_goal_conditioned")
    sd = adapter_sd if family_adapter else clip_sd
    e = _engine(capi, meta, model_type, reduce, precision, sd)
    path = tmp_path / "ob.bin"
    ob.tofile(path)
    T, F = ob.shape[:2]
    assert e.embedding_dim == (13 * 512 if family_adapter else 512)
    emb = _embed_three_ways(e, ob, path)
    ob_dev = torch.from_numpy(ob).cuda()
    enc = e.encode_image(ob_dev).cpu()
    if family_adapter:
        assert torch.allclose(torch.nn.functional.normalize(torch.from_numpy(emb), dim=1), enc, rtol=0, atol=1e-6)
    else:
        assert np.array_equal(emb, enc.numpy())
    emb_dev = torch.from_numpy(emb).cuda()
    off_t = torch.from_numpy(off)
    for grouped in ((False,) if e.goal else (False, True)):
        _text(capi, e, sd, GROUPS if grouped else GROUPS[:1], grouped)
        want = [t.cpu().numpy() for t in e.label(ob_dev, off_t, F)]
        got = [t.cpu().numpy() for t in e.label_embeddings(emb_dev, off_t, F)]
        lead = (len(GROUPS),) if grouped else ()
        assert [a.shape for a in got] == [lead + (T,), lead + (T,), lead + (T, F), lead + (T, F)]
        for i, (a, b) in enumerate(zip(got, want)):
            assert a.shape == b.shape and np.array_equal(a, b), (grouped, i)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("saved_by,relabeled_by", [("clip_ft", "clip_multiscale_ensemble"),
                                                   ("clip", "clip_goal_conditioned")])
def test_embedding_serves_every_head_of_its_family(capi, saved_by, relabeled_by):
    meta, ob, off, clip_sd, adapter_sd = _inputs("g6_clipft_b16_64")
    sd = clip_sd if saved_by == "clip" else adapter_sd
    src = _engine(capi, meta, saved_by, "mean", "16bit", sd)
    emb = src.embed_host(ob)
    src.close()
    dst = _engine(capi, meta, relabeled_by, "mean", "16bit", sd)
    _text(capi, dst, sd, GROUPS[:1], False)
    F = ob.shape[1]
    off_t = torch.from_numpy(off)
    want = [t.cpu().numpy() for t in dst.label(torch.from_numpy(ob).cuda(), off_t, F)]
    got = [t.cpu().numpy() for t in dst.label_embeddings(torch.from_numpy(emb).cuda(), off_t, F)]
    for i, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(a, b), i
    dst.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type", ["clip", "clip_ft"])
def test_relabel_needs_no_image_weights_and_makes_two_launches(capi, model_type):
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from test_instruction_sets import COINRUN_TYPES
    meta, ob, off, clip_sd, adapter_sd = _inputs("g6_clipft_b16_64")
    sd = clip_sd if model_type == "clip" else adapter_sd
    full = _engine(capi, meta, model_type, "first", "16bit", sd)
    emb = torch.from_numpy(full.embed_host(ob)).cuda()
    bare = _engine(capi, meta, model_type, "first", "16bit", sd, load=False)
    assert bare.missing_weights()                                           # no image-side weight was ever set
    texts = [[get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t)]
             for t in COINRUN_TYPES]
    F = ob.shape[1]
    off_t = torch.from_numpy(off)
    for groups in (texts[:1], texts):
        for e in (full, bare):
            _text(capi, e, sd, groups, len(groups) > 1)
        want = [t.cpu().numpy() for t in full.label(torch.from_numpy(ob).cuda(), off_t, F)]
        l0 = bare.launch_count
        got = [t.cpu().numpy() for t in bare.label_embeddings(emb, off_t, F)]
        assert bare.launch_count - l0 == 2, len(groups)
        for i, (a, b) in enumerate(zip(got, want)):
            assert np.array_equal(a, b), (len(groups), i)
    assert bare.missing_weights()
    full.close()
    bare.close()


@pytest.mark.gpu
def test_c_abi_refusals(capi):
    import ctypes as C
    from arp_b200.weights import random_clip_state_dict
    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4)
    lib, h = e._lib, e._h
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    emb = torch.zeros(3, 512, device="cuda")
    off = torch.tensor([0, 3], dtype=torch.int64, device="cuda")
    out = torch.empty(3, 4, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    # a text head without text
    assert lib.arp_label_embeddings(h, p(emb), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_ERR_STATE
    e.set_text(torch.nn.functional.normalize(torch.randn(1, 512), dim=1), 14.3)
    assert lib.arp_label_embeddings(None, p(emb), 3, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_embeddings(h, None, 3, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_embeddings(h, p(emb), -1, p(off), 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_embeddings(h, p(emb), 3, None, 1, 4, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_embeddings(h, p(emb), 3, p(off), 1, 0, None, None, None, None, stream) == capi.ARP_ERR_INVALID
    assert lib.arp_label_embeddings(h, p(emb), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == capi.ARP_OK
    e.load_state_dict(random_clip_state_dict("ViT-B/32", 0, "cuda"))
    frames = np.zeros((2, 64, 64, 3), np.uint8)
    host = np.empty((2, 512), np.float32)
    hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    assert lib.arp_embed_host(None, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_host(h, hp(frames), 2, 64 * 64 * 3, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_host(h, None, 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_host(h, hp(frames), -1, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_file(h, -1, 0, 2, 64 * 64 * 3, hp(host)) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_file(h, 0, 0, 2, 64 * 64 * 3, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_host(h, hp(frames), 2, 64 * 64 * 3, hp(host)) == capi.ARP_OK
    assert lib.arp_embedding_dim(None) == 0 and lib.arp_embedding_dim(h) == 512
    e.close()
    goal = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4, head=capi.HEAD_CLIP_GOAL)
    assert goal._lib.arp_label_embeddings(goal._h, p(emb), 3, p(off), 1, 4, None, None, p(out), p(out), stream) == \
        capi.ARP_OK                                                          # goal heads take no text
    goal.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type", ["clip", "clip_ft"])
def test_drop_in_relabels_from_embeddings_without_frames(tmp_path, model_type):
    """label_reward(embeddings="save") writes the bytes of embeddings=None; with the frames zeroed, embeddings="load"
    reproduces them, extra instruction sets included."""
    from arp_b200.label_reward import embedding_key, label_reward
    from arp_b200.store import NpyStore
    from arp_b200.synth import make_dataset, write_dataset
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    sd = random_clip_state_dict("ViT-B/32", 0, "cpu")
    ckpt = random_adapter_state_dict("ViT-B/32", seed=1, device="cpu", clip_sd=sd) if model_type != "clip" else None
    data = make_dataset(n_episodes=4, len_lo=3, len_hi=11, size=64, num_frames=4, seed=7, tail_rows=2)

    def store(name):
        s = NpyStore(tmp_path / name, "w")
        write_dataset(s, data)
        s.close()
        return tmp_path / name

    def run(path, embeddings, extra=None):
        label_reward("coinrun", "hard", 500, 0, TEXT, str(tmp_path), data_path=str(path), model_type=model_type,
                     clip_state_dict=sd, model_ckpt_dir=ckpt, arch="ViT-B/32", max_batch=8, env_type="none",
                     reduce="mean", tokenizer="standin", extra_instructions=extra, embeddings=embeddings)

    plain, saved = store("plain"), store("saved")
    run(plain, None, EXTRA)
    run(saved, "save", EXTRA)
    want, got = _read(plain), _read(saved)
    key = embedding_key("ob", model_type)
    assert sorted(got) == sorted(list(want) + [key, key + "_sig"])
    for k in want:
        assert got[k].tobytes() == want[k].tobytes() and got[k].dtype == want[k].dtype, k
    _zero_frames(saved)
    for k in want:
        os.unlink(saved / f"{k}.npy")
    run(saved, "load", EXTRA)
    again = _read(saved)
    for k in want:
        assert again[k].tobytes() == want[k].tobytes(), k
