"""Several instruction sets ("text groups") labeled from one encoder pass.

CPU: the drop-in refuses what one pass cannot label before it opens the dataset or builds an engine; the CLI resolves
--extra_inst_types like --inst_type; the sharded host path writes the same 2G datasets as a single process.
GPU (-m gpu): group g of a grouped call is bit for bit the same call after set_text(group g's rows), through every entry
point, for every text head; the launch count does not depend on G; the drop-in writes the 2G reference datasets."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_sharding_gloo import _free_port, _make_store

COINRUN_TYPES = ("none", "random1", "random2", "misinfo", "misinfo2", "misinfo3", "misinfo4")


# ------------------------------------------------------------------------------------------------
# CPU: refusals, CLI, sharded host path
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model_type,inst_type,extra", [
    ("clip", "none", {"none": "another text"}),                        # an extra with the primary's key
    ("clip", "misinfo", {"random1": "x", "misinfo": "y"}),             # likewise, suffixed
    ("clip_goal_conditioned", "none", {"random1": "x"}),               # goal heads take no text
    ("clip_ft_goal_conditioned", "none", {"random1": "x"}),
    ("clip", "none", {f"t{i}": "x" for i in range(16)}),               # 17 instruction sets
    ("clip", "none", {"random1": ["x"] * 17}),                         # 17 texts in one set
    ("clip", "none", {"random1": []}),                                 # an empty set
    ("clip", "none", {f"t{i}": ["x"] * 16 for i in range(4)}),         # 65 texts in all
])
def test_label_reward_refuses_before_opening_anything(tmp_path, model_type, inst_type, extra):
    from arp_b200.label_reward import label_reward
    with pytest.raises(ValueError, match="extra_instructions"):
        label_reward("coinrun", "hard", 500, 0, "the goal is to collect the coin.", str(tmp_path),
                     data_path=str(tmp_path / "does_not_exist"), model_type=model_type, inst_type=inst_type,
                     extra_instructions=extra, model_ckpt_dir=str(tmp_path / "ckpt.pt"))


def test_labeler_refuses_before_building_an_engine(monkeypatch):
    from arp_b200 import capi
    from arp_b200.label_reward import RewardLabeler

    def no_engine(**kw):
        raise AssertionError("an engine was built")
    monkeypatch.setattr(capi, "Engine", no_engine)
    with pytest.raises(ValueError, match="goal-conditioned"):
        RewardLabeler("clip_goal_conditioned", None, (64, 64), extra_instructions={"random1": "x"})
    with pytest.raises(ValueError, match="instruction sets"):
        RewardLabeler("clip", "x", (64, 64), extra_instructions={f"t{i}": "x" for i in range(16)})


def test_cli_resolves_extra_inst_types(monkeypatch):
    from arp_b200 import label_reward as lr
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    seen = {}
    monkeypatch.setattr(lr, "label_reward", lambda **kw: seen.update(kw))
    monkeypatch.setattr(sys, "argv", ["label_reward", "--env_name", "coinrun", "--extra_inst_types", "random1,misinfo"])
    lr.main()
    assert seen["text"] == get_clip_instruct("coinrun") and seen["inst_type"] == "none"
    assert seen["extra_instructions"] == {"random1": get_clip_special_instruct("coinrun", "random1"),
                                          "misinfo": get_clip_special_instruct("coinrun", "misinfo")}
    assert list(seen["extra_instructions"]) == ["random1", "misinfo"]
    # --inst_type keeps its meaning, "none" among the extras is the goal instruction
    monkeypatch.setattr(sys, "argv", ["label_reward", "--inst_type", "misinfo2", "--extra_inst_types", "none"])
    lr.main()
    assert seen["text"] == get_clip_special_instruct("coinrun", "misinfo2")
    assert seen["extra_instructions"] == {"none": get_clip_instruct("coinrun")}
    monkeypatch.setattr(sys, "argv", ["label_reward"])
    lr.main()
    assert seen["extra_instructions"] is None


class _GroupStubLabeler:
    """Deterministic per-frame stand-in with a group axis (test-only; the product has no CPU path): group g's reward is
    the frame mean scaled by a number derived from the group's texts."""
    goal = False

    class _Eng:
        device = torch.device("cpu")

    def __init__(self, model_type, text, frame_hw, **kw):
        from arp_b200.label_reward import _text_groups
        self.engine = self._Eng()
        self.groups = _text_groups(model_type, text, kw.get("extra_instructions"))
        self.grouped = bool(kw.get("extra_instructions"))

    def label_slab(self, ob, ep_offsets, num_frames):
        ob = np.asarray(ob)
        last = ob[:, -1] if ob.ndim == 5 else ob
        base = last.reshape(len(last), -1).astype(np.float64).mean(axis=1)
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

    def close(self):
        pass


EXTRA = {"random1": "His voice echoed through the empty hallway.",
         "misinfo": ["The agent must go to the far right of the level.", "The goal is to reach the saw."]}


def _label_groups(path, distributed):
    import arp_b200.label_reward as lr
    real = lr.RewardLabeler
    lr.RewardLabeler = _GroupStubLabeler
    try:
        lr.label_reward("coinrun", "hard", 500, 0, "the goal is to collect the coin.", ".", data_path=str(path),
                        model_type="clip", env_type="none", slab_frames=16, distributed=distributed,
                        extra_instructions=EXTRA)
    finally:
        lr.RewardLabeler = real


def _worker_groups(rank, world, port, path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _label_groups(path, True)
    finally:
        dist.destroy_process_group()


def test_grouped_host_path_gloo_equals_single_process(tmp_path):
    from arp_b200.store import NpyStore
    single, multi = tmp_path / "single", tmp_path / "multi"
    _make_store(single)
    _make_store(multi)
    _label_groups(single, False)
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker_groups, args=(r, 2, port, multi)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    a, b = NpyStore(single, "r"), NpyStore(multi, "r")
    keys = sorted(k for k in a.keys() if k.startswith("ob_"))
    assert keys == sorted(["ob_clip_reward", "ob_clip_pos_rtg", "ob_clip_reward_random1", "ob_clip_pos_rtg_random1",
                           "ob_clip_reward_misinfo", "ob_clip_pos_rtg_misinfo"])
    assert sorted(k for k in b.keys() if k.startswith("ob_")) == keys
    for k in keys:
        x, y = np.array(a[k][:]), np.array(b[k][:])
        assert x.shape == y.shape and x.dtype == y.dtype == np.float32 and np.array_equal(x, y), k
    assert not np.array_equal(np.array(a["ob_clip_reward"][:]), np.array(a["ob_clip_reward_misinfo"][:]))
    a.close()
    b.close()


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
# ragged groups: 1, 3, 2 and 16 texts
GROUPS = [["the goal is to collect the coin."],
          ["His voice echoed through the empty hallway.", "The agent must go to the far right of the level.",
           "The goal is to collect the red strawberry."],
          ["The goal is to reach the saw.", "The goal is to jump as high as you can."],
          [f"instruction number {i}: navigate to object {i % 5} and avoid hazard {i % 3}." for i in range(16)]]


@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


def _case(capi, golden, model_type, reduce, precision, max_batch=6):
    """(engine, per-group (emb, scale), ob [T,F,H,W,3], episode offsets) on a golden fixture's seeded inputs"""
    from _util import load_golden, rebuild_inputs
    from arp_b200.label_reward import _head_for
    from arp_b200.text_tower import adapter_text_embedding, clip_text_embedding
    from arp_b200.tokenizer import tokenize
    from oracle import port
    meta, _ = load_golden(golden)
    data, clip_sd, adapter_sd = rebuild_inputs(meta)
    head, pre = _head_for(model_type)
    size = meta["data"]["size"]
    e = capi.Engine(device=0, patch=32 if meta["arch"].endswith("/32") else 16, in_h=size, in_w=size, preprocess=pre,
                    head=head, reduce=capi.REDUCE_MEAN if reduce == "mean" else capi.REDUCE_FIRST, max_batch=max_batch,
                    precision=capi.precision_enum(precision))
    sd = adapter_sd if e.adapter else clip_sd
    assert not e.load_state_dict(sd)
    if e.adapter:
        embs = [adapter_text_embedding(sd, tokenize(g), e.device, ensemble=head == capi.HEAD_ADAPTER_ENSEMBLE)
                for g in GROUPS]
    else:
        embs = [clip_text_embedding(sd, tokenize(g), e.device) for g in GROUPS]
    idx = port.episode_index(data["done"][:, -1])
    ob = np.ascontiguousarray(data["ob"][:idx[-1]])
    return e, embs, ob, np.asarray(idx, np.int64)


def _every_entry_point(e, ob, off, path):
    """{entry point: outputs} for the same frames through label, label_host (pinned, pageable), label_file and
    compute_reward"""
    T, S = ob.shape[:2]
    F = S
    frame = int(np.prod(ob.shape[2:]))
    ob_dev = torch.from_numpy(ob).cuda()
    out = {"label": [t.cpu().numpy() for t in e.label(ob_dev, torch.from_numpy(off), F)],
           "host_pinned": list(e.label_host(torch.from_numpy(ob).pin_memory(), off, F)),
           "host_pageable": list(e.label_host(ob, off, F))}
    fd = os.open(path, os.O_RDONLY)
    try:
        out["file"] = list(e.label_file(fd, (S - 1) * frame, T, S * frame, off, F))
    finally:
        os.close(fd)
    r, lg = e.compute_reward(ob_dev, want_logits=True)
    out["compute_reward"] = [r.cpu().numpy(), lg.cpu().numpy()]
    return out


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
    ("g6_clipft_b16_64", "clip", "mean", "fp32resid"),
    ("g6_clipft_b16_64", "clip_ft", "mean", "fp32"),
])
def test_grouped_equals_separate_bit_for_bit(capi, tmp_path, golden, model_type, reduce, precision):
    e, embs, ob, off = _case(capi, golden, model_type, reduce, precision)
    path = tmp_path / "ob.bin"
    ob.tofile(path)
    T, F, G = ob.shape[0], ob.shape[1], len(GROUPS)
    e.set_text_groups([x for x, _ in embs], embs[0][1])
    assert e.n_groups == G
    grouped = _every_entry_point(e, ob, off, path)
    for name in ("label", "host_pinned", "host_pageable", "file"):
        assert [a.shape for a in grouped[name]] == [(G, T), (G, T), (G, T, F), (G, T, F)], name
    assert grouped["compute_reward"][0].shape == (G, T)
    assert grouped["compute_reward"][1].shape == (T, sum(map(len, GROUPS)))
    t0 = 0
    for g, (emb, scale) in enumerate(embs):
        e.set_text(emb, scale)
        assert e.n_groups == 1
        sep = _every_entry_point(e, ob, off, path)
        for name in ("label", "host_pinned", "host_pageable", "file"):
            for i, (a, b) in enumerate(zip(grouped[name], sep[name])):
                assert a[g].shape == b.shape and np.array_equal(a[g], b), (name, i, g)
        assert np.array_equal(grouped["compute_reward"][0][g], sep["compute_reward"][0]), g
        n = len(GROUPS[g])
        assert np.array_equal(grouped["compute_reward"][1][:, t0:t0 + n], sep["compute_reward"][1]), g
        t0 += n
    # the groups are different instructions: their rewards differ
    assert not np.array_equal(grouped["label"][0][0], grouped["label"][0][3])
    e.close()


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_groups(capi):
    """One encoder pass, one head launch per chunk and one scan launch per call, whatever G is."""
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from arp_b200.text_tower import clip_text_embedding
    from arp_b200.tokenizer import tokenize
    from arp_b200.weights import random_clip_state_dict
    e = capi.Engine(device=0, patch=16, in_h=64, in_w=64, max_batch=8)
    sd = random_clip_state_dict("ViT-B/16", 0, "cuda")
    e.load_state_dict(sd)
    texts = [get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t)
             for t in COINRUN_TYPES]
    embs = [clip_text_embedding(sd, tokenize([t]), e.device) for t in texts]
    off = torch.tensor([0, 7, 20, 29], dtype=torch.int64)
    ob = torch.from_numpy(np.random.default_rng(0).integers(0, 256, size=(29, 4, 64, 64, 3), dtype=np.uint8)).cuda()
    e.set_text(*embs[0])
    e.label(ob, off, 4)                                     # weights are finalised by the first call
    l0 = e.launch_count
    one = e.label(ob, off, 4)
    l1 = e.launch_count
    e.set_text_groups([x for x, _ in embs], embs[0][1])
    seven = e.label(ob, off, 4)
    l2 = e.launch_count
    assert l2 - l1 == l1 - l0 > 0
    assert seven[0].shape == (7, 29) and seven[3].shape == (7, 29, 4)
    assert all(torch.equal(a[0], b) for a, b in zip(seven, one))
    e.close()


@pytest.mark.gpu
def test_set_text_groups_refusals(capi):
    import ctypes as C
    from arp_b200.weights import random_clip_state_dict
    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4)
    e.load_state_dict(random_clip_state_dict("ViT-B/32", 0, "cuda"))
    unit = lambda n, d=512: torch.nn.functional.normalize(torch.randn(n, d), dim=1)  # noqa: E731

    def refused(fn):
        with pytest.raises(capi.ArpError) as err:
            fn()
        assert err.value.code == capi.ARP_ERR_INVALID

    refused(lambda: e.set_text_groups([unit(2), unit(0)], 14.3))                     # an empty group
    refused(lambda: e.set_text_groups([unit(17)], 14.3))                             # 17 texts in a group
    refused(lambda: e.set_text_groups([unit(1)] * 17, 14.3))                         # 17 groups
    refused(lambda: e.set_text_groups([unit(13)] * 5, 14.3))                         # 65 texts in all
    refused(lambda: e.set_text_groups([unit(2, 256)], 14.3))                         # wrong dim
    t = unit(4).cuda()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for bad in ([1, 2, 4], [0, 5, 4], [0, 2, 5]):                                    # offsets: start, order, end
        off = np.asarray(bad, np.int32)
        refused(lambda: e._check(e._lib.arp_set_text_groups(e._h, C.c_void_p(t.data_ptr()), 4, 512,
                                                              C.c_void_p(off.ctypes.data), 2, 14.3, stream)))
    frames = np.random.default_rng(0).integers(0, 256, size=(2, 64, 64, 3), dtype=np.uint8)
    e.set_text(unit(2), 14.3)
    single = e.online_reward(frames)["reward"]
    e.set_text_groups([unit(2), unit(1)], 14.3)
    assert e.n_groups == 2
    refused(lambda: e.online_reward(frames))                                         # no grouped online reward
    e.set_text(unit(2), 14.3)                                                        # back to one group
    assert e.n_groups == 1 and e.online_reward(frames)["reward"].shape == single.shape
    r = e.compute_reward(torch.from_numpy(frames[:, None]).cuda())
    assert r.shape == (2,)
    e.close()
    goal = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4, head=capi.HEAD_CLIP_GOAL)
    refused(lambda: goal.set_text_groups([unit(1)], 14.3))
    goal.close()


@pytest.mark.gpu
def test_drop_in_writes_every_instruction_set(tmp_path):
    """label_reward(..., extra_instructions=...) on a memory-mapped store writes exactly the 2G keys; each pair equals a
    separate label_reward call with that text and inst_type; a second call assigns in place and gives the same bits."""
    from arp_b200.label_reward import label_reward
    from arp_b200.store import NpyStore
    from arp_b200.synth import make_dataset, write_dataset
    from arp_b200.weights import random_clip_state_dict
    sd = random_clip_state_dict("ViT-B/32", 0, "cpu")
    data = make_dataset(n_episodes=4, len_lo=3, len_hi=11, size=64, num_frames=4, seed=7, tail_rows=2)
    primary = "the goal is to collect the coin."
    extra = {"random1": "His voice echoed through the empty hallway.",
             "misinfo": ["The agent must go to the far right of the level.", "The goal is to reach the saw."]}

    def store(name):
        s = NpyStore(tmp_path / name, "w")
        write_dataset(s, data)
        s.close()
        return tmp_path / name

    def run(path, text, inst_type, extra_instructions=None):
        label_reward("coinrun", "hard", 500, 0, text, str(tmp_path), data_path=str(path), model_type="clip",
                     inst_type=inst_type, clip_state_dict=sd, arch="ViT-B/32", max_batch=8, env_type="none",
                     reduce="mean", tokenizer="standin", extra_instructions=extra_instructions)

    def read(path):
        s = NpyStore(path, "r")
        out = {k: np.array(s[k][:]) for k in s.keys() if k.startswith("ob_")}
        s.close()
        return out

    grouped, separate = store("grouped"), store("separate")
    run(grouped, primary, "none", extra)
    got = read(grouped)
    assert sorted(got) == sorted(["ob_clip_reward", "ob_clip_pos_rtg", "ob_clip_reward_random1", "ob_clip_pos_rtg_random1",
                                  "ob_clip_reward_misinfo", "ob_clip_pos_rtg_misinfo"])
    run(separate, primary, "none")
    for inst_type, text in extra.items():
        run(separate, text, inst_type)
    want = read(separate)
    assert sorted(want) == sorted(got)
    for k in got:
        assert got[k].dtype == want[k].dtype == np.float32 and np.array_equal(got[k], want[k]), k
    run(grouped, primary, "none", extra)                   # the datasets exist now: assigned in place
    again = read(grouped)
    assert all(np.array_equal(again[k], got[k]) for k in got)
