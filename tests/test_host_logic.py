"""Host-side logic of the drop-in: episode index, instruction lookup, store, slabbing, sharding partition."""
from pathlib import Path

import numpy as np
import pytest
import torch

from arp_b200 import instructions
from arp_b200.label_reward import _head_for, _slabs, center_crop, episode_index
from arp_b200.sharding import partition_episodes
from arp_b200.store import NpyStore, open_store
from arp_b200.synth import make_dataset, stack_frames, write_dataset


def test_episode_index_matches_oracle(tmp_path):
    from oracle import port
    d = make_dataset(n_episodes=7, len_lo=1, len_hi=6, size=64, num_frames=4, seed=3, tail_rows=3)
    s = NpyStore(tmp_path / "ds", "w")
    write_dataset(s, d)
    len_data, F, idx = episode_index(s)
    assert (len_data, F) == d["done"].shape and idx == port.episode_index(d["done"][:, -1])
    assert idx[-1] == int(d["lengths"].sum()) and len_data == idx[-1] + 3     # tail rows are never labeled
    s.close()


def test_episode_index_key_fallbacks(tmp_path):
    s = NpyStore(tmp_path / "a", "w")
    with pytest.raises(ValueError):                     # label_reward.py:78
        episode_index(s)
    done = np.zeros((6, 2), np.float32)
    done[[2, 5], -1] = 1
    s.create_dataset("is_terminal", data=done)
    assert episode_index(s)[2] == [0, 3, 6]
    s.close()
    t = NpyStore(tmp_path / "b", "w")                   # "time" layout fallback (:84-87)
    t.create_dataset("done", data=np.zeros(4, np.float32))          # 1-D -> the try block fails
    time = np.zeros((9, 2, 1), np.float32)
    time[[0, 4], -1, 0] = 1.0
    t.create_dataset("time", data=time)
    assert episode_index(t) == (9, 2, [0, 4, 9])
    t.close()


def test_instruction_strings():
    assert instructions.get_clip_instruct("coinrun") == "the goal is to collect the coin."
    assert instructions.get_clip_instruct("maze_redline_yellowgem") == "navigate a maze to collect the red line."
    assert instructions.get_clip_instruct("nope") is None
    assert instructions.get_clip_special_instruct("coinrun_aisc", "misinfo3") == "The goal is to reach the saw."
    with pytest.raises(ValueError):
        instructions.get_clip_special_instruct("maze", "misinfo2")


@pytest.mark.reference
def test_instruction_strings_equal_reference():
    from oracle import stubs
    stubs.import_reference()
    import arp_dt.data_procgen as ref
    for env in ("coinrun", "coinrun_aisc", "maze", "maze_aisc", "maze_yellowline", "maze_redline_yellowgem", "x"):
        assert instructions.get_clip_instruct(env) == ref.get_clip_instruct(env)
        for inst in ("random1", "random2", "misinfo", "misinfo2", "misinfo3", "misinfo4", "zzz"):
            try:
                want = ref.get_clip_special_instruct(env, inst)
            except ValueError:
                with pytest.raises(ValueError):
                    instructions.get_clip_special_instruct(env, inst)
                continue
            assert instructions.get_clip_special_instruct(env, inst) == want
    from arp_dt.assets.procgen_instruct import PROCGEN_POS_NEG_INSTRUCT
    for k, v in instructions.POS_NEG.items():
        assert PROCGEN_POS_NEG_INSTRUCT[k] == v
    # the stored table that test_instruction_strings_match_golden checks everywhere is the reference's too
    import json
    from oracle.make_golden_instructions import GOLDEN, reference_table
    gold = json.loads(GOLDEN.read_text())
    assert {k: gold[k] for k in ("clip_instruct", "clip_special_instruct", "pos_neg")} == reference_table()


def test_instruction_strings_match_golden():
    """Every lookup of tests/golden/instructions.json (oracle/make_golden_instructions.py): 7 envs x 7 instruction types,
    the refusals included, and every positive / negative prompt list."""
    import json
    from oracle.make_golden_instructions import ENVS, GOLDEN, INSTS, RAISES
    gold = json.loads(GOLDEN.read_text())
    assert list(gold["clip_instruct"]) == list(ENVS) and list(gold["clip_special_instruct"]) == list(ENVS)
    for env in ENVS:
        assert instructions.get_clip_instruct(env) == gold["clip_instruct"][env], env
        assert list(gold["clip_special_instruct"][env]) == list(INSTS)
        for inst, want in gold["clip_special_instruct"][env].items():
            if want == RAISES:
                with pytest.raises(ValueError):
                    instructions.get_clip_special_instruct(env, inst)
            else:
                assert instructions.get_clip_special_instruct(env, inst) == want, (env, inst)
    assert instructions.POS_NEG == gold["pos_neg"]


def test_model_type_dispatch():
    from arp_b200 import capi
    assert _head_for("clip") == (capi.HEAD_CLIP, capi.PRE_PIL_BICUBIC)
    assert _head_for("clip_goal_conditioned") == (capi.HEAD_CLIP_GOAL, capi.PRE_PIL_BICUBIC)
    assert _head_for("clip_ft") == (capi.HEAD_ADAPTER, capi.PRE_BILINEAR)
    assert _head_for("clip_multiscale_ensemble") == (capi.HEAD_ADAPTER_ENSEMBLE, capi.PRE_BILINEAR)
    assert _head_for("clip_ft_goal_conditioned") == (capi.HEAD_ADAPTER_GOAL, capi.PRE_BILINEAR)
    with pytest.raises(ValueError):
        _head_for("r3m")


def test_center_crop_matches_reference_formula():
    x = np.arange(2 * 9 * 9 * 3).reshape(2, 9, 9, 3)
    y = center_crop(x, (4, 4))
    assert y.shape == (2, 4, 4, 3) and np.array_equal(y, x[:, 2:6, 2:6])


def test_store_roundtrip_and_resize(tmp_path):
    s = open_store(tmp_path / "ds", "a")
    assert isinstance(s, NpyStore) and s.get("nope") is None and not s.get("nope")
    a = np.arange(12, dtype=np.float32).reshape(3, 4)
    ds = s.create_dataset("k", data=a, maxshape=(5, 4), chunks=(1, 4), compression="gzip")
    assert bool(ds) and ds.shape == (3, 4)
    with pytest.raises(ValueError):
        s.create_dataset("k", data=a)
    ds.resize(5, axis=0)
    ds[-2:] = np.ones((2, 4), np.float32)
    ds[[0, 1]] = np.zeros((2, 4), np.float32)
    with pytest.raises(ValueError):
        ds.resize(6, axis=0)
    s.close()
    r = open_store(tmp_path / "ds", "r")
    got = np.array(r["k"][:])
    assert got.shape == (5, 4) and got[:2].sum() == 0 and np.array_equal(got[2], a[2]) and got[3:].sum() == 8
    assert np.array_equal(r["k"][:, -1], got[:, -1]) and np.array_equal(r["k"][[0, 2], -1], got[[0, 2], -1])
    r.close()


def test_stack_frames_layout():
    x = np.arange(5)
    assert stack_frames(x, 3).tolist() == [[0, 0, 0], [0, 0, 1], [0, 1, 2], [1, 2, 3], [2, 3, 4]]


def test_slabs_cover_episodes_in_order():
    off = np.array([0, 10, 25, 26, 90, 100])
    slabs = list(_slabs(off, 0, 5, 30))
    assert slabs[0][0] == 0 and slabs[-1][1] == 5
    assert all(a[1] == b[0] for a, b in zip(slabs, slabs[1:]))
    assert slabs == [(0, 3), (3, 4), (4, 5)]            # whole episodes, grouped up to the frame budget
    assert list(_slabs(off, 2, 2, 30)) == []


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_partition_is_contiguous_and_balanced(world):
    rng = np.random.default_rng(world)
    lens = rng.integers(32, 256, size=500)
    off = np.concatenate([[0], np.cumsum(lens)])
    parts = partition_episodes(off, world)
    assert len(parts) == world and parts[0][0] == 0 and parts[-1][1] == 500
    assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
    frames = [off[b] - off[a] for a, b in parts]
    assert max(frames) - min(frames) <= 256 and sum(frames) == off[-1]
    # fewer episodes than ranks: empty ranges, still a partition
    small = partition_episodes(np.array([0, 5, 9]), 4)
    assert small[0][0] == 0 and small[-1][1] == 2 and all(a[1] == b[0] for a, b in zip(small, small[1:]))


def test_destacked_sidecar_roundtrip(tmp_path):
    """SURVEY.md §8(f)3: "<key>_last" holds exactly ob[:, -1]; _rows_array prefers it and ignores a stale one."""
    from arp_b200.label_reward import SIDECAR_SUFFIX, _rows_array, write_destacked_sidecar
    from arp_b200.store import NpyStore
    from arp_b200.synth import make_dataset, write_dataset
    data = make_dataset(n_episodes=3, len_lo=2, len_hi=6, size=64, num_frames=4, seed=9)
    s = NpyStore(tmp_path / "ds", "w")
    write_dataset(s, data)
    key = write_destacked_sidecar(s, "ob", rows_per_pass=5)
    assert key == "ob" + SIDECAR_SUFFIX and write_destacked_sidecar(s, "ob") == key      # idempotent
    s.close()
    s = NpyStore(tmp_path / "ds", "r")
    T = data["ob"].shape[0]
    assert s[key].shape == (T, 64, 64, 3) and np.array_equal(np.array(s[key][:]), data["ob"][:, -1])
    a = _rows_array(s["ob"], 1, T - 1, s[key])
    b = _rows_array(s["ob"], 1, T - 1)
    assert a.shape == (T - 2, 64, 64, 3) and np.array_equal(a, b[:, -1] if b.ndim == 5 else b)
    s.close()


# ---- property tests (hypothesis): ragged, empty and degenerate episode layouts -------------------------------------
from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=200, deadline=None)
@given(lens=st.lists(st.integers(0, 999), min_size=0, max_size=60), world=st.integers(1, 9), first=st.integers(0, 50))
def test_partition_properties(lens, world, first):
    """Any episode layout (zero-length episodes, fewer episodes than ranks, a non-zero first offset): the ranges are a
    contiguous partition in file order, and no rank is further from its fair share than the longest episode."""
    off = first + np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    parts = partition_episodes(off, world)
    n = len(lens)
    assert len(parts) == world and parts[0][0] == 0 and parts[-1][1] == n
    assert all(a <= b for a, b in parts) and all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
    total = int(off[-1] - off[0])
    longest = max(lens, default=0)
    ends = [int(off[b] - off[0]) for _, b in parts]
    for k, e in enumerate(ends[:-1], start=1):
        assert abs(e - total * k / world) <= longest       # every cut sits within one episode of its ideal place


@settings(max_examples=200, deadline=None)
@given(lens=st.lists(st.integers(0, 400), min_size=1, max_size=40), budget=st.integers(1, 600), data=st.data())
def test_slabs_properties(lens, budget, data):
    """Slabs are whole episodes in order, cover exactly [e_lo, e_hi), and only a single over-long episode may exceed
    the frame budget."""
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    n = len(lens)
    e_lo = data.draw(st.integers(0, n))
    e_hi = data.draw(st.integers(e_lo, n))
    slabs = list(_slabs(off, e_lo, e_hi, budget))
    if e_lo == e_hi:
        assert slabs == []
        return
    assert slabs[0][0] == e_lo and slabs[-1][1] == e_hi
    assert all(a < b for a, b in slabs) and all(a[1] == b[0] for a, b in zip(slabs, slabs[1:]))
    for a, b in slabs:
        assert off[b] - off[a] <= budget or b == a + 1


def test_tokenizer_refuses_the_standin_unless_opted_in(monkeypatch):
    """VERDICT r1 #7 / ADVICE: with openai/CLIP's tokenizer missing, real weights + stand-in ids would give garbage
    rewards silently. The stand-in must be an explicit choice (tokenizer="standin" or ARP_ALLOW_STANDIN_TOKENIZER=1)."""
    import sys
    from arp_b200 import tokenizer as tk
    shims = str(Path(__file__).resolve().parents[1] / "oracle" / "shims")
    if shims not in sys.path:
        sys.path.insert(0, shims)
    import clip as shim                                    # the oracle's stand-in package must not count as the real one
    assert getattr(shim, "__arp_oracle_shim__", False) and tk._real_tokenizer() is None
    monkeypatch.delenv("ARP_ALLOW_STANDIN_TOKENIZER", raising=False)
    with pytest.raises(tk.TokenizerUnavailable):
        tk.tokenize(["the goal is to collect the coin."])
    with pytest.raises(tk.TokenizerUnavailable):
        tk.resolve(None)(["x"])
    with pytest.raises(tk.TokenizerUnavailable):
        tk.resolve("clip")(["x"])
    t = tk.resolve("standin")(["a b", "c"])
    assert t.shape == (2, 77) and int(t[0, 0]) == tk.SOT and int(t[0].max()) == tk.EOT
    assert torch.equal(tk.resolve(lambda texts: torch.ones(len(texts), 77, dtype=torch.int32))(["q"]),
                       torch.ones(1, 77, dtype=torch.int32))
    monkeypatch.setenv("ARP_ALLOW_STANDIN_TOKENIZER", "1")
    assert torch.equal(tk.tokenize(["a b", "c"]), t)
    with pytest.raises(ValueError):
        tk.resolve("bpe")


def test_label_reward_refuses_without_a_tokenizer(tmp_path, monkeypatch):
    """The drop-in itself: a CLIP state_dict that is NOT flagged as an experiment + no `clip` package -> refuse before
    any frame is scored (the text embedding is built first)."""
    from arp_b200 import capi, tokenizer as tk
    from arp_b200.label_reward import RewardLabeler
    monkeypatch.delenv("ARP_ALLOW_STANDIN_TOKENIZER", raising=False)

    class FakeEngine:                                       # no GPU here: stop right after construction
        device, goal = torch.device("cpu"), False
        def __init__(self, **kw): pass
        def load_state_dict(self, sd, strict=False): return []
    monkeypatch.setattr(capi, "Engine", FakeEngine)
    with pytest.raises(tk.TokenizerUnavailable):
        RewardLabeler("clip", "the goal is to collect the coin.", (64, 64), clip_state_dict={"visual.proj": torch.zeros(1)})


def test_precision_names_are_one_table(monkeypatch):
    """label_reward, OnlineClip and FrozenClip accept exactly the names of capi.PRECISIONS and hand the engine the same
    enum for each; an unknown name is refused with ValueError when the object is built, before the library is used."""
    from arp_b200 import capi, label_reward
    from arp_b200.finetune import FrozenClip
    from arp_b200.online import OnlineClip
    from arp_b200.weights import random_clip_state_dict
    assert sorted(capi.PRECISIONS) == ["16bit", "bf16", "fp16", "fp32", "fp32resid"]
    built = []

    class FakeEngine:                                       # no GPU here: record what the engine would be built with
        device, goal = torch.device("cpu"), True
        def __init__(self, **kw):
            self.kw = kw
            built.append(kw)
        def load_state_dict(self, sd, strict=False): return []
        def close(self): pass

    def no_library():
        raise AssertionError("the native library was used")
    monkeypatch.setattr(capi, "Engine", FakeEngine)
    monkeypatch.setattr(capi, "load_library", no_library)
    monkeypatch.setattr(label_reward, "_ENGINE_CACHE", {})   # the labeler's handle cache: start and leave it untouched
    sd = random_clip_state_dict("ViT-B/32", 0, device="cpu", with_text=False)
    entry_points = {
        "label_reward": lambda p: label_reward.RewardLabeler("clip_goal_conditioned", None, (64, 64), clip_state_dict=sd,
                                                             arch="ViT-B/32", precision=p).engine,
        "online": lambda p: OnlineClip("clip", clip_state_dict=sd, arch="ViT-B/32", precision=p)._engine(64, 64),
        "finetune": lambda p: FrozenClip(sd, arch="ViT-B/32", precision=p)._get_engine(torch.device("cuda", 0)),
    }
    for name, make in entry_points.items():
        for p, enum in capi.PRECISIONS.items():
            assert make(p).kw["precision"] == enum, (name, p)
        n = len(built)
        for bad in ("bf32", "FP32", "fp16 ", "", None):
            with pytest.raises(ValueError, match="precision must be one of"):
                make(bad)
        assert len(built) == n, name
