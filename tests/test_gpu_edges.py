"""Edge cases and size-independent properties of the labeling path (-m gpu), through the C ABI.

What the domain offers at sizes the CPU oracle cannot reach: a frame's reward may not depend on where the frame sits
(which chunk, which row of a GEMM tile, which episode), re-labeling is idempotent, and the return-to-go our library
produced must be reproduced bit for bit by the oracle's scan over OUR rewards."""
import os
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


@pytest.fixture(scope="module")
def weights():
    from arp_b200.weights import random_clip_state_dict
    return random_clip_state_dict("ViT-B/16", 0, "cuda")


def _engine(capi, weights, n_text=1, **kw):
    e = capi.Engine(device=0, patch=16, in_h=kw.pop("size", 64), in_w=kw.pop("size_w", 64), **kw)
    e.load_state_dict(weights)
    g = torch.Generator().manual_seed(1)
    e.set_text(torch.nn.functional.normalize(torch.randn(n_text, 512, generator=g), dim=1), 1 / 0.07)
    return e


def _oracle_scan(r, off, F):
    from oracle import cport
    g = np.empty_like(r)
    rs = np.empty((len(r), F), np.float32)
    gs = np.empty((len(r), F), np.float32)
    for lo, hi in zip(off[:-1], off[1:]):
        g[lo:hi] = cport.discount_cumsum(r[lo:hi])
        rs[lo:hi] = cport.stack_outputs(r[lo:hi], F)
        gs[lo:hi] = cport.stack_outputs(g[lo:hi], F)
    return g, rs, gs


def test_empty_dataset_and_empty_episode_list(capi, weights):
    e = _engine(capi, weights, max_batch=8)
    ob = torch.zeros(0, 4, 64, 64, 3, dtype=torch.uint8, device="cuda")
    r, g, rs, gs = e.label(ob, torch.tensor([0]), 4)
    assert r.shape == (0,) and g.shape == (0,) and rs.shape == (0, 4) and gs.shape == (0, 4)
    h = e.label_host(np.zeros((0, 4, 64, 64, 3), np.uint8), np.array([0], np.int64), 4)
    assert all(a.shape[0] == 0 for a in h)
    # frames but no finished episode (no `done` yet): rewards are computed, nothing is scanned
    ob = torch.randint(0, 256, (5, 4, 64, 64, 3), dtype=torch.uint8, device="cuda")
    r2 = e.compute_reward(ob)
    assert r2.shape == (5,) and torch.isfinite(r2).all()
    # zero-length episodes between real ones (consecutive equal offsets) are skipped, not mis-scanned
    r3, g3, _, _ = e.label(ob, torch.tensor([0, 2, 2, 5]), 4)
    ref_g, _, _ = _oracle_scan(r3.cpu().numpy(), np.array([0, 2, 5]), 4)
    assert np.array_equal(g3.cpu().numpy(), ref_g) and torch.equal(r3, r2)
    e.close()


def test_reward_does_not_depend_on_chunk_size(capi, weights):
    """41 frames labeled with chunks of 3, 16 and 64 frames (ragged last chunk each time): identical bits."""
    rng = np.random.default_rng(3)
    ob = torch.from_numpy(rng.integers(0, 256, size=(41, 1, 64, 64, 3), dtype=np.uint8)).cuda()
    got = []
    for mb in (3, 16, 64):
        e = _engine(capi, weights, max_batch=mb)
        got.append(e.compute_reward(ob).cpu().numpy())
        e.close()
    assert np.array_equal(got[0], got[1]) and np.array_equal(got[1], got[2])


def test_position_independence_and_scan_at_scale(capi, weights):
    """12 288 frames = 192 distinct frames x 64 copies in shuffled order, 1024-frame chunks (the bench's chunk size),
    episodes of 1..999 frames: every copy of a frame gets the same bits wherever it lands; the rtg / stacks equal the
    oracle's scan over our rewards; labeling twice gives the same bits."""
    rng = np.random.default_rng(4)
    base = rng.integers(0, 256, size=(192, 64, 64, 3), dtype=np.uint8)
    idx = rng.permutation(np.repeat(np.arange(192), 64))
    ob = torch.from_numpy(base[idx]).cuda()
    lens = [999, 1, 1, 998, 1000 - 999] + rng.integers(1, 400, size=40).tolist()
    off = np.concatenate([[0], np.cumsum(lens)])
    off = off[off <= len(idx)].astype(np.int64)
    e = _engine(capi, weights, max_batch=1024)
    r, g, rs, gs = (t.cpu().numpy() for t in e.label(ob, torch.from_numpy(off), 8))
    first = np.zeros(192, np.float32)
    first[idx[::-1]] = r[::-1]
    assert np.array_equal(r, first[idx])                                  # same frame -> same bits, any position
    assert len(np.unique(r)) > 150                                        # and the frames do differ from each other
    n = int(off[-1])
    ref_g, ref_rs, ref_gs = _oracle_scan(r[:n], off, 8)
    assert np.array_equal(g[:n], ref_g) and np.array_equal(rs[:n], ref_rs) and np.array_equal(gs[:n], ref_gs)
    r2, g2, _, _ = (t.cpu().numpy() for t in e.label(ob, torch.from_numpy(off), 8))
    assert np.array_equal(r, r2) and np.array_equal(g[:n], g2[:n])
    e.close()


def test_max_instruction_count(capi, weights):
    e = _engine(capi, weights, n_text=capi.MAX_TEXT, max_batch=8, reduce=capi.REDUCE_MEAN)
    ob = torch.randint(0, 256, (6, 1, 64, 64, 3), dtype=torch.uint8, device="cuda")
    r, lg = e.compute_reward(ob, want_logits=True)
    assert lg.shape == (6, capi.MAX_TEXT)
    assert torch.allclose(r, lg.mean(dim=1), rtol=0, atol=1e-6)
    with pytest.raises(capi.ArpError) as ei:
        e.set_text(torch.zeros(capi.MAX_TEXT + 1, 512), 1.0)
    assert ei.value.code == capi.ARP_ERR_INVALID
    e.close()


@pytest.mark.parametrize("size", [50, 100, 200, 300, 512])
def test_decode_odd_frame_sizes_bit_exact(capi, size):
    """Sizes Procgen does not produce but the reference's transform accepts: row lengths that are not a multiple of 16
    bytes (50, 100), up-scaling (50), 5-tap / 7-tap / 11-tap Pillow kernels (200 / 300 / 512 -> 224)."""
    from oracle import port
    rng = np.random.default_rng(size)
    ob = rng.integers(0, 256, size=(3, 2, size, size, 3), dtype=np.uint8)
    ob[1, -1] = np.where(rng.random((size, size, 3)) < 0.5, 0, 255).astype(np.uint8)
    e = capi.Engine(device=0, patch=16, in_h=size, in_w=size, max_batch=4)
    out = e.decode_only(torch.from_numpy(ob).cuda()).cpu().numpy()
    tf = port.transform_pil(False, size)
    for t in range(3):
        assert np.array_equal(out[t], tf(ob[t, -1]).numpy()), f"frame {t}"
    e.close()


def test_crop_larger_than_the_frame_is_refused_loudly(capi):
    """use_crop takes CenterCrop(W // 2) (label_reward.py:96,104): on a frame shorter than that torchvision would zero-pad;
    the library refuses instead of inventing pixels."""
    with pytest.raises(capi.ArpError) as ei:
        capi.Engine(device=0, patch=16, in_h=40, in_w=128, use_crop=True, max_batch=4)
    assert ei.value.code == capi.ARP_ERR_INVALID and "crop" in str(ei.value)


def test_label_host_pageable_stager_equals_pinned(capi):
    """arp_label_host gathers pageable (e.g. memory-mapped) frames through its pinned ring with worker threads and copies
    pinned frames directly; both must give the bits of the device entry point. Ragged on purpose: max_batch 100 is not a
    multiple of the 64-frame staging slot, T = 457 is not a multiple of max_batch, rows are strided (F = 3)."""
    from arp_b200.weights import random_clip_state_dict
    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=100)
    e.load_state_dict(random_clip_state_dict("ViT-B/32", 0, "cuda"))
    e.set_text(torch.nn.functional.normalize(torch.randn(1, 512), dim=1), 14.3)
    rng = np.random.default_rng(3)
    lens = rng.integers(1, 60, size=16)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    T = int(off[-1]) + 5
    ob = rng.integers(0, 256, size=(T, 3, 64, 64, 3), dtype=np.uint8)
    pageable = e.label_host(ob, off, 4)
    pinned_t = torch.from_numpy(ob).pin_memory()
    pinned = e.label_host(pinned_t, off, 4)
    dev = [t.cpu().numpy() for t in e.label(torch.from_numpy(ob).cuda(), torch.from_numpy(off), 4)]
    n = int(off[-1])
    for a, b, c in zip(pageable, pinned, dev):
        assert np.array_equal(a[:n], b[:n]) and np.array_equal(a[:n], c[:n])
    # twice in a row (ring slots and their events are reused across calls)
    again = e.label_host(ob, off, 4)
    assert all(np.array_equal(a[:n], b[:n]) for a, b in zip(pageable, again))
    # and straight from a file (arp_label_file: the gather threads pread the last stacked frame of every row)
    import os
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ob.npy")
        np.save(path, ob)
        mm = np.load(path, mmap_mode="r")
        frame = 64 * 64 * 3
        fd = os.open(path, os.O_RDONLY)
        try:
            filed = e.label_file(fd, mm.offset + 2 * frame, T, 3 * frame, off, 4)
            with pytest.raises(capi.ArpError):                       # reading past the end of the file is an error, not zeros
                e.label_file(fd, mm.offset + 2 * frame + 3 * frame * 10, T, 3 * frame, off, 4)
        finally:
            os.close(fd)
    assert all(np.array_equal(a[:n], b[:n]) for a, b in zip(pageable, filed))
    e.close()


@pytest.mark.parametrize("H,W,crop", [(64, 96, False), (96, 64, False), (200, 256, False), (256, 200, False),
                                      (224, 300, False), (100, 37, False), (128, 160, True)])
def test_decode_non_square_frames_bit_exact(capi, H, W, crop):
    """Resize(224) takes the SHORTER side to 224 and CenterCrop(224) cuts the longer one (label_reward.py:113-114); with
    use_crop the square CenterCrop(W // 2) comes first (:96-97). Against the reference's own torchvision / PIL calls."""
    from oracle import port
    e = capi.Engine(device=0, patch=16, in_h=H, in_w=W, use_crop=crop, max_batch=4)
    rng = np.random.default_rng(H * 1000 + W)
    ob = rng.integers(0, 256, size=(3, 2, H, W, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:H, 0:W]
    ob[0, -1] = np.stack([yy * 255 // H, xx * 255 // W, (yy + xx) * 255 // (H + W)], -1).astype(np.uint8)
    out = e.decode_only(torch.from_numpy(ob).cuda()).cpu().numpy()
    tf = port.transform_pil(crop, W)
    for t in range(3):
        assert np.array_equal(out[t], tf(ob[t, -1]).numpy()), f"frame {t}"
    assert np.array_equal(out[1], port.transform_restated(ob[1, -1], crop))
    e.close()


_JITTER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from arp_b200 import capi
eng = capi.Engine(device=0, max_batch=8)
worst = 0.0
for rep in range(6):
    for B, L in ((40, 197), (13, 197), (1, 197), (30, 50)):
        g = torch.Generator(device="cuda").manual_seed(1000 * rep + B)
        qkv = (torch.randn(B * L, 2304, device="cuda", generator=g) * 1.5).to(capi.operand_dtype())
        out = eng.attention(qkv, B, L)
        torch.cuda.synchronize()
        q, k, v = qkv.float().view(B, L, 3, 12, 64).permute(2, 0, 3, 1, 4)
        ref = (torch.softmax(q @ k.transpose(-1, -2) * 0.125, -1) @ v).permute(0, 2, 1, 3).reshape(B * L, 768)
        assert torch.isfinite(out.float()).all(), (rep, B, L)
        worst = max(worst, float((out.float() - ref).abs().max() / ref.abs().max()))
eng.close()
print("JITTER_WORST", worst)
"""


@pytest.mark.gpu
def test_attention_protocol_survives_jitter(tmp_path):
    """The attention kernel's barrier protocol (turns, shared O accumulator, split smem rings) must not depend on the
    warps' usual relative speeds: the -DARP_ATTN_JITTER build sleeps a random 0..8 us at every hand-off. Several items
    per CTA (B = 40: 480 items over 148 CTAs) so that every ring and every parity wraps. A protocol hole shows up as a
    watchdog trap, a hang (timeout) or wrong numbers. Found the hard way: a single O-drained barrier shared by both
    slots let a waiter run two phases ahead of it as soon as the epilogue warps were slowed down; later a single
    "tile 1's turn begins" barrier let its waiter fall two phases behind (this test caught that one)."""
    import subprocess
    import sys
    from arp_b200.build import build_jitter
    lib = build_jitter()
    script = tmp_path / "jitter.py"
    script.write_text(_JITTER_SCRIPT)
    root = str(Path(__file__).resolve().parents[1])
    res = subprocess.run([sys.executable, str(script), root], env={**os.environ, "ARP_B200_LIB": str(lib)},
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    worst = float(res.stdout.split("JITTER_WORST")[1])
    assert worst < 2e-2
