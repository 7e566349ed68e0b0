"""Seven CoinRun instruction sets labeled in one pass versus one pass per set (B200).

    python tools/instruction_sets_bench.py [--frames 16384] [--rounds 3] [--out FILE]

bench.py's default configuration (CLIP ViT-B/16, 256x256 frames, rows of two stacked frames scored with the row stride,
pinned host frames through arp_label_host, max_batch 1024, random-init weights, stand-in token ids) on the first episodes
of bench.py's synthetic CoinRun-shaped dataset with at least --frames frames. After one untimed round, each round times,
in this order:
    g1          one pass with one instruction set (set_text + label_host)
    g7          one pass with the seven CoinRun instruction sets (set_text_groups + label_host)
    sequential  seven passes, one per set (set_text + label_host, seven times)
Every time is host wall clock ending in a device synchronise. The grouped outputs must equal the sequential ones bit for
bit. Prints one JSON line (also written to --out) with the median and every sample of each arm, the kernel launches of
each arm's call(s), and the card's name, power limit and SM clock read right after the timed rounds.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

INST_TYPES = ("none", "random1", "random2", "misinfo", "misinfo2", "misinfo3", "misinfo4")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16384, help="at least this many frames (whole episodes)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--num-frames", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("instruction_sets_bench.py needs a B200: arp_b200 has no CPU path")

    from bench import episode_offsets
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from arp_b200.text_tower import clip_text_embedding
    from arp_b200.tokenizer import tokenize
    from arp_b200.weights import random_clip_state_dict
    build()
    dev = torch.device("cuda", 0)
    size, S, F = 256, 2, args.num_frames
    off_all = episode_offsets(500, seed=1)
    n_eps = int(np.searchsorted(off_all, args.frames, side="left"))
    off = off_all[:n_eps + 1].copy()
    T = int(off[-1])

    eng = capi.Engine(device=0, patch=16, in_h=size, in_w=size, max_batch=1024, precision=capi.PREC_16BIT)
    sd = random_clip_state_dict("ViT-B/16", seed=0, device="cpu")
    eng.load_state_dict(sd)
    texts = [get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t) for t in INST_TYPES]
    embs = [clip_text_embedding(sd, tokenize([t], standin=True), dev) for t in texts]
    scale = embs[0][1]

    gen = torch.Generator(device=dev).manual_seed(1234)
    ob = torch.empty(T, S, size, size, 3, dtype=torch.uint8, pin_memory=True)
    for t0 in range(0, T, 2048):
        blk = ob[t0:t0 + 2048]
        blk.copy_(torch.randint(0, 256, blk.shape, dtype=torch.uint8, device=dev, generator=gen).cpu())

    G = len(embs)

    def outputs(lead=()):
        return (np.empty(lead + (T,), np.float32), np.empty(lead + (T,), np.float32),
                np.empty(lead + (T, F), np.float32), np.empty(lead + (T, F), np.float32))
    out1, out7, outs = outputs(), outputs((G,)), [outputs() for _ in range(G)]

    def g1():
        eng.set_text(*embs[0])
        eng.label_host(ob, off, F, out=out1)

    def g7():
        eng.set_text_groups([e for e, _ in embs], scale)
        eng.label_host(ob, off, F, out=out7)

    def sequential():
        for (e, s), o in zip(embs, outs):
            eng.set_text(e, s)
            eng.label_host(ob, off, F, out=o)

    arms = {"g1": g1, "g7": g7, "sequential": sequential}
    secs = {k: [] for k in arms}
    launches = {}

    def run(name, fn, record):
        torch.cuda.synchronize()
        l0 = eng.launch_count
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        launches[name] = eng.launch_count - l0
        if record:
            secs[name].append(dt)

    for r in range(args.rounds + 1):           # round 0 warms every shape up and is not recorded
        for name, fn in arms.items():
            run(name, fn, r > 0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()

    for g in range(G):
        for a, b in zip(out7, outs[g]):
            assert np.array_equal(a[g], b), f"group {g} differs from its own pass"
    assert all(np.array_equal(a, b) for a, b in zip(out1, outs[0]))

    med = {k: float(np.median(v)) for k, v in secs.items()}
    line = {
        "tool": "tools/instruction_sets_bench.py", "frames": T, "episodes": n_eps, "frame": [size, size, 3],
        "stack_in_memory": S, "num_frames": F, "max_batch": 1024, "precision": "16bit", "api": "arp_label_host",
        "pinned_host": bool(ob.is_pinned()), "groups": G, "inst_types": list(INST_TYPES), "rounds": args.rounds,
        "seconds": {k: round(v, 4) for k, v in med.items()},
        "seconds_samples": {k: [round(x, 4) for x in v] for k, v in secs.items()},
        "frames_per_s": {k: round(T / v) for k, v in med.items()},
        "g7_over_g1": round(med["g7"] / med["g1"], 4), "sequential_over_g7": round(med["sequential"] / med["g7"], 3),
        "launches": launches, "bit_identical": True,
        "gpu": q,
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
