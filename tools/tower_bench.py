"""What relabeling with a new fine-tuned adapter from stored CLIP tower records costs and saves (B200).

    python tools/tower_bench.py [--frames 16384] [--rounds 3] [--out FILE]

The pinned 256x256 set of tools/embeddings_bench.py (CLIP ViT-B/16, rows of two stacked frames scored with the row
stride, max_batch 1024, random-init weights, stand-in token ids, the seven CoinRun instruction sets) on the first
episodes of bench.py's synthetic dataset with at least --frames frames, labeled by clip_ft with adapter checkpoint A.
Adapter checkpoint B is another random adapter of the same CLIP. After one untimed round, each round times, alternating:
    label7          arp_label_host with checkpoint A and the seven sets
    save_tower      what embeddings="save_tower" costs: arp_embed_tower_host, the records to the device,
                    arp_label_tower with the seven sets, its outputs to the host (checkpoint A)
    relabel_b       what a new checkpoint costs from the records: the records (pinned host) to the device,
                    arp_label_tower on an engine that holds only checkpoint B's image-adapter tensors, outputs to the host
Host wall clock ending in a device synchronise. Then arp_label_tower alone as CUDA-event time of the call with the
records on the device, over --reps calls, with its FLOP/s against the adapter's 0.468 GFLOP per frame. Last,
label_reward(embeddings="load_tower") with checkpoint B against embeddings=None with B on one NpyStore of the same frames
(one per row), after one embeddings="save_tower" call with A, median of --rounds alternating calls. Outputs are checked
bit for bit. Prints one JSON line (also written to --out) with the card's name, power limit and SM clock read in the
same run.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

INST_TYPES = ("none", "random1", "random2", "misinfo", "misinfo2", "misinfo3", "misinfo4")
# image_intermediate_linear 9216 -> 6144, AdapterMLP 6656 -> 13312 -> 6656: 2 * (9216*6144 + 2*6656*13312) per frame
ADAPTER_FLOP_PER_FRAME = 2.0 * (9216 * 6144 + 2 * 6656 * 13312)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16384, help="at least this many frames (whole episodes)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--num-frames", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tower_bench.py needs a B200: arp_b200 has no CPU path")

    from bench import episode_offsets
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from arp_b200.label_reward import _IMAGE_ADAPTER_PREFIXES, label_reward, release_cached_engine
    from arp_b200.store import NpyStore
    from arp_b200.text_tower import adapter_text_embedding
    from arp_b200.tokenizer import tokenize
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    build()
    dev = torch.device("cuda", 0)
    size, S, F = 256, 2, args.num_frames
    off_all = episode_offsets(500, seed=1)
    n_eps = int(np.searchsorted(off_all, args.frames, side="left"))
    off = off_all[:n_eps + 1].copy()
    T = int(off[-1])

    clip_sd = random_clip_state_dict("ViT-B/16", seed=0, device="cpu")
    ckpt_a = random_adapter_state_dict("ViT-B/16", seed=1, device="cpu", clip_sd=clip_sd)
    ckpt_b = random_adapter_state_dict("ViT-B/16", seed=2, device="cpu", clip_sd=clip_sd)
    texts = [get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t) for t in INST_TYPES]
    G = len(texts)

    def engine(sd, adapter_only):
        e = capi.Engine(device=0, patch=16, in_h=size, in_w=size, preprocess=capi.PRE_BILINEAR, head=capi.HEAD_ADAPTER,
                        max_batch=1024, precision=capi.PREC_16BIT)
        e.load_state_dict({k: v for k, v in sd.items() if k.startswith(_IMAGE_ADAPTER_PREFIXES)} if adapter_only else sd)
        embs = [adapter_text_embedding(sd, tokenize([t], standin=True), dev) for t in texts]
        e.set_text_groups([x for x, _ in embs], embs[0][1])
        return e

    eng_a, eng_b = engine(ckpt_a, False), engine(ckpt_b, True)
    assert eng_b.missing_weights(), "engine B must hold no visual.* weight"

    gen = torch.Generator(device=dev).manual_seed(1234)
    ob = torch.empty(T, S, size, size, 3, dtype=torch.uint8, pin_memory=True)
    for t0 in range(0, T, 2048):
        blk = ob[t0:t0 + 2048]
        blk.copy_(torch.randint(0, 256, blk.shape, dtype=torch.uint8, device=dev, generator=gen).cpu())
    off_dev = torch.from_numpy(off).to(dev)
    lead = (G,)
    out7 = (np.empty(lead + (T,), np.float32), np.empty(lead + (T,), np.float32),
            np.empty(lead + (T, F), np.float32), np.empty(lead + (T, F), np.float32))
    rec_host = torch.empty(T, eng_a.tower_dim, dtype=torch.float32, pin_memory=True)
    saved = {}

    def label7():
        eng_a.label_host(ob, off, F, out=out7)

    def save_tower():
        eng_a.embed_tower_host(ob, out=rec_host.numpy())
        res = eng_a.label_tower(rec_host.to(dev, non_blocking=True), off_dev, F)
        saved["a"] = [t.cpu().numpy() for t in res]

    def relabel_b():
        res = eng_b.label_tower(rec_host.to(dev, non_blocking=True), off_dev, F)
        saved["b"] = [t.cpu().numpy() for t in res]

    arms = {"label7": label7, "save_tower": save_tower, "relabel_b": relabel_b}
    secs = {k: [] for k in arms}
    for r in range(args.rounds + 1):           # round 0 warms every shape up and is not recorded
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            if r > 0:
                secs[name].append(time.perf_counter() - t0)
    for a, b in zip(saved["a"], out7):
        assert np.array_equal(a, b), "labels from tower records differ from labels from frames"
    assert not np.array_equal(saved["b"][0], out7[0]), "checkpoint B labels like checkpoint A"

    # arp_label_tower alone: CUDA events around the call, the records on the device
    rec_dev = rec_host.to(dev)
    for _ in range(3):
        eng_b.label_tower(rec_dev, off_dev, F)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
    for a, b in ev:
        a.record()
        eng_b.label_tower(rec_dev, off_dev, F)
        b.record()
    torch.cuda.synchronize()
    ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
    l0 = eng_b.launch_count
    eng_b.label_tower(rec_dev, off_dev, F)
    launches = eng_b.launch_count - l0
    flop = ADAPTER_FLOP_PER_FRAME * T
    kernel = {"ms": round(ms, 3), "gflop": round(flop / 1e9, 1), "TFLOP_per_s": round(flop / ms / 1e9, 1),
              "record_bytes": T * eng_b.tower_dim * 4, "launches": launches, "groups": G}
    del rec_dev
    eng_a.close()
    eng_b.close()

    # the drop-in on an NpyStore of the same frames (one per row): a new checkpoint B from the records saved with A
    with tempfile.TemporaryDirectory() as d:
        path = Path(d) / "ds"
        s = NpyStore(path, "w")
        s.create_dataset("done", data=np.zeros((T, F), np.float32))
        done = s["done"]
        done[off[1:] - 1, -1] = 1.0
        s.close()
        mm = np.lib.format.open_memmap(path / "ob.npy", mode="w+", dtype=np.uint8, shape=(T, 1, size, size, 3))
        for t0 in range(0, T, 2048):
            mm[t0:t0 + 2048, 0] = ob[t0:t0 + 2048, S - 1].numpy()
        mm.flush()
        del mm

        def run(embeddings, ckpt):
            label_reward("coinrun", "hard", 500, 0, texts[0], d, data_path=str(path), model_type="clip_ft",
                         model_ckpt_dir=ckpt, arch="ViT-B/16", max_batch=1024, env_type="none", tokenizer="standin",
                         extra_instructions={t: x for t, x in zip(INST_TYPES[1:], texts[1:])}, embeddings=embeddings)

        def datasets():
            st = NpyStore(path, "r")
            out = {k: np.array(st[k][:]) for k in st.keys() if k.startswith("ob_clip_ft_")}
            st.close()
            return out

        run("save_tower", ckpt_a)
        dsecs = {"none": [], "load_tower": []}
        ref = None
        for r in range(args.rounds + 1):
            for mode in ("none", "load_tower"):
                t0 = time.perf_counter()
                run(None if mode == "none" else "load_tower", ckpt_b)
                torch.cuda.synchronize()
                if r > 0:
                    dsecs[mode].append(time.perf_counter() - t0)
                got = datasets()
                ref = got if ref is None else ref
                assert all(np.array_equal(got[k], ref[k]) for k in ref), mode
        release_cached_engine()
        drop = {"seconds": {k: round(float(np.median(v)), 4) for k, v in dsecs.items()},
                "seconds_samples": {k: [round(x, 4) for x in v] for k, v in dsecs.items()},
                "datasets": len(ref), "bit_identical": True}
        drop["load_tower_over_none"] = round(drop["seconds"]["load_tower"] / drop["seconds"]["none"], 4)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    med = {k: float(np.median(v)) for k, v in secs.items()}
    line = {
        "tool": "tools/tower_bench.py", "frames": T, "episodes": n_eps, "frame": [size, size, 3],
        "stack_in_memory": S, "num_frames": F, "max_batch": 1024, "precision": "16bit", "model_type": "clip_ft",
        "pinned_host": bool(ob.is_pinned()), "groups": G, "rounds": args.rounds,
        "seconds": {k: round(v, 4) for k, v in med.items()},
        "seconds_samples": {k: [round(x, 4) for x in v] for k, v in secs.items()},
        "save_tower_over_label7": round(med["save_tower"] / med["label7"], 4),
        "relabel_b_over_label7": round(med["relabel_b"] / med["label7"], 4),
        "label_tower": kernel, "drop_in_npystore": drop, "bit_identical": True, "gpu": q,
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
