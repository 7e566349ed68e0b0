"""What relabeling from stored embeddings costs and saves (B200).

    python tools/embeddings_bench.py [--frames 16384] [--rounds 3] [--out FILE]

The pinned 256x256 set of tools/instruction_sets_bench.py (bench.py's configuration: CLIP ViT-B/16, rows of two stacked
frames scored with the row stride, max_batch 1024, random-init weights, stand-in token ids, the seven CoinRun instruction
sets), on the first episodes of bench.py's synthetic dataset with at least --frames frames. After one untimed round,
each round times, alternating:
    label7          arp_label_host with the seven sets (set_text_groups + label_host)
    save            what embeddings="save" costs: arp_embed_host, the embeddings to the device, arp_label_embeddings with
                    the seven sets, its outputs to the host
    embed           arp_embed_host alone (the embedding pass against arp_label_host's pass over the same frames)
Host wall clock ending in a device synchronise. Then arp_label_embeddings alone, as CUDA-event time of the call (its two
kernels) over --reps calls with the embeddings already on the device, for the clip embedding of this set and for a
random adapter-width (13*512) embedding of the same rows, at G = 1 and G = 7; achieved GB/s = (T*dim*4 + the outputs)
over that time, against the 6 544 GB/s a device-to-device copy reached on a B200. Last, label_reward(embeddings="load")
against embeddings=None on one NpyStore of the same frames (stored one per row, so the file is 3.2 GB at 16 513 frames),
after one embeddings="save" call, median of --rounds alternating calls. Outputs are checked bit for bit. Prints one JSON
line (also written to --out) with the card's name, power limit and SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
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
COPY_GBPS = 6544.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16384, help="at least this many frames (whole episodes)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--num-frames", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("embeddings_bench.py needs a B200: arp_b200 has no CPU path")

    from bench import episode_offsets
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from arp_b200.label_reward import label_reward, release_cached_engine
    from arp_b200.store import NpyStore
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
    G = len(embs)
    eng.set_text_groups([e for e, _ in embs], scale)

    gen = torch.Generator(device=dev).manual_seed(1234)
    ob = torch.empty(T, S, size, size, 3, dtype=torch.uint8, pin_memory=True)
    for t0 in range(0, T, 2048):
        blk = ob[t0:t0 + 2048]
        blk.copy_(torch.randint(0, 256, blk.shape, dtype=torch.uint8, device=dev, generator=gen).cpu())
    off_dev = torch.from_numpy(off).to(dev)
    lead = (G,)
    out7 = (np.empty(lead + (T,), np.float32), np.empty(lead + (T,), np.float32),
            np.empty(lead + (T, F), np.float32), np.empty(lead + (T, F), np.float32))
    emb_host = torch.empty(T, eng.embedding_dim, dtype=torch.float32, pin_memory=True).numpy()
    saved = {}

    def label7():
        eng.label_host(ob, off, F, out=out7)

    def save():
        eng.embed_host(ob, out=emb_host)
        res = eng.label_embeddings(torch.from_numpy(emb_host).to(dev, non_blocking=True), off_dev, F)
        saved["out"] = [t.cpu().numpy() for t in res]

    def embed():
        eng.embed_host(ob, out=emb_host)

    arms = {"label7": label7, "save": save, "embed": embed}
    secs = {k: [] for k in arms}
    for r in range(args.rounds + 1):           # round 0 warms every shape up and is not recorded
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            if r > 0:
                secs[name].append(time.perf_counter() - t0)
    for a, b in zip(saved["out"], out7):
        assert np.array_equal(a, b), "labels from embeddings differ from labels from frames"

    # arp_label_embeddings alone: CUDA events around the call, the embeddings on the device
    def kernel_time(e, emb_dev, groups):
        if groups == 1:
            e.set_text(*groups_emb(e)[0])
        else:
            e.set_text_groups([x for x, _ in groups_emb(e)], scale)
        for _ in range(3):
            e.label_embeddings(emb_dev, off_dev, F)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
        for a, b in ev:
            a.record()
            e.label_embeddings(emb_dev, off_dev, F)
            b.record()
        torch.cuda.synchronize()
        ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
        nbytes = T * e.embedding_dim * 4 + groups * T * 4 * (2 + 2 * F)
        return {"ms": round(ms, 4), "bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1),
                "of_copy_bandwidth": round(nbytes / ms / 1e6 / COPY_GBPS, 3)}

    adapter = capi.Engine(device=0, patch=16, in_h=size, in_w=size, max_batch=8, head=capi.HEAD_ADAPTER)   # no weights
    ad_text = [torch.nn.functional.normalize(torch.randn(1, adapter.embedding_dim, generator=torch.Generator().manual_seed(i)),
                                             dim=1) for i in range(G)]

    def groups_emb(e):
        return embs if e is eng else [(t, scale) for t in ad_text]

    clip_emb = torch.from_numpy(emb_host).to(dev)
    ad_emb = torch.randn(T, adapter.embedding_dim, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    relabel = {"clip_g1": kernel_time(eng, clip_emb, 1), "clip_g7": kernel_time(eng, clip_emb, G),
               "adapter_g1": kernel_time(adapter, ad_emb, 1), "adapter_g7": kernel_time(adapter, ad_emb, G)}
    l0 = eng.launch_count
    eng.label_embeddings(clip_emb, off_dev, F)
    relabel_launches = eng.launch_count - l0
    adapter.close()
    del ad_emb, clip_emb
    eng.close()

    # the drop-in on an NpyStore of the same frames (one per row)
    drop = {}
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

        def run(embeddings):
            label_reward("coinrun", "hard", 500, 0, texts[0], d, data_path=str(path), model_type="clip",
                         clip_state_dict=sd, arch="ViT-B/16", max_batch=1024, env_type="none", tokenizer="standin",
                         extra_instructions={t: x for t, x in zip(INST_TYPES[1:], texts[1:])}, embeddings=embeddings)

        def datasets():
            st = NpyStore(path, "r")
            out = {k: np.array(st[k][:]) for k in st.keys() if k.startswith("ob_clip_") and "emb" not in k}
            st.close()
            return out

        run("save")
        ref = datasets()
        dsecs = {"none": [], "load": []}
        for r in range(args.rounds + 1):
            for mode in ("none", "load"):
                t0 = time.perf_counter()
                run(None if mode == "none" else "load")
                torch.cuda.synchronize()
                if r > 0:
                    dsecs[mode].append(time.perf_counter() - t0)
                got = datasets()
                assert all(np.array_equal(got[k], ref[k]) for k in ref), mode
        release_cached_engine()
        drop = {"seconds": {k: round(float(np.median(v)), 4) for k, v in dsecs.items()},
                "seconds_samples": {k: [round(x, 4) for x in v] for k, v in dsecs.items()},
                "datasets": len(ref), "bit_identical": True}
        drop["load_over_none"] = round(drop["seconds"]["load"] / drop["seconds"]["none"], 4)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    med = {k: float(np.median(v)) for k, v in secs.items()}
    line = {
        "tool": "tools/embeddings_bench.py", "frames": T, "episodes": n_eps, "frame": [size, size, 3],
        "stack_in_memory": S, "num_frames": F, "max_batch": 1024, "precision": "16bit", "pinned_host": bool(ob.is_pinned()),
        "groups": G, "rounds": args.rounds,
        "seconds": {k: round(v, 4) for k, v in med.items()},
        "seconds_samples": {k: [round(x, 4) for x in v] for k, v in secs.items()},
        "save_over_label7": round(med["save"] / med["label7"], 4), "embed_over_label7": round(med["embed"] / med["label7"], 4),
        "label_embeddings": relabel, "label_embeddings_launches": relabel_launches, "copy_GB_per_s": COPY_GBPS,
        "drop_in_npystore": drop, "bit_identical": True, "gpu": q,
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
