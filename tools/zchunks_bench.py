"""Gzip datasets of other chunk shapes: the compressed-chunk path against the row path, the uncompressed file and the host.

    python tools/zchunks_bench.py [--rows 16384] [--rounds 3] [--out FILE]

Geometries: 64x64 with F = 4 and 256x256 with F = 8, procgen-like frames (arp_b200/synth.py), every chunk compressed with
zlib.compress(chunk, 4) (h5py's default gzip level). Layouts:
- row: (1, F, H, W, 3), the recorder's (arp_label_zfile applies too);
- frames8: (8, 1, H, W, 3), frames split along F;
- auto: the chunk shape h5py picks when create_dataset gets no chunks= (h5py's guess_chunk, restated below):
  (2048, 1, 8, 8, 1) at 64x64 and (1024, 1, 16, 16, 1) at 256x256.
Row t's frames come from a pool of --pool distinct rows (row t % pool); the pool size divides every multi-row chunk
extent or is divided by it, so a chunk's content depends only on its origin modulo the pool and each distinct chunk is
compressed once. Each chunk is still its own stream in the file and is read and inflated on its own. Only the chunks
that hold frame F-1 are written (the others are never read, and the call gets only the needed part of the table).
Reported per layout, medians of --rounds alternating rounds with outputs checked bit for bit:
- arp_label_zchunks rows/s, arp_label_file on the same rows uncompressed (a sparse file of the scored frames), and
  arp_label_zfile for the row layout;
- inflated bytes per scored frame (a row-chunk serving two max_batch batches is inflated in both);
- the inflate and gather kernels' device time per batch inside label_zchunks (torch.profiler kernel records, in a
  call of their own), and the gather kernel alone by CUDA events through arp_gather_frames on one batch of chunks;
- host zlib.decompress alone of the chunks that the scored frames of the first row-chunks (at least 512 rows) need, on 1
  and 4 threads;
- at 64x64, the drop-in's h5py slab path end to end (label_reward._label_rows: a reader thread one slab of 2048 rows
  ahead of label_slab) with h5py's read replaced by one-thread zlib inflate of the same chunks, which is what h5py does
  for ds[lo:hi, -1] without its own overheads, so an upper bound on the h5py path's rate.
Prints one JSON line (also written to --out) with the card's name, power limit, current and maximum SM clock read in
the same run.
ViT-B/16, clip head, 16-bit path, max_batch 1024, one instruction.
"""
import argparse
import itertools
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

B = 1024


def gpu_info():
    """name, power limit, current SM clock, maximum SM clock"""
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                           "-i", "0"], capture_output=True, text=True).stdout.strip()


def guess_chunk(shape, typesize=1):
    """h5py's automatic chunk shape (h5py/_hl/filters.py guess_chunk, BSD licence) for a fixed-size dataset"""
    base, lo, hi = 16 * 1024, 8 * 1024, 1024 * 1024
    chunks = np.array(shape, dtype="=f8")
    target = min(max(base * 2 ** np.log10(np.prod(chunks) * typesize / (1024. * 1024)), lo), hi)
    idx = 0
    while True:
        cb = np.prod(chunks) * typesize
        if (cb < target or abs(cb - target) / target < 0.5) and cb < hi:
            break
        if np.prod(chunks) == 1:
            break
        chunks[idx % len(shape)] = np.ceil(chunks[idx % len(shape)] / 2.0)
        idx += 1
    return tuple(int(x) for x in chunks)


def make_pool(size, F, n):
    from arp_b200.synth import make_dataset
    d = make_dataset(n_episodes=n // 40 + 1, len_lo=40, len_hi=60, size=size, num_frames=F, seed=0, kind="structured")
    assert len(d["ob"]) >= n
    return np.ascontiguousarray(d["ob"][:n])


def needed_origins(shape, chunks):
    """origins of the chunks holding frame F-1 of every row, in (row-chunk, H, W, C) order"""
    F = shape[1]
    fc = (F - 1) // chunks[1] * chunks[1]
    return [(r, fc) + o for r in range(0, shape[0], chunks[0])
            for o in itertools.product(*[range(0, s, c) for s, c in zip(shape[2:], chunks[2:])])]


def chunk_data(pool, o, chunks):
    part = pool[(slice(None),) + tuple(slice(a, a + c) for a, c in zip(o[1:], chunks[1:]))]
    return np.ascontiguousarray(part[(o[0] + np.arange(chunks[0])) % len(pool)])


def inflated_per_frame(T, chunks, nsp, vol):
    """bytes inflated per scored frame: every batch inflates every chunk of each row-chunk it touches"""
    total = sum(((min(T, t0 + B) - 1) // chunks[0] - t0 // chunks[0] + 1) * nsp * vol for t0 in range(0, T, B))
    return total / T


class _ZlibRows:
    """the rows of a chunked gzip dataset as the drop-in's h5py path reads them (`ds[lo:hi, -1]`): on one thread, every
    chunk holding frame F-1 of the rows is zlib-inflated and its part copied into the frames. A lower bound on h5py's
    own cost for the same read (h5py adds its chunk index walk, its selection machinery and a chunk cache)."""

    def __init__(self, shape, chunks, streams, P):
        self.shape, self.chunks, self.streams, self.P = shape, chunks, streams, P

    def __getitem__(self, idx):
        rows, _ = idx
        lo, hi = rows.start, rows.stop
        (cT, cF, cH, cW, cC), (_, F, H, W, C) = self.chunks, self.shape
        out = np.empty((hi - lo, H, W, C), np.uint8)
        fc = (F - 1) // cF * cF
        for r0 in range(lo // cT * cT, hi, cT):
            for o in itertools.product(range(0, H, cH), range(0, W, cW), range(0, C, cC)):
                ch = np.frombuffer(zlib.decompress(self.streams[(r0 % self.P, fc) + o]), np.uint8).reshape(self.chunks)
                a, b = max(lo, r0), min(hi, r0 + cT)
                out[a - lo:b - lo, o[0]:o[0] + cH, o[1]:o[1] + cW, o[2]:o[2] + cC] = ch[a - r0:b - r0, F - 1 - fc]
        return out


def host_path(e, shape, chunks, streams, P, ep, F, slab_frames):
    """seconds of the drop-in's slab path (label_reward._label_rows with a reader thread one slab ahead) on
    _ZlibRows, and its outputs"""
    from arp_b200.label_reward import _label_rows

    class _Labeler:
        goal = False

        def label_slab(self, ob, rel, num_frames):
            return e.label_host(ob, rel, num_frames)

    t = time.perf_counter()
    out = _label_rows(_Labeler(), _ZlibRows(shape, chunks, streams, P), None, ep, 0, len(ep) - 1, F, slab_frames)
    return time.perf_counter() - t, out


def kernel_ms(fn):
    """device time of inflate_rows_kernel and gather_frames_kernel in one call of fn, from torch.profiler's kernel
    records (a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ms = {"inflate": 0.0, "gather": 0.0}
    for ev in prof.key_averages():
        for k, tag in (("inflate", "inflate_rows_kernel"), ("gather", "gather_frames_kernel")):
            if tag in ev.key:
                ms[k] += getattr(ev, "self_device_time_total", 0.0) / 1e3
    return ms


def layout(capi, e, pool, name, chunks, T, rounds, workdir, fr, ref_args):
    P, F, H, W = pool.shape[:4]
    shape = (T,) + pool.shape[1:]
    assert all(P % c == 0 or c % P == 0 for c in (chunks[0],)), (P, chunks)
    origins = needed_origins(shape, chunks)
    keys = sorted({(o[0] % P,) + o[1:] for o in origins})
    with ThreadPoolExecutor(16) as ex:
        streams = dict(zip(keys, ex.map(lambda k: zlib.compress(chunk_data(pool, k, chunks).tobytes(), 4), keys)))
    path = workdir / f"{name}{H}.bin"
    off, nb = np.empty(len(origins), np.int64), np.empty(len(origins), np.int64)
    with open(path, "wb") as f:
        for i, o in enumerate(origins):
            s = streams[(o[0] % P,) + o[1:]]
            off[i], nb[i] = f.tell(), len(s)
            f.write(s)
    org = np.array(origins, np.int64)
    vol = int(np.prod(chunks))
    nsp = int(np.prod([s // c for s, c in zip(shape[2:], chunks[2:])]))
    ep, frame = ref_args["ep"], H * W * 3
    fz = os.open(path, os.O_RDONLY)
    calls = {"label_file": lambda: e.label_file(fr, (F - 1) * frame, T, F * frame, ep, F),
             "label_zchunks": lambda: e.label_zchunks(fz, (shape, chunks), org, off, nb, 0, T, ep, F)}
    if chunks[0] == 1 and chunks[1:] == shape[1:]:
        calls["label_zfile"] = lambda: e.label_zfile(fz, off, nb, F * frame, ep, F)
    try:
        ref = calls["label_file"]()
        bit = all(all(np.array_equal(a, b) for a, b in zip(fn(), ref)) for k, fn in calls.items() if k != "label_file")
        secs = {k: [] for k in calls}
        for _ in range(rounds):
            for k, fn in calls.items():
                t = time.perf_counter()
                fn()
                secs[k].append(time.perf_counter() - t)
        kernels = kernel_ms(calls["label_zchunks"])
        host_s = None
        if H <= 64:
            # the h5py slab path at its best: slabs of 2048 rows so that reading overlaps labeling, zlib without h5py
            ref_pairs = calls["label_file"]()
            host_s, pairs = host_path(e, shape, chunks, streams, P, ep, F, 2048)
            bit = bit and all(np.array_equal(a, b) for a, b in zip(pairs, (ref_pairs[2], ref_pairs[3])))
    finally:
        os.close(fz)
    med = {k: float(np.median(v)) for k, v in secs.items()}

    # the gather kernel alone on batch 0's chunks (inflated on the host), CUDA events; the dense layouts launch none
    dense = chunks[0] == 1 and chunks[2:] == shape[2:]
    gather_ms = 0.0
    if not dense:
        n_rc = (B - 1) // chunks[0] + 1
        dev = torch.from_numpy(np.concatenate([chunk_data(pool, o, chunks).ravel()
                                               for o in origins[:n_rc * nsp]])).cuda()
        out = e.gather_frames((shape, chunks), 0, B, dev)
        assert np.array_equal(out.cpu().numpy(), pool[np.arange(B) % P, -1])
        reps = 20
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            e.gather_frames((shape, chunks), 0, B, dev)
        t1.record()
        torch.cuda.synchronize()
        gather_ms = t0.elapsed_time(t1) / reps
        del dev, out

    # host: zlib.decompress alone of the chunks the first 512 rows' scored frames need
    n_rc = (512 - 1) // chunks[0] + 1
    rows = n_rc * chunks[0]                       # the rows whose scored frames those chunks hold
    sample = [streams[(o[0] % P,) + o[1:]] for o in origins[:n_rc * nsp]]
    host = {}
    for threads in (1, 4):
        t = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(zlib.decompress, sample))
        host[f"threads_{threads}_rows_per_s"] = round(rows / (time.perf_counter() - t), 1)
    batches = -(-T // B)
    return {
        "layout": name, "chunks": list(chunks), "chunk_bytes": vol, "needed_chunks": len(origins),
        "compressed_bytes_per_needed_chunk": round(float(nb.mean()), 1),
        "inflated_bytes_per_scored_frame": round(inflated_per_frame(T, chunks, nsp, vol), 1),
        "gather_launch": not dense,
        "rows_per_s": {k: round(T / v, 1) for k, v in med.items()},
        "seconds_samples": {k: [round(x, 4) for x in v] for k, v in secs.items()},
        "zchunks_over_file": round(med["label_zchunks"] / med["label_file"], 3),
        "inflate_kernel_ms_per_batch": round(kernels["inflate"] / batches, 3),
        "gather_kernel_ms_per_batch": round(kernels["gather"] / batches, 3),
        "gather_kernel_alone_ms_per_batch": round(gather_ms, 3),
        "host_zlib": host,
        "host_slab_path_rows_per_s": round(T / host_s, 1) if host_s else None,
        "bit_identical": bool(bit),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16384)
    ap.add_argument("--pool", type=int, default=512, help="distinct rows")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "zchunks_bench measures the B200 path: it needs a GPU"
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.weights import random_clip_state_dict
    build()
    sd = random_clip_state_dict("ViT-B/16", 0, "cpu")
    T = args.rows
    res = []
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        for size, F in ((64, 4), (256, 8)):
            pool = make_pool(size, F, args.pool)
            e = capi.Engine(device=0, patch=16, in_h=size, in_w=size, max_batch=B)
            e.load_state_dict(sd)
            e.set_text(torch.nn.functional.normalize(torch.randn(1, 512, generator=torch.Generator().manual_seed(0)),
                                                     dim=1), 100.0)
            rpath = d / f"r{size}.bin"
            row_bytes, frame = pool[0].nbytes, pool[0, 0].nbytes
            with open(rpath, "wb") as f:              # only the scored frames, at their row offsets (the rest is a hole)
                for t in range(T):
                    f.seek(t * row_bytes + (F - 1) * frame)
                    f.write(pool[t % len(pool), -1].tobytes())
                f.truncate(T * row_bytes)
            ep = np.append(np.arange(0, T, 40), T).astype(np.int64)
            fr = os.open(rpath, os.O_RDONLY)
            auto = guess_chunk((T,) + pool.shape[1:])
            geo = {"frame": [size, size, 3], "num_frames": F, "rows": T, "distinct_rows": len(pool), "layouts": []}
            try:
                for name, chunks in (("row", (1,) + pool.shape[1:]), ("frames8", (8, 1, size, size, 3)),
                                     ("auto", auto)):
                    geo["layouts"].append(layout(capi, e, pool, name, chunks, T, args.rounds, d, fr, {"ep": ep}))
                    print(json.dumps(geo["layouts"][-1]), flush=True)
            finally:
                os.close(fr)
            res.append(geo)
            e.close()
            del pool
    line = {"tool": "tools/zchunks_bench.py", "arch": "ViT-B/16", "model_type": "clip", "precision": "16bit",
            "max_batch": B, "zlib_level": 4, "stager_threads": 4, "rounds": args.rounds, "geometries": res,
            "gpu": gpu_info()}
    s = json.dumps(line)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
