"""Gzip-chunked rows: the device inflate against the host, and the labeling call end to end.

    python tools/zrows_bench.py [--rows 16384] [--rounds 3] [--out FILE]

For each geometry (64x64 with F = 4 stacked frames, 256x256 with F = 8), procgen-like frames (arp_b200/synth.py) are
stacked into rows as the recorder stores them and every row is compressed with zlib.compress(row, 4), the level h5py's
compression="gzip" uses by default. Distinct rows are drawn from a pool of --pool episodes' rows and repeated to reach
--rows rows (compressing 16 k rows of 1.5 MB on one host thread would take minutes); every row is still its own stream
in the file and is read and inflated on its own. Reported per geometry:
- inflate_rows_kernel alone (arp_inflate_rows on one max_batch chunk already on the device), CUDA events, in rows/s and
  inflated GB/s;
- arp_label_zfile end to end (pread of the compressed rows, H2D, inflate, encoder, head, scan) against arp_label_file on
  the same rows stored uncompressed (a sparse file holding only the scored frames, which is all arp_label_file reads),
  medians of --rounds, with the outputs checked bit for bit;
- the host path the drop-in takes today: zlib.decompress of whole rows on one thread, and on the stager's 4 threads;
- the compression ratio;
- bound_by: the slower device stage alone (inflate kernel or the label_file pass). The two run in series on the
  compute stream, so label_zfile takes about the sum of their times.
Prints one JSON line (also written to --out) with the card's name, power limit and SM clock read in the same run.
ViT-B/16, clip head, 16-bit path, max_batch 1024, one instruction.
"""
import argparse
import ctypes as C
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


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()


def make_rows(size, F, pool_eps, seed=0):
    from arp_b200.synth import make_dataset
    d = make_dataset(n_episodes=pool_eps, len_lo=20, len_hi=60, size=size, num_frames=F, seed=seed, kind="structured")
    return np.ascontiguousarray(d["ob"])


def geometry(capi, e, size, F, n_rows, pool_eps, rounds, workdir):
    pool = make_rows(size, F, pool_eps)
    with ThreadPoolExecutor(16) as ex:
        streams = list(ex.map(lambda r: zlib.compress(r.tobytes(), 4), pool))
    P = len(pool)
    idx = np.arange(n_rows) % P
    row_bytes, frame = pool[0].nbytes, pool[0, 0].nbytes
    # episodes of 40 rows over the whole table
    ep = np.append(np.arange(0, n_rows, 40), n_rows).astype(np.int64)
    zpath, rpath = workdir / f"z{size}.bin", workdir / f"r{size}.bin"
    off = np.empty(n_rows, np.int64)
    nb = np.empty(n_rows, np.int64)
    with open(zpath, "wb") as f:
        for t in range(n_rows):
            s = streams[idx[t]]
            off[t], nb[t] = f.tell(), len(s)
            f.write(s)
    with open(rpath, "wb") as f:                  # only the scored frames, at their row offsets (the rest is a hole)
        for t in range(n_rows):
            f.seek(t * row_bytes + (F - 1) * frame)
            f.write(pool[idx[t], -1].tobytes())
        f.truncate(n_rows * row_bytes)

    # inflate kernel alone: one max_batch chunk of compressed rows on the device
    B = e.cfg.max_batch
    src = torch.frombuffer(bytearray(b"".join(streams[i] for i in idx[:B])), dtype=torch.uint8).cuda()
    soff = torch.from_numpy(np.concatenate([[0], np.cumsum(nb[:B])[:-1]]).astype(np.int64)).cuda()
    sb = torch.from_numpy(nb[:B].copy()).cuda()
    out = torch.empty((B, row_bytes), dtype=torch.uint8, device="cuda")
    status = torch.empty(B, dtype=torch.int32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def inflate():
        assert e._lib.arp_inflate_rows(e._h, p(src), p(soff), p(sb), B, row_bytes, p(out), p(status), stream) == 0
    inflate()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0
    m = min(P, B)
    assert out[:m].cpu().numpy().tobytes() == pool[:m].tobytes()
    reps = 10
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        inflate()
    t1.record()
    torch.cuda.synchronize()
    k_s = t0.elapsed_time(t1) / 1e3 / reps
    kernel = {"rows": B, "ms": round(k_s * 1e3, 3), "rows_per_s": round(B / k_s, 1),
              "inflated_GB_per_s": round(B * row_bytes / k_s / 1e9, 2),
              "compressed_GB_per_s": round(float(nb[:B].sum()) / k_s / 1e9, 3)}

    # end to end
    fz, fr = os.open(zpath, os.O_RDONLY), os.open(rpath, os.O_RDONLY)
    try:
        ref = e.label_file(fr, (F - 1) * frame, n_rows, row_bytes, ep, F)
        got = e.label_zfile(fz, off, nb, row_bytes, ep, F)
        bit = all(np.array_equal(a, b) for a, b in zip(got, ref))
        secs = {"label_file": [], "label_zfile": []}
        for _ in range(rounds):
            for name, fn in (("label_file", lambda: e.label_file(fr, (F - 1) * frame, n_rows, row_bytes, ep, F)),
                             ("label_zfile", lambda: e.label_zfile(fz, off, nb, row_bytes, ep, F))):
                t = time.perf_counter()
                fn()
                secs[name].append(time.perf_counter() - t)
    finally:
        os.close(fz)
        os.close(fr)
    med = {k: float(np.median(v)) for k, v in secs.items()}

    # host baseline: whole-row zlib.decompress (what h5py does per chunk), 1 thread and the stager's 4
    sample = [streams[i] for i in idx[:min(n_rows, 512)]]
    host = {}
    for threads in (1, 4):
        t = time.perf_counter()
        if threads == 1:
            for s in sample:
                zlib.decompress(s)
        else:
            with ThreadPoolExecutor(threads) as ex:
                list(ex.map(zlib.decompress, sample))
        dt = time.perf_counter() - t
        host[f"threads_{threads}"] = {"rows_per_s": round(len(sample) / dt, 1),
                                      "inflated_GB_per_s": round(len(sample) * row_bytes / dt / 1e9, 3)}
    zfile_rps, file_rps = n_rows / med["label_zfile"], n_rows / med["label_file"]
    return {
        "frame": [size, size, 3], "num_frames": F, "rows": n_rows, "distinct_rows": P, "row_bytes": row_bytes,
        "compressed_bytes_per_row": round(float(nb.mean()), 1),
        "compression_ratio": round(row_bytes * n_rows / float(nb.sum()), 2),
        "inflate_kernel": kernel,
        "seconds": {k: round(v, 4) for k, v in med.items()},
        "seconds_samples": {k: [round(x, 4) for x in v] for k, v in secs.items()},
        "label_zfile_rows_per_s": round(zfile_rps, 1), "label_file_rows_per_s": round(file_rps, 1),
        "label_zfile_over_label_file": round(med["label_zfile"] / med["label_file"], 3),
        "host_zlib": host,
        # the slower of the two device stages measured alone; they run in series on the compute stream, so label_zfile
        # takes about the sum of their times
        "bound_by": "inflate" if kernel["rows_per_s"] < file_rps else "encoder",
        "bit_identical": bool(bit),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16384)
    ap.add_argument("--pool", type=int, default=12, help="episodes of distinct rows (20-60 rows each)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "zrows_bench measures the B200 path: it needs a GPU"
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.weights import random_clip_state_dict
    build()
    sd = random_clip_state_dict("ViT-B/16", 0, "cpu")
    res = []
    with tempfile.TemporaryDirectory() as d:
        for size, F in ((64, 4), (256, 8)):
            e = capi.Engine(device=0, patch=16, in_h=size, in_w=size, max_batch=1024)
            e.load_state_dict(sd)
            e.set_text(torch.nn.functional.normalize(torch.randn(1, 512, generator=torch.Generator().manual_seed(0)),
                                                     dim=1), 100.0)
            res.append(geometry(capi, e, size, F, args.rows, args.pool, args.rounds, Path(d)))
            e.close()
    line = {"tool": "tools/zrows_bench.py", "arch": "ViT-B/16", "model_type": "clip", "precision": "16bit",
            "max_batch": 1024, "zlib_level": 4, "stager_threads": 4, "rounds": args.rounds, "geometries": res,
            "gpu": gpu_info()}
    s = json.dumps(line)
    print(s)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
