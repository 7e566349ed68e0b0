"""Headline benchmark: reward-labeled frames/s of the ARP labeler hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                         # the reference algorithm on host cores

Workload (BASELINE.json configs[1]): CLIP ViT-B/16, model_type="clip", 500 synthetic CoinRun-shaped episodes (lengths
rng(1).integers(32,256), ~72k frames) of 256x256 uint8 frames, random-init weights. A "step" is one pass of the hot path
over the whole dataset shard:  decode -> ViT-B/16 -> cosine reward -> per-episode return-to-go scan + window stack.
Frames are kept in the reference's STACKED layout ob[T, S, H, W, 3] (data/PPG/trajectory_recorder.py) with S =
--stack-in-memory rows (default 2; the recorder's 8 would need 113 GB per rank): only the last stacked frame of a row is
scored (label_reward.py:268), so every copy / decode below walks the rows with stride S*H*W*3 exactly as on a real file.

`value`            frames/s with the stacked frames already resident in HBM (arp_label on device buffers);
`e2e`              frames/s through the host-buffer C-ABI call (arp_label_host): pinned host frames are copied H2D
                   (strided cudaMemcpy2DAsync) inside the timed region and the four result arrays are copied back;
`entrypoint_e2e`   wall clock of the drop-in itself, arp_b200.label_reward.label_reward(), on a memory-mapped on-disk
                   store of the same rows: store open, weight upload, text tower, every frame from pageable page-cache
                   memory through the native stager, labels written back;
`roofline`         the tcgen05 GEMM kernel (all launches of one step), algorithmic FLOPs / CUDA-event time;
`cpu_baseline`     the oracle port (CPU restatement of the reference) on a bounded sample, rank 0, N=1;
`gpu_eager_baseline` the reference's CUDA route (label_reward.py:89,126-146: clip.load -> fp16 PyTorch / cuBLAS) — the
                   CLIP restatement in eager fp16 on the same GPU, model forward only at batch 1024, rank 0, N=1;
`strong_scaling`   BASELINE configs[4]: 10k episodes of 64x64 frames partitioned over the N ranks (fixed total work),
                   one NCCL gather, bit-exact scan check of the gathered arrays on rank 0.
With N>1 (torchrun) every rank labels its own 500-episode shard (weak scaling) and the per-frame reward / return-to-go
arrays are gathered to rank 0 with one NCCL collective inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

GFLOP_PER_FRAME_B16 = 35.127  # SURVEY.md §8(d)
TEXT = "the goal is to collect the coin."


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--episodes", type=int, default=500)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--num-frames", type=int, default=8, help="F of the stacked outputs (label_reward.py:81)")
    ap.add_argument("--stack-in-memory", type=int, default=2, help="stacked frames per row kept in memory / on disk")
    ap.add_argument("--max-batch", type=int, default=1024)
    ap.add_argument("--precision", default="16bit", choices=["16bit", "fp32resid"],
                    help="tensor-core mode: 16-bit residual stream + folded LayerNorm (default) or fp32 residual stream")
    ap.add_argument("--cpu-sample-frames", type=int, default=400)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--strong-episodes", type=int, default=10_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-entrypoint", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float32), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_MAX_BYTES = 60 * 10**6     # array data; with the .npy headers a dump stays under 64 MB


def dump_outputs(d: Path, arrays: dict) -> None:
    """Writes every tensor of `arrays` to d/<name>.npy as float32. Above DUMP_MAX_BYTES in all, each array keeps the same
    fraction of its rows, drawn with a fixed seed and kept in order, so runs with the same arguments stay comparable."""
    d.mkdir(parents=True, exist_ok=True)
    total = sum(a.numel() * 4 for a in arrays.values())
    frac = min(1.0, DUMP_MAX_BYTES / max(total, 1))
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if frac < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * frac), replace=False))]
        np.save(d / f"{name}.npy", a)


def episode_offsets(n_episodes: int, seed: int) -> np.ndarray:
    lens = np.random.default_rng(seed).integers(32, 256, size=n_episodes)
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)


def workload_config(args) -> dict:
    """Identical on both arms (the reference arm's bounded sample is described under cpu_baseline.sample only)."""
    frames = int(episode_offsets(args.episodes, seed=1)[-1])
    return {"workload": f"CLIP ViT-B/16 model_type=clip labeling of {args.episodes} synthetic CoinRun-shaped episodes "
                        f"at {args.size}x{args.size} (BASELINE configs[1]), random-init weights",
            "episodes_per_gpu": args.episodes, "frames_per_gpu": frames, "frame": [args.size, args.size, 3],
            "num_frames": args.num_frames, "stack_in_memory": args.stack_in_memory,
            "layout": "ob[T, stack_in_memory, H, W, 3], last stacked frame scored, row stride stack_in_memory*H*W*3",
            "max_batch": args.max_batch, "precision": args.precision, "parallelism": f"episode-sharded x{args.gpus}",
            "cache": "inputs (>= 14 GB/GPU of scored frames) far exceed the 126 MB L2; no flush needed"}


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference algorithm (oracle port) on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_reference_rate(args, n_frames: int, threads: int | None = None):
    """Times oracle.port.label_reward_port (torch CPU fp32 + PIL + numpy loops, i.e. the reference's own
    algorithm) on the first episodes of the same synthetic dataset, >= n_frames frames. Returns
    (frames/s, frames, cores, rewards, frames_u8, offsets, state_dict)."""
    from oracle import port
    from arp_b200.weights import random_clip_state_dict
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    off = episode_offsets(args.episodes, seed=1)
    n_eps = int(np.searchsorted(off, n_frames, side="left"))
    n_eps = max(1, min(n_eps, args.episodes))
    T = int(off[n_eps])
    rng = np.random.default_rng(1234)
    frames = rng.integers(0, 256, size=(T, 1, args.size, args.size, 3), dtype=np.uint8)
    done = np.zeros((T, args.num_frames), np.float32)
    done[off[1:n_eps + 1] - 1, -1] = 1.0
    model = port.clip_shim.build("ViT-B/16", seed=0)
    sd = random_clip_state_dict("ViT-B/16", seed=0, device="cpu")
    model.load_state_dict(sd, strict=True)
    model = model.float().eval()
    data = {"ob": frames, "done": done}
    # untimed warm-up on a handful of frames (thread pool, oneDNN primitive caches) so the sample measures steady state
    warm = {"ob": frames[:4], "done": np.concatenate([np.zeros((3, args.num_frames), np.float32),
                                                       np.eye(1, args.num_frames, args.num_frames - 1, dtype=np.float32)])}
    port.label_reward_port(warm, model=model, model_type="clip", text=TEXT)
    t0 = time.perf_counter()
    out = port.label_reward_port(data, model=model, model_type="clip", text=TEXT)
    secs = time.perf_counter() - t0
    return T / secs, T, threads, out, frames, off[:n_eps + 1], sd


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rates = []
    frames = 0
    for i in range(args.warmup + args.steps):
        rate, frames, cores, *_ = cpu_reference_rate(args, max(16, args.cpu_sample_frames // 2))
        if i >= args.warmup:
            rates.append(rate)
    v = float(np.mean(rates))
    sample = (f"each step = the first episodes of the same synthetic dataset, {frames} frames, oracle/port.py (the "
              f"reference's algorithm: torch CPU fp32 + PIL + python scan loops) on {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": "reward-labeled frames/sec", "value": v, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * frames / v,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------------------
# stated baselines and side measurements of our arm
# ---------------------------------------------------------------------------------------------------
def gpu_eager_rate(dev, sd, batch: int = 1024, iters: int = 3) -> dict:
    """The reference's own CUDA route (label_reward.py:89 device = cuda, :126 clip.load -> fp16 weights, :141 model
    forward): the CLIP restatement in PyTorch eager fp16 on this GPU, image tower + logits at `batch` preprocessed
    frames. PIL preprocessing (4 ms / frame on one host thread in the reference) is NOT included: model forward only."""
    from oracle import port
    model = port.clip_shim.build("ViT-B/16", seed=0)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    # openai/CLIP's convert_weights (what clip.load does on a CUDA device): Linear / Conv / attention weights and the two
    # projections in fp16, LayerNorm parameters and arithmetic stay fp32
    for m in model.modules():
        if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)):
            m.half()
        if isinstance(m, torch.nn.MultiheadAttention):
            for prm in (m.in_proj_weight, m.in_proj_bias, m.out_proj.weight, m.out_proj.bias):
                prm.data = prm.data.half()
    model.text_projection.data = model.text_projection.data.half()
    model.visual.proj.data = model.visual.proj.data.half()
    text = port.clip_shim.tokenize([TEXT]).to(dev)
    x = torch.randn(batch, 3, 224, 224, device=dev, dtype=torch.float16)
    with torch.no_grad():
        for _ in range(2):
            model(x, text)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            model(x, text)
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    del model, x
    torch.cuda.empty_cache()
    return {"value": batch / (ms * 1e-3), "unit": "frames/s", "batch": batch, "ms_per_batch": ms, "dtype": "fp16",
            "what": "oracle CLIP restatement (openai/CLIP d50d76d) in PyTorch eager fp16 on the same B200: model(image, "
                    "text) forward only, preprocessed inputs resident (the reference's CUDA route without its PIL "
                    "preprocessing and per-episode Python loop)"}


def entrypoint_rate(args, ob_host: torch.Tensor, off_np: np.ndarray, sd, local: int, want: np.ndarray) -> dict:
    """Wall clock of label_reward() on a memory-mapped NpyStore holding the same stacked rows (page cache warm)."""
    from arp_b200.label_reward import label_reward
    from arp_b200.store import NpyStore
    T = ob_host.shape[0]
    need = ob_host.numel() + (1 << 28)
    base = None
    for cand in (os.environ.get("ARP_BENCH_TMP"), "/dev/shm", tempfile.gettempdir()):
        if cand and os.path.isdir(cand) and shutil.disk_usage(cand).free > need:
            base = cand
            break
    if base is None:
        return {"unavailable": f"no scratch directory with {need / 1e9:.0f} GB free"}
    d = Path(tempfile.mkdtemp(prefix="arp_bench_store_", dir=base))
    try:
        t0 = time.perf_counter()
        mm = np.lib.format.open_memmap(d / "ob.npy", mode="w+", dtype=np.uint8, shape=tuple(ob_host.shape))
        src = ob_host.numpy()
        for lo in range(0, T, 2048):
            mm[lo:lo + 2048] = src[lo:lo + 2048]
        mm.flush()
        del mm
        done = np.zeros((T, args.num_frames), np.float32)
        done[off_np[1:] - 1, -1] = 1.0
        np.save(d / "done.npy", done)
        write_s = time.perf_counter() - t0
        kw = dict(env_name="coinrun", distribution_mode="hard", num_levels=500, start_level=0, text=TEXT, base_path=".",
                  data_path=str(d), model_type="clip", clip_state_dict=sd, env_type="none", max_batch=args.max_batch,
                  device=local, distributed=False, precision=args.precision, tokenizer="standin")
        secs = []
        for _ in range(2):                                   # first call creates the datasets, second overwrites in place
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            label_reward(**kw)
            secs.append(time.perf_counter() - t0)
        s = NpyStore(d, "r")
        got = np.array(s["ob_clip_reward"][:])[:, -1]
        s.close()
        return {"value": T / min(secs), "unit": "frames/s", "seconds_per_call": secs, "frames": T,
                "store": f"NpyStore (np.memmap) under {base}, {ob_host.numel() / 1e9:.1f} GB, written in {write_s:.1f} s, "
                         "page cache warm", "equals_device_path": bool(np.array_equal(got, want)),
                "api": "arp_b200.label_reward.label_reward(...) — the reference's entry point signature"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def strong_scaling(args, capi, eng_kw, sd, emb, scale, dev, world: int, rank: int, dist) -> dict:
    """BASELINE configs[4]: `strong_episodes` episodes of 64x64 frames, total work fixed, episodes partitioned over the
    ranks at the boundaries nearest k*T/N (sharding.partition_episodes), one gather of [rows, 2] to rank 0."""
    from arp_b200.sharding import gather_rows, partition_episodes
    off = episode_offsets(args.strong_episodes, seed=7)
    T_all = int(off[-1])
    shards = partition_episodes(off, world)
    e_lo, e_hi = shards[rank]
    lo, hi = int(off[e_lo]), int(off[e_hi])
    T = hi - lo
    eng = capi.Engine(**{**eng_kw, "in_h": 64, "in_w": 64})
    eng.load_state_dict(sd)
    eng.set_text(emb, scale)
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    ob = torch.empty(T, 1, 64, 64, 3, dtype=torch.uint8, device=dev)
    for t0 in range(0, T, 1 << 16):
        ob[t0:t0 + (1 << 16)] = torch.randint(0, 256, ob[t0:t0 + (1 << 16)].shape, dtype=torch.uint8, device=dev, generator=gen)
    off_dev = torch.from_numpy(off[e_lo:e_hi + 1] - lo).to(dev)
    rows = [int(off[b] - off[a]) for a, b in shards]
    F = args.num_frames

    def step():
        r, g, rs, gs = eng.label(ob, off_dev, F)
        both = torch.stack([r, g], dim=1)
        return gather_rows(both, rows, dst=0) if world > 1 else both

    eng.label(ob[:4096], torch.tensor([0, 4096]), F)                 # warm the 64x64 decode tables / kernels
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    full = step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        # episode boundaries / scan order survive the partition + gather: re-scan the gathered rewards in one piece
        g_full, _, _ = eng.scan_only(full[:, 0].contiguous(), torch.from_numpy(off), 1)
        exact = bool(torch.equal(g_full, full[:, 1].contiguous()))
        out = {"workload": f"{args.strong_episodes} synthetic episodes at 64x64 (BASELINE configs[4]), total work fixed",
               "frames_total": T_all, "n_gpus": world, "seconds": float(ms) * 1e-3, "value": T_all / (float(ms) * 1e-3),
               "unit": "frames/s", "scaling": "strong", "rows_per_rank": rows,
               "rtg_of_gathered_rewards_bit_exact": exact, "timing": "one pass, CUDA events, max over ranks, gather inside"}
    eng.close()
    del ob
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    from arp_b200 import capi
    from arp_b200.build import build
    from arp_b200.sharding import gather_rows
    from arp_b200.text_tower import clip_text_embedding
    from arp_b200.tokenizer import tokenize
    from arp_b200.weights import random_clip_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        sys.exit("bench.py needs a B200: arp_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    build()

    F, S = args.num_frames, args.stack_in_memory
    off_np = episode_offsets(args.episodes, seed=1 + rank)
    T = int(off_np[-1])
    eng_kw = dict(device=local, patch=16, in_h=args.size, in_w=args.size, max_batch=args.max_batch,
                  precision=capi.PREC_F32RESID if args.precision == "fp32resid" else capi.PREC_16BIT)
    eng = capi.Engine(**eng_kw)
    sd = random_clip_state_dict("ViT-B/16", seed=0, device="cpu")   # CPU generator: same weights as the CPU arm
    eng.load_state_dict(sd)
    emb, scale = clip_text_embedding(sd, tokenize([TEXT], standin=True), dev)   # random-init weights: stand-in token ids
    eng.set_text(emb, scale)

    # synthetic frames, generated on the device in the stacked layout [T, S, H, W, 3]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    ob = torch.empty(T, S, args.size, args.size, 3, dtype=torch.uint8, device=dev)
    for t0 in range(0, T, 2048):
        ob[t0:t0 + 2048] = torch.randint(0, 256, ob[t0:t0 + 2048].shape, dtype=torch.uint8, device=dev, generator=gen)
    off = torch.from_numpy(off_np).to(dev)
    rows = [int(episode_offsets(args.episodes, seed=1 + r)[-1]) for r in range(world)]

    def step_device():
        """(reward, rtg, reward_stacked, rtg_stacked) of this rank, then with N>1 the gathered [rows, 2] (None off rank 0)"""
        out = eng.label(ob, off, F)
        if world > 1:
            return (*out, gather_rows(torch.stack(out[:2], dim=1), rows, dst=0))      # the path's only collective
        return out

    def timed(fn, k):
        """(milliseconds for k calls of fn, what the last call returned)"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            last = None                 # free the previous step's outputs before the next step, as if they were not kept
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), last

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    total_ms, last = timed(step_device, args.steps)
    launches = eng.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        arrays = dict(zip(("reward", "rtg", "reward_stacked", "rtg_stacked"), last))
        if world > 1:
            arrays.update(reward_all_ranks=last[4][:, 0], rtg_all_ranks=last[4][:, 1])
        dump_outputs(Path(args.dump_outputs), arrays)
    del last
    ms_per_step = total_ms / args.steps
    total_frames = sum(rows)
    value = total_frames / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel: one more step with per-launch CUDA events ----
    eng.profile_begin()
    step_device()
    prof = eng.profile_end()
    peaks = measured_peaks()
    gemm = prof["gemm"]
    achieved = gemm["flops"] / (gemm["total_ms"] * 1e-3) / 1e12
    traffic = None
    tpath = ROOT / "profiles" / "roofline_traffic.json"
    if tpath.exists():
        traffic = json.loads(tpath.read_text())
    step_kernel_ms = sum(v["total_ms"] for v in prof.values())
    roofline = {
        "bound": "tensor", "kernel": "gemm_tcgen05_kernel (all linear layers of one step)",
        "achieved": achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
        "frac": achieved / peaks["bf16_tflops_sustained"],
        "peak_source": f"{peaks['source']} (sustained cuBLAS bf16; tcgen05 kind::f16 runs fp16 and bf16 at the same rate)",
        "launches_per_step": gemm["launches"], "flops_per_launch_avg": gemm["flops"] / max(gemm["launches"], 1),
        "avg_launch_ms": gemm["total_ms"] / max(gemm["launches"], 1),
        "traffic": None if traffic is None else traffic.get("gemm_dram_bytes_per_launch"),
        "share_of_step": gemm["total_ms"] / step_kernel_ms,
        "by_class_ms": {k: round(v["total_ms"], 3) for k, v in prof.items() if v["launches"]},
        "hbm_bound_classes": {k: {"achieved_gbs": v["bytes"] / (v["total_ms"] * 1e-3) / 1e9,
                                  "frac_of_hbm_peak": v["bytes"] / (v["total_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"]}
                              for k, v in prof.items() if k in ("layernorm", "decode", "scan", "attention") and v["launches"]},
        # the reference's work per frame (SURVEY.md §8d: 35.127 GFLOP) over our time, and what we actually execute
        # (the last block is computed for the class-token row only, DESIGN.md): both per GPU
        "whole_step_tflops_reference_work": total_frames / world * GFLOP_PER_FRAME_B16 / (ms_per_step * 1e-3) / 1e3,
        "whole_step_tflops_executed": sum(v["flops"] for v in prof.values()) / (ms_per_step * 1e-3) / 1e12,
    }
    roofline["whole_step_frac_of_sustained_reference_work"] = \
        roofline["whole_step_tflops_reference_work"] / peaks["bf16_tflops_sustained"]

    # ---- end to end through the host-buffer entry point (C ABI), then through the drop-in itself ----
    e2e = entry = None
    r_dev = step_device()[0].cpu().numpy()
    if not args.no_e2e:
        pinned = True
        try:
            ob_host = torch.empty(ob.shape, dtype=torch.uint8, pin_memory=True)
        except RuntimeError:
            ob_host, pinned = torch.empty(ob.shape, dtype=torch.uint8), False
        ob_host.copy_(ob)
        outs = (np.empty(T, np.float32), np.empty(T, np.float32), np.empty((T, F), np.float32),
                np.empty((T, F), np.float32))

        def step_host():
            eng.label_host(ob_host, off_np, F, out=outs)
            if world > 1:
                both = torch.from_numpy(np.stack([outs[0], outs[1]], axis=1)).to(dev)
                gather_rows(both, rows, dst=0)

        step_host()
        assert np.array_equal(outs[0], r_dev), "host and device entry points disagree"
        t_e2e = []
        for _ in range(max(1, args.e2e_steps)):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step_host()
            torch.cuda.synchronize()
            t_e2e.append(time.perf_counter() - t0)
        te = torch.tensor([float(np.mean(t_e2e))], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        frame_bytes = args.size * args.size * 3
        e2e = {"value": total_frames / float(te), "unit": "frames/s", "steps": len(t_e2e),
               "h2d_bytes_per_step": int(total_frames * frame_bytes + (args.episodes + 1) * 8 * world),
               "d2h_bytes_per_step": int(total_frames * 4 * (2 + 2 * F)),
               "pinned_host": pinned, "host_row_stride_bytes": S * frame_bytes,
               "api": "arp_label_host (C ABI, host buffers, strided rows of the stacked layout)"}
        if rank == 0 and world == 1 and not args.no_entrypoint:
            del ob                                           # the store needs the host RAM / page cache more than we need HBM
            torch.cuda.empty_cache()
            ob = None
            try:
                entry = entrypoint_rate(args, ob_host, off_np, sd, local, r_dev)
            except Exception as e:  # noqa: BLE001 — a side measurement must not lose the headline
                entry = {"unavailable": f"{type(e).__name__}: {e}"}
        del ob_host

    # ---- stated baselines, rank 0, N=1 only ----
    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, n, cores, out, frames, off_s, sd_cpu = cpu_reference_rate(args, args.cpu_sample_frames)
        # parity on the same sample, same weights (reported, the tests are the gate)
        r_gpu = eng.compute_reward(torch.from_numpy(frames).to(dev)).cpu().numpy()
        dcos = float(np.abs(r_gpu - out["reward"]).max() / scale)
        cpu = {"value": rate, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": f"first {len(off_s) - 1} episodes ({n} frames) of the same synthetic workload; "
                         f"oracle/port.py (torch CPU fp32 + PIL + python scan loops)",
               "parity_max_abs_dcos_on_sample": dcos}
    if rank == 0 and world == 1 and not args.no_eager_baseline:
        try:
            eager = gpu_eager_rate(dev, sd)
        except Exception as e:  # noqa: BLE001
            eager = {"unavailable": f"{type(e).__name__}: {e}"}

    # ---- strong scaling of configs[4] (every N, including 1) ----
    strong = None
    if not args.no_strong:
        if ob is not None:
            del ob
            torch.cuda.empty_cache()
        strong = strong_scaling(args, capi, eng_kw, sd, emb, scale, dev, world, rank, dist)

    if rank == 0:
        print(json.dumps({
            "metric": "reward-labeled frames/sec", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16" if capi.operand_dtype() == torch.float16 else "bf16", "data": "synthetic",
            "config": workload_config(args), "clocks": clocks, "e2e": e2e, "entrypoint_e2e": entry,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "gpu_eager_baseline": eager,
            "strong_scaling": strong,
        }))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
