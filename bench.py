#!/usr/bin/env python
"""bench.py -- PESQ + STOI/ESTOI audio-seconds scored per second on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--seconds S] [--dump-outputs DIR]

Workload (BASELINE.json configs[4]): PESQ + STOI/ESTOI of a batch of 8192 x 10 s synthetic
speech-like pairs at 16 kHz, batch-sharded over the N ranks (strong scaling: 8192 / N items per
GPU), only the per-item scores gathered with one NCCL all-gather.  One "step" = one PESQ call plus
one STOI call over the whole (sharded) batch = 81 920 audio-seconds.

  value  : device-resident inputs -> scores on device (+ all-gather), CUDA events on the launching
           stream, barrier + synchronize on both sides, max over ranks.
  e2e    : the same through the public API `PESQ(...)(clean, denoised)` / `STOI(...)(clean, denoised)`
           with pinned HOST tensors: the library's host entry point copies H->D in chunks overlapped
           with compute and copies the scores back, every step.
  roofline: dominant kernel (largest device time in the step, measured live with CUDA events around
           every launch): algorithmic bytes of its metric call (8 B per sample pair = 128 000 B per
           audio-second, SURVEY.md 8d) / its average duration, against MEASURED_PEAKS.json's hbm_gbs.
  roofline_call: the same per metric CALL (all kernels of the PESQ call / of the STOI call against the bytes
           the call must read), roofline_step for the whole step -- the dominant kernel's fraction is not the path's.
  parity : outside the timed region, a seeded sample of the SAME device tensors (>= 32 items per rank, spread over
           the shard) is scored by the float64 oracle port and, when oracle/_ref is staged, by the unmodified
           reference; reports max |dPESQ|, |dSTOI|, |dESTOI|, K equality, the smallest silent-frame decision margin
           of the whole batch and, for N > 1, that the all-gathered rows equal rank-local scoring bit for bit.
  cpu_baseline / --impl reference: the reference's own CPU path (oracle/_ref: the unmodified reference modules,
           `PESQ(16000, use_gpu=False)` + `STOI(16000, use_gpu=False)` on 64-item chunks) on the host cores, on a
           bounded sample of the same workload; the numpy port (oracle/) beside it / as fallback.
  --dump-outputs DIR: the score table the last timed step returned, one float32 file per column
           (DIR/pesq.npy, stoi.npy, estoi.npy, item order).  The inputs are a pure function of the arguments, so two
           builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "PESQ+STOI audio-seconds scored/sec"
UNIT = "audio-s/s"
FS = 16000
BYTES_PER_AUDIO_SECOND_PER_METRIC = 2 * 4 * FS   # two fp32 signals read once (SURVEY.md 8d)


# ------------------------------------------------------------------------------------------ data
def make_shard(batch: int, n: int, seed: int, device):
    """Synthetic speech-like pairs (recipe of fast_speech_enhancement_metrics_b200.synth): a pool of
    seeded numpy items (low-passed noise x syllabic envelope + -60 dB floor), expanded on the GPU
    with a per-item circular shift and gain; degraded = clean + white noise at SNR ~ U[-5, 25] dB."""
    import numpy as np
    import torch

    from fast_speech_enhancement_metrics_b200.synth import synth_batch
    pool = min(batch, 256)
    base, _, _ = synth_batch(seed, pool, n)
    base = torch.from_numpy(base).to(device)
    g = torch.Generator(device=device).manual_seed(seed)
    clean = torch.empty(batch, n, dtype=torch.float32, device=device)
    for i0 in range(0, batch, pool):
        cnt = min(pool, batch - i0)
        shift = int(torch.randint(0, n, (1,), generator=g, device=device).item())
        gain = 0.5 + torch.rand(cnt, 1, generator=g, device=device)
        clean[i0:i0 + cnt] = torch.roll(base[:cnt], shifts=shift, dims=1) * gain
    deg = torch.empty_like(clean)
    snr = torch.rand(batch, 1, generator=g, device=device) * 30.0 - 5.0
    step = 512
    for i0 in range(0, batch, step):
        c = clean[i0:i0 + step]
        noise = torch.randn(c.shape, generator=g, device=device)
        scale = (c.pow(2).mean(1, keepdim=True) / 10.0 ** (snr[i0:i0 + step] / 10.0)).sqrt()
        deg[i0:i0 + step] = c + noise * scale
    return clean, deg


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ CPU baseline
def workload_string(batch: int, seconds: float, gpus: int) -> str:
    """config.workload: identical in the GPU arm and the reference arm."""
    return ("PESQ + STOI/ESTOI, %d x %.0f s @16 kHz, batch-sharded over %d GPU(s) (BASELINE configs[4])"
            % (batch, seconds, gpus))


def newest_traffic_file():
    """profiles/rNN_dram_traffic.json of the latest round (written by tools/ncu_launches_summary.py from the ncu
    launch list of THIS code), else None."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_dram_traffic.json")))
    return files[-1] if files else None


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args, emit):
    """The reference's own CPU implementation of the path on the host cores (oracle/_ref when staged, else the
    numpy port), every step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import cpu_arm
    cores = cpu_arm.host_cores()
    n = int(args.seconds * FS)
    kind = cpu_arm.pick_kind()
    procs, threads, items = cpu_arm.plan(kind, cores)
    arm = cpu_arm.CpuArm(kind, n, procs, threads, items)
    times = []
    for step in range(args.warmup + args.steps):
        dt = arm.step()
        if step >= args.warmup:
            times.append(dt)
    finite = arm.finite
    arm.close()
    audio_s = arm.audio_seconds_per_step
    total = sum(times)
    value = audio_s * len(times) / total
    sample = ("%d worker processes x %d items x %.0f s per step; %s; inputs pre-generated"
              % (procs, items, args.seconds, cpu_arm._describe(kind, threads)))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32" if kind == "reference" else "f64",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": workload_string(args.batch, args.seconds, args.gpus),
                   "batch_total": args.batch, "samples": n, "sample_rate": FS,
                   "sample_items_per_step": procs * items,
                   "note": "each step scores a bounded sample of the workload on the host cores"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "procs": procs,
                         "threads_per_proc": threads, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "finite_score_fraction": finite,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------ NUMA placement
def bind_to_gpu_cpus(gpu_index: int):
    """Pin this rank to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is allocated: the
    e2e leg is bound by pinned host->device copies, and a pinned buffer is placed (first touch) on the NUMA node of
    the thread that allocates it.  Returns a short description for the bench line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (v >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no local cpus reported"
        os.sched_setaffinity(0, cpus)
        try:
            node = pynvml.nvmlDeviceGetNumaNodeId(h)
        except Exception:
            node = None
        return "bound to %d cpus local to gpu %d (numa node %s)" % (len(cpus), gpu_index, node)
    except Exception as exc:
        return "not bound (%r)" % (exc,)


# ------------------------------------------------------------------------------------------ parity at the workload
def parity_block(pesq, stoi, clean, deg, gathered, lo, hi, world, device, items):
    """Outside the timed region: the rank's shard is scored once more (same kernels, same chunk grid as the timed
    steps), a seeded sample of `items` rows spread over the shard is checked against the float64 oracle port and --
    when oracle/_ref is staged -- the unmodified reference, and the all-gathered table of the last timed step is
    compared bit for bit with rank-local scoring.  Bars (BASELINE.md section 5): 1e-3 / 1e-4 / exact."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from oracle import make_ref, pesq_oracle, stoi_oracle
    local_b = clean.shape[0]
    mos, _ = pesq.score_tensors(clean, deg)
    sc, kept, _ = stoi.score_tensors(clean, deg)
    margin = stoi.mask_margin()
    local = torch.stack([mos, sc[0], sc[1]], dim=1)
    torch.cuda.synchronize()
    # bit-for-bit (NaN-safe): compare the raw words
    gather_equal = bool(torch.equal(gathered[lo:hi].contiguous().view(torch.int32), local.contiguous().view(torch.int32)))
    idx = np.unique(np.linspace(0, local_b - 1, min(items, local_b)).round().astype(np.int64))
    tidx = torch.from_numpy(idx).to(device)
    c = clean[tidx].cpu()
    d = deg[tidx].cpu()
    got = local[tidx].double().cpu().numpy()
    k_got = kept[tidx].cpu().numpy()

    def maxabs(a, b):
        both_nan = np.isnan(a) & np.isnan(b)
        diff = np.where(both_nan, 0.0, np.abs(a - b))
        return float(np.max(np.where(np.isnan(diff), np.inf, diff))) if len(a) else 0.0

    o_p = pesq_oracle.pesq_batch(c.numpy(), d.numpy())
    o_s, o_e, o_k = stoi_oracle.stoi_batch(c.numpy(), d.numpy(), FS)
    stats = [maxabs(got[:, 0], o_p), maxabs(got[:, 1], o_s), maxabs(got[:, 2], o_e)]
    k_equal = bool(np.array_equal(k_got, o_k))
    ref_stats = [-1.0, -1.0, -1.0]
    ref_extra = [0.0, 0.0]          # items whose |dPESQ| vs the reference exceeds the bar; max |reference - oracle| over those
    ref_unexplained = 0.0           # ... of which the reference itself is within the bar of the oracle (a real discrepancy)
    if make_ref.available():
        RP, RS = make_ref.load()
        rp = np.array([r["PESQ"] for r in RP(FS, use_gpu=False)(c, d)])
        rs = RS(FS, use_gpu=False)(c, d)
        ref_stats = [maxabs(got[:, 0], rp),
                     maxabs(got[:, 1], np.array([r["STOI"] for r in rs])),
                     maxabs(got[:, 2], np.array([r["ESTOI"] for r in rs]))]
        over = np.abs(got[:, 0] - rp) > 1e-3
        if over.any():
            ref_extra = [float(over.sum()), float(np.max(np.abs(rp[over] - o_p[over])))]
            ref_unexplained = float((over & (np.abs(rp - o_p) <= 1e-3)).sum())
    finite_margin = margin[torch.isfinite(margin)]
    mmin = float(finite_margin.min()) if finite_margin.numel() else float("inf")
    near = int((margin < 1e-4).sum())
    red_max = torch.tensor(stats + ref_stats + [0.0 if k_equal else 1.0, 0.0 if gather_equal else 1.0, -mmin],
                           dtype=torch.float64, device=device)
    red_sum = torch.tensor([float(len(idx)), float(near), ref_extra[0], ref_unexplained], dtype=torch.float64, device=device)
    red_max = torch.cat([red_max, torch.tensor([ref_extra[1]], dtype=torch.float64, device=device)])
    if world > 1:
        dist.all_reduce(red_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(red_sum, op=dist.ReduceOp.SUM)
    m = red_max.tolist()
    out = {"pesq_max_abs": m[0], "stoi_max_abs": m[1], "estoi_max_abs": m[2], "k_equal": m[6] == 0.0,
           "items": int(red_sum[0].item()), "vs": "float64 oracle port (oracle/), sample spread over every rank's shard",
           "bars": {"pesq": 1e-3, "stoi": 1e-4, "estoi": 1e-4, "k": "exact"},
           "mask_margin_min_db": -m[8], "items_with_margin_below_1e-4_db": int(red_sum[1].item()),
           "gathered_rows_equal_rank_local_bitwise": m[7] == 0.0}
    if m[3] >= 0.0:
        n_over = int(red_sum[2].item())
        out["vs_reference"] = {"pesq_max_abs": m[3], "stoi_max_abs": m[4], "estoi_max_abs": m[5],
                               "vs": "oracle/_ref: unmodified reference, use_gpu=False, same sample",
                               "pesq_items_above_1e-3": n_over, "ok": bool(m[3] <= 1e-3 and m[4] <= 1e-4 and m[5] <= 1e-4)}
        if n_over:
            # the reference runs its order-10 IIR in float32 direct form (PESQ.py:80-81,94): its own output carries
            # ~1e-4 of PESQ noise and, on rare items, flips one of PESQ's hard thresholds.  For the items above the bar:
            # how far the REFERENCE is from the float64 evaluation of its own algorithm (the CUDA path is within
            # `pesq_max_abs` of that evaluation on every item)
            out["vs_reference"]["reference_vs_oracle_max_abs_on_those_items"] = m[9]
            # 0 = on every item above the bar the reference is itself more than the bar away from the float64 evaluation
            out["vs_reference"]["items_above_1e-3_not_explained_by_reference_noise"] = int(red_sum[3].item())
    # the pinned checker is the float64 oracle (tests/test_oracle_vs_golden.py pins it on the reference's outputs)
    out["ok"] = bool(m[0] <= 1e-3 and m[1] <= 1e-4 and m[2] <= 1e-4 and out["k_equal"]
                     and out["gathered_rows_equal_rank_local_bitwise"])
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path: str, table) -> None:
    """Writes the [batch, 3] score table (PESQ, STOI, ESTOI) as float32 columns.  Above 64 MB in all, a fixed seeded
    sample of the rows is written instead, with their item indices in items.npy (float64)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    keep = DUMP_LIMIT_BYTES // (table.shape[1] * 4 + 8)
    if table.shape[0] > keep:
        idx = np.sort(np.random.default_rng(0).choice(table.shape[0], keep, replace=False))
        table = table[idx]
        np.save(os.path.join(path, "items.npy"), idx.astype(np.float64))
    for j, name in enumerate(("pesq", "stoi", "estoi")):
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(table[:, j], dtype=np.float32))


# ------------------------------------------------------------------------------------------ main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="total items over all ranks")
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the direct entry points instead of the CUDA-graph path")
    ap.add_argument("--parity-items", type=int, default=32, help="items per rank scored by the oracle (outside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the scores of the last timed step to DIR/{pesq,stoi,estoi}.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the scores of the GPU path; the reference arm keeps none")
    args.warmup = max(args.warmup, 0)
    # stdout carries exactly ONE JSON line (rank 0): anything libraries print there (e.g. NCCL's version banner) is
    # sent to stderr by pointing fd 1 at fd 2 until the line is written
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line: dict):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)

    if args.impl == "reference":
        return run_reference(args, emit)

    import numpy as np
    import torch
    import torch.distributed as dist

    from fast_speech_enhancement_metrics_b200 import PESQ, STOI, CapturedScorer, _lib
    from fast_speech_enhancement_metrics_b200.dist import gather_scores, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.gpus > 1:
        print("bench.py: --gpus %d needs torchrun (WORLD_SIZE is 1); running 1 rank" % args.gpus, file=sys.stderr)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # multi-GPU: NUMA-local pinned buffers by default (FSEM_BIND_NUMA=0 disables)
    numa = "off"
    if os.environ.get("FSEM_BIND_NUMA", "1" if world > 1 else "0") == "1":
        numa = bind_to_gpu_cpus(local_rank)
    n = int(args.seconds * FS)
    lo, hi = shard_range(args.batch, world, rank)
    local_b = hi - lo
    audio_s_total = args.batch * n / FS

    pesq = PESQ(FS, use_gpu=True)
    stoi = STOI(FS, use_gpu=True)
    clean, deg = make_shard(local_b, n, 1000 + rank, device)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gathered = torch.empty(args.batch, 3, dtype=torch.float32, device=device)

    # The timed step is the library's captured-scoring path (public API CapturedScorer = C ABI fsem_graph_*): ONE CUDA
    # graph per step whose PESQ chain and STOI chain are parallel branches (the tails of one chain's kernels fill
    # with the other's: x1.01 at 8192 items per GPU, x1.08 at 1024), then the all-gather of the score rows.
    # --no-graph times the direct entry points (fsem_pesq_score + fsem_stoi_score back to back on one stream).
    scorer = None if args.no_graph else CapturedScorer(pesq, stoi, clean, deg)

    def step_direct():
        mos, _ = pesq.score_tensors(clean, deg)
        sc, _, _ = stoi.score_tensors(clean, deg)
        return torch.stack([mos, sc[0], sc[1]], dim=1)

    def step_device():
        if scorer is not None:
            local = scorer.replay()[0].t().contiguous()
        else:
            local = step_direct()
        return gather_scores(local, args.batch, world, out=gathered)

    # ---- value: device-resident inputs
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = step_device()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = _lib.launch_count() - launches0
    # ---- per-kernel times: the same kernels launched directly (one stream, one CUDA-event pair around every launch,
    # fsem_profile_*), right after the timed region and under the same clocks; events cannot bracket the nodes of a
    # graph whose branches run concurrently.  Rank-local, no collective.
    _lib.profile_reset()
    _lib.profile_enable(True)
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pv0.record()
    for _ in range(args.steps):
        step_direct()
    pv1.record()
    torch.cuda.synchronize()
    direct_ms_per_step = pv0.elapsed_time(pv1) / args.steps
    _lib.profile_enable(False)
    prof = _lib.profile_read()
    if rank == 0 and len(sampler.lines) < 4:
        # a short timed region can end before nvidia-smi has sampled a few times: keep the same load running (untimed)
        # until there are enough samples to report the clocks under load
        t_end = time.perf_counter() + 1.0
        while time.perf_counter() < t_end and len(sampler.lines) < 6:
            step_direct()                           # rank-local work only: no collective outside the timed steps
            torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = audio_s_total / (ms_per_step * 1e-3)
    scores = out.cpu().numpy()
    finite = float(np.isfinite(scores).mean())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scores)

    # ---- parity at this workload, on these tensors (outside the timed region)
    parity = None
    if not args.no_parity:
        parity = parity_block(pesq, stoi, clean, deg, out, lo, hi, world, device, args.parity_items)

    # ---- e2e: public API with pinned host tensors (H2D + compute + D2H every step)
    e2e = None
    if not args.no_e2e:
        hc = torch.empty(clean.shape, dtype=torch.float32, pin_memory=True).copy_(clean)
        hd = torch.empty(deg.shape, dtype=torch.float32, pin_memory=True).copy_(deg)
        torch.cuda.synchronize()

        from fast_speech_enhancement_metrics_b200 import score_pesq_stoi

        def finish(rows):
            local = torch.tensor(rows, dtype=torch.float32)
            if world > 1:
                return gather_scores(local.to(device), args.batch, world, out=gathered).cpu()
            return local

        def step_fused():        # one upload, both metrics (C ABI fsem_pesq_stoi_score_host_f32)
            r = score_pesq_stoi(pesq, stoi, hc, hd)
            return finish([[a["PESQ"], a["STOI"], a["ESTOI"]] for a in r])

        def step_separate():     # the reference's two calls, each uploading both signals
            p = pesq(hc, hd)
            s = stoi(hc, hd)
            return finish([[a["PESQ"], b["STOI"], b["ESTOI"]] for a, b in zip(p, s)])

        per_call_ms = {}

        def time_e2e(fn, steps, label):
            import gc
            fn()
            # every call builds 8192 result dicts: a generation-2 garbage collection landing inside a timed call costs
            # ~45 ms of pure interpreter time (seen as one 145 ms call among 99 ms ones); collect now, not in the loop
            gc.collect()
            gc.disable()
            barrier()
            calls = []
            t0 = time.perf_counter()
            for _ in range(steps):
                t1 = time.perf_counter()
                fn()
                calls.append(round((time.perf_counter() - t1) * 1e3, 2))
            barrier()
            gc.enable()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            per_call_ms[label] = calls                      # rank 0's wall time of every timed call
            return audio_s_total * steps / float(dt.item())

        e_steps = max(1, min(args.steps, 3))
        v_fused = time_e2e(step_fused, e_steps, "fused")
        v_sep = time_e2e(step_separate, e_steps, "separate_calls")
        del hc, hd
        # the same call on int16 PCM (SURVEY.md 8f rank 2: ingest formats): 2 bytes per sample over PCIe, widened on
        # the device.  Informational -- the headline e2e above is the float32 contract of the reference API.
        scale = 32767.0 / float(torch.maximum(clean.abs().max(), deg.abs().max()))
        hc = torch.empty(clean.shape, dtype=torch.int16, pin_memory=True).copy_((clean * scale).round().to(torch.int16))
        hd = torch.empty(deg.shape, dtype=torch.int16, pin_memory=True).copy_((deg * scale).round().to(torch.int16))
        torch.cuda.synchronize()
        v_i16 = time_e2e(step_fused, e_steps, "int16_ingest")
        e2e = {"value": v_fused, "unit": UNIT,
               "h2d_bytes_per_step": int(2 * args.batch * n * 4),          # both signals, uploaded once
               "d2h_bytes_per_step": int(args.batch * 24),                 # mos, stoi, estoi, K, 2 x status
               "steps": e_steps, "per_call_ms": per_call_ms,
               "api": "score_pesq_stoi(PESQ(16000), STOI(16000), clean_cpu, deg_cpu) with pinned host tensors "
                      "(C ABI fsem_pesq_stoi_score_host_f32: one upload, both metrics)",
               "separate_calls": {"value": v_sep, "unit": UNIT, "h2d_bytes_per_step": int(2 * 2 * args.batch * n * 4),
                                  "api": "PESQ(16000)(clean_cpu, deg_cpu) + STOI(16000)(clean_cpu, deg_cpu): "
                                         "the reference's two calls, each uploading both signals"},
               "int16_ingest": {"value": v_i16, "unit": UNIT, "h2d_bytes_per_step": int(2 * args.batch * n * 2),
                                "api": "score_pesq_stoi on pinned int16 PCM tensors (C ABI fsem_score_host, "
                                       "FSEM_DTYPE_I16): same samples quantised to 16 bit, widened on the device"}}
        del hc, hd

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    kernels = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps} for k, v in prof.items()}
    top = max(prof.items(), key=lambda kv: kv[1][0])
    top_name, (top_ms, top_cnt) = top
    local_audio_s = local_b * n / FS
    alg_bytes = BYTES_PER_AUDIO_SECOND_PER_METRIC * local_audio_s          # per launch (one launch per metric call)
    top_avg_ms = top_ms / max(top_cnt, 1)
    achieved = alg_bytes / (top_avg_ms * 1e-3) / 1e9
    # DRAM traffic per launch: from the ncu launch list of THIS round's code (profiles/rNN_dram_traffic.json, written
    # by tools/ncu_launches_summary.py); measured at tj["items"] items x 10 s, linear in the item count
    traffic, traffic_src, tj = None, None, None
    traffic_path = newest_traffic_file()
    if traffic_path:
        tj = json.load(open(traffic_path))
        per_launch = tj.get("bytes_per_launch", {}).get(top_name)
        if per_launch is not None:
            traffic = per_launch * (local_b * args.seconds) / (tj.get("items", 8192) * 10.0)
            traffic_src = os.path.relpath(traffic_path, ROOT)
    roofline = {"bound": "hbm", "kernel": top_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": top_avg_ms,
                "note": "dominant kernel only (one of the kernels of its metric call): see roofline_call / "
                        "roofline_step for the path; the path is FP32-issue / shared-memory bound (SURVEY 7.2), the "
                        "HBM fraction is reported because the metric asks for it"}
    # issue / FP32-pipe / LSU utilisation of the dominant kernel from the same round's `ncu --set full` capture (north_star:
    # "achieved HBM GB/s ... and FP32-pipe utilisation"): the path is bound by these, not by HBM
    import glob
    pipe_files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_ncu_pipes.json")))
    if pipe_files:
        pj = json.load(open(pipe_files[-1])).get("kernels", {})
        if top_name in pj:
            roofline["pipes"] = dict(pj[top_name], source=os.path.relpath(pipe_files[-1], ROOT))
    # per metric CALL: all kernels of the call against the bytes the call must read
    roofline_call = {}
    for call, prefix in (("PESQ", "pesq_"), ("STOI", "stoi_")):
        call_ms = sum(v[0] for k, v in prof.items() if k.startswith(prefix)) / args.steps
        if call_ms > 0:
            tr = None
            if tj is not None:
                tr = sum(b for k, b in tj.get("bytes_per_launch", {}).items() if k.startswith(prefix))
                tr = tr * (local_b * args.seconds) / (tj.get("items", 8192) * 10.0)
            roofline_call[call] = {"ms": call_ms, "achieved": alg_bytes / (call_ms * 1e-3) / 1e9, "peak": peak,
                                   "unit": "GB/s", "frac": alg_bytes / (call_ms * 1e-3) / 1e9 / peak,
                                   "algorithmic_bytes": alg_bytes, "traffic": tr}
    # what binds the step: device time each resource is busy, summed over the kernels (utilisation from the round's
    # `ncu --set full` capture x this run's kernel times; DRAM = the launch list's bytes at the measured copy bandwidth)
    pipe_time = None
    if pipe_files:
        lsu = issue = 0.0
        for k, v in kernels.items():
            pk = pj.get(k)
            if pk and v["ms_per_step"] > 0:
                lsu += pk.get("lsu_data_pipe_pct", 0.0) / 100.0 * v["ms_per_step"]
                issue += pk.get("issue_active_pct", 0.0) / 100.0 * v["ms_per_step"]
        pipe_time = {"lsu_data_pipe_ms": lsu, "issue_slots_ms": issue, "source": os.path.relpath(pipe_files[-1], ROOT)}
        if tj is not None:
            tot = sum(tj.get("bytes_per_launch", {}).values()) * (local_b * args.seconds) / (tj.get("items", 8192) * 10.0)
            pipe_time["dram_ms_at_measured_peak"] = tot / (peak * 1e9) * 1e3
            pipe_time["dram_bytes_per_step"] = tot
    step_bytes = 2 * BYTES_PER_AUDIO_SECOND_PER_METRIC * local_audio_s
    roofline_step = {"achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                     "algorithmic_bytes_per_step_per_gpu": step_bytes, "resource_busy_ms": pipe_time}

    cpu = None
    if not args.no_cpu and world == 1:
        from oracle import cpu_arm
        cores = cpu_arm.host_cores()
        kind = cpu_arm.pick_kind()
        cpu = cpu_arm.measure(kind, n, cores)                  # 1 warm-up + best of 3 steps of 64-item chunks
        if kind == "reference":                                # the numpy port beside it (round-1 baseline)
            port = cpu_arm.measure("port", n, cores, repeats=2, single_process=False)
            cpu["port"] = {k: port[k] for k in ("value", "unit", "procs", "seconds", "sample")}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.batch, args.seconds, world),
                   "batch_total": args.batch, "batch_per_gpu": local_b, "samples": n, "sample_rate": FS,
                   "l2": "inputs (%.1f GB per GPU) exceed L2; no flush" % (2 * local_b * n * 4 / 1e9),
                   "collective": "all_gather of [batch/N, 3] fp32 scores (NCCL)" if world > 1 else "none",
                   "step": "direct calls" if args.no_graph else "one CUDA graph (fsem_graph_launch) + score gather",
                   "numa": numa},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "roofline_call": roofline_call, "roofline_step": roofline_step, "kernels": kernels,
        "kernels_from": {"pass": "direct entry points on one stream, one CUDA-event pair per launch, run right after the timed "
                                 "region (the timed steps replay the CUDA graph, whose concurrent branches events cannot bracket)",
                         "direct_ms_per_step": direct_ms_per_step,
                         "timed_path": "direct calls" if args.no_graph else "CapturedScorer.replay (fsem_graph_launch): PESQ and STOI chains as parallel graph branches"},
        "cpu_baseline": cpu, "parity": parity, "finite_score_fraction": finite,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
