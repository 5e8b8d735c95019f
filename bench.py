#!/usr/bin/env python
"""bench.py -- GCUPS of the DP-relaxation hot path on the BASELINE.json workload.

Workload (BASELINE.json configs[1] / configs[4]): ecoli x sboydii, semi-global,
affine (Gotoh) gaps (same=2, diff=-1, gapInit=-2, gapExtend=-1), score-only,
~4.64 Mbp x 4.6 Mbp.  The bundled genomes are missing from the reference mount,
so seeded synthetic stand-ins are used (anyseq_b200/workloads.py) unless
sequences/ecoli.fna and sequences/sboydii.fna exist.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

One JSON line on stdout (rank 0).  A "step" = one complete score-only alignment
of the pair.  N > 1 (torchrun): the pair is split into N column strips, one per
GPU, chained by the strip-boundary column over NVLink (strong scaling); `value`
is ONE alignment at a time (barrier between steps, every alignment pays the
wavefront fill) -- BASELINE configs[4]; the throughput of a stream of alignments
(several side by side per launch) is reported separately under "stream".

    python bench.py --workload reads [--pairs 10000000]    BASELINE configs[3]: batched reads x windows

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float64; float32 for per-pair
scores, at most 64 MB in all), so that two builds can be compared output for output on the same seeded inputs.

  value     whole-job GCUPS, sequences resident in HBM, device time (CUDA events
            recorded by the library on the stream it launches on), max over ranks
  e2e       same metric through the C ABI with HOST buffers (H2D + D2H inside)
  roofline  integer/DPX issue roofline (SURVEY.md 8d) measured live on this GPU
  cpu_baseline  the oracle's restated reference CPU path on a bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCORING = dict(same=2, diff=-1, gap_init=-2, gap_extend=-1)
MODE = "semiglobal"
OPS_PER_CELL_AFFINE = 7        # SURVEY.md 8(d): algorithmic 32-bit integer ops per Gotoh cell
# what the strip kernel actually issues per Gotoh cell at full width (decoupled cell form, K = 32, two-row tiles; counted
# in the SASS of the unguarded step loop with tools/sass_stats.py: 445 instructions, 285 on the ALU pipe, per 64 cells;
# ncu on the whole launch: 7.14 warp-instructions per 32 cells, ALU pipe 94 % busy)
ISSUED_PER_CELL = 445 / 64.0
ALU_PER_CELL = 285 / 64.0
METRIC = "GCUPS (score-only ecoli x sboydii affine)"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The contract is ONE JSON line on stdout.  Libraries print to fd 1 behind Python's
# back (NCCL announces its version there), so fd 1 is pointed at stderr for the
# whole run and the JSON line goes to a private duplicate of the original stdout.
_JSON_OUT = None


def _claim_stdout():
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


DUMP_LIMIT_BYTES = 64 << 20
DUMP_MAX_PAIRS = 2_000_000     # --workload reads: 2 schemes x 4 B + an 8 B index per pair = 32 MB


def dump_outputs(directory, arrays):
    """--dump-outputs: one <name>.npy per array (float32 / float64 only)"""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"bench.py: wrote {', '.join(sorted(arrays))} to {directory}")


def result_arrays(score, end_i, end_j):
    return {"score": np.array([score], dtype=np.float64), "end_cell": np.array([end_i, end_j], dtype=np.float64)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "250"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        clk, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                clk.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for nm, v in zip(names, r[3:7]):
                if v == "Active":
                    reasons.add(nm)
        if not clk:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(clk)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_median": float(np.median(pw)), "samples": len(clk)}


def cpu_baseline(q, s, sample_rows, sample_cols, threads):
    """restated reference CPU path (oracle port: 1024x1024 block wavefront, scalar
    inner loop, Gotoh as defined by the build) on a bounded sample of the workload"""
    from oracle import oracle as O
    qs, ss = q[:sample_rows], s[:sample_cols]
    t0 = time.perf_counter()
    sc = O.score_affine(MODE, qs, ss, SCORING["same"], SCORING["diff"], SCORING["gap_init"],
                        SCORING["gap_extend"], threads=threads)
    dt = time.perf_counter() - t0
    return len(qs) * len(ss) / dt / 1e9, dt, sc


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path on the host
    cores.  AnyDSL/Impala cannot be built here (DESIGN.md), so this is the oracle's
    restatement of iteration_cpu/scoring_cpu (kind "port") with all host threads."""
    if rank != 0:
        return 0
    from anyseq_b200 import workloads as W
    q, s, desc = W.whole_genome_pair(args.scale)
    threads = os.cpu_count() or 1
    side = int(args.cpu_sample) or 150000
    times = []
    for i in range(args.warmup + args.steps):
        g, dt, sc = cpu_baseline(q, s, side, side, threads)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result_arrays(*sc))
    ms = 1e3 * float(np.mean(times))
    val = side * side / (ms * 1e-3) / 1e9
    sample = f"first {side} x {side} cells of the workload per step ({side*side:.3g} cells), all {threads} host threads"
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GCUPS", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": desc + "; semiglobal affine (2,-1,-2,-1) score-only", "sample": sample},
        "cpu_baseline": {"value": val, "unit": "GCUPS", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)
    return 0


def golden_c2():
    """frozen CPU result of the full-size workload (tools/freeze_fullsize.py -> tests/golden/fullsize.json)"""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "fullsize.json")) as f:
            return json.load(f).get("c2_semiglobal_affine")
    except Exception:
        return None


def run_reads(args, rank, world, local_rank):
    """BASELINE configs[3]: npairs random 150 bp reads vs 500 bp windows, global + semiglobal Gotoh, score only; the
    pairs are sharded over the ranks by contiguous ranges (no data-path collective, SURVEY 8e).  Inputs are 2-bit
    packed (anyseq_score_batch_packed2).  value: device-resident, device time; e2e: pinned host arrays through the
    C ABI (H2D of every chunk and D2H of the scores inside)."""
    import torch
    import anyseq_b200 as A
    from anyseq_b200 import capi, workloads as W
    from anyseq_b200.multigpu import pair_ranges

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    RL, WL = 150, 500
    QB, SB = (RL + 3) // 4, (WL + 3) // 4
    npairs = int(args.pairs)
    p0, p1 = pair_ranges(npairs, world)[rank]
    mine = p1 - p0
    al = A.Aligner(local_rank)
    info = al.device_info()
    scoring = A.affine_scoring_scheme(**SCORING)
    # synthetic pairs generated chunk by chunk (seed = 7 + global chunk index, so every rank count sees the same pairs),
    # packed on the host, kept in PINNED host memory and copied to the device once for the resident runs
    CH = 250_000
    h_q = torch.empty((mine, QB), dtype=torch.uint8).pin_memory()
    h_s = torch.empty((mine, SB), dtype=torch.uint8).pin_memory()
    sample = None                      # rank 0 keeps the unpacked first pairs for the oracle check
    t_gen = time.perf_counter()

    def gen_chunk(c):
        lo, hi = c * CH, min((c + 1) * CH, npairs)
        q, qo, s, so = W.read_batch(hi - lo, RL, WL, seed=7 + c)
        a, b = max(p0, lo) - lo, min(p1, hi) - lo
        q, s = q.reshape(-1, RL)[a:b], s.reshape(-1, WL)[a:b]
        keep = (q[:int(args.oracle_pairs)].copy(), s[:int(args.oracle_pairs)].copy()) if (rank == 0 and lo + a == p0) else None
        return lo + a, A.pack2(q), A.pack2(s), keep

    from concurrent.futures import ThreadPoolExecutor
    chunks = range(p0 // CH, (p1 - 1) // CH + 1) if mine > 0 else range(0)
    with ThreadPoolExecutor(max_workers=max(1, min(8, (os.cpu_count() or 8) // max(1, min(world, 8))))) as ex:
        for first, pq, ps, keep in ex.map(gen_chunk, chunks):
            h_q[first - p0: first - p0 + len(pq)] = torch.from_numpy(pq)
            h_s[first - p0: first - p0 + len(ps)] = torch.from_numpy(ps)
            if keep is not None:
                sample = keep
    log(f"[rank {rank}] generated + packed {mine} pairs in {time.perf_counter() - t_gen:.1f} s")
    d_q, d_s = h_q.cuda(), h_s.cuda()
    d_sc = torch.zeros(mine, dtype=torch.int32, device="cuda")
    h_sc = torch.zeros(mine, dtype=torch.int32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    pb_dev = capi.PackedBatch(d_q.data_ptr(), d_s.data_ptr(), None, None, None, None, RL, WL, QB, SB, mine)
    pb_host = capi.PackedBatch(h_q.data_ptr(), h_s.data_ptr(), None, None, None, None, RL, WL, QB, SB, mine)
    cells = float(npairs) * RL * WL
    modes = ("global", "semiglobal")

    def step_resident(mode):
        flush.zero_()
        torch.cuda.synchronize()
        return al.score_batch_packed2(mode, pb_dev, d_sc.data_ptr(), scoring, device=True)

    # --dump-outputs: the scores of a fixed, seeded sample of the pairs (all of them up to DUMP_MAX_PAIRS)
    dumped = {}
    if args.dump_outputs:
        pick = np.arange(npairs) if npairs <= DUMP_MAX_PAIRS else \
            np.sort(np.random.default_rng(0).choice(npairs, DUMP_MAX_PAIRS, replace=False))
        mine_pick = torch.from_numpy(pick[(pick >= p0) & (pick < p1)] - p0).cuda()

    results = {}
    sampler = ClockSampler(local_rank)
    for mi, mode in enumerate(modes):
        for _ in range(args.warmup):
            step_resident(mode)
        barrier()
        if rank == 0 and mi == 0:
            sampler.start()
        ms, nl = 0.0, 0
        for _ in range(args.steps):
            r = step_resident(mode)
            ms += r.kernel_ms
            nl += r.kernel_launches
        barrier()
        if args.dump_outputs:
            got = d_sc[mine_pick].float().cpu().numpy()        # |score| < 2**24: exact in float32
            if dist is not None:
                parts = [None] * world
                dist.all_gather_object(parts, got)
                got = np.concatenate(parts)                     # ranks hold contiguous, ascending pair ranges
            dumped[f"scores_{mode}"] = got
        chk = int(d_sc.to(torch.int64).sum().item())          # 64-bit checksum of this rank's scores
        # e2e: pinned host arrays through the C ABI
        e2e_steps = max(1, min(args.steps, 3))
        al.score_batch_packed2(mode, pb_host, h_sc.data_ptr(), scoring)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            al.score_batch_packed2(mode, pb_host, h_sc.data_ptr(), scoring)
        barrier()
        dt = time.perf_counter() - t0
        same = bool(torch.equal(h_sc, d_sc.cpu()))
        t = torch.tensor([ms, dt * 1e3, float(chk), float(nl), 1.0 if same else 0.0], dtype=torch.float64, device="cuda")
        tmax, tsum = t.clone(), t.clone()
        if dist is not None:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_step = tmax[0].item() / args.steps
        results[mode] = {"gcups": cells / (ms_step * 1e-3) / 1e9, "ms_per_step": ms_step,
                         "e2e_gcups": cells * e2e_steps / (tmax[1].item() * 1e-3) / 1e9,
                         "checksum": int(tsum[2].item()), "launches": int(tsum[3].item()),
                         "e2e_scores_equal_resident": bool(tsum[4].item() == world)}
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**dumped, "pair_index": pick.astype(np.float64)})
    # oracle check on the first pairs of rank 0 (both schemes) + CPU baseline timing of the same sample
    from oracle import oracle as O
    sq, ss = sample
    k = len(sq)
    qo = np.arange(k + 1, dtype=np.int64) * RL
    so = np.arange(k + 1, dtype=np.int64) * WL
    threads = os.cpu_count() or 1
    check = {}
    cpu = None
    for mode in modes:
        t0 = time.perf_counter()
        want = O.score_batch(mode, sq.reshape(-1), qo, ss.reshape(-1), so, SCORING["same"], SCORING["diff"],
                             SCORING["gap_init"], SCORING["gap_extend"], threads=threads)
        dt = time.perf_counter() - t0
        al.score_batch_packed2(mode, pb_dev, d_sc.data_ptr(), scoring, device=True)
        got = d_sc[:k].cpu().numpy()
        check[mode] = {"pairs": k, "equal": bool(np.array_equal(got, want))}
        if not check[mode]["equal"]:
            raise SystemExit(f"bench.py: GPU batch scores differ from the oracle ({mode})")
        if mode == "semiglobal":
            cpu = {"value": k * RL * WL / dt / 1e9, "unit": "GCUPS", "cores": threads, "kind": "port",
                   "sample": f"first {k} pairs ({dt:.1f} s), restated reference CPU path pair by pair, {threads} threads"}
    main_mode = "semiglobal"
    r = results[main_mode]
    out = {
        "metric": "GCUPS (batched 150 bp reads x 500 bp windows, affine, score-only)", "value": r["gcups"], "unit": "GCUPS",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int16x2 (packed halves; int32 fallback)",
        "data": "synthetic",
        "config": {"workload": f"{npairs} pairs: random {RL} bp reads vs {WL} bp windows holding a mutated copy (seed 7 + chunk), "
                               "semiglobal + global Gotoh (2,-1,-2,-1), score-only; 2-bit packed input",
                   "pairs": npairs, "pairs_per_rank": mine, "cells_per_step": cells,
                   "partition": f"contiguous ranges of pairs over {world} rank(s), no data-path collective",
                   "l2": "L2 flushed (256 MiB memset) before every timed step",
                   "timing": "CUDA events on the library's launch stream, summed over steps, max over ranks"},
        "per_scheme": results, "oracle_check": check, "clocks": clocks,
        "e2e": {"value": r["e2e_gcups"], "unit": "GCUPS", "h2d_bytes_per_step": int(mine * (QB + SB)),
                "d2h_bytes_per_step": int(mine * 4), "note": "per rank; pinned host arrays, chunks copied under the kernels"},
        "gpu_launches": r["launches"], "cpu_baseline": cpu, "device": info["name"], "sm_count": info["sm_count"],
    }
    emit(out)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="genome", choices=["genome", "reads"],
                    help="genome: BASELINE configs[1]/[4] (the headline); reads: configs[3], batched short pairs")
    ap.add_argument("--pairs", type=int, default=10_000_000, help="--workload reads: number of pairs")
    ap.add_argument("--oracle-pairs", type=int, default=100_000, help="--workload reads: pairs checked against the oracle")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (development only)")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="side of the CPU-baseline sample (default: 250000 for the cpu_baseline leg, "
                         "150000 per step for --impl reference)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--pairs-per-launch", type=int, default=4,
                    help="N > 1, 'stream' leg: consecutive alignments relaxed side by side in one launch per rank")
    ap.add_argument("--stream-steps", type=int, default=-1,
                    help="N > 1: alignments of the streamed leg (default: 2 launches of --pairs-per-launch; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32/float64, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    _claim_stdout()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (anyseq_b200 has no CPU fallback)")
    if args.workload == "reads":
        return run_reads(args, rank, world, local_rank)

    import anyseq_b200 as A
    from anyseq_b200 import workloads as W
    from anyseq_b200.multigpu import StripWavefront, column_slices

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    q, s, desc = W.whole_genome_pair(args.scale)
    m, n = len(q), len(s)
    cells = float(m) * float(n)
    scoring = A.affine_scoring_scheme(**SCORING)
    al = A.Aligner(local_rank)
    info = al.device_info()

    slices = column_slices(n, world)              # equal slices (see multigpu.column_slices for why not shrinking ones)
    c0, c1 = slices[rank]
    h_q = torch.from_numpy(q).pin_memory()
    h_s = torch.from_numpy(np.ascontiguousarray(s[c0:c1])).pin_memory()
    d_q = h_q.cuda()
    d_s = h_s.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    # the timed steps: ONE alignment at a time over all ranks (one inbox per rank boundary, barrier between steps)
    wave = StripWavefront(al, rank, world, m, dist, depth=1, pairs_per_launch=1)
    torch.cuda.synchronize()
    wave.reset()

    def step_resident():
        flush.zero_()
        if dist is not None:
            dist.barrier()          # every rank has finished the previous alignment
        torch.cuda.synchronize()
        return wave.run(MODE, scoring, d_q.data_ptr(), m, d_s.data_ptr(), c0, c1, n)

    # ---- value: inputs resident in HBM -----------------------------------------
    for _ in range(args.warmup):
        part = step_resident()
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if rank == 0:
        sampler.start()
    t_wall0 = time.perf_counter()
    ev0.record()
    dev_ms, launches = 0.0, 0
    for _ in range(args.steps):
        part = step_resident()
        dev_ms += part.kernel_ms
        launches += part.kernel_launches
    # wave.run() returns after its kernels have finished (the call synchronises its stream), so an event
    # on the idle torch stream is a device timestamp of "this rank's last step is done"
    ev1.record()
    ev1.synchronize()
    span_ms = ev0.elapsed_time(ev1)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    res = wave.combine(MODE, scoring, part)
    if world == 1:
        span_ms = dev_ms           # one rank: the sum of the per-call CUDA-event times (excludes the L2 flush)
    t = torch.tensor([span_ms, t_wall * 1e3, dev_ms], dtype=torch.float64, device="cuda")
    lt = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_ms_max, kern_ms_max = t.tolist()
    ms_per_step = dev_ms_max / args.steps
    value = cells / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: host buffers through the C ABI (H2D of the rank's sequences + D2H of its result inside) -------------
    e2e = None
    if not args.no_e2e:
        e2e_steps = max(1, min(args.steps, 3))

        def step_e2e():
            if world == 1:
                return al.score(MODE, h_q.numpy(), h_s.numpy(), scoring)       # anyseq_score
            if dist is not None:
                dist.barrier()
            p_ = wave.run_host(MODE, scoring, h_q.numpy(), h_s.numpy(), c0, c1, n)    # anyseq_score_strip
            return wave.combine(MODE, scoring, p_)                              # every rank's partial reaches every host

        step_e2e()   # warm-up
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r_e2e = step_e2e()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = tt.item()
        if (r_e2e.score, r_e2e.end_i, r_e2e.end_j) != (res.score, res.end_i, res.end_j):
            raise SystemExit("bench.py: e2e result differs from the resident result")
        e2e = {"value": cells * e2e_steps / dt / 1e9, "unit": "GCUPS",
               "h2d_bytes_per_step": int(m + (c1 - c0)), "d2h_bytes_per_step": 160, "steps": e2e_steps,
               "score": int(r_e2e.score), "api": "anyseq_score (host buffers)" if world == 1 else
               "anyseq_score_strip (host buffers, per rank) + anyseq_strip_combine"}

    # ---- N > 1: a STREAM of alignments (not the headline): several side by side per launch, two inbox sets ----------
    stream = None
    if world > 1 and args.stream_steps != 0:
        ppl = max(1, args.pairs_per_launch)
        nst = args.stream_steps if args.stream_steps > 0 else 2 * ppl
        wave.close()
        wave2 = StripWavefront(al, rank, world, m, dist, depth=2, pairs_per_launch=ppl)
        wave2.reset()

        def launch(k):
            flush.zero_()
            torch.cuda.synchronize()
            if k > 1:
                return wave2.run_multi(MODE, scoring, [d_q.data_ptr()] * k, m, [d_s.data_ptr()] * k, c0, c1, n)
            return [wave2.run(MODE, scoring, d_q.data_ptr(), m, d_s.data_ptr(), c0, c1, n)]

        launch(ppl)      # warm-up
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        left = nst
        while left > 0:
            k = min(ppl, left)
            parts = launch(k)
            left -= k
        e1.record()
        e1.synchronize()
        sp = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(sp, op=dist.ReduceOp.MAX)
        barrier()
        sres = wave2.combine(MODE, scoring, parts[-1])
        stream = {"gcups": cells * nst / (sp.item() * 1e-3) / 1e9, "alignments": nst, "pairs_per_launch": ppl,
                  "score": int(sres.score),
                  "note": "consecutive alignments stream through the ranks back to back (two inbox sets + neighbour run "
                          "tokens), several side by side per launch; the wavefront fill is paid once per stream"}
        wave2.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result_arrays(res.score, res.end_i, res.end_j))

    # ---- parity inside the bench: the frozen CPU result of the FULL-SIZE workload, and the CPU sample scored on the GPU
    gold = golden_c2() if args.scale == 1.0 else None
    golden = None
    if gold is not None and (gold["m"], gold["n"]) == (m, n):
        golden = {"cpu": [gold["score"], gold["end_i"], gold["end_j"]], "gpu": [int(res.score), int(res.end_i), int(res.end_j)],
                  "by": gold["by"], "equal": [gold["score"], gold["end_i"], gold["end_j"]] == [int(res.score), int(res.end_i), int(res.end_j)]}
        if not golden["equal"]:
            raise SystemExit(f"bench.py: full-size result {golden['gpu']} differs from the frozen CPU result {golden['cpu']}")

    # ---- roofline: integer/DPX issue rate measured on this GPU -------------------
    peak_alu, _ = al.measure_int_peak(0)          # VIADDMNMX/VIMNMX3 only, lane-ops/s
    peak_mix7, _ = al.measure_int_peak(2)         # the 7-op all-ALU Gotoh mix, lane-ops/s
    peak_cells_dual, _ = al.measure_int_peak(5)   # the coupled 3 ALU + 3 IMAD cell, cells/s
    cells_per_s_gpu = cells / (ms_per_step * 1e-3) / world
    achieved_ops = cells_per_s_gpu * OPS_PER_CELL_AFFINE
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_peak = info["sm_count"] * 128.0 * sm_mhz * 1e6          # lane-issue slots per second (4 schedulers x 32 lanes)
    alu_peak = info["sm_count"] * 64.0 * sm_mhz * 1e6             # ALU-pipe lane-ops per second (16 lanes x 4 sub-partitions)
    roofline = {
        "bound": "int_alu",
        "achieved": achieved_ops / 1e12, "peak": peak_alu / 1e12, "unit": "Tlaneop/s (int32, per GPU)",
        "frac": achieved_ops / peak_alu,
        # dram__bytes_read.sum + dram__bytes_write.sum of ONE strip-kernel launch at this workload (ncu --set full,
        # profiles/r02_strip_kernel_fullsize_ncu_full.txt): 134.2 MB + 171.3 MB; only valid for N = 1
        "traffic": 305_494_272 if (world == 1 and args.scale == 1.0) else None,
        "traffic_unit": "bytes of DRAM traffic per launch (algorithmic input: m + n = 9.24 MB; the border records live in L2)",
        "ops_per_cell": OPS_PER_CELL_AFFINE,
        "peak_source": "measured live: anyseq_measure_int_peak(kind=0), dependency-free VIADDMNMX/VIMNMX3 loop",
        # the binding roofs of the kernel as built (instruction counts per cell from the SASS of its steady-state loop,
        # tools/sass_stats.py; DESIGN.md 3.1): issue slots (128 lanes/clk/SM) and the ALU pipe (64 lanes/clk/SM)
        "issue_slot_frac": cells_per_s_gpu * ISSUED_PER_CELL / issue_peak,
        "issue_slot_frac_algorithmic_7_ops": cells_per_s_gpu * OPS_PER_CELL_AFFINE / issue_peak,
        "alu_pipe_frac": cells_per_s_gpu * ALU_PER_CELL / alu_peak,
        "instr_per_cell": {"issued": ISSUED_PER_CELL, "alu_pipe": ALU_PER_CELL, "source": "SASS of the unguarded step loop"},
        "peak_gcups_alu7": peak_alu / OPS_PER_CELL_AFFINE / 1e9,
        "peak_gcups_mix7_measured": peak_mix7 / OPS_PER_CELL_AFFINE / 1e9,
        "peak_gcups_dual_pipe_mix": peak_cells_dual / 1e9,
        "frac_of_dual_pipe_mix": (value / world) / (peak_cells_dual / 1e9),
        "hbm": {"achieved_gbs": (305_494_272 / (ms_per_step * 1e-3) / 1e9) if (world == 1 and args.scale == 1.0) else None,
                "peak_gbs": 6452.8, "note": "DRAM traffic of the strip kernel / step time; far below the HBM roofline by design"},
    }

    cpu = None
    parity = None
    if not args.no_cpu:
        threads = os.cpu_count() or 1
        side = int(args.cpu_sample) or 250000
        g, dt, sc_cpu = cpu_baseline(q, s, side, side, threads)
        # the same sample on the GPU: score AND end cell must equal the restated reference CPU path, every run
        r_gpu = al.score(MODE, q[:side], s[:side], scoring)
        parity = {"sample": f"first {min(side, m)} x {min(side, n)} cells", "cpu": list(sc_cpu),
                  "gpu": [int(r_gpu.score), int(r_gpu.end_i), int(r_gpu.end_j)],
                  "equal": list(sc_cpu) == [int(r_gpu.score), int(r_gpu.end_i), int(r_gpu.end_j)]}
        if not parity["equal"]:
            raise SystemExit(f"bench.py: GPU {parity['gpu']} differs from the oracle {parity['cpu']} on the CPU sample")
        # the reference's own team size is 4 threads (src/backend/backend_cpu.impala:13): reported beside it
        side4 = max(1024, side // 2)
        g4, dt4, _ = cpu_baseline(q, s, side4, side4, 4)
        cpu = {"value": g, "unit": "GCUPS", "cores": threads, "kind": "port",
               "sample": f"first {side} x {side} cells of the workload ({dt:.1f} s), restated reference CPU path "
                         f"(1024x1024 block wavefront, scalar inner loop), {threads} threads",
               "reference_team_of_4_threads": {"value": g4, "unit": "GCUPS", "cores": 4,
                                               "sample": f"first {side4} x {side4} cells ({dt4:.1f} s)"}}

    out = {
        "metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": desc + "; semiglobal affine (same=2,diff=-1,gapInit=-2,gapExtend=-1) score-only",
                   "rows": m, "cols": n, "cells_per_step": cells,
                   "partition": (f"ONE pair, {world} column strips, boundary column streamed over NVLink by the kernel "
                                 "(peer stores, no collective); one alignment at a time, barrier between steps") if world > 1 else "1 GPU",
                   "l2": "L2 flushed (256 MiB memset) before every timed step",
                   "timing": ("CUDA events on the library's launch stream, summed over steps" if world == 1 else
                              "CUDA events around the K steps on every rank, max over ranks"),
                   "kernel_ms_per_step_max_over_ranks": kern_ms_max / args.steps},
        "wall_ms_per_step": wall_ms_max / args.steps,
        "score": int(res.score), "end_cell": [int(res.end_i), int(res.end_j)],
        "golden_fullsize": golden, "parity_check": parity, "stream": stream,
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(lt.item()),
        "roofline": roofline, "cpu_baseline": cpu,
        "device": info["name"], "sm_count": info["sm_count"],
    }
    emit(out)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
