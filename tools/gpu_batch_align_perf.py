#!/usr/bin/env python
"""throughput of the batch full-matrix traceback (anyseq_align_batch_device) on the C4 workload shape
(reads 150 vs windows 500), against score-only batches and a per-pair anyseq_align_full loop

  tools/gpu_batch_align_perf.py [npairs]"""
import os, subprocess, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import anyseq_b200 as A
from anyseq_b200 import workloads as W
from oracle import oracle as O

npairs = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
lq, ls = 150, 500
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}", flush=True)
qd, qo, sd, so = W.read_batch(npairs, lq, ls)
dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
total = npairs * (lq + ls)
scores = torch.zeros(npairs, dtype=torch.int32, device="cuda")
ref = torch.zeros(npairs, dtype=torch.int32, device="cuda")
ends = torch.zeros(2 * npairs, dtype=torch.int32, device="cuda")
starts = torch.zeros(2 * npairs, dtype=torch.int32, device="cuda")
oq = torch.zeros(total, dtype=torch.uint8, device="cuda")
os_ = torch.zeros(total, dtype=torch.uint8, device="cuda")
al = A.Aligner()
O.build()
cells = float(lq) * ls * npairs
for mode in ("global", "semiglobal", "local"):
    for sch in (A.linear_scoring_scheme(), A.affine_scoring_scheme()):
        best = 1e30
        for rep in range(3):
            r = al.align_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), npairs,
                                      scores.data_ptr(), ends.data_ptr(), starts.data_ptr(), oq.data_ptr(),
                                      os_.data_ptr(), sch)
            best = min(best, r.kernel_ms)
        sbest = 1e30
        for rep in range(3):
            r = al.score_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), npairs,
                                      ref.data_ptr(), sch)
            sbest = min(sbest, r.kernel_ms)
        chk = int(scores.to(torch.int64).sum())
        sref = int(ref.to(torch.int64).sum())
        fnv = O.fnv1a64(np.concatenate([oq.cpu().numpy(), os_.cpu().numpy()]))
        # per-pair baseline: anyseq_align_full over the first 1000 pairs
        nb = min(1000, npairs)
        t0 = time.perf_counter()
        for p in range(nb):
            al.align_full(mode, qd[p * lq:(p + 1) * lq], sd[p * ls:(p + 1) * ls], sch)
        per_pair = (time.perf_counter() - t0) / nb
        pps = npairs / (best / 1e3)
        print(f"align_batch {npairs} pairs {mode} affine={sch.affine}: {best:.2f} ms {cells / best / 1e6:.1f} GCUPS "
              f"{pps:.3g} pairs/s checksum={chk} rows_fnv={fnv:016x} | score_batch {sbest:.2f} ms checksum={sref} "
              f"({'equal' if sref == chk else 'DIFFERENT'}), traceback/score time {best / sbest:.2f}x | align_full loop "
              f"{1 / per_pair:.0f} pairs/s, batch {pps * per_pair:.0f}x", flush=True)
        assert sref == chk
