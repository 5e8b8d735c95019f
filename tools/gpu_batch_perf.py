#!/usr/bin/env python
"""throughput of the batch kernel on the C4 workload shape (reads 150 vs windows 500)

  tools/gpu_batch_perf.py [npairs [window length, default 500]]"""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import anyseq_b200 as A
from anyseq_b200 import workloads as W
npairs = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
wlen = int(sys.argv[2]) if len(sys.argv) > 2 else 500
qd, qo, sd, so = W.read_batch(npairs, 150, wlen)
dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
out = torch.zeros(npairs, dtype=torch.int32, device="cuda")
al = A.Aligner()
cells = 150.0 * wlen * npairs
for mode in ("global", "semiglobal", "local"):
    for sch in (A.affine_scoring_scheme(), A.linear_scoring_scheme()):
        best = 1e30
        for rep in range(3):
            r = al.score_batch_device(mode, dq.data_ptr(), dqo.data_ptr(), ds.data_ptr(), dso.data_ptr(), npairs, out.data_ptr(), sch)
            best = min(best, r.kernel_ms)
        print(f"batch {npairs} pairs {mode} affine={sch.affine}: {best:.2f} ms {cells/best/1e6:.1f} GCUPS checksum={int(out.to(torch.int64).sum())}", flush=True)

# end to end through the host entry point (pageable caller memory -> pinned chunk pipeline -> scores)
if os.environ.get("E2E", "1") != "0":
    tile = int(os.environ.get("TILE", "1"))          # C4 at full size: 10^7 pairs = 10 x the generated 10^6
    if tile > 1:
        qd, sd = np.tile(qd, tile), np.tile(sd, tile)
        qo = np.arange(npairs * tile + 1, dtype=np.int64) * 150
        so = np.arange(npairs * tile + 1, dtype=np.int64) * wlen
    n_all = npairs * tile
    sch = A.affine_scoring_scheme()
    for threads in (1, 4, 8):
        al.set_option("batch_copy_threads", threads)
        best = 1e30
        for rep in range(3):
            t0 = time.perf_counter()
            sc, r = al.score_batch("semiglobal", qd, qo, sd, so, sch)
            best = min(best, time.perf_counter() - t0)
        print(f"host e2e {n_all} pairs semiglobal affine, {threads} staging threads: {best*1e3:.1f} ms wall "
              f"{150.0*wlen*n_all/best/1e9:.1f} GCUPS (kernels {r.kernel_ms:.1f} ms, {r.kernel_launches} launches, "
              f"H2D {(qd.nbytes+sd.nbytes+qo.nbytes+so.nbytes)/best/1e9:.1f} GB/s) checksum={int(sc.astype(np.int64).sum())}", flush=True)
