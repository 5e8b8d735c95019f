#!/usr/bin/env python
"""kernel time of batch scores with end cells (anyseq_score_batch_ends) on the C4 workload shape (reads 150 vs windows
500, device-resident), against score-only batches and the full-matrix traceback batch (anyseq_align_batch), for byte
and 2-bit packed input; best of three after a warm-up

  tools/gpu_batch_ends_perf.py [npairs]"""
import os, subprocess, sys
import numpy as np, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import anyseq_b200 as A
from anyseq_b200 import capi
from anyseq_b200 import workloads as W

npairs = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
lq, ls = 150, 500
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card}", flush=True)
qd, qo, sd, so = W.read_batch(npairs, lq, ls)
dq, dqo, ds, dso = (torch.from_numpy(x).cuda() for x in (qd, qo, sd, so))
q2, s2 = A.pack2(qd.reshape(npairs, lq)), A.pack2(sd.reshape(npairs, ls))
dq2, ds2 = torch.from_numpy(q2).cuda(), torch.from_numpy(s2).cuda()
pb = capi.PackedBatch(dq2.data_ptr(), ds2.data_ptr(), None, None, None, None, lq, ls, q2.shape[1], s2.shape[1], npairs)
scores = torch.zeros(npairs, dtype=torch.int32, device="cuda")
ref = torch.zeros(npairs, dtype=torch.int32, device="cuda")
ends = torch.zeros(2 * npairs, dtype=torch.int32, device="cuda")
aends = torch.zeros(2 * npairs, dtype=torch.int32, device="cuda")
total = npairs * (lq + ls)
oq = torch.zeros(total, dtype=torch.uint8, device="cuda")
os_ = torch.zeros(total, dtype=torch.uint8, device="cuda")
al = A.Aligner()
cells = float(lq) * ls * npairs
P = lambda t: t.data_ptr()     # noqa: E731


def best(fn):
    fn()                                    # warm-up
    return min(fn().kernel_ms for _ in range(3))


for mode in ("global", "semiglobal", "local"):
    for sch in (A.linear_scoring_scheme(), A.affine_scoring_scheme()):
        t_score = best(lambda: al.score_batch_device(mode, P(dq), P(dqo), P(ds), P(dso), npairs, P(ref), sch))
        t_ends = best(lambda: al.score_batch_ends_device(mode, P(dq), P(dqo), P(ds), P(dso), npairs, P(scores), P(ends), sch))
        assert torch.equal(scores, ref), (mode, sch)
        t_align = best(lambda: al.align_batch_device(mode, P(dq), P(dqo), P(ds), P(dso), npairs, P(scores), P(aends), 0,
                                                     P(oq), P(os_), sch))
        same_ends = torch.equal(ends, aends)
        t_p2 = best(lambda: al.score_batch_packed2(mode, pb, P(ref), sch, device=True))
        t_p2e = best(lambda: al.score_batch_packed2(mode, pb, P(scores), sch, device=True, ends=P(aends)))
        assert torch.equal(scores, ref) and torch.equal(ends, aends), (mode, sch)
        g = lambda t: cells / t / 1e6        # noqa: E731  GCUPS
        print(f"{mode:10s} affine={int(sch.affine)} | bytes: score {t_score:8.2f} ms {g(t_score):7.1f} GCUPS, "
              f"ends {t_ends:8.2f} ms {g(t_ends):7.1f} GCUPS ({t_score / t_ends:.3f}x), align_batch {t_align:8.2f} ms "
              f"(ends {npairs / t_ends * 1e3:.3g} pairs/s = {t_align / t_ends:.2f}x align_batch, same ends: {same_ends}) | "
              f"2-bit: score {t_p2:8.2f} ms, ends {t_p2e:8.2f} ms ({t_p2 / t_p2e:.3f}x)", flush=True)
