#!/usr/bin/env python
"""Timeline of ONE training step as it really ran on the GPU (drvae_trace_begin / _end: every kernel stamps the
global timer at its first CTA's start and its last CTA's end).  Workload: bench.py's default ensemble shard.

    python tools/trace_step.py [--models 32] [--kind drvae] > profiles/rNN_trace.txt
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from drvae_b200.init import init_state_dict  # noqa: E402
from drvae_b200.plan import Plan, anneal_coef  # noqa: E402
from drvae_b200.synth import synthetic_batch  # noqa: E402

README = dict(dim_x=978, dim_y=2, dim_z1=100, dim_z3=100, enc_z1=[800], dec_x=[600], enc_z3=[200], dec_z1=[200])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--models", type=int, default=32)
    ap.add_argument("--kind", default="drvae")
    ap.add_argument("--batch", type=int, default=150)
    args = ap.parse_args()
    M = args.models
    plan = Plan(args.kind, L=2, max_batch=args.batch, n_models=M, **README)
    fields = {"drvae": ("x1", "x2", "y", "has_x2", "has_y"), "pvae": ("x1", "x2", "has_x2"), "vfae": ("x1", "y", "has_y")}[args.kind]
    host = {k: [] for k in fields}
    for m in range(M):
        plan.load_state_dict(init_state_dict(args.kind, seed=1000 + m, **README), model=m)
        b = synthetic_batch(args.batch, README["dim_x"], seed=m)
        for k in fields:
            host[k].append(b[k])
    devb = {k: torch.stack(v).contiguous().cuda() for k, v in host.items()}
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for it in range(5):
            plan.train_step(devb, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=0)
        torch.cuda.synchronize()
        plan.trace_begin()
        for it in range(5, 8):
            plan.train_step(devb, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=0)
        rec = plan.trace_end()
    plan.dwa_stats(True)
    with torch.cuda.stream(s):
        for it in range(8, 12):
            plan.train_step(devb, plan.hparams(step=it, beta_pert=anneal_coef(it, 1, 0)), seed=0)
    st = plan.dwa_stats(False)
    tot = max(1, st["cta_total"])
    print("# grouped dW+Adam role waits, fraction of CTA time (4 steps): " + ", ".join("%s %.3f" % (k, v / tot) for k, v in st.items() if k != "cta_total")
          + "; CTA cycles per launch and CTA %.0f" % (tot / 4 / 148))
    per = len(rec) // 3
    step = rec[2 * per:]  # the third traced step
    t0 = min(r[2] for r in step)
    t1 = max(r[3] for r in step)
    print("# %s, %d models x %d rows, one step: %d launches, %.1f us from first kernel start to last kernel end" % (
        args.kind, M, args.batch, len(step), (t1 - t0) / 1e3))
    print("# %-4s %-34s %10s %10s %9s" % ("idx", "kernel", "start_us", "end_us", "dur_us"))
    busy = 0
    for i, tag, a, b in sorted(step, key=lambda r: r[2]):
        print("  %-4d %-34s %10.1f %10.1f %9.1f" % (i - step[0][0], tag, (a - t0) / 1e3, (b - t0) / 1e3, (b - a) / 1e3))
        busy += b - a
    print("# sum of kernel durations %.1f us" % (busy / 1e3))


if __name__ == "__main__":
    main()
