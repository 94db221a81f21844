#!/usr/bin/env python
"""A/B measurement helper (never a bench number): one engine on the named shape, `--warmup` untimed outer iterations,
then `--iters` iterations timed with CUDA events on the engine's stream and the per-kernel CUDA-event table.  The variant
is the library PRIMALCR_LIB names (default: the in-tree build); `--tag` labels the JSON line."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="netflix")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--lam", type=float, default=5000.0)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=2)
    ap.add_argument("--tag", default="")
    ap.add_argument("--top", type=int, default=14)
    args = ap.parse_args()
    import torch
    from primalcr_b200 import api
    from primalcr_b200.data import synth_dataset
    ds = synth_dataset(args.workload, scale=args.scale, device="cuda", test_per_user=0)
    torch.cuda.empty_cache()
    U = api.reference_init(ds.d1, args.k)
    V = U[:ds.d2].copy() if ds.d2 <= ds.d1 else api.reference_init(ds.d2, args.k)
    e = api.Engine(api.Parameter(solver_type=2, k=args.k, lambda_=args.lam, maxiter=1, do_predict=0))
    e.set_levels(np.arange(1, 6))
    e.set_train(ds.train); e.set_factors(U, V)
    objs = [e.initial_objective()]
    for _ in range(args.warmup):
        objs.append(e.outer_iteration())
    stream = torch.cuda.ExternalStream(e.stream_ptr(), device=torch.device("cuda", 0))
    e.profile_enable(True); e.profile_reset()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    for _ in range(args.iters):
        objs.append(e.outer_iteration())
    ev1.record(stream)
    torch.cuda.synchronize()
    sec = ev0.elapsed_time(ev1) / 1e3 / args.iters
    prof = e.profile(); e.profile_enable(False)
    kern = sorted(((v["ms"] / args.iters, n, v["launches"] / args.iters) for n, v in prof.items()), reverse=True)
    out = dict(tag=args.tag, env={k: v for k, v in os.environ.items() if k.startswith("PRIMALCR_")}, workload=args.workload,
               scale=args.scale, k=args.k, nnz=ds.train.nnz, sec_per_iter=sec, objective=objs, counters=e.counters(),
               kernels={n: [round(ms, 3), l] for ms, n, l in kern[:args.top]},
               kernel_ms_total=round(sum(ms for ms, _, _ in kern), 2))
    e.close()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
