"""Held-out ranking evaluation at Netflix shape on one GPU: primalcr_rank_heldout against a torch composition.

    python tools/rankeval_bench.py --out result.json [--reps 3] [--scale 1.0]

Workload: synth_dataset("netflix") (480,189 users x 17,770 items, 1e8 training ratings, 10 held-out ratings per user with
at least 20), k = 100, the training set excluded, two sets of factors:
  * "trained": the reference init after 3 Primal-CR++ outer iterations through the library (lambda 5000);
  * "random": seeded N(0,1) factors, where held-out items rank uniformly and most candidates take the histogram path.
The synthetic set picks which items a user rates from item popularity alone, independent of the ratings' ground truth,
so a model of the ratings ranks held-out items mid-catalog too (AUC near 0.5, reported with the metrics): on this data
the trained factors do not reach the case where most candidates beat no held-out entry.
For each it reports
  * wall_s: host clock around the synchronous library call (validation, copies, kernel), warm (one untimed call first);
  * kernel_ms: the rank_kernel time from torch.profiler with CUDA activities, in a separate pass;
  * tflops: 2 * units * d2 * k / kernel time (fp64, achieved; a unit is a user and up to 64 of its held-out entries);
  * torch_s: the ranks composed from torch on the same GPU, U / V / exclusion / held-out set already resident: user
    blocks of U_blk @ V.T (cuBLAS fp64), excluded entries set to -inf, rank = 1 + the number of row entries greater than
    the held-out score; timed alternately with the library call;
  * agreement with torch: a rank may differ only inside the near-tie window [1 + #(S > h + tol), #(S >= h - tol)], with
    tol = 1e-12 * |U[u]| * max_i |V[i]| (a bound of the row's largest |score|);
  * the card's name, power limit and maximum SM clock from nvidia-smi, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from primalcr_b200 import api  # noqa: E402
from primalcr_b200.data import synth_dataset  # noqa: E402

UNIT = 64      # held-out entries per unit of rank_kernel (pcr::RANK_UNIT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    keys = [s.strip() for s in q[0].split(",")]
    return [dict(zip(keys, (s.strip() for s in line.split(",")))) for line in q[1:]][0]


class TorchRanks:
    """The held-out ranks from cuBLAS fp64 scores in user blocks, everything resident on the GPU."""

    def __init__(self, X, T, block):
        self.X, self.T, self.block = X, T, block
        self.x_user = torch.from_numpy(X.users()).cuda(); self.x_item = torch.from_numpy(X.item.astype(np.int64)).cuda()
        self.t_user = torch.from_numpy(T.users()).cuda(); self.t_item = torch.from_numpy(T.item.astype(np.int64)).cuda()
        self.t_j = torch.from_numpy(np.arange(T.nnz) - np.repeat(T.row_ptr[:-1], T.lens())).cuda()
        self.maxlen = int(T.lens().max())

    def blocks(self, Ug, Vg):
        X, T = self.X, self.T
        for b0 in range(0, Ug.shape[0], self.block):
            b1 = min(Ug.shape[0], b0 + self.block)
            e0, e1 = int(T.row_ptr[b0]), int(T.row_ptr[b1])
            if e0 == e1:
                continue
            S = Ug[b0:b1] @ Vg.T
            eu = self.t_user[e0:e1] - b0; ej = self.t_j[e0:e1]
            h = S[eu, self.t_item[e0:e1]]
            x0, x1 = int(X.row_ptr[b0]), int(X.row_ptr[b1])
            S[self.x_user[x0:x1] - b0, self.x_item[x0:x1]] = -float("inf")
            Hb = torch.full((b1 - b0, self.maxlen), float("inf"), dtype=torch.float64, device="cuda")
            Hb[eu, ej] = h
            yield b0, e0, e1, eu, ej, S, Hb

    def ranks(self, Ug, Vg):
        out = torch.empty(self.T.nnz, dtype=torch.int64, device="cuda")
        for _, e0, e1, eu, ej, S, Hb in self.blocks(Ug, Vg):
            cnt = (S[:, None, :] > Hb[:, :, None]).sum(-1)
            out[e0:e1] = 1 + cnt[eu, ej]
        return out

    def agreement(self, Ug, Vg, lib_ranks):
        r = torch.from_numpy(lib_ranks.astype(np.int64)).cuda()
        tr = self.ranks(Ug, Vg)
        ok = torch.empty(self.T.nnz, dtype=torch.bool, device="cuda")
        vmax = Vg.norm(dim=1).max()
        for b0, e0, e1, eu, ej, S, Hb in self.blocks(Ug, Vg):
            tol = (1e-12 * Ug[b0:b0 + S.shape[0]].norm(dim=1) * vmax)[:, None, None]
            lo = 1 + (S[:, None, :] > Hb[:, :, None] + tol).sum(-1)
            hi = (S[:, None, :] >= Hb[:, :, None] - tol).sum(-1)
            rr = r[e0:e1]
            ok[e0:e1] = (rr == tr[e0:e1]) | ((lo[eu, ej] <= rr) & (rr <= hi[eu, ej]))
        return float((r == tr).double().mean()), float(ok.double().mean())


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        if "rank_kernel" in e.key:
            t = getattr(e, "device_time_total", None)
            total += t if t is not None else e.cuda_time_total
    return total / 1e3


def trained_factors(ds, k, lam, iters):
    U = api.reference_init(ds.d1, k); V = api.reference_init(ds.d2, k)
    e = api.Engine(api.Parameter(solver_type=api.PCRPP, k=k, lambda_=lam, maxiter=iters, do_predict=0))
    try:
        e.set_train(ds.train); e.set_factors(U, V)
        e.initial_objective()
        for _ in range(iters):
            e.outer_iteration()
        return e.get_factors()
    finally:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--iters", type=int, default=3, help="Primal-CR++ outer iterations of the trained factors")
    ap.add_argument("--block", type=int, default=4096, help="users per cuBLAS block of the torch composition")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rankeval_bench needs a CUDA device")
    info = gpu_info()
    ds = synth_dataset("netflix", scale=a.scale, device="cuda")
    X, T = ds.train, ds.test
    units = int(np.sum((T.lens() + UNIT - 1) // UNIT))
    flop = 2.0 * units * X.d2 * a.k
    tr = TorchRanks(X, T, a.block)
    rng = np.random.default_rng(20240601)
    factor_sets = [("trained", lambda: trained_factors(ds, a.k, 5000.0, a.iters)),
                   ("random", lambda: (rng.standard_normal((X.d1, a.k)), rng.standard_normal((X.d2, a.k))))]
    res = dict(shape="netflix", scale=a.scale, d1=X.d1, d2=X.d2, k=a.k, nnz_excluded=X.nnz, nnz_heldout=T.nnz,
               units=units, gpu=info, runs=[])
    for name, make in factor_sets:
        U, V = make()
        U = np.ascontiguousarray(U); V = np.ascontiguousarray(V)
        Ug = torch.from_numpy(U).cuda(); Vg = torch.from_numpy(V).cuda()
        api.heldout_ranks(U, V, T, exclude=X)                              # warm-up of the same shape
        tr.ranks(Ug, Vg); torch.cuda.synchronize()
        lib_wall, torch_wall = [], []
        for _ in range(a.reps):                                          # alternate the two
            t0 = time.perf_counter(); r, _ = api.heldout_ranks(U, V, T, exclude=X); lib_wall.append(time.perf_counter() - t0)
            torch.cuda.synchronize()
            t0 = time.perf_counter(); tr.ranks(Ug, Vg); torch.cuda.synchronize(); torch_wall.append(time.perf_counter() - t0)
        kms = [kernel_ms(lambda: api.heldout_ranks(U, V, T, exclude=X)) for _ in range(2)]
        exact, agree = tr.agreement(Ug, Vg, r)
        m = api.ranking_metrics(r, T, exclude=X, cutoffs=(10, 100))
        run = dict(factors=name, wall_s=lib_wall, kernel_ms=kms, tflops=flop / (min(kms) * 1e-3) / 1e12, torch_s=torch_wall,
                   speedup_kernel_vs_torch=min(torch_wall) / (min(kms) * 1e-3), agree_entries=agree,
                   exact_rank_match=exact, median_rank=float(np.median(r)), metrics=m)
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
        del Ug, Vg
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
