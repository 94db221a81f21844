"""Top-N recommendation at Netflix shape on one GPU: primalcr_recommend against torch (cuBLAS fp64 + torch.topk).

    python tools/recommend_bench.py --out result.json [--n 10 100] [--reps 3]

Workload: synth_dataset("netflix") (480,189 users x 17,770 items, 1e8 training ratings), k = 100, seeded N(0,1) factors,
every user, the training set excluded.  For each N it reports
  * wall_s: host clock around the synchronous library call (validation, copies, kernel), warm (one untimed call first);
  * kernel_ms: the topn_kernel time from torch.profiler with CUDA activities, in a separate pass;
  * tflops: 2 * n_users * d2 * k / kernel time (fp64, achieved; no peak is claimed);
  * torch_s: the same selection composed from torch on the same GPU, U / V / exclusion already resident: user blocks of
    U_blk @ V.T (cuBLAS fp64), excluded entries set to -inf, torch.topk; timed alternately with the library call;
  * agreement of the two item lists, position by position, where a differing item counts as agreeing when the two scores
    are within 1e-12 * |U[u]| * max_i |V[i]| (a bound of the row's largest |score|; near ties may swap places);
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    keys = [s.strip() for s in q[0].split(",")]
    return [dict(zip(keys, (s.strip() for s in line.split(",")))) for line in q[1:]][0]


def torch_topn(Ug, Vg, n, user_of, item_g, row_ptr, block):
    d1 = Ug.shape[0]
    items = torch.empty((d1, n), dtype=torch.int64, device="cuda")
    scores = torch.empty((d1, n), dtype=torch.float64, device="cuda")
    for b0 in range(0, d1, block):
        b1 = min(d1, b0 + block)
        S = Ug[b0:b1] @ Vg.T
        e0, e1 = int(row_ptr[b0]), int(row_ptr[b1])
        S[user_of[e0:e1] - b0, item_g[e0:e1]] = -float("inf")
        v, i = torch.topk(S, n, dim=1)
        items[b0:b1] = i; scores[b0:b1] = v
        del S
    return items, scores


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        if "topn_kernel" in e.key:
            t = getattr(e, "device_time_total", None)
            total += t if t is not None else e.cuda_time_total
    return total / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, nargs="+", default=[10, 100])
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--block", type=int, default=32768, help="users per cuBLAS block of the torch composition")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_bench needs a CUDA device")
    info = gpu_info()
    ds = synth_dataset("netflix", scale=a.scale, device="cuda")
    X = ds.train
    rng = np.random.default_rng(20240601)
    U = rng.standard_normal((X.d1, a.k)); V = rng.standard_normal((X.d2, a.k))
    Ug = torch.from_numpy(U).cuda(); Vg = torch.from_numpy(V).cuda()
    item_g = torch.from_numpy(X.item.astype(np.int64)).cuda()
    user_of = torch.from_numpy(X.users()).cuda()
    flop = 2.0 * X.d1 * X.d2 * a.k
    res = dict(shape="netflix", scale=a.scale, d1=X.d1, d2=X.d2, k=a.k, nnz_excluded=X.nnz, gpu=info, runs=[])
    for n in a.n:
        api.recommend(U, V, n, exclude=X)                                  # warm-up of the same shape
        torch_topn(Ug, Vg, n, user_of, item_g, X.row_ptr, a.block); torch.cuda.synchronize()
        lib_wall, torch_wall = [], []
        for _ in range(a.reps):                                          # alternate the two
            t0 = time.perf_counter(); it, sc = api.recommend(U, V, n, exclude=X); lib_wall.append(time.perf_counter() - t0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ti, ts = torch_topn(Ug, Vg, n, user_of, item_g, X.row_ptr, a.block)
            torch.cuda.synchronize(); torch_wall.append(time.perf_counter() - t0)
        kms = [kernel_ms(lambda: api.recommend(U, V, n, exclude=X)) for _ in range(2)]
        itg = torch.from_numpy(it.astype(np.int64)).cuda(); scg = torch.from_numpy(sc).cuda()
        # |U[u].V[i]| <= |U[u]| max_i |V[i]|: a bound of the row's largest |score|, so the tolerance is slightly loose
        tol = 1e-12 * (Ug.norm(dim=1) * Vg.norm(dim=1).max())[:, None]
        agree = (itg == ti) | ((scg - ts).abs() <= tol)
        run = dict(n=n, wall_s=lib_wall, kernel_ms=kms, tflops=flop / (min(kms) * 1e-3) / 1e12,
                   torch_s=torch_wall, speedup_kernel_vs_torch=min(torch_wall) / (min(kms) * 1e-3),
                   agree_positions=float(agree.double().mean()), agree_rows=float(agree.all(1).double().mean()),
                   exact_item_match=float((itg == ti).double().mean()))
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
