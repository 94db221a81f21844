"""Similar items / users (primalcr_similar, cosine) on one GPU against a torch composition on the same card.

    python tools/similar_bench.py --outdir profiles [--shapes netflix_items netflix_users yahoo_items] [--reps 3]

Shapes (k = 100, seeded N(0,1) factors, no exclusion):
  * netflix_items: 17,770 x 100, every item a query, N = 10 and 100;
  * netflix_users: 480,189 x 100 (384 MB, more than L2), a seeded sample of 50,000 users as queries, N = 10 and 100;
  * yahoo_items:   625,000 x 100, every item a query, N = 10.
For each shape and N, written to <outdir>/similar_<shape>.json:
  * wall_s: host clock around the synchronous library call (validation, upload, kernels, copy back), warm;
  * kernel_ms: device time of the call's kernels (row_norms + similar_kernel, whose device symbol is
    pcr::topn_kernel<NMAX, UG, CAP, true, true>) from torch.profiler's CUDA activities, in a pass of its own;
    tflops = 2 * n_queries * n * k / kernel time (fp64, achieved; no peak is claimed);
  * torch_ms: CUDA events around the torch composition with M already on the device: rows normalised, query blocks of
    Mn[q] @ Mn.T (cuBLAS fp64), each query's own row set to -inf, torch.topk; alternated with the library call;
  * exact_id_match: the fraction of positions where the two id lists agree, and agree_positions, where a differing id
    still counts when the two scores are within 1e-12 (near ties may swap places between the two roundings);
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

SHAPES = {
    "netflix_items": dict(n=17_770, queries=None, topn=(10, 100)),
    "netflix_users": dict(n=480_189, queries=50_000, topn=(10, 100)),
    "yahoo_items": dict(n=625_000, queries=None, topn=(10,)),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    keys = [s.strip() for s in q[0].split(",")]
    return [dict(zip(keys, (s.strip() for s in line.split(",")))) for line in q[1:]][0]


def torch_similar(Mn, q, n, block):
    items = torch.empty((len(q), n), dtype=torch.int64, device="cuda")
    scores = torch.empty((len(q), n), dtype=torch.float64, device="cuda")
    for b0 in range(0, len(q), block):
        qb = q[b0:b0 + block]
        S = Mn[qb] @ Mn.T
        S[torch.arange(len(qb), device="cuda"), qb] = -float("inf")
        v, i = torch.topk(S, n, dim=1)
        items[b0:b0 + block] = i; scores[b0:b0 + block] = v
        del S
    return items, scores


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for e in prof.key_averages():
        if "topn_kernel" in e.key or "row_norms" in e.key:     # similar_kernel is topn_kernel<..., SELF, COS> on the device
            t = getattr(e, "device_time_total", None)
            total += t if t is not None else e.cuda_time_total
    return total / 1e3


def run_shape(name, cfg, k, reps, seed):
    rng = np.random.default_rng(seed)
    n = cfg["n"]
    M = rng.standard_normal((n, k))
    q = None if cfg["queries"] is None else np.sort(rng.choice(n, size=cfg["queries"], replace=False)).astype(np.int32)
    nq = n if q is None else len(q)
    Mg = torch.from_numpy(M).cuda()
    Mn = Mg / Mg.norm(dim=1, keepdim=True)
    qg = torch.arange(n, device="cuda") if q is None else torch.from_numpy(q.astype(np.int64)).cuda()
    block = max(1, min(nq, int(16e9 // (8 * n))))        # 16 GB of scores per cuBLAS block
    flop = 2.0 * nq * n * k
    res = dict(shape=name, n=n, k=k, n_queries=nq, measure="cosine", torch_block=block, runs=[])
    for topn in cfg["topn"]:
        call = lambda: api.similar(M, topn, measure="cosine", queries=q)     # noqa: E731
        call()                                                               # warm-up of the same shape
        torch_similar(Mn, qg, topn, block); torch.cuda.synchronize()
        lib_wall, torch_ms = [], []
        for _ in range(reps):                                                # alternate the two
            t0 = time.perf_counter(); ids, sc = call(); lib_wall.append(time.perf_counter() - t0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ti, ts = torch_similar(Mn, qg, topn, block)
            e1.record(); torch.cuda.synchronize(); torch_ms.append(e0.elapsed_time(e1))
        kms = [kernel_ms(call) for _ in range(2)]
        idg = torch.from_numpy(ids.astype(np.int64)).cuda(); scg = torch.from_numpy(sc).cuda()
        same = idg == ti
        agree = same | ((scg - ts).abs() <= 1e-12)
        run = dict(topn=topn, wall_s=lib_wall, kernel_ms=kms, tflops=flop / (min(kms) * 1e-3) / 1e12, torch_ms=torch_ms,
                   speedup_kernel_vs_torch=min(torch_ms) / min(kms), exact_id_match=float(same.double().mean()),
                   rows_identical=float(same.all(1).double().mean()), agree_positions=float(agree.double().mean()))
        res["runs"].append(run)
        print(name, json.dumps(run), flush=True)
        del idg, scg, ti, ts
    del Mg, Mn
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--outdir", required=True)
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES), choices=list(SHAPES))
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("similar_bench needs a CUDA device")
    os.makedirs(a.outdir, exist_ok=True)
    for i, name in enumerate(a.shapes):
        res = run_shape(name, SHAPES[name], a.k, a.reps, seed=20261022 + i)
        res["gpu"] = gpu_info()
        with open(os.path.join(a.outdir, "similar_%s.json" % name), "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res["gpu"]), flush=True)


if __name__ == "__main__":
    main()
