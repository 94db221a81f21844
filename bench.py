#!/usr/bin/env python
"""bench.py -- seconds per Primal-CR++ outer iteration (update_V + update_U), k=100, Netflix-shape synthetic.

    python bench.py --gpus N --steps K --warmup W            # our B200 path   (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU implementation

One JSON line on stdout (rank 0).  A "step" is one outer iteration over the whole (sharded) rating set:
  value  = device-timed seconds per outer iteration with ratings/factors resident in HBM (max over ranks), iterations
           W+1 .. W+K from the reference init (the driver's window);
  e2e    = the same metric through the reference-facing call (host CSR + host U,V in, W+K iterations from the same init,
           host U,V out), host<->device copies and the one-time CSR/CSC preparation inside the timed region, divided by
           W+K; `e2e.device_same_window` is the device-timed mean over the SAME iterations 1 .. W+K, so
           e2e.value - e2e.device_same_window is exactly what the copies and the setup cost per iteration;
           `e2e.shim` is the call through the real C++ drop-in (reference containers in pageable memory, oracle/shim_e2e.cpp);
  roofline      = dominant kernel's algorithmic bytes / CUDA-event time vs the measured HBM peak (`frac_kind`
                  "algorithmic_vs_hbm": it exceeds 1 when the gathered rows come from L2), with the ncu DRAM bytes and L2
                  counters of the same kernel beside it (profiles/r02_traffic.json, regenerated from this round's capture);
  cpu_baseline  = the reference's race-free `omp-pmf-train-rf` (oracle/_ref) on two bounded user samples, extrapolated with
                  the affine model t(n) = a + b n they determine (the plain nnz-ratio figure is kept as `linear_value`);
  parity        = the engine vs the unmodified reference (race-free harness) on the first ~2 M ratings of the same data.

--dump-outputs DIR writes what the timed path returned after its last step (objective, counters, U and V; rows of a
factor larger than its budget are a fixed seeded sample, indices beside them) as DIR/*.npy, so two builds can be compared
output for output: the workload and the init are deterministic functions of the arguments.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the tree may be read-only: nothing of a bench run lands in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sec_per_outer_iter_primalcrpp_k100_netflix_shape"
_REAL_STDOUT = None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        self.ready = threading.Event()
        self.window = [None, None]      # perf_counter bounds of the timed region

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "hw_power_brake": 0x80}
            self.ready.set()
            while not self.stop_flag:
                now = time.perf_counter()
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((now, mhz, r))
                time.sleep(0.02)
        except Exception as ex:      # pragma: no cover - NVML missing
            self.reasons.add("nvml_unavailable:%s" % type(ex).__name__)
            self.ready.set()
        self.names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20,
                      "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80}

    def summary(self):
        t0, t1 = self.window
        inside = [s for s in self.samples if t0 is None or (t0 <= s[0] <= t1)] or self.samples[-1:]
        for _, _, r in inside:
            for n, bit in getattr(self, "names", {}).items():
                if r & bit:
                    self.reasons.add(n)
        return {"sm_mhz": float(np.median([s[1] for s in inside])) if inside else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(inside)}


# --------------------------------------------------------------------------------------------- workload

def make_workload(args, device):
    from primalcr_b200.data import synth_dataset
    t = time.time()
    ds = synth_dataset(args.workload, scale=args.scale, device=device, test_per_user=0)
    log("[bench] %s: d1=%d d2=%d nnz=%d (max len %d) generated on %s in %.1fs" % (
        ds.name, ds.d1, ds.d2, ds.train.nnz, int(ds.train.lens().max()), device, time.time() - t))
    return ds


def reference_init_cached(n, k):
    from primalcr_b200 import api
    return api.reference_init(n, k)


# --------------------------------------------------------------------------------------------- CPU reference arm

# the race-free build (obj_u_new made loop-local, oracle/Makefile): with -n > 1 the stock binary's line search reads
# another thread's objective (pcrpp.cpp:822-832), so its work per iteration is not reproducible
REF_EXE = "omp-pmf-train-rf"
# measured on the GPU box's 16 host cores (round 1): ~1.6e-6 s per rating and iteration at k=100
REF_SEC_PER_RATING_ITER_16C = 1.6e-6


def reference_sample_nnz(args, iters, nnz, budget_s):
    """Ratings in the reference's timing sample: 10 % of the workload (SURVEY 8d) unless `iters` iterations of it would
    not finish within `budget_s`; never below 2 M."""
    if args.ref_sample_nnz > 0:
        return min(args.ref_sample_nnz, nnz)
    cores = os.cpu_count() or 1
    per = REF_SEC_PER_RATING_ITER_16C * 16.0 / min(cores, 16) * (args.k / 100.0)
    fit = int(budget_s / max(iters, 1) / per)
    return int(min(nnz, max(2_000_000, min(nnz // 10, fit))))


def run_reference_cli(ds_sample, k, lam, iters, threads):
    """Times the reference's own omp-pmf-train (oracle/_ref) on `ds_sample`; returns per-iteration seconds."""
    from primalcr_b200.data import write_reference_dir
    exe = os.path.join(ROOT, "oracle", "_ref", REF_EXE)
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "data")
        write_reference_dir(d, ds_sample)
        cmd = [exe, "-s", "2", "-k", str(k), "-l", str(lam), "-t", str(iters), "-p", "0", "-n", str(threads), d,
               os.path.join(tmp, "model")]
        out = subprocess.run(cmd, cwd=tmp, capture_output=True, text=True, check=True).stdout
    times = [float(m.group(2)) for m in re.finditer(r"^Iter (\d+) time (\S+) obj", out, re.M)]
    return np.diff(np.array(times)), out       # times[0] is "Iter 0 time 0"


def run_oracle_port(ds_sample, k, lam, iters):
    from oracle import bindings as ob
    from primalcr_b200 import api
    R = ds_sample.train
    X = ob.Csr(R.d1, R.d2, R.row_ptr, R.item.astype(np.int64), R.rating)
    U = api.reference_init(R.d1, k); V = api.reference_init(R.d2, k)
    per = []
    O = ob.oracle()
    for _ in range(iters):
        t = time.time()
        res = O.train(2, X, None, U, V, lam, 1, do_predict=0)
        per.append(time.time() - t)
        U, V = res["U"], res["V"]
    return np.array(per)


def head_sample(ds, sample_nnz):
    from primalcr_b200.data import Dataset, Ratings
    rp = ds.train.row_ptr
    n_users = int(np.searchsorted(rp, min(sample_nnz, ds.train.nnz), side="left"))
    n_users = max(1, min(n_users, ds.d1))
    return Dataset(ds.train.slice_users(0, n_users), Ratings.empty(n_users, ds.d2), "sample"), n_users


def cpu_baseline(ds, args, iters, sample_nnz, skip=0):
    """Reference CPU time per outer iteration on a bounded user sample, extrapolated to the full workload.

    The reference's iteration cost is affine in the ratings, t(n) = a + b n: the V-side CG works on d2 x k vectors whatever
    the number of users (a is 1-2 s at Netflix-shape, measured), so scaling a small sample by the nnz ratio OVERSTATES the
    full-size time (2 M ratings x50: 160 s, 10 M x10: 96 s on the same box).  A second, three times smaller sample is timed
    for two iterations and the pair gives a and b; `value` = a + b N, the plain ratio figure is reported beside it."""
    sample, n_users = head_sample(ds, sample_nnz)
    cores = os.cpu_count() or 1
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", REF_EXE))
    t = time.time()
    N = ds.train.nnz
    if have_ref:
        per, _ = run_reference_cli(sample, args.k, args.lam, iters, cores)
        kind = "reference"
    else:       # oracle/_ref is built wherever /root/reference is mounted and travels with the repo: this is the fallback
        per = run_oracle_port(sample, args.k, args.lam, iters)       # for a tree that never saw the reference
        kind, cores = "port", 1
    factor = N / max(sample.train.nnz, 1)
    t_main = float(np.mean(per[skip:]))
    fit = {"model": "linear", "a_s": 0.0, "b_s_per_rating": t_main / max(sample.train.nnz, 1)}
    if have_ref and sample.train.nnz >= 1_500_000 and sample.train.nnz < N:
        small, n_small = head_sample(ds, sample.train.nnz // 3)
        per_s, _ = run_reference_cli(small, args.k, args.lam, 3, cores)
        t_small = float(np.mean(per_s[1:]))
        b = (t_main - t_small) / max(sample.train.nnz - small.train.nnz, 1)
        a = t_main - b * sample.train.nnz
        if b > 0 and a >= 0:
            fit = {"model": "affine", "a_s": a, "b_s_per_rating": b, "small_sample_nnz": int(small.train.nnz),
                   "small_sample_s_per_iter": t_small}
    value = fit["a_s"] + fit["b_s_per_rating"] * N
    log("[bench] cpu %s: %d users / %d ratings, per-iter %s s; %s fit a=%.2f s b=%.3f us/rating -> %.1f s at %d ratings "
        "(nnz ratio x%.1f would say %.1f s); %.1fs total" % (kind, n_users, sample.train.nnz, np.round(per, 3).tolist(), fit["model"],
                                                             fit["a_s"], fit["b_s_per_rating"] * 1e6, value, N, factor, t_main * factor,
                                                             time.time() - t))
    return {"per_iter_sample_s": per.tolist(), "factor": factor, "kind": kind, "cores": cores, "value": value, "fit": fit,
            "linear_value": t_main * factor,
            "sample": "first %d users (%d ratings, %.4f of the workload) of the same synthetic set, %s (race-free build of the "
                      "reference) -s 2 -k %d -l %g -p 0 -n %d; extrapolated with t(n) = a + b n (%s fit: a = %.2f s, b = %.3f "
                      "us/rating; second sample of %s ratings); scaling by the nnz ratio %.1f alone would give %.1f s" % (
                          n_users, sample.train.nnz, sample.train.nnz / N, REF_EXE, args.k, args.lam, cores, fit["model"],
                          fit["a_s"], fit["b_s_per_rating"] * 1e6, fit.get("small_sample_nnz", "-"), factor, t_main * factor)}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ds = make_workload(args, "cpu" if args.scale <= 0.05 else _gen_device())
    iters = args.warmup + args.steps
    cb = cpu_baseline(ds, args, iters, reference_sample_nnz(args, iters, ds.train.nnz, budget_s=150.0), skip=args.warmup)
    per = np.array(cb["per_iter_sample_s"])[args.warmup:]
    value = float(cb["value"])
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": value * 1e3, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, ds),
        "cpu_baseline": {"value": value, "unit": "s", "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"]},
        "e2e": {"value": value, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "extrapolation": {"factor": cb["factor"], "measured_s_per_step_on_sample": float(per.mean()), "fit": cb["fit"],
                          "linear_value": cb["linear_value"],
                          "note": "value = a + b * nnz with a, b fitted on two user samples (the reference's iteration time is "
                                  "affine in the ratings; scaling the sample by the nnz ratio alone gives linear_value, an "
                                  "overestimate); a full-size CPU iteration takes over a minute, %d of them would not fit a "
                                  "bench run, so steps x value exceeds this run's wall time" % iters},
    }
    _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()
    return 0


def _gen_device():
    try:
        import torch
        return "cuda" if torch.cuda.is_available() else "cpu"
    except Exception:
        return "cpu"


def workload_config(args, ds):
    return {"workload": "%s, %d users x %d items, %d ratings (levels 1-5), Primal-CR++ -s 2 -k %d -l %g, reference init" % (
                ds.name, ds.d1, ds.d2, ds.train.nnz, args.k, args.lam),
            "solver": "Primal-CR++", "k": args.k, "lambda": args.lam, "d1": ds.d1, "d2": ds.d2, "nnz": ds.train.nnz,
            "parallelism": "users sharded over %d GPU(s) by nnz, V replicated, NCCL allreduce of d2 x k sums" % args.gpus,
            "l2_policy": "working set (>= 9 GB of ratings + factors per pass at full size) exceeds the 126 MB L2; no flush needed"}


# --------------------------------------------------------------------------------------------- parity / shim legs

def parity_check(ds, args, device, sample_nnz=2_000_000, iters=2):
    """The engine against the UNMODIFIED reference (race-free harness, all host threads) on the first ~2 M ratings of the
    bench's own data, same init: objective per outer iteration at full precision and training NDCG@10 / pairwise error."""
    from oracle import bindings as ob
    from primalcr_b200 import api
    R = ob.reference_rf()
    if R is None:
        return {"unavailable": "oracle/_ref/libref_harness_rf.so not built (needs /root/reference at build time)"}
    sample, n_users = head_sample(ds, sample_nnz)
    X = ob.Csr(sample.d1, sample.d2, sample.train.row_ptr, sample.train.item.astype(np.int64), sample.train.rating)
    U0 = api.reference_init(sample.d1, args.k); V0 = api.reference_init(sample.d2, args.k)
    t = time.time()
    ref = R.train(2, X, None, U0, V0, args.lam, iters, do_predict=1, threads=os.cpu_count() or 1)
    t_ref = time.time() - t
    e = api.Engine(api.Parameter(solver_type=api.PCRPP, k=args.k, lambda_=args.lam, maxiter=iters, device=device))
    e.set_levels(np.arange(1, 6, dtype=np.int64)); e.set_train(sample.train); e.set_factors(U0, V0)
    objs = [e.initial_objective()]; evals = [e.eval(0)]
    for _ in range(iters):
        objs.append(e.outer_iteration()); evals.append(e.eval(0))
    e.close()
    objs = np.array(objs); evals = np.array(evals)
    out = {"obj_rel_err": float(np.max(np.abs(objs - ref["obj"]) / np.abs(ref["obj"]))),
           "ndcg_abs_err": float(np.max(np.abs(evals[:, 1] - ref["evals"][:, 1]))),
           "pairwise_err_abs_err": float(np.max(np.abs(evals[:, 0] - ref["evals"][:, 0]))),
           "tolerance": {"obj_rel": 1e-6, "ndcg_abs": 1e-4},
           "objective": objs.tolist(), "reference_objective": ref["obj"].tolist(),
           "sample": "first %d users (%d ratings) of the bench data, k=%d, %d outer iterations, reference = unmodified pcrpp.cpp "
                     "(race-free objects) on %d threads (%.0f s)" % (n_users, sample.train.nnz, args.k, iters, os.cpu_count() or 1, t_ref)}
    out["ok"] = bool(out["obj_rel_err"] < 1e-6 and out["ndcg_abs_err"] < 1e-4)
    log("[bench] parity vs reference on %d ratings: obj rel err %.2e, ndcg abs err %.2e" % (
        sample.train.nnz, out["obj_rel_err"], out["ndcg_abs_err"]))
    return out


def shim_e2e(shard, args, iters):
    """e2e through the real drop-in: oracle/_ref/shim-e2e fills the reference's own containers (smat_t, mat_t =
    vector<vector<double>> in pageable memory, initial()) and calls pcrpp() = our shim + libprimalcr_b200.so once."""
    exe = os.path.join(ROOT, "oracle", "_ref", "shim-e2e")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/shim-e2e not built (needs /root/reference at build time)"}
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        path = os.path.join(tmp, "csr.bin")
        with open(path, "wb") as f:
            np.array([shard.d1, shard.d2, shard.nnz], np.int64).tofile(f)
            shard.row_ptr.astype(np.int64).tofile(f); shard.item.astype(np.int32).tofile(f); shard.rating.astype(np.float64).tofile(f)
        r = subprocess.run([exe, path, str(args.k), str(args.lam), str(iters)], capture_output=True, text=True)
    for l in r.stderr.splitlines():
        if l.startswith("[primalcr"):
            log("[bench] shim " + l)
    m = re.search(r"SHIM_E2E seconds=(\S+) iters=(\d+)", r.stdout)
    if r.returncode != 0 or not m:
        return {"unavailable": "shim-e2e failed: rc=%d %s" % (r.returncode, r.stderr[-300:])}
    total = float(m.group(1))
    objs = [float(x.group(1)) for x in re.finditer(r"^Iter \d+ time \S+ obj (\S+)", r.stdout, re.M)]
    log("[bench] shim e2e: pcrpp() call %.3f s for %d iterations" % (total, iters))
    return {"value": total / iters, "unit": "s", "call_seconds": total, "iterations": iters, "objective_last": objs[-1] if objs else None,
            "note": "wall time of ONE pcrpp(smat_t&, mat_t&, mat_t&, testset_t&, parameter&) call through primalcr_b200/shim/"
                    "pcr_shim.cpp with the reference's containers in pageable memory (flattening vector<vector<double>>, "
                    "H2D, setup, Iter-0 objective + %d iterations, D2H, un-flattening) / iterations" % iters}


# --------------------------------------------------------------------------------------------- output dump

# per-factor byte budgets of --dump-outputs (64 MB in all with the indices): Netflix-shape V (14 MB) fits whole,
# U (384 MB) is sampled
DUMP_U_BYTES, DUMP_V_BYTES = 32_000_000, 24_000_000
DUMP_SEED = 20170813


def dump_rows(n, k, budget, seed):
    """Sorted row indices of an (n, k) float64 factor to dump: all of them if they fit `budget` bytes, else a seeded sample."""
    cap = max(1, budget // (8 * k))
    if n <= cap:
        return np.arange(n, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n, size=cap, replace=False))


def dump_outputs(path, obj, counters, U_rows, U, V, k):
    """Writes the last step's outputs as float64 .npy files: objective (1,), counters (8, api.Counters order; rank 0's), U / V
    rows and their global indices."""
    os.makedirs(path, exist_ok=True)
    v_rows = dump_rows(V.shape[0], k, DUMP_V_BYTES, DUMP_SEED + 1)
    out = {"objective": np.array([obj], np.float64),
           "counters": np.array(list(counters.values()), np.float64),
           "U": U, "U_rows": U_rows.astype(np.float64), "V": V[v_rows], "V_rows": v_rows.astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float64))
    log("[bench] outputs of the last timed step written to %s (%s, %.1f MB)" % (
        path, ", ".join("%s%s" % (n, list(a.shape)) for n, a in out.items()), sum(a.nbytes for a in out.values()) / 1e6))


# --------------------------------------------------------------------------------------------- our arm

def main_ours(args):
    import torch
    import torch.distributed as dist
    from primalcr_b200 import api
    from primalcr_b200.data import shard_bounds

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: primalcr_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api.lib()                                   # fail loudly if the extension is missing

    ds = make_workload(args, "cuda")
    torch.cuda.empty_cache()
    k, lam = args.k, args.lam
    bounds = shard_bounds(ds.train.row_ptr, world)
    u0, u1 = int(bounds[rank]), int(bounds[rank + 1])
    shard = ds.train.slice_users(u0, u1)
    t = time.time()
    U_full = reference_init_cached(ds.d1, k)
    V_host = U_full[:ds.d2].copy() if ds.d2 <= ds.d1 else reference_init_cached(ds.d2, k)
    U_host = np.ascontiguousarray(U_full[u0:u1]); del U_full
    log("[bench] rank %d: users [%d,%d) nnz=%d; reference init in %.1fs" % (rank, u0, u1, shard.nnz, time.time() - t))
    levels = np.arange(1, 6, dtype=np.int64)

    # pinned host copies (the e2e leg copies from these inside its timed region)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_rp, h_it, h_ra = pin(shard.row_ptr.astype(np.int64)), pin(shard.item.astype(np.int32)), pin(shard.rating)
    h_U, h_V = pin(U_host), pin(V_host)

    def fresh_uid():
        """A ncclUniqueId serves ONE communicator: rank 0 makes a new one per engine, torch.distributed carries it."""
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(api.Engine.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        return bytes(buf.cpu().numpy().tobytes())

    comm_ready = [False]

    def new_engine(maxiter):
        p = api.Parameter(solver_type=api.PCRPP, k=k, lambda_=lam, maxiter=maxiter, do_predict=0, device=local)
        e = api.Engine(p)
        e.set_levels(levels)
        if world > 1:
            # the NCCL communicator is per-process state (created once, cached by the library): later solver calls of
            # the same process re-attach to it, exactly as a long-lived host application would
            e.comm_init(rank, world, None if comm_ready[0] else fresh_uid())
            comm_ready[0] = True
        return e

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # ---------------- device-resident leg
    eng = new_engine(args.steps)
    eng.set_train_raw(shard.d1, shard.d2, shard.nnz, h_rp, h_it, h_ra)
    eng.set_factors(h_U, h_V)
    stream = torch.cuda.ExternalStream(eng.stream_ptr(), device=torch.device("cuda", local))
    ev_init = torch.cuda.Event(enable_timing=True)
    barrier()
    ev_init.record(stream)            # start of the window the e2e leg covers: "Iter 0" objective + iterations 1 .. W+K
    obj0 = eng.initial_objective()
    objs = [obj0]
    for _ in range(args.warmup):
        objs.append(eng.outer_iteration())
    eng.profile_enable(True); eng.profile_reset()
    launches0 = eng.launch_count()
    sampler = ClockSampler(local); sampler.start(); sampler.ready.wait(10)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    counters = []
    barrier()
    sampler.window[0] = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        objs.append(eng.outer_iteration())
        counters.append(eng.counters())
    ev1.record(stream)
    barrier()
    sampler.window[1] = time.perf_counter()
    sampler.stop_flag = True; sampler.join()
    sec = max_over_ranks(ev0.elapsed_time(ev1) / 1e3) / args.steps
    n_all = args.warmup + args.steps
    sec_same_window = max_over_ranks(ev_init.elapsed_time(ev1) / 1e3) / n_all
    launches = eng.launch_count() - launches0
    prof = eng.profile()
    eng.profile_enable(False)
    dev_bytes = eng.device_bytes()
    dump = None
    if args.dump_outputs:       # copied back after the timed window
        U_out, V_out = eng.get_factors()
        rows = dump_rows(ds.d1, k, DUMP_U_BYTES, DUMP_SEED)
        rows = rows[(rows >= u0) & (rows < u1)]
        dump = (rows, U_out[rows - u0], V_out)
        del U_out
    eng.close(); del eng
    torch.cuda.empty_cache()

    # ---------------- end-to-end leg: host buffers in, the SAME W+K iterations from the same init, host factors out
    outU = torch.empty_like(h_U).pin_memory(); outV = torch.empty_like(h_V).pin_memory()
    barrier()
    t0 = time.perf_counter()
    e2 = new_engine(n_all)
    t1 = time.perf_counter()
    e2.set_train_raw(shard.d1, shard.d2, shard.nnz, h_rp, h_it, h_ra)
    t2 = time.perf_counter()
    e2.set_factors(h_U, h_V)
    t3 = time.perf_counter()
    e2.run(log=None)
    t4 = time.perf_counter()
    e2.get_factors(outU, outV)
    barrier()
    t5 = time.perf_counter()
    e2e_sec = max_over_ranks(t5 - t0) / n_all
    e2e_phases = {"create": t1 - t0, "set_train": t2 - t1, "set_factors": t3 - t2, "run": t4 - t3, "get_factors": t5 - t4}
    log("[bench] rank %d e2e phases (s): %s" % (rank, {k_: round(v_, 4) for k_, v_ in e2e_phases.items()}))
    e2.close()
    h2d = (h_rp.numel() * 8 + h_it.numel() * 4 + h_ra.numel() * 8 + h_U.numel() * 8 + h_V.numel() * 8) / n_all
    d2h = (outU.numel() * 8 + outV.numel() * 8) / n_all
    torch.cuda.empty_cache()

    per_rank = None
    if world > 1:      # per-rank kernel totals (load balance of the user shards), gathered before the ranks part ways
        mine = {"nnz": int(shard.nnz), "users": int(u1 - u0), "sec": ev0.elapsed_time(ev1) / 1e3 / args.steps,
                "kernels": {n: round(v["ms"] / args.steps, 3) for n, v in prof.items() if v["ms"] / args.steps >= 0.05}}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered
    if dump is not None:
        rows, U_rows = dump[0], dump[1]
        if world > 1:           # each rank holds the sampled rows of its own users
            parts = [None] * world
            dist.all_gather_object(parts, (rows, U_rows))
            rows = np.concatenate([p[0] for p in parts]); U_rows = np.concatenate([p[1] for p in parts])
        if rank == 0:
            dump_outputs(args.dump_outputs, objs[-1], counters[-1], rows, U_rows, dump[2], k)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---------------- roofline
    peak, peak_src = peaks()
    N, d1 = ds.train.nnz, ds.d1
    b_pass = N * (8 * k + 12) + 8 * k * d1
    its = []
    for c in counters:     # rank 0's counters; the len-weighted means use rank 0's shard
        tv, lv = c["v_cg_iters"], c["v_ls_trials"]
        cu = c["u_cg_len_sum"] / max(shard.nnz, 1); lu = c["u_ls_len_sum"] / max(shard.nnz, 1)
        pi = 3 + 2 * tv + lv + 2 * cu + lu
        s = 3 + lv + lu
        its.append(dict(T_V=tv, L_V=lv, c_U=cu, l_U=lu, passes=pi, sorts=s, b_alg=pi * b_pass + s * 32 * N))
    b_alg = float(np.mean([i["b_alg"] for i in its]))
    hot = {n: v for n, v in prof.items() if v["bytes"] > 0}
    top = max(hot, key=lambda n: hot[n]["ms"]) if hot else None
    roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None}
    if top:
        a = hot[top]["bytes"] / (hot[top]["ms"] / 1e3) / 1e9
        roof.update(kernel=top, achieved=a, frac=a / peak, launches=hot[top]["launches"],
                    avg_launch_ms=hot[top]["ms"] / hot[top]["launches"],
                    bytes_per_launch=hot[top]["bytes"] / hot[top]["launches"],
                    share_of_step=hot[top]["ms"] / 1e3 / (sec * args.steps))
    roof["frac_kind"] = ("algorithmic_vs_hbm: SURVEY 8d's logical row touches per launch / launch time / measured HBM peak; "
                         "the gathered rows are served from L2/L1, so this is NOT an HBM utilisation and may exceed 1 -- "
                         "see dram_frac and l2 for what the memory system delivered")
    # ncu figures of THIS round's tree (one `ncu --set full` capture per kernel + one dram-bytes launch list of a whole
    # iteration; tools/gpu/r02_capture.sh, summarised by tools/ncu_summary.py traffic): a profiler cannot run inside a bench run
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    traffic = json.load(open(tpath)) if os.path.exists(tpath) else {}
    same_workload = world == 1 and args.workload == "netflix" and args.scale == 1.0 and k == 100
    if top and same_workload and top in traffic.get("kernels", {}):
        tk = traffic["kernels"][top]
        roof["traffic"] = tk["dram_bytes_per_launch"]        # dram__bytes_read.sum + dram__bytes_write.sum per launch
        roof["dram_achieved"] = roof["traffic"] / (roof["avg_launch_ms"] / 1e3) / 1e9   # what the HBM actually delivered
        roof["dram_frac"] = roof["dram_achieved"] / peak
        roof["l2"] = {"lts_throughput_pct": tk.get("lts_throughput_pct"), "l2_hit_pct": tk.get("l2_hit_pct"),
                      "l1tex_hit_pct": tk.get("l1tex_hit_pct"), "dram_read_bytes_per_launch": tk.get("dram_read_bytes_per_launch"),
                      "note": "the binding resource of the N*k gathers is the L2 -> SM path, not HBM"}
        roof["traffic_source"] = traffic.get("_note")
    it_dram = traffic.get("iteration", {}).get("dram_bytes") if same_workload else None
    roof.update(peak_source=peak_src,
                iteration={"b_alg_bytes": b_alg, "achieved": b_alg / sec / 1e9 * 1.0, "frac": b_alg / sec / 1e9 / peak / world,
                           "frac_kind": "algorithmic_vs_hbm",
                           "dram_bytes": it_dram, "dram_frac": (it_dram / sec / 1e9 / peak) if it_dram else None,
                           "note": "B_alg = passes*[N(8k+12)+8k*d1] + sorts*32N (SURVEY 8d); frac is per GPU; dram_bytes = ncu "
                                   "dram read+write summed over every launch of one outer iteration",
                           "counters": its[-1]})
    kern = sorted(((v["ms"], n, v["launches"], v["bytes"]) for n, v in prof.items()), reverse=True)
    roof["kernels"] = [{"name": n, "ms_per_step": ms / args.steps, "launches_per_step": l / args.steps,
                        "gbs": (b / (ms / 1e3) / 1e9 if b > 0 and ms > 0 else None)} for ms, n, l, b in kern[:40]]

    # the side legs (CPU baseline, parity vs the reference, drop-in e2e) must never cost the run its main line
    cb = parity = shim = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            c = cpu_baseline(ds, args, 2, reference_sample_nnz(args, 2, ds.train.nnz, budget_s=40.0), skip=1)
            cb = {"value": float(c["value"]), "unit": "s", "cores": c["cores"], "kind": c["kind"], "sample": c["sample"],
                  "fit": c["fit"], "linear_value": c["linear_value"]}
        except Exception as ex:
            cb = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
        try:
            parity = parity_check(ds, args, local)
        except Exception as ex:
            parity = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
    if world == 1 and not args.no_shim_e2e:
        try:
            shim = shim_e2e(shard, args, n_all)
        except Exception as ex:
            shim = {"unavailable": "%s: %s" % (type(ex).__name__, str(ex)[:200])}

    line = {
        "metric": METRIC, "value": sec, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, ds),
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_sec, "unit": "s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "phases_s": e2e_phases, "iterations": n_all, "device_same_window": sec_same_window,
                "shim": shim,
                "note": "whole pcrpp()-style call through the C ABI from pinned host buffers (upload CSR+U+V, build CSC and work "
                        "lists, Iter-0 objective + iterations 1..%d from the reference init, download U+V) / %d; "
                        "device_same_window = device-timed mean of the same iterations with everything resident "
                        "(`value` covers iterations %d..%d only)" % (n_all, n_all, args.warmup + 1, n_all)},
        "gpu_launches": int(launches),
        "roofline": roof, "cpu_baseline": cb, "parity": parity, "per_rank": per_rank,
        "objective": objs, "device_bytes": dev_bytes,
    }
    _REAL_STDOUT.write(json.dumps(line) + "\n"); _REAL_STDOUT.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    # libraries (NCCL's version banner, ...) may write to fd 1: keep the real stdout for the ONE JSON line only
    global _REAL_STDOUT
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="netflix")
    ap.add_argument("--scale", type=float, default=1.0, help="user/rating subsample factor of the named shape")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--lam", type=float, default=5000.0)
    ap.add_argument("--ref-sample-nnz", type=int, default=0,
                    help="ratings in the reference's timing sample (0: 10 %% of the workload, less if that would not fit the run)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline and parity legs")
    ap.add_argument("--no-shim-e2e", action="store_true", help="skip the e2e run through the C++ drop-in shim")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    global METRIC
    if not (args.workload == "netflix" and args.k == 100):
        METRIC = "sec_per_outer_iter_primalcrpp_k%d_%s_shape" % (args.k, args.workload)
    if args.impl == "reference":
        return main_reference(args)
    return main_ours(args)


if __name__ == "__main__":
    sys.exit(main())
