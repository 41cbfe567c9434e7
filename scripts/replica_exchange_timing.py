"""Price and effect of a replica exchange (ReplicaSet.exchange = allgather + adopt(best), ig_adopt_gathered), 8 chains on one GPU:

1. exchange() at each workload: pack + all-gather + header compaction from the library's CUDA events (the `ms` of
   ig_allgather_best), adoption alone as a host clock around adopt() between two device synchronisations.
2. the first step of an adopted chain (a full refresh, kind 1) against the incremental step that follows it: one-step cycles
   of one adopted chain, device time from the chain's own CUDA events (get_stats()["ms_step"]).
3. the search effect at T: from a bomb, 10 cycles (nuisance step from cycle 5 on, as full_em), exchange after every cycle
   against the all-gather alone, 3 seed sets; the best-of-8 likelihood after each cycle.
Prints one JSON line (GPU name and power limit read in the same run) and writes it to --out when given.

    python scripts/replica_exchange_timing.py --workloads T,G --out profiles/r4_replica_exchange_timing.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ","
    name, power = (x.strip() for x in first.split(",", 1))
    return name, power


def sync():
    import torch
    torch.cuda.synchronize()


def replica_set(level, p8, n_chains, seed0):
    from instagraal_b200.cuda_lib_gl_single import sampler
    from instagraal_b200.replicas import ReplicaSet
    first = sampler(*level.sampler_args())
    first.set_param_simu(p8)
    rs = ReplicaSet(first, n_chains, seeds=np.arange(n_chains, dtype=np.uint64) + seed0)
    rs.bomb(seed0=seed0)
    return rs


def orders(nf, n_chains, n_steps, seed):
    rng = np.random.RandomState(seed)
    return np.stack([rng.permutation(nf)[:n_steps] for _ in range(n_chains)]).astype(np.int32)


def exchange_cost(name, n_chains, reps, warm_steps):
    from instagraal_b200.synth import make_workload, workload_params
    level = make_workload(name)
    rs = replica_set(level, workload_params(level), n_chains, 1000)
    out = {"n_frags": int(level.n_frags), "chains": n_chains, "reps": reps,
           "record_bytes_per_chain": 128 + 64 * int(level.n_frags)}
    gather, adopt, total, first, incr, first_full, incr_full = [], [], [], [], [], [], []
    for r in range(reps + 1):   # rep 0 warms the graphs of both step kinds
        rs.run_cycle(orders(level.n_frags, n_chains, warm_steps, 10 + r), 5, cycle=2 * r)
        sync()
        g0 = rs.gather_ms
        t0 = time.perf_counter()
        best, lik, nc = rs.allgather()
        t1 = time.perf_counter()
        rs.adopt(best)
        sync()
        t2 = time.perf_counter()
        ch = rs.chains[1 if best != 1 else 2]   # an adopted chain, stepping alone
        o = orders(level.n_frags, 1, 2, 90 + r)[0]
        ch.get_stats(reset=True)
        ch.run_cycle_device(o[:1], 5, seed=7, cycle=2 * r + 1)
        st1 = ch.get_stats(reset=True)
        ch.run_cycle_device(o[1:2], 5, seed=7, cycle=2 * r + 1)
        st0 = ch.get_stats(reset=True)
        if r == 0:
            continue
        gather.append(rs.gather_ms - g0)
        adopt.append((t2 - t1) * 1e3)
        total.append((t2 - t0) * 1e3)
        first.append(st1["ms_step"])
        incr.append(st0["ms_step"])
        first_full.append(st1["full_refreshes"])
        incr_full.append(st0["full_refreshes"])
    med = lambda v: float(np.median(v))   # noqa: E731
    out.update({
        "pack_gather_ms_median": med(gather), "pack_gather_ms_min": float(np.min(gather)),
        "adopt_ms_median": med(adopt), "adopt_ms_min": float(np.min(adopt)),
        "exchange_wall_ms_median": med(total),
        "first_step_after_adopt_ms_median": med(first), "incremental_step_ms_median": med(incr),
        "first_step_full_refreshes": int(sum(first_full)), "incremental_step_full_refreshes": int(sum(incr_full)),
    })
    rs.free()
    return out


def search_effect(n_chains, n_cycles, seed_sets):
    from instagraal_b200.synth import make_workload, workload_params
    level = make_workload("T")
    p8 = workload_params(level)
    res = {"workload": "T", "n_frags": int(level.n_frags), "chains": n_chains, "cycles": n_cycles,
           "nuisance_from_cycle": 5, "runs": []}
    for s in seed_sets:
        run = {"seed_set": s}
        for mode in ("exchange", "allgather_only"):
            rs = replica_set(level, p8, n_chains, 100 * s)
            best_lik = []
            t0 = time.perf_counter()
            for j in range(n_cycles):
                rs.run_cycle(orders(level.n_frags, n_chains, level.n_frags, 1000 * s + j), 5, cycle=j, nuisance=j >= 5)
                _best, lik, _nc = rs.exchange() if mode == "exchange" else rs.allgather()
                best_lik.append(float(lik.max()))
            sync()
            run[mode] = best_lik
            run[mode + "_wall_s"] = time.perf_counter() - t0
            rs.free()
        run["exchange_minus_allgather_only_last"] = run["exchange"][-1] - run["allgather_only"][-1]
        res["runs"].append(run)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,G")
    ap.add_argument("--chains", type=int, default=8)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warm-steps", type=int, default=64)
    ap.add_argument("--cycles", type=int, default=10)
    ap.add_argument("--seed-sets", default="1,2,3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("replica_exchange_timing: no CUDA device (this measurement has no CPU mode)")
    name, power = gpu_info()
    res = {"script": "scripts/replica_exchange_timing.py", "gpu": name, "power_limit": power,
           "exchange_cost_start": "bomb, then one cycle of --warm-steps steps per chain before every exchange"}
    for w in args.workloads.split(","):
        res["exchange_" + w] = exchange_cost(w, args.chains, args.reps, args.warm_steps)
    res["search_T"] = search_effect(args.chains, args.cycles, [int(x) for x in args.seed_sets.split(",")])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
