"""Price and effect of tempering (sampler.set_chain_temperature, ReplicaSet.set_ladder / swap_temperatures):

1. device time per step at T = 0 against T > 0, the two alternated block by block on one chain in this one run, at T and G,
   5 and 16 neighbours (16 = a wide step of two batches); device time from the chain's CUDA events (get_stats()["ms_step"]).
2. the cost of swap_temperatures() (one all-gather + the decision + setting the temperatures) on 8 chains of T, host clock
   between two device synchronisations, against allgather() alone.
3. the search effect at T: 8 chains, 10 cycles from a bomb (nuisance step from cycle 5 on, as full_em), 3 seed sets:
   8 independent argmax chains (all-gather only), exchange of the best chain after every cycle (DESIGN.md 6a), and the ladder
   [0, g * geomspace(0.5, 50, 7)] with a swap round after every cycle.  g = the median best-minus-second-best score gap of
   one calibration cycle of host-mode steps from a bomb (all_scores).  Best-of-8 live log-likelihood per cycle and the
   acceptance per rung pair.
Prints one JSON line (GPU name and power limit read in the same run) and writes it to --out when given.

    python scripts/tempering_timing.py --out profiles/r5_tempering.json
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


def chain(level, p8, seed):
    from instagraal_b200.cuda_lib_gl_single import sampler
    s = sampler(*level.sampler_args())
    s.set_param_simu(p8)
    np.random.seed(seed)
    s.bomb_the_genome()
    return s


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


def score_gap(level, p8, n_neigh=5, seed=7):
    """median over the steps of one host-mode cycle from a bomb of (best - second best) scored proposal"""
    s = chain(level, p8, seed)
    gaps = []
    for a in np.random.RandomState(seed).permutation(level.n_frags):
        s.step_sampler(int(a), n_neigh, np.float32(0.01))
        v = np.sort(s.all_scores[(s.all_scores != 0) & ~np.isnan(s.all_scores)])[::-1]
        if len(v) >= 2:
            gaps.append(float(v[0] - v[1]))
    s.free_gpu()
    return float(np.median(gaps))


def step_cost(level, n_neigh, T_hot, blocks, steps):
    from instagraal_b200.synth import workload_params
    s = chain(level, workload_params(level), 11)
    rng = np.random.RandomState(5)
    out = {"n_frags": int(level.n_frags), "n_neighbours": n_neigh, "T_hot": T_hot, "blocks": blocks, "steps_per_block": steps}
    ms = {0: [], 1: []}
    for b in range(blocks + 1):   # block 0 warms the graphs of both temperatures
        for hot in (0, 1):
            s.set_chain_temperature(T_hot if hot else 0.0)
            s.run_cycle_device(rng.permutation(level.n_frags)[:steps].astype(np.int32), n_neigh, seed=b, cycle=2 * b + hot)
            st = s.get_stats(reset=True)
            if b:
                ms[hot].append(st["ms_step"] / st["steps"])
    s.free_gpu()
    out["ms_per_step_T0"] = ms[0]
    out["ms_per_step_hot"] = ms[1]
    out["median_T0"] = float(np.median(ms[0]))
    out["median_hot"] = float(np.median(ms[1]))
    out["hot_over_T0"] = out["median_hot"] / out["median_T0"]
    return out


def swap_cost(level, p8, ladder, n_chains, reps):
    rs = replica_set(level, p8, n_chains, 300)
    rs.set_ladder(ladder)
    rs.run_cycle(orders(level.n_frags, n_chains, 64, 1), 5, cycle=0)
    gather, swap = [], []
    for r in range(reps + 1):
        sync()
        t0 = time.perf_counter()
        rs.allgather()
        sync()
        t1 = time.perf_counter()
        rs.swap_temperatures()
        sync()
        t2 = time.perf_counter()
        if r:
            gather.append(1e3 * (t1 - t0))
            swap.append(1e3 * (t2 - t1))
    rs.free()
    return {"chains": n_chains, "reps": reps, "allgather_ms_median": float(np.median(gather)),
            "swap_temperatures_ms_median": float(np.median(swap)), "allgather_ms": gather, "swap_temperatures_ms": swap}


def search_effect(level, p8, ladder, n_chains, n_cycles, seed_sets):
    res = {"workload": "T", "n_frags": int(level.n_frags), "chains": n_chains, "cycles": n_cycles,
           "nuisance_from_cycle": 5, "ladder": list(map(float, ladder)), "runs": []}
    for s in seed_sets:
        run = {"seed_set": s}
        for mode in ("independent", "exchange", "tempering"):
            rs = replica_set(level, p8, n_chains, 100 * s)
            if mode == "tempering":
                rs.set_ladder(ladder, swap_seed=s)
            best = []
            t0 = time.perf_counter()
            for j in range(n_cycles):
                rs.run_cycle(orders(level.n_frags, n_chains, level.n_frags, 1000 * s + j), 5, cycle=j, nuisance=j >= 5)
                if mode == "exchange":
                    rs.exchange()
                elif mode == "tempering":
                    rs.swap_temperatures()
                else:
                    rs.allgather()
                best.append(float(rs.gathered_live_likelihood().max()))
            sync()
            run[mode] = best
            run[mode + "_wall_s"] = time.perf_counter() - t0
            if mode == "tempering":
                run["swap_tried"] = rs.swap_stats["tried"].tolist()
                run["swap_accepted"] = rs.swap_stats["accepted"].tolist()
            rs.free()
        run["tempering_minus_independent_last"] = run["tempering"][-1] - run["independent"][-1]
        run["tempering_minus_exchange_last"] = run["tempering"][-1] - run["exchange"][-1]
        res["runs"].append(run)
    tried = np.sum([r["swap_tried"] for r in res["runs"]], axis=0)
    acc = np.sum([r["swap_accepted"] for r in res["runs"]], axis=0)
    res["acceptance_per_pair"] = (acc / np.maximum(tried, 1)).tolist()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,G")
    ap.add_argument("--neighbours", default="5,16")
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--chains", type=int, default=8)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cycles", type=int, default=10)
    ap.add_argument("--seed-sets", default="1,2,3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tempering_timing: no CUDA device (this measurement has no CPU mode)")
    from instagraal_b200.synth import make_workload, workload_params
    name, power = gpu_info()
    res = {"script": "scripts/tempering_timing.py", "gpu": name, "power_limit": power}
    level = make_workload("T")
    p8 = workload_params(level)
    g = score_gap(level, p8)
    ladder = [0.0] + (g * np.geomspace(0.5, 50.0, args.chains - 1)).tolist()
    res["score_gap_g_T"] = g
    for w in args.workloads.split(","):
        lw = level if w == "T" else make_workload(w)
        for k in (int(x) for x in args.neighbours.split(",")):
            res["step_%s_n%d" % (w, k)] = step_cost(lw, k, 5.0 * g, args.blocks, args.steps)
    res["swap_T"] = swap_cost(level, p8, ladder, args.chains, args.reps)
    res["search_T"] = search_effect(level, p8, ladder, args.chains, args.cycles, [int(x) for x in args.seed_sets.split(",")])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
