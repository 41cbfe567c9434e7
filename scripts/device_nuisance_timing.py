"""Cost of a step + nuisance step (full_em from cycle 5 on, IG:242-252) end to end: the host loop (step_sampler +
step_nuisance_parameters: host RNG, scipy fsolve, two blocking calls) against the production RNG mode with the nuisance step
on the device (run_cycle_device(nuisance=True)), plus run_cycle_device without it and 8 chains of one GPU with it
(ReplicaSet.run_cycle(nuisance=True)).  Start: bomb + 2 device cycles, as bench.py builds its mid-assembly state.
Prints one JSON line (GPU name and power limit read in the same run).

    python scripts/device_nuisance_timing.py --workloads T,G --steps 2000 --chain-steps 500
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


def measure(name, steps, chain_steps, n_chains):
    from instagraal_b200.cuda_lib_gl_single import sampler
    from instagraal_b200.replicas import ReplicaSet
    from instagraal_b200.synth import make_workload, workload_params
    level = make_workload(name)
    p8 = workload_params(level)
    s = sampler(*level.sampler_args())
    s.set_param_simu(p8)
    np.random.seed(1000)
    s.bomb_the_genome()
    frs = np.arange(level.n_frags)
    for c in range(2):
        np.random.shuffle(frs)
        s.run_cycle_device(frs, 5, seed=1000, cycle=c)
    st_mid, valid_mid = s._get_state(), s.get_valid_insert()
    rng = np.random.RandomState(7)
    order = rng.permutation(level.n_frags).astype(np.int32)
    order = np.concatenate([order] * (1 + (steps + 64) // level.n_frags))
    dt = np.float32(0.01)

    def reset():
        s._set_state(st_mid)
        s.set_valid_insert(valid_mid)
        s.set_param_simu(p8)
        s.param_simu_test = s.param_simu

    out = {"n_frags": int(level.n_frags), "nnz": int(level.sparse_matrix.nnz), "steps": steps}
    # host loop: step_sampler + step_nuisance_parameters (warm-up: 64 pairs)
    reset()
    np.random.seed(5)
    for i in range(64):
        s.step_sampler(int(order[i]), 5, dt)
        s.step_nuisance_parameters(dt, i, 64)
    reset()
    acc = 0
    sync()
    t0 = time.perf_counter()
    for i in range(steps):
        s.step_sampler(int(order[i]), 5, dt)
        acc += int(s.step_nuisance_parameters(dt, i, steps)[6])
    sync()
    out["host_loop_ms_per_step_pair"] = (time.perf_counter() - t0) * 1e3 / steps
    out["host_loop_acceptance"] = acc / steps
    # device: run_cycle_device without and with the nuisance step (one warm-up call each: graph capture)
    for nuis, key in ((False, "device_cycle_ms_per_step"), (True, "device_nuisance_ms_per_step_pair")):
        reset()
        s.run_cycle_device(order[:64], 5, seed=11, cycle=900, nuisance=nuis)
        reset()
        sync()
        t0 = time.perf_counter()
        r = s.run_cycle_device(order[:steps], 5, seed=11, cycle=901, nuisance=nuis)
        sync()
        out[key] = (time.perf_counter() - t0) * 1e3 / steps
        if nuis:
            out["device_acceptance"] = float(r[1]["success"].mean())
            out["device_invalid"] = float((r[1]["valid"] == 0).mean())
    s.set_device_nuisance(False)
    # 8 chains on this GPU with the nuisance step
    reset()
    rs = ReplicaSet(s, n_chains, seeds=np.arange(n_chains) + 40)
    for c in rs.chains:
        c._set_state(st_mid)
        c.set_valid_insert(valid_mid)
    frags = np.stack([np.roll(order[:chain_steps], 17 * i) for i in range(n_chains)]).astype(np.int32)
    rs.run_cycle(frags[:, :32], 5, cycle=950, nuisance=True)
    sync()
    t0 = time.perf_counter()
    steps_rec, nuis_rec = rs.run_cycle(frags, 5, cycle=951, nuisance=True)
    sync()
    dt_s = time.perf_counter() - t0
    out["chains"] = n_chains
    out["chains_steps_per_chain"] = chain_steps
    out["chains_nuisance_proposals_per_s"] = n_chains * chain_steps / dt_s
    out["chains_scored_proposals_per_s"] = float(steps_rec["n_proposals"].sum()) / dt_s
    out["chains_acceptance"] = float(nuis_rec["success"].mean())
    rs.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,G")
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--chain-steps", type=int, default=500)
    ap.add_argument("--chains", type=int, default=8)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_nuisance_timing: no CUDA device (this measurement has no CPU mode)")
    name, power = gpu_info()
    res = {"script": "scripts/device_nuisance_timing.py", "gpu": name, "power_limit": power,
           "start": "mid-assembly: bomb + 2 run_cycle_device cycles (seed 1000), as bench.py"}
    for w in args.workloads.split(","):
        res[w] = measure(w, args.steps, args.chain_steps, args.chains)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
