"""Cost of steps with more candidate neighbours than one scoring pass takes (IG_MAX_CANDS = 8; up to IG_MAX_NEIGHBOURS =
64, scored in batches of 8 plus a re-score of the winning batch): steps/s and scored proposals/s for n in {5, 8, 12, 16,
32, 64} through step_sampler (one blocking call per step, host-drawn neighbours) and run_cycle_device (device draws, one
call per cycle), mid-assembly (bomb + 2 device cycles, as bench.py) and assembled (the level's initial scaffold), plus the
device memory one more chain of the level takes after running such steps (cudaMemGetInfo before / after a clone).
Writes JSON under profiles/ (GPU name and power limit read in the same run) and prints it.

    python scripts/wide_neighbourhood_timing.py --workloads T,G --steps 300 --out profiles/r4_wide_neighbourhood_timing.json
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
NS = (5, 8, 12, 16, 32, 64)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    first = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ","
    name, power = (x.strip() for x in first.split(",", 1))
    return name, power


def sync():
    import torch
    torch.cuda.synchronize()


def mem_free():
    import torch
    sync()
    return torch.cuda.mem_get_info()[0]


def measure(name, steps):
    from instagraal_b200.cuda_lib_gl_single import sampler
    from instagraal_b200.synth import make_workload, workload_params
    level = make_workload(name)
    p8 = workload_params(level)
    s = sampler(*level.sampler_args())
    s.set_param_simu(p8)
    st0, valid0 = s._get_state(), s.get_valid_insert()
    np.random.seed(1000)
    s.bomb_the_genome()
    frs = np.arange(level.n_frags)
    for c in range(2):
        np.random.shuffle(frs)
        s.run_cycle_device(frs, 5, seed=1000, cycle=c)
    starts = {"mid_assembly": (s._get_state(), s.get_valid_insert()), "assembled": (st0, valid0)}
    order = np.random.RandomState(7).permutation(level.n_frags).astype(np.int32)
    order = np.concatenate([order] * (1 + (steps + 64) // level.n_frags))
    dt = np.float32(0.01)
    out = {"n_frags": int(level.n_frags), "nnz": int(level.sparse_matrix.nnz), "steps": steps}
    for start, (st, valid) in starts.items():
        res = {}
        for n in NS:
            r = {}
            # step_sampler: host draws (return_neighbours), one blocking library call per step; 16 warm-up steps
            s._set_state(st); s.set_valid_insert(valid)
            np.random.seed(5)
            for i in range(16):
                s.step_sampler(int(order[i]), n, dt)
            s._set_state(st); s.set_valid_insert(valid)
            s.step_sampler(int(order[-1]), n, dt)   # the full refresh after set_state, outside the window
            p0 = s.n_proposals_scored
            sync()
            t0 = time.perf_counter()
            for i in range(steps):
                s.step_sampler(int(order[i]), n, dt)
            sync()
            el = time.perf_counter() - t0
            r["step_sampler_steps_per_s"] = steps / el
            r["step_sampler_proposals_per_s"] = (s.n_proposals_scored - p0) / el
            # run_cycle_device: one call for the whole run (warm-up call: graph capture)
            s._set_state(st); s.set_valid_insert(valid)
            s.run_cycle_device(order[:32], n, seed=11, cycle=900)
            s._set_state(st); s.set_valid_insert(valid)
            s.run_cycle_device(order[:1], n, seed=11, cycle=901)   # the full refresh after set_state, outside the window
            sync()
            t0 = time.perf_counter()
            rec = s.run_cycle_device(order[:steps], n, seed=11, cycle=902)
            sync()
            el = time.perf_counter() - t0
            r["run_cycle_device_steps_per_s"] = steps / el
            r["run_cycle_device_proposals_per_s"] = float(rec["n_proposals"].sum()) / el
            r["mean_candidates_per_step"] = float(s.last_cycle_plan(steps)[:, 0].mean())
            res[str(n)] = r
        out[start] = res
    # device memory of one more chain of this level that runs steps of n neighbours (the level's arrays are shared)
    mem = {}
    for n in NS:
        f0 = mem_free()
        c = sampler.clone_of(s)
        c.step_sampler(int(order[0]), n, dt)
        c.run_cycle_device(order[:64], n, seed=3, cycle=0)
        mem[str(n)] = (f0 - mem_free()) / 2**20
        c.free_gpu()
    out["device_mib_per_extra_chain"] = mem
    s.free_gpu()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="T,G")
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_wide_neighbourhood_timing.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wide_neighbourhood_timing: no CUDA device (this measurement has no CPU mode)")
    name, power = gpu_info()
    res = {"script": "scripts/wide_neighbourhood_timing.py", "gpu": name, "power_limit": power,
           "starts": {"mid_assembly": "bomb + 2 run_cycle_device cycles (seed 1000), as bench.py",
                      "assembled": "the level's initial scaffold"}}
    for w in args.workloads.split(","):
        res[w] = measure(w, args.steps)
    txt = json.dumps(res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
