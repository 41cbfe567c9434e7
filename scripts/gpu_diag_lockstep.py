#!/usr/bin/env python3
"""Diagnostic: lockstep of the product vs the reference kernels (cubin) on a workload; at the first step whose scores
differ by more than --tol, prints the per-proposal differences for the default path, the row-per-warp path (IG_SCORING_PATH=rows)
and the NumPy oracle.   python scripts/gpu_diag_lockstep.py --workload T --steps 900"""
import argparse, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="T"); ap.add_argument("--steps", type=int, default=900)
ap.add_argument("--seed", type=int, default=3); ap.add_argument("--tol", type=float, default=1e-9)
ap.add_argument("--max-report", type=int, default=3)
a = ap.parse_args()
from instagraal_b200.synth import make_workload, workload_params
from test_bench_configs import burnt_state
from test_gpu_parity import GpuImpl
from oracle.ref_replay import RefReplaySampler
from oracle.sampler_oracle import return_neighbours, setup_distri_frags, OracleSampler
from instagraal_b200._lib import FIELDS13
level = make_workload(a.workload); p8 = workload_params(level)
st = burnt_state(level, p8, 2, 1000, "bomb")
ref = RefReplaySampler(level, p8, backend="gpu")
mine = GpuImpl(level)
os.environ["IG_SCORING_PATH"] = "rows"
rowp = GpuImpl(level)
del os.environ["IG_SCORING_PATH"]
for i in (mine, rowp): i.set_params(p8)
ref.set_state(st)
distri = setup_distri_frags(level.sub_sampled_sparse_matrix, level.n_frags)
frs = np.random.RandomState(a.seed).permutation(level.n_frags)
np.random.seed(a.seed)
state = np.ascontiguousarray(st, dtype=np.int32)
t = rep = 0
for f in frs:
    if t >= a.steps: break
    f = int(f)
    cands = sorted(int(c) for c in return_neighbours(distri, level.n_frags, f, 5) if int(c) != f)
    if not cands: continue
    valid = ref.valid_insert.get().copy()
    for i in (mine, rowp): i.set_state(state); i.set_valid(valid)
    ref.step_sampler(f, cands)
    sa = np.asarray(ref.all_scores, dtype=np.float64)
    sb = np.asarray(mine.step(f, cands)["scores"], dtype=np.float64)
    sc = np.asarray(rowp.step(f, cands)["scores"], dtype=np.float64)
    nz = sa != 0
    def rel(x): return float(np.max(np.abs(sa[nz] - x[nz]) / np.abs(sa[nz]))) if np.array_equal(sa != 0, x != 0) else float("inf")
    rb, rc = rel(sb), rel(sc)
    if max(rb, rc) > a.tol:
        o = OracleSampler(level, p8)
        o.live = {k: state[i].copy() for i, k in enumerate(FIELDS13)}
        o.valid = [int(x) for x in valid]
        o.step_sampler(f, 5, candidates=cands)
        so = np.asarray(o.all_scores, dtype=np.float64)
        print("STEP", t, "frag", f, "cands", cands, "rel flat", rb, "rel rowpath", rc, "rel oracle", rel(so), "n_sub", mine.s.n_sub_vals, "ref n_sub", getattr(ref, "n_sub_list", None))
        print("  contigs:", {c: (int(state[2][c]), int(state[0][c]), int(state[9][c])) for c in [f] + cands})
        for k in range(len(cands)):
            for op in range(24):
                g = k * 24 + op
                if sa[g] != 0 and (abs(sa[g] - sb[g]) > a.tol * abs(sa[g]) or abs(sa[g] - sc[g]) > a.tol * abs(sa[g])):
                    print("   cand %d op %2d ref %.10e flat-ref %+.4e row-ref %+.4e oracle-ref %+.4e" % (k, op, sa[g], sb[g] - sa[g], sc[g] - sa[g], so[g] - sa[g]))
        rep += 1
        if rep >= a.max_report: break
    state = ref.get_state()
    t += 1
print("done", t, "steps,", rep, "mismatching steps")
