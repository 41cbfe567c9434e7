"""GPU-vs-GPU parity ON THE BENCHMARKED CONFIGS (BASELINE.json configs[1..3] = workloads T, Y3, G): the
product (through the C ABI) against the reference's OWN kernels (oracle/_ref/ref_kernels.cubin, built from
/root/reference by oracle/Makefile) driven in the reference's launch order (oracle/ref_replay.py, validated
against the golden vectors on the CPU backend).

Teacher = the reference: every step starts from the reference's state.  Per step
  * the set of scored proposals is identical,
  * every score agrees to 1e-9 relative (same libdevice powf/log10; the tolerance covers f64 summation order --
    the reference itself uses double atomics),
  * the chosen (op, B) is identical -- then the 13 x NF integer state, dist, n_contigs and mean contig length
    are compared bit for bit -- or the two choices are tied at 1e-9 relative in the reference's own scores.

The same harness measures what `rigid_pruning` (deviation D2) costs in accuracy on the 1 Gb level:
    err[m] = |score_rigid[m] - score_ref[m]|  against  |score_ref[m] - score_ref[best]|  and  |score_ref[m] - L(current)|
and writes the numbers to gpurun_out/rigid_error_<workload>.json (summarised in DESIGN.md).
"""
import json
import os

import numpy as np
import pytest

from instagraal_b200.synth import make_workload, workload_params
from parity_common import FIELDS13, OracleTeacher, score_tol, state_mismatch_modulo_length_ties

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG_E = 0.43429448190325182


def _cubin():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_kernels.cubin"))


_levels = {}


def level_of(name):
    if name not in _levels:
        _levels.clear()   # one large level in host memory at a time
        _levels[name] = make_workload(name)
    return _levels[name]


def burnt_state(level, p8, n_cycles, seed, start):
    """the scaffold the bench starts its timed region from: bomb + n_cycles of MCMC (device RNG), or the true assembly"""
    from test_gpu_parity import make_sampler
    if start == "true":
        return level.true_state()
    s = make_sampler(level)
    s.set_param_simu(p8)
    np.random.seed(seed)
    s.bomb_the_genome()
    frs = np.arange(level.n_frags)
    for c in range(n_cycles):
        np.random.shuffle(frs)
        s.run_cycle_device(frs, 5, seed=seed, cycle=c)
    st = s._get_state()
    s.free_gpu()
    return st


def current_total_likelihood(s):
    """L(current scaffold) = Lnz + Lz as eval_likelihood_4_nuisance assembles it (CL:1296-1344) under the live parameters"""
    import ctypes as C
    from instagraal_b200 import _lib as L
    out = np.zeros(3, dtype=np.float64)
    p = np.ascontiguousarray(np.array(list(s.param_simu[0]), dtype=np.float32))
    L.check(s._h, L.lib().ig_full_likelihood(s._h, p.ctypes.data_as(C.c_void_p), 0, out.ctypes.data_as(C.c_void_p)), "ig_full_likelihood")
    v_inter = float(p[7])
    return out[0] + out[1] * LOG_E + LOG_E * (float(s.n_pixl_sub_mat) - np.int32(out[2])) * -1.0 * v_inter


def lockstep_vs_reference_kernels(level, p8, state13, n_steps, seed, probes=(), raw_slice_order=False):
    """returns dict(worst_rel, ties, same, probe_stats).

    The reference's kernels run with the order of the sliced contacts inside a row pinned to ascending column
    (RefReplaySampler(canonical_slice_order=True)): on a GPU that order is decided by the execution order of slice_sp_mat's
    atomicAdd and changes from run to run, and through eval_sub_likelihood's last-block quirk (KA:4362) it changes the scores
    of the uniq positions >= n_sub % 64.  raw_slice_order=True keeps the reference's own (arbitrary) order and checks that
    every disagreement is confined to exactly those positions (then nothing else of the step is compared).

    Where the reference's kernels are not built, the teacher is its NumPy port (parity_common.OracleTeacher) and scores,
    ties and the chosen move's likelihood are compared at the port's tolerance."""
    from oracle.ref_replay import RefReplaySampler
    from oracle.sampler_oracle import return_neighbours, setup_distri_frags
    from test_gpu_parity import GpuImpl
    kernels = _cubin()
    assert kernels or not raw_slice_order
    ref = RefReplaySampler(level, p8, backend="gpu", canonical_slice_order=not raw_slice_order) if kernels else OracleTeacher(level, p8)
    tie = 1e-9 if kernels else 2e-8
    order_dependent_steps = 0
    mine = GpuImpl(level)
    extra = {name: GpuImpl(level, **kw) for name, kw in probes}
    for impl in [mine] + list(extra.values()):
        impl.set_params(p8)
    ref.set_state(state13)
    distri = setup_distri_frags(level.sub_sampled_sparse_matrix, level.n_frags)
    rng = np.random.RandomState(seed)
    frs = rng.permutation(level.n_frags)
    np.random.seed(seed)
    worst, ties, same = 0.0, 0, 0
    stats = {name: dict(err_abs=[], err_vs_best=[], err_vs_cur=[], flips=0) for name in extra}
    state = np.ascontiguousarray(state13, dtype=np.int32)
    t = 0
    for f in frs:
        if t >= n_steps:
            break
        f = int(f)
        cands = sorted(int(c) for c in return_neighbours(distri, level.n_frags, f, 5) if int(c) != f)
        if not cands:
            continue
        valid = ref.valid_insert.get().copy()
        mine.set_state(state)
        mine.set_valid(valid)
        l_cur = None
        for name, impl in extra.items():
            impl.set_state(state)
            impl.set_valid(valid)
            if l_cur is None:
                l_cur = current_total_likelihood(impl.s)
                impl.set_state(state)   # (ig_full_likelihood refreshed the coordinates; start the step from scratch)
                impl.set_valid(valid)
        o, dist, op, b, mean_len, nc = ref.step_sampler(f, cands)
        sa = np.asarray(ref.all_scores, dtype=np.float64)
        r = mine.step(f, cands)
        sb = np.asarray(r["scores"], dtype=np.float64)
        assert np.array_equal(sa != 0, sb != 0), (t, f, cands)
        nz = sa != 0
        relv = np.zeros_like(sa)
        relv[nz] = np.abs(sa[nz] - sb[nz]) / np.abs(sa[nz])
        if raw_slice_order and relv.max() >= 1e-9:
            n_sub = mine.s.n_sub_vals
            for g in np.nonzero(relv >= 1e-9)[0]:
                k, op = divmod(int(g), 24)
                pos_in_uniq = int(np.count_nonzero(nz[k * 24:k * 24 + op]))
                r = int(n_sub[k]) % 64
                assert r > 0 and pos_in_uniq >= r, ("disagreement outside the order-dependent uniq positions", t, f, cands, k, op, pos_in_uniq, r, float(relv[g]))
            order_dependent_steps += 1
            state = ref.get_state()
            t += 1
            continue
        rel = float(relv.max())
        worst = max(worst, rel)
        if kernels:
            assert rel < 1e-9, (t, f, cands, rel)
        else:
            assert np.all(np.abs(sa[nz] - sb[nz]) <= score_tol(sa[nz])), (t, f, cands, rel)
        gid_ref = cands.index(int(b)) * 24 + int(op)
        gid = cands.index(int(r["B"])) * 24 + int(r["op"])
        new_state = ref.get_state()
        if gid == gid_ref:
            same += 1
            got = mine.get_state()
            bad = state_mismatch_modulo_length_ties(got, new_state)   # (on a GPU the reference's labels of equal-length contigs are arbitrary)
            assert not bad, (t, f, cands, op, b, bad)
            assert float(r["dist"]) == float(dist), (t, r["dist"], dist)
            assert int(r["n_contigs"]) == int(nc), (t, r["n_contigs"], nc)
            assert np.float32(r["mean_len"]) == np.float32(mean_len), (t, r["mean_len"], mean_len)
            assert abs(float(r["o"]) - float(o)) <= tie * abs(float(o)), (t, r["o"], o)
        else:
            gap = abs(sa[gid] - sa[gid_ref])
            assert gap <= tie * abs(sa[gid_ref]), ("different move without a tie", t, gid, gid_ref, float(gap))
            ties += 1
        for name, impl in extra.items():
            rr = impl.step(f, cands)
            sr = np.asarray(rr["scores"], dtype=np.float64)
            assert np.array_equal(sa != 0, sr != 0), (name, t)
            err = np.abs(sr[nz] - sa[nz])
            best = sa[nz].max()
            st_ = stats[name]
            st_["err_abs"].append(float(err.max()))
            st_["err_vs_best"].append(float(np.max(err / np.maximum(np.abs(sa[nz] - best), 1e-3))))
            st_["err_vs_cur"].append(float(np.max(err / np.maximum(np.abs(sa[nz] - l_cur), 1e-3))))
            gid_r = cands.index(int(rr["B"])) * 24 + int(rr["op"])
            if gid_r != gid_ref and abs(sa[gid_r] - sa[gid_ref]) > 1e-9 * abs(sa[gid_ref]):
                st_["flips"] += 1
        state = new_state
        t += 1
    for impl in [mine] + list(extra.values()):
        impl.s.free_gpu()
    return dict(worst_rel=worst, ties=ties, same=same, steps=t, probes=stats, order_dependent_steps=order_dependent_steps)


def _dump(name, obj):
    d = os.path.join(ROOT, "gpurun_out")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, name), "w") as fh:
        json.dump(obj, fh, indent=1)


def _probe_summary(stats):
    out = {}
    for name, st in stats.items():
        out[name] = {k: {"max": float(np.max(v)), "median": float(np.median(v))} for k, v in st.items() if k != "flips" and len(v)}
        out[name]["different_move_without_tie"] = st["flips"]
    return out


def test_T_full_cycle_from_the_bench_state(built):
    """config T: one full MCMC cycle (NF steps) from the bench's burnt-in state (bomb + 2 cycles)"""
    level = level_of("T")
    p8 = workload_params(level)
    st = burnt_state(level, p8, 2, 1000, "bomb")
    res = lockstep_vs_reference_kernels(level, p8, st, level.n_frags, seed=3, probes=(("rigid", dict(rigid_pruning=True)),))
    _dump("rigid_error_T.json", dict(workload="T", steps=res["steps"], ties=res["ties"], worst_rel=res["worst_rel"],
                                     probes=_probe_summary(res["probes"])))
    assert res["steps"] >= level.n_frags - 5
    assert res["same"] >= 0.9 * res["steps"], res


@pytest.mark.skipif(not _cubin(), reason="reference cubin not built")
def test_T_reference_own_slice_order_only_moves_the_last_block_positions(built):
    """The reference with its OWN order of the sliced contacts (atomic order on the GPU, not reproducible run to run): over
    400 steps every disagreement with the product sits on uniq positions >= n_sub % 64 of a candidate -- the proposals whose
    sum drops the final 64-thread block (KA:4362), i.e. whose value depends on WHICH contacts happen to be last."""
    level = level_of("T")
    p8 = workload_params(level)
    st = burnt_state(level, p8, 2, 1000, "bomb")
    res = lockstep_vs_reference_kernels(level, p8, st, 400, seed=3, raw_slice_order=True)
    _dump("reference_slice_order_T.json", dict(workload="T", steps=res["steps"], order_dependent_steps=res["order_dependent_steps"],
                                               ties=res["ties"], worst_rel_elsewhere=res["worst_rel"]))
    assert res["steps"] == 400


def test_Y3_200_steps(built):
    level = level_of("Y3")
    p8 = workload_params(level)
    st = burnt_state(level, p8, 2, 1000, "bomb")
    res = lockstep_vs_reference_kernels(level, p8, st, 200, seed=4)
    assert res["steps"] == 200 and res["same"] >= 0.9 * res["steps"], res


@pytest.mark.parametrize("start", ["bomb", "true"])
def test_G_steps_and_rigid_pruning_error(built, start):
    """config G (the ~1 Gb level the north-star target is stated on): 10 steps from the mid-assembly start (bomb + 3
    cycles) and from the fully assembled start; also measures the score error of rigid pruning (D2).  With the reference's
    NumPy port as teacher (~30 s a step at this level on one host core) the default is 3 steps."""
    level = level_of("G")
    p8 = workload_params(level)
    n_burn = int(os.environ.get("IG_TEST_G_BURN", "3"))
    st = burnt_state(level, p8, n_burn, 1000, start)
    n_steps = int(os.environ.get("IG_TEST_G_STEPS", "10" if _cubin() else "3"))
    res = lockstep_vs_reference_kernels(level, p8, st, n_steps, seed=5, probes=(("rigid", dict(rigid_pruning=True)),))
    _dump("rigid_error_G_%s.json" % start, dict(workload="G", start=start, burn_cycles=n_burn, steps=res["steps"], ties=res["ties"],
                                               worst_rel=res["worst_rel"], n_contigs=int((st[0] == 0).sum()),
                                               probes=_probe_summary(res["probes"])))
    assert res["steps"] == n_steps, res
