"""Steps of more than IG_MAX_CANDS (8) candidate neighbours, up to IG_MAX_NEIGHBOURS (64): ig_step_wide, ig_run_cycle_wide and
the wide device plans of ig_run_cycle_device / ig_run_cycles_device_multi, through sampler.step_sampler, run_cycle,
run_cycle_device and ReplicaSet.run_cycle.  CPU: the wide device draws (NumPy restatement) and the limits.  GPU: lockstep
with the oracle (which has no candidate limit) on every scoring path, and equality with the narrow code where both apply."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from instagraal_b200.synth import WORKLOADS, SynthSpec, make_level
from oracle import device_rng
from parity_common import FIELDS13

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = np.float32(0.01)


# ---------------------------------------------------------------------------------------------------------------- CPU
def _weights(nf, rng, n_min=0, n_max=40):
    """a neighbour-weight CSR like neighbour_weights_csr: per fragment a few weighted neighbours (some with zero weight),
    a few fragments without any"""
    ptr, idx, cdf, nnz = [0], [], [], []
    for a in range(nf):
        k = int(rng.randint(n_min, n_max + 1)) if a % 7 else 0
        nb = rng.choice(np.setdiff1d(np.arange(nf), [a]), k, replace=False)
        w = rng.gamma(0.7, size=k)
        w[rng.rand(k) < 0.1] = 0.0
        if k and w.sum() == 0:
            w[0] = 1.0
        pk = w / w.sum() if k else w
        idx.append(nb.astype(np.int32))
        cdf.append(np.cumsum(pk))
        nnz.append(int(np.count_nonzero(pk)))
        ptr.append(ptr[-1] + k)
    return (np.array(ptr, np.int64), np.concatenate(idx).astype(np.int32), np.concatenate(cdf), np.array(nnz, np.int32))


def test_wide_plan_first_eight_draws_are_the_narrow_plan():
    """draw i keeps the counter (t, cycle, i, attempt): the narrow plan's candidates are among the wide plan's, and for
    delta <= 8 the wide plan is the narrow plan padded with zeros"""
    rng = np.random.RandomState(3)
    nf = 90
    ptr, idx, cdf, nnz = _weights(nf, rng)
    frags = rng.permutation(nf).astype(np.int32)
    seed = 0x0123_4567_89AB_CDEF
    for cycle in (0, 7):
        narrow = device_rng.draw_plan(frags, 8, nf, ptr, idx, cdf, nnz, seed, cycle)
        for delta in (9, 12, 24, 64):
            wide = device_rng.draw_plan(frags, delta, nf, ptr, idx, cdf, nnz, seed, cycle, max_cands=64)
            assert wide.shape == (nf, 66)
            for t in range(nf):
                n_w, n_n = wide[t, 0], narrow[t, 0]
                got = set(wide[t, 2:2 + n_w].tolist())
                assert set(narrow[t, 2:2 + n_n].tolist()) <= got, (cycle, delta, t)
                assert n_w <= delta and np.all(wide[t, 2 + n_w:] == 0)
                assert list(wide[t, 2:2 + n_w]) == sorted(got) and frags[t] not in got
                a = frags[t]
                want_n = min(delta, int(nnz[a])) if ptr[a + 1] > ptr[a] else min(delta, nf - 1)
                assert n_w == want_n, (t, n_w, want_n)
        for delta in (1, 5, 8):
            wide = device_rng.draw_plan(frags, delta, nf, ptr, idx, cdf, nnz, seed, cycle, max_cands=64)
            small = device_rng.draw_plan(frags, delta, nf, ptr, idx, cdf, nnz, seed, cycle)
            assert np.array_equal(wide[:, :10], small) and not wide[:, 10:].any()


def test_wide_plan_draw_frequencies_follow_the_weights():
    """inclusion frequencies of a 12-of-30 draw without replacement equal those of NumPy's choice(replace=False, p)
    (what return_neighbours does), over many steps and seeds"""
    rng = np.random.RandomState(8)
    nf, a = 40, 0
    nb = np.arange(1, 31, dtype=np.int32)
    w = rng.gamma(0.8, size=30)
    w[[3, 17]] = 0.0
    pk = w / w.sum()
    ptr = np.zeros(nf + 1, np.int64)
    ptr[a + 1:] = 30
    cdf = np.cumsum(pk)
    nnz = np.zeros(nf, np.int32)
    nnz[a] = 28
    n_rep, delta = 1500, 12
    got = np.zeros(nf)
    for seed in (1, 2):
        plan = device_rng.draw_plan(np.zeros(n_rep, np.int32), delta, nf, ptr, nb, cdf, nnz, seed, 0, max_cands=64)
        assert np.all(plan[:, 0] == delta)
        for row in plan:
            got[row[2:2 + delta]] += 1
    got /= 2 * n_rep
    ref = np.zeros(nf)
    rs = np.random.RandomState(5)
    n_ref = 6000
    for _ in range(n_ref):
        ref[rs.choice(nb, delta, replace=False, p=pk)] += 1
    ref /= n_ref
    assert got[1 + 3] == 0 and got[1 + 17] == 0
    assert np.max(np.abs(got - ref)) < 0.05, np.max(np.abs(got - ref))


def test_neighbour_limit_is_sixty_four():
    from instagraal_b200 import _lib as L
    from instagraal_b200.cuda_lib_gl_single import sampler
    hdr = open(os.path.join(ROOT, "include", "instagraal_b200.h")).read()
    assert int(re.search(r"#define IG_MAX_NEIGHBOURS (\d+)", hdr).group(1)) == L.IG_MAX_NEIGHBOURS == 64
    assert int(re.search(r"#define IG_MAX_CANDS (\d+)", hdr).group(1)) == L.IG_MAX_CANDS == 8
    assert sampler._usable_candidates(None, 0, range(0, 65)) == list(range(1, 65))   # the visited fragment is dropped
    with pytest.raises(ValueError, match="at most 64"):
        sampler._usable_candidates(None, 0, range(1, 66))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _mk(level, **kw):
    from test_gpu_parity import make_sampler
    return make_sampler(level, **kw)


def _wide_lockstep(level, p8, n_steps, seed, n_neigh, rigid=False, path=None):
    """product and oracle advance together on steps of exactly n_neigh random candidates; besides the checks of
    test_gpu_parity._lockstep: the chosen move is the first index of the maximum non-zero score, its score is the step's
    likelihood, and the carried validity list equals the oracle's before any resynchronisation (quirk Q3).  rigid: scores
    within the rigid mode's coordinate-rounding noise; path: the scoring path the product must have taken.  Returns (ties,
    steps won by a candidate of batch >= 1)."""
    from test_gpu_parity import _oracle, assert_scoring_path
    s = _mk(level, rigid_pruning=rigid)
    s.set_param_simu(p8)
    o = _oracle(level, p8)
    np.random.seed(seed)
    s.bomb_the_genome()
    o.live = {k: s._get_state()[i].copy() for i, k in enumerate(FIELDS13)}
    o.valid = [int(x) for x in s.get_valid_insert()]
    rng = np.random.RandomState(seed + 1000)
    ties = later = 0
    for _ in range(n_steps):
        a = int(rng.randint(level.n_frags))
        cands = sorted(int(c) for c in rng.choice(level.n_frags, n_neigh + 1, replace=False) if c != a)[:n_neigh]
        r = s.step_sampler(a, n_neigh, DT, candidates=cands)
        ro = o.step_sampler(a, n_neigh, candidates=cands)
        want, got = o.all_scores, s.all_scores
        assert len(got) == 24 * n_neigh and len(s.n_uniq) == n_neigh and len(s.n_sub_vals) == n_neigh
        assert np.array_equal(want != 0, got != 0), (a, cands)
        nz = want != 0
        if rigid:
            tol = 2e-6 * np.abs(want[nz]) + 1e-9
        else:
            tol = 1e-5 * np.abs(want[nz] - want[nz].max()) + 2e-8 * np.abs(want[nz]) + 1e-9
        assert np.all(np.abs(got[nz] - want[nz]) <= tol), (a, cands, float(np.max(np.abs(got[nz] - want[nz]))))
        gid = cands.index(int(r[3])) * 24 + int(r[2])
        assert gid == int(np.argmax(np.where(got != 0, got, -np.inf))), (a, gid)
        assert float(r[0]) == got[gid]
        later += gid >= 8 * 24
        st = s._get_state()
        if (int(r[2]), int(r[3])) == (int(ro[2]), int(ro[3])):
            for i, k in enumerate(FIELDS13):
                assert np.array_equal(st[i], o.live[k]), (a, k)
            assert float(r[1]) == float(ro[1]) and int(r[5]) == int(ro[5])
            assert list(s.get_valid_insert()) == [int(x) for x in o.valid], (a, cands)
        else:
            gid_o = cands.index(int(ro[3])) * 24 + int(ro[2])
            gap = abs(want[gid] - want[gid_o])
            assert gap <= (4e-6 if rigid else 2e-8) * abs(want[gid_o]) + 1e-9, "diverged without a tie"
            ties += 1
            o.live = {k: st[i].copy() for i, k in enumerate(FIELDS13)}
        o.valid = [int(x) for x in s.get_valid_insert()]
    if path:
        assert_scoring_path(s, path, rigid)
    s.free_gpu()
    return ties, later


@pytest.mark.gpu
@pytest.mark.parametrize("n_neigh", [9, 12, 16, 24])
def test_wide_lockstep_toy(built, n_neigh):
    from test_gpu_parity import P8
    ties, later = _wide_lockstep(make_level(WORKLOADS["toy"]), P8, 40, seed=n_neigh, n_neigh=n_neigh, path="flat")
    assert ties <= 20


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"IG_SCORING_PATH": "rows"}, {"IG_SCORING_PATH": "rows", "IG_FORCE_SPLIT": "24,1"}])
@pytest.mark.parametrize("n_neigh", [9, 12, 16, 24])
def test_wide_lockstep_large_level_paths_on_toy(built, env, n_neigh, monkeypatch):
    """the two-pass affected-row list and the row-per-warp kernel of the largest levels (rows path), with its adaptive
    and its whole-row work split"""
    from test_gpu_parity import P8_RIPPE
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ties, _ = _wide_lockstep(make_level(WORKLOADS["toy"]), P8_RIPPE, 30, seed=40 + n_neigh, n_neigh=n_neigh, path="rows")
    assert ties <= 15


@pytest.mark.gpu
@pytest.mark.parametrize("n_neigh", [9, 12, 16, 24])
def test_wide_lockstep_medium_level(built, n_neigh):
    """6000 fragments / 18k sub-fragments: the two-pass affected-row list and the streaming path of large levels, which
    leaves the candidates that involve a circular contig to the row-per-warp kernel"""
    from test_gpu_parity import P8_RIPPE
    level = make_level(SynthSpec(n_frags=6000, n_contigs=12, n_chrom=2, max_offset=300, lambda1=30.0, trans_per_row=2.0, seed=11))
    ties, _ = _wide_lockstep(level, P8_RIPPE, 4, seed=3, n_neigh=n_neigh, path="stream")
    assert ties <= 2


@pytest.mark.gpu
@pytest.mark.parametrize("rigid", [True, False])
@pytest.mark.parametrize("n_neigh", [9, 12, 16, 24])
def test_wide_lockstep_streaming_path(built, n_neigh, rigid, monkeypatch):
    from test_gpu_parity import P8
    monkeypatch.setenv("IG_SCORING_PATH", "stream")
    ties, _ = _wide_lockstep(make_level(WORKLOADS["toy"]), P8, 30, seed=70 + n_neigh, n_neigh=n_neigh, rigid=rigid, path="stream")
    assert ties <= 15


@pytest.mark.gpu
def test_wide_step_first_batch_equals_narrow_step_and_winner_is_global_first_argmax(built):
    """from the same state, the first 8 x 24 scores of a 20-candidate step are bit for bit those of an 8-candidate step on
    the first 8 candidates; the applied move is the first index of the maximum over all 480 scores (its score is the
    step's likelihood), and over the run candidates of later batches win some steps"""
    from test_gpu_parity import P8
    level = make_level(WORKLOADS["toy"])
    w, n8 = _mk(level), _mk(level)
    for s in (w, n8):
        s.set_param_simu(P8)
    np.random.seed(12)
    w.bomb_the_genome()
    rng = np.random.RandomState(13)
    later = 0
    for t in range(60):
        st, valid = w._get_state(), w.get_valid_insert()
        for s in (w, n8):   # both refresh fully: same summation order
            s._set_state(st)
            s.set_valid_insert(valid)
        a = int(rng.randint(level.n_frags))
        cands = sorted(int(c) for c in rng.choice(level.n_frags, 21, replace=False) if c != a)[:20]
        n8.step_sampler(a, 8, DT, candidates=cands[:8])
        r = w.step_sampler(a, 20, DT, candidates=cands)
        assert np.array_equal(w.all_scores[:8 * 24].view(np.int64), n8.all_scores.view(np.int64)), t
        assert w.n_uniq[:8] == n8.n_uniq and w.n_sub_vals[:8] == n8.n_sub_vals
        sc = w.all_scores
        gid = cands.index(int(r[3])) * 24 + int(r[2])
        assert gid == int(np.argmax(np.where(sc != 0, sc, -np.inf))) and float(r[0]) == sc[gid]
        assert w._res.cand_index == gid // 24
        later += gid >= 8 * 24
    assert later >= 3, later
    for s in (w, n8):
        s.free_gpu()


@pytest.mark.gpu
def test_wide_incremental_likelihood_equals_full_recompute(built):
    """200+ steps of 12 candidates (winners in later batches included): incremental maintenance after a re-scored batch
    == the full recomputation every step, up to f64 summation order"""
    from test_gpu_parity import P8_RIPPE
    level = make_level(WORKLOADS["T"])
    runs = []
    for refresh, graph in ((1, False), (0, True)):
        s = _mk(level)
        s.set_options(refresh_every=refresh, use_graph=graph)
        s.set_param_simu(P8_RIPPE)
        np.random.seed(11)
        s.bomb_the_genome()
        rng = np.random.RandomState(5)
        out = []
        for _ in range(220):
            a = int(rng.randint(level.n_frags))
            cands = sorted(int(c) for c in rng.choice(level.n_frags, 13, replace=False) if c != a)[:12]
            r = s.step_sampler(a, 12, DT, candidates=cands)
            out.append((float(r[0]), int(r[2]), int(r[3]), int(r[5]), np.sort(s.all_scores[s.all_scores != 0])[-2:].copy()))
        runs.append(out)
        if refresh == 0:
            assert s.get_stats()["full_refreshes"] <= 1
        s.free_gpu()
    n_same = 0
    for a, b in zip(*runs):
        if a[1:4] != b[1:4]:
            top = a[4]
            assert abs(top[-1] - top[-2]) <= 1e-9 * abs(top[-1]), ("diverged without a tie", n_same, a, b)
            break
        assert abs(a[0] - b[0]) <= 1e-9 * abs(a[0]), (n_same, a[0], b[0])
        n_same += 1
    assert n_same >= 200, n_same


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [True, False])
def test_wide_run_cycle_equals_stepwise(built, use_graph):
    """ig_run_cycle_wide (steps of 3 to 30 candidates, narrow and wide mixed in one cycle) == the same steps through
    step_sampler, records and final state bit for bit"""
    from test_gpu_parity import P8
    level = make_level(WORKLOADS["toy"])
    rng = np.random.RandomState(21)
    perm = np.random.RandomState(1).permutation(level.n_frags).astype(np.int32)
    frs = np.concatenate([rng.permutation(level.n_frags) for _ in range(2)])
    cands = []
    for f in frs:
        n = int(rng.choice([3, 8, 9, 12, 17, 30]))
        cands.append(sorted(int(c) for c in rng.choice(level.n_frags, n + 1, replace=False) if c != f)[:n])
    res = []
    from instagraal_b200 import _lib as L
    for mode in ("step", "cycle"):
        s = _mk(level)
        s.set_options(use_graph=use_graph)
        s.set_param_simu(P8)
        L.check(s._h, L.lib().ig_bomb(s._h, perm.ctypes.data_as(C.c_void_p)), "ig_bomb")
        if mode == "step":
            out = [s.step_sampler(int(f), len(c), DT, candidates=c) for f, c in zip(frs, cands)]
            rec = [(float(o[0]), float(o[1]), int(o[2]), int(o[3]), int(o[5])) for o in out]
            n_prop = s.n_proposals_scored
        else:
            out = s.run_cycle(frs, 5, candidates=cands)
            rec = [(float(r["likelihood"]), float(r["dist"]), int(r["op_sampled"]), int(r["id_f_sampled"]), int(r["n_contigs"]))
                   for r in out]
            n_prop = int(out["n_proposals"].sum())
            plan = s.last_cycle_plan(len(frs))
            assert plan.shape == (len(frs), 32)
            assert all(plan[t, 2:2 + plan[t, 0]].tolist() == cands[t] for t in range(len(frs)))
            assert np.array_equal(out["cand_index"], [cands[t].index(int(out["id_f_sampled"][t])) for t in range(len(frs))])
        res.append((rec, n_prop, s._get_state(), s.get_valid_insert()))
        s.free_gpu()
    assert res[0][0] == res[1][0]
    assert res[0][1] == res[1][1]
    assert np.array_equal(res[0][2], res[1][2])
    assert np.array_equal(res[0][3], res[1][3])


def _bombed(level, p8, seed=4):
    s = _mk(level)
    s.set_param_simu(p8)
    np.random.seed(seed)
    s.bomb_the_genome()
    return s


@pytest.mark.gpu
def test_wide_device_cycle_matches_restated_plan_and_host_plan_run(built):
    """run_cycle_device(n_neighbours=12): the plan equals draw_plan(max_cands=64), and the chain equals run_cycle fed that
    plan on a separate handle, bit for bit"""
    from test_gpu_parity import P8_RIPPE
    level = make_level(WORKLOADS["toy"])
    a, b = _bombed(level, P8_RIPPE), _bombed(level, P8_RIPPE)
    rng = np.random.RandomState(22)
    seed = 0x1234_5678_9ABC_DEF0
    n_wide = 0
    for cyc in range(2):
        frags = rng.permutation(level.n_frags).astype(np.int32)
        out_dev = a.run_cycle_device(frags, 12, seed=seed, cycle=cyc)
        plan = a.last_cycle_plan(len(frags), width=64)
        ptr, idx, cdf, nnz = a.neighbour_weights_csr()
        want = device_rng.draw_plan(frags, 12, level.n_frags, ptr, idx, cdf, nnz, seed, cyc, max_cands=64)
        assert np.array_equal(plan, want)
        assert np.array_equal(a.last_cycle_plan(len(frags)), want[:, :14])
        n_wide += int((plan[:, 0] > 8).sum())
        cands = [plan[t, 2:2 + plan[t, 0]].tolist() for t in range(len(frags))]
        out_host = b.run_cycle(frags, 12, candidates=cands)
        for f in ("op_sampled", "id_f_sampled", "cand_index", "n_contigs", "sum_l_cont", "n_proposals", "likelihood", "dist"):
            assert np.array_equal(out_dev[f], out_host[f]), f
        assert np.array_equal(a._get_state(), b._get_state())
        assert np.array_equal(a.get_valid_insert(), b.get_valid_insert())
    assert n_wide > 0
    for s in (a, b):
        s.free_gpu()


@pytest.mark.gpu
def test_wide_device_cycle_with_nuisance_equals_host_driven_sequence(built):
    """run_cycle_device(n_neighbours=12, nuisance=True) on handle a; handle b runs a's plan through step_sampler, evaluates
    a's nuisance proposals and takes a's decisions: likelihoods, moves, parameters and scaffold agree bit for bit"""
    from instagraal_b200.cuda_lib_gl_single import PARAM_SIMU_RIPPE
    from test_gpu_parity import P8_RIPPE
    level = make_level(WORKLOADS["toy"])
    a, b = _bombed(level, P8_RIPPE), _bombed(level, P8_RIPPE)
    rng = np.random.RandomState(23)
    seed = 99
    n_acc = 0
    for cycle in range(2):
        frags = rng.permutation(level.n_frags).astype(np.int32)
        steps, nuis = a.run_cycle_device(frags, 12, seed=seed, cycle=cycle, nuisance=True)
        plan = a.last_cycle_plan(len(frags))
        ptr, idx, cdf, nnz = a.neighbour_weights_csr()
        assert np.array_equal(plan, device_rng.draw_plan(frags, 12, level.n_frags, ptr, idx, cdf, nnz, seed, cycle, max_cands=12))
        for t in range(len(frags)):
            r = nuis[t]
            cands = plan[t, 2:2 + plan[t, 0]].tolist()
            o, dist, op, fid, _ml, n_contigs = b.step_sampler(int(plan[t, 1]), 12, DT, candidates=cands)
            assert o == steps["likelihood"][t] and dist == steps["dist"][t], (cycle, t)
            assert op == steps["op_sampled"][t] and fid == steps["id_f_sampled"][t] and n_contigs == steps["n_contigs"][t]
            b.param_simu_test = np.array([tuple(r["p_test"].tolist())], dtype=PARAM_SIMU_RIPPE)
            l_nuis = b.eval_likelihood_4_nuisance()
            assert l_nuis == r["likelihood_nuis"] or (np.isnan(l_nuis) and np.isnan(r["likelihood_nuis"])), (cycle, t)
            if r["success"]:
                b.set_param_simu(r["p_test"])
                b.likelihood_t = l_nuis
                n_acc += 1
        assert np.array_equal(np.array(list(a.param_simu[0]), np.float32), np.array(list(b.param_simu[0]), np.float32))
        assert np.array_equal(a._get_state(), b._get_state()), cycle
    assert n_acc > 0
    for s in (a, b):
        s.free_gpu()


@pytest.mark.gpu
@pytest.mark.parametrize("nuisance", [False, True])
def test_wide_replica_set_equals_separate_handles(built, nuisance):
    from instagraal_b200.replicas import ReplicaSet
    from test_gpu_parity import P8_RIPPE
    level = make_level(WORKLOADS["toy"])
    n = 3
    rng = np.random.RandomState(77)
    frags = np.stack([rng.permutation(level.n_frags) for _ in range(n)]).astype(np.int32)
    seeds = np.array([5, 6, 7], dtype=np.uint64)
    want, want_state = [], []
    for i in range(n):
        s = _mk(level)
        s.set_gpu_share(3)   # what ReplicaSet gives each of 3 chains
        s.set_param_simu(P8_RIPPE)
        np.random.seed(200 + i)
        s.bomb_the_genome()
        r = s.run_cycle_device(frags[i], 12, seed=int(seeds[i]), cycle=5, nuisance=nuisance)
        want.append(r)
        want_state.append(s._get_state())
        s.free_gpu()
    first = _mk(level)
    first.set_param_simu(P8_RIPPE)
    rs = ReplicaSet(first, n, seeds=seeds)
    rs.bomb(seed0=200)
    got = rs.run_cycle(frags, 12, cycle=5, nuisance=nuisance)
    for i in range(n):
        g, w = (got[0][i], want[i][0]) if nuisance else (got[i], want[i])
        for key in ("likelihood", "dist", "op_sampled", "id_f_sampled", "cand_index", "n_contigs", "n_proposals"):
            assert np.array_equal(g[key], w[key]), (i, key)
        if nuisance:
            assert got[1][i].tobytes() == want[i][1].tobytes(), i
        assert np.array_equal(rs.chains[i]._get_state(), want_state[i]), i
        assert rs.chains[i].last_cycle_plan(len(frags[i])).shape == (len(frags[i]), 14)
    rs.free()


@pytest.mark.gpu
def test_wide_refusals(built):
    """more than 64 neighbours, a candidate array narrower than a step's list, a candidate equal to the visited fragment"""
    from instagraal_b200 import _lib as L
    from test_gpu_parity import P8
    level = make_level(WORKLOADS["toy"])
    s = _bombed(level, P8)
    lib = L.lib()
    c65 = np.arange(1, 66, dtype=np.int32)
    res = L.ig_step_result()
    buf = np.zeros(65 * 24)
    nb = np.zeros(65, np.int32)
    ptr = lambda x: x.ctypes.data_as(C.c_void_p)   # noqa: E731
    assert lib.ig_step_wide(s._h, 0, ptr(c65), 65, C.byref(res), ptr(buf), ptr(nb), ptr(nb)) == -1
    assert b"64" in lib.ig_last_error(s._h)
    c12 = np.arange(1, 13, dtype=np.int32)
    c12[5] = 0
    assert lib.ig_step_wide(s._h, 0, ptr(c12), 12, C.byref(res), ptr(buf), ptr(nb), ptr(nb)) == -1
    assert b"visited fragment" in lib.ig_last_error(s._h)
    frags = np.array([0, 1], np.int32)
    cands = np.arange(2, 2 + 2 * 12, dtype=np.int32).reshape(2, 12)
    nc = np.array([12, 12], np.int32)
    out = np.zeros(2, dtype=L.CYCLE_DTYPE)
    assert lib.ig_run_cycle_wide(s._h, 2, ptr(frags), ptr(cands), 10, ptr(nc), ptr(out)) == -1
    assert b"width" in lib.ig_last_error(s._h)
    assert lib.ig_run_cycle_wide(s._h, 2, ptr(frags), ptr(cands), 65, ptr(nc), ptr(out)) == -1
    cands[1, 3] = 1
    assert lib.ig_run_cycle_wide(s._h, 2, ptr(frags), ptr(cands), 12, ptr(nc), ptr(out)) == -1
    assert b"visited fragment" in lib.ig_last_error(s._h)
    with pytest.raises(RuntimeError, match="n_neighbours out of range"):
        s.run_cycle_device(np.arange(10, dtype=np.int32), 65, seed=1)
    with pytest.raises(ValueError, match="at most 64"):
        s.step_sampler(0, 65, DT, candidates=list(range(1, 66)))
    # nothing was changed by the refused calls: a valid wide step still runs
    s.step_sampler(0, 12, DT, candidates=list(range(1, 13)))
    assert len(s.all_scores) == 12 * 24
    s.free_gpu()
