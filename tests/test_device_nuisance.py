"""The nuisance-parameter step of the production RNG mode (ig_set_device_nuisance, sampler.run_cycle_device(nuisance=True),
ReplicaSet.run_cycle(nuisance=True)): its NumPy restatement (oracle/device_nuisance.py) on the CPU, then the device against
the restatement and against the host-driven sequence fed the same numbers."""
import math
import types
import warnings

import numpy as np
import pytest
from scipy.optimize import brentq, fsolve

from oracle import device_nuisance as dn
from oracle import device_rng

P8 = np.array([2.2354, 1.4933294, 0.06928191, -0.9384134, 2.0, 386.88467, 65.71848, 0.01698581], dtype=np.float32)
P8_RIPPE = np.array([50.0, 9.6, np.float32(0.53 * (9.6 / 50.0) ** -1.5 * 50.0 ** -3), -1.5, 2.0, 900.0, 4.0e5, 0.02],
                    dtype=np.float32)


def _rippe(x, kuhn, lm, slope, dd, A):
    q = lm * x / kuhn
    return A * (0.53 * kuhn ** -3.0 * q ** slope * math.exp((dd - 2.0) / (q * q + dd)))


def _param_grid():
    """realistic parameter sets: the two P8 of the tests, each moved by -2, 0, +2 proposal sigmas in fact / slope / d_nuc"""
    out = []
    for base in (P8, P8_RIPPE):
        kuhn, lm, c1, slope, d, d_max, fact, v = (float(x) for x in base)
        for kf in (-2, 0, 2):
            for ks in (-2, 0, 2):
                for kv in (-2, 0, 2):
                    out.append((kuhn, lm, slope + ks * 0.005, fact + kf * fact / 100.0, v + kv * v / 100.0))
    return out


# ------------------------------------------------------------------ CPU: the restatement
def test_draw_frequencies_and_normal_moments():
    ids, zs = [], []
    for t in range(20000):
        i, u, z = dn.draws(t, 3, 12345)
        assert 0.0 <= u < 1.0
        ids.append(i)
        zs.append(z)
    f = np.bincount(ids, minlength=4) / len(ids)
    assert np.all(np.abs(f - 0.25) < 0.02), f
    zs = np.array(zs)
    assert abs(zs.mean()) < 0.03 and abs(zs.var() - 1.0) < 0.05, (zs.mean(), zs.var())


def test_nuisance_counters_are_disjoint_from_neighbour_counters():
    """k_draw_plan uses draw indices < IG_MAX_CANDS (8) and attempts < 256; the nuisance step uses draw >= 2^31, attempt 0"""
    ca, cb = dn.counters(17, 2)
    for c in (ca, cb):
        assert c[2] >= 0x80000000 and c[2] > 8 and c[3] == 0
    # the same (t, cycle, key) gives unrelated words in the two domains
    key = (99, 0)
    assert device_rng.philox4x32_10((17, 2, 0, 0), key) != device_rng.philox4x32_10(ca, key)


def test_root_closed_form_d2_matches_brentq():
    for kuhn, lm, slope, fact, v in _param_grid():
        x = dn.dmax_root(kuhn, lm, slope, 2.0, fact, v)
        assert x is not None and x > 0
        f = lambda s: _rippe(s, kuhn, lm, slope, 2.0, fact) - v   # noqa: E731
        lo, hi = x / 4.0, x * 4.0
        want = brentq(f, lo, hi, xtol=1e-300, rtol=4 * np.finfo(float).eps)
        assert abs(x - want) <= 1e-12 * want, (kuhn, lm, slope, fact, v, x, want)


@pytest.mark.parametrize("dd", [1.8, 2.37, 3.0])
def test_root_newton_d_not_2_matches_brentq(dd):
    for kuhn, lm, slope, fact, v in _param_grid():
        x = dn.dmax_root(kuhn, lm, slope, dd, fact, v)
        assert x is not None and x > 0
        f = lambda s: _rippe(s, kuhn, lm, slope, dd, fact) - v   # noqa: E731
        want = brentq(f, x / 4.0, x * 4.0, xtol=1e-300, rtol=4 * np.finfo(float).eps)
        assert abs(x - want) <= 1e-12 * want, (dd, kuhn, lm, slope, fact, v, x, want)


def test_root_against_fsolve_where_it_converges():
    from instagraal_b200 import rippe_fit
    n_cmp = 0
    for kuhn, lm, slope, fact, v in _param_grid():
        p32 = [np.float32(kuhn), np.float32(lm), np.float32(slope), np.float32(2.0), np.float32(fact)]
        x = dn.dmax_root(*p32[:4], p32[4], np.float32(v))
        for x0 in (x * 0.9, x * 1.1):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                sol, info, ier, msg = fsolve(rippe_fit.residual_4_max_dist, x0, args=([*p32[:4], p32[4], np.float32(v)],),
                                             full_output=True)
            if ier != 1:
                continue
            got = rippe_fit.estimate_max_dist_intra_nuis(p32, np.float32(v), x0)
            assert abs(abs(got) - x) <= 1e-6 * x, (kuhn, lm, slope, fact, v, got, x)
            n_cmp += 1
    assert n_cmp > 20


def test_root_flags_no_root_and_invalid_inputs():
    k, lm, s, A, y = 50.0, 9.6, -1.5, 4e5, 0.02
    assert dn.dmax_root(k, lm, 0.0, 2.0, A, y) is None            # slope 0: no root
    assert dn.dmax_root(k, lm, 0.01, 2.0, A, y) is None           # slope > 0
    assert dn.dmax_root(k, lm, s, 2.0, -1.0, y) is None           # fact <= 0
    assert dn.dmax_root(k, lm, s, 2.0, A, 0.0) is None            # d_nuc <= 0
    assert dn.dmax_root(k, lm, s, 2.0, A, -0.5) is None
    assert dn.dmax_root(k, lm, float("nan"), 2.0, A, y) is None   # non-finite
    assert dn.dmax_root(k, lm, s, 2.0, float("inf"), y) is None
    assert dn.dmax_root(k, lm, -1e-4, 2.0, A, y) is None          # root far beyond any double: x^(1/slope) overflows
    p = P8_RIPPE.copy()
    for id_modif, draw in ((0, -1e9), (1, 5.0), (3, -1.0), (2, -1e4)):
        q, valid = dn.propose(p, id_modif, draw)
        assert not valid, (id_modif, draw, q)


def _stub(p8):
    from instagraal_b200.cuda_lib_gl_single import PARAM_SIMU_RIPPE
    return types.SimpleNamespace(param_simu=np.array([tuple(np.asarray(p8, dtype=np.float32).tolist())], dtype=PARAM_SIMU_RIPPE))


def test_proposal_bit_identical_to_nuisance_finish_except_d_max():
    from instagraal_b200.cuda_lib_gl_single import sampler
    rng = np.random.RandomState(5)
    n = 0
    for base in (P8, P8_RIPPE):
        for it in range(60):
            p = base.copy()
            p[3] = np.float32(p[3] + rng.normal(0, 0.01))
            p[6] = np.float32(p[6] * (1 + rng.normal(0, 0.02)))
            p[7] = np.float32(p[7] * (1 + rng.normal(0, 0.02)))
            p[5] = np.float32(p[5] + rng.normal(0, 50))
            for id_modif in range(4):
                z = rng.normal()
                draw = dn.draw_of(id_modif, z, p)
                with warnings.catch_warnings(), np.errstate(all="ignore"):
                    warnings.simplefilter("ignore", RuntimeWarning)
                    want = sampler._nuisance_finish(_stub(p), id_modif, draw)
                got, valid = dn.propose(p, id_modif, draw)
                w = np.array(list(want[0]), dtype=np.float32)
                keep = [0, 1, 2, 3, 4, 6, 7] if id_modif != 2 else list(range(8))
                assert np.array_equal(got[keep].view(np.uint32), w[keep].view(np.uint32)), (id_modif, draw, got, w)
                assert valid
                n += 1
    assert n == 480


def test_sigma_agrees_with_nuisance_draws():
    """the restated sigma rounds each float32 operation once.  _nuisance_draws' NumPy float32 log10 may be an ulp off, which
    10 ** x amplifies (about 9 float32 ulps of sigma per ulp of x near x = 3.6): the two agree to 1e-5 relative"""
    for v in (P8[6], P8[7], P8_RIPPE[6], P8_RIPPE[7], np.float32(3.3e-3), np.float32(1234.5)):
        want = np.float32(10 ** (np.log10(v) - 2))
        got = dn.sigma(v)
        assert abs(float(got) - float(want)) <= 1e-5 * float(want), (v, got, want)
        assert abs(float(got) - float(v) / 100.0) <= 1e-5 * float(v) / 100.0


# ------------------------------------------------------------------ GPU
def _bombed(level, p8, seed=2, **kw):
    from test_gpu_parity import make_sampler
    s = make_sampler(level, **kw)
    s.set_param_simu(p8)
    np.random.seed(seed)
    s.bomb_the_genome()
    return s


def _orders(nf, n_cycles, seed=3):
    rng = np.random.RandomState(seed)
    return [rng.permutation(nf).astype(np.int32) for _ in range(n_cycles)]


def _restated_chain(p0, rec, cycle, seed):
    """replays the records through the restatement: every field but the likelihood is predicted from the live parameters"""
    p = np.asarray(p0, dtype=np.float32).copy()
    for t, r in enumerate(rec):
        id_modif, u, draw, q, valid = dn.step(p, t, cycle, seed)
        yield t, r, p.copy(), (id_modif, u, draw, q, valid)
        if r["accepted"]:
            p = r["p_test"].copy()


def _ulps(a, b):
    a, b = np.float32(a), np.float32(b)
    if np.isnan(a) and np.isnan(b):
        return 0
    ia, ib = int(a.view(np.int32)), int(b.view(np.int32))
    ia = ia if ia >= 0 else -(ia & 0x7FFFFFFF)
    ib = ib if ib >= 0 else -(ib & 0x7FFFFFFF)
    return abs(ia - ib)


@pytest.mark.gpu
def test_device_draws_equal_restatement(built):
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    s = _bombed(level, P8_RIPPE)
    seed = 2024
    p = P8_RIPPE.copy()
    n_seen = n_acc = 0
    for cycle, frags in enumerate(_orders(level.n_frags, 2)):
        steps, nuis = s.run_cycle_device(frags, 5, seed=seed, cycle=cycle, nuisance=True)
        rec = s.last_nuisance_records(len(frags))
        for t, r, p_live, (id_modif, u, draw, q, valid) in _restated_chain(p, rec, cycle, seed):
            assert r["id_modif"] == id_modif and r["u"] == u and bool(r["valid"]) == valid, (cycle, t)
            assert abs(r["draw"] - draw) <= 1e-13 * abs(draw), (cycle, t, r["draw"], draw)
            for i in range(8):
                lim = 1 if i == 5 else 2
                assert _ulps(r["p_test"][i], q[i]) <= lim, (cycle, t, i, r["p_test"][i], q[i])
            ratio_log = r["likelihood_nuis"] - steps["likelihood"][t]
            if valid and abs(math.exp(min(ratio_log, 700.0)) - u) > 1e-12:
                assert bool(r["accepted"]) == (math.exp(min(ratio_log, 700.0)) >= u), (cycle, t)
            if not valid:
                assert not r["accepted"]
            n_seen += 1
            n_acc += int(r["accepted"])
        p = np.array(list(s.param_simu[0]), dtype=np.float32)
        assert np.array_equal(nuis["success"], rec["accepted"])
    assert n_seen == 2 * level.n_frags and 0 < n_acc < n_seen
    s.free_gpu()


def _host_replay(level, p8, frags_per_cycle, seed, refresh_every=None):
    """handle a: device nuisance cycles; handle b: step_sampler with a's plan, then eval_likelihood_4_nuisance on a's
    proposal and the Metropolis decision with a's u -- everything must agree bit for bit"""
    from instagraal_b200.cuda_lib_gl_single import PARAM_SIMU_RIPPE
    a = _bombed(level, p8)
    b = _bombed(level, p8)
    if refresh_every is not None:
        a.set_options(refresh_every=refresh_every)
        b.set_options(refresh_every=refresh_every)
    dt = np.float32(0.01)
    n_acc_then_step = 0
    for cycle, frags in enumerate(frags_per_cycle):
        steps, nuis = a.run_cycle_device(frags, 5, seed=seed, cycle=cycle, nuisance=True)
        plan = a.last_cycle_plan(len(frags))
        for t in range(len(frags)):
            r = nuis[t]
            cands = plan[t, 2:2 + plan[t, 0]].tolist()
            o, dist, op, fid, mean_len, n_contigs = b.step_sampler(int(plan[t, 1]), 5, dt, candidates=cands)
            assert o == steps["likelihood"][t] and dist == steps["dist"][t], (cycle, t)
            assert op == steps["op_sampled"][t] and fid == steps["id_f_sampled"][t] and n_contigs == steps["n_contigs"][t]
            b.param_simu_test = np.array([tuple(r["p_test"].tolist())], dtype=PARAM_SIMU_RIPPE)
            l_nuis = b.eval_likelihood_4_nuisance()
            assert l_nuis == r["likelihood_nuis"] or (np.isnan(l_nuis) and np.isnan(r["likelihood_nuis"])), (cycle, t)
            with np.errstate(over="ignore", invalid="ignore"):
                acc = bool(r["valid"]) and bool(np.exp((l_nuis - b.likelihood_t) / 1.0) >= r["u"])
            assert acc == bool(r["accepted"]), (cycle, t)
            if acc:
                b.set_param_simu(r["p_test"])
                b.likelihood_t = l_nuis
                if t + 1 < len(frags):
                    n_acc_then_step += 1
            assert b.likelihood_t == r["likelihood_t"]
            live = np.array(list(b.param_simu[0]), dtype=np.float32)
            assert (live[6], live[4], live[5], live[7], live[3]) == (r["fact"], r["d"], r["d_max"], r["d_nuc"], r["slope"])
        assert np.array_equal(np.array(list(a.param_simu[0]), dtype=np.float32), np.array(list(b.param_simu[0]), dtype=np.float32))
        assert np.array_equal(a._get_state(), b._get_state()), cycle
    a.free_gpu()
    b.free_gpu()
    return n_acc_then_step


@pytest.mark.gpu
@pytest.mark.parametrize("workload,refresh_every,n_frags", [("toy", None, None), ("T", None, 300), ("toy", 1, None)])
def test_device_nuisance_cycle_equals_host_driven_sequence(built, workload, refresh_every, n_frags):
    from instagraal_b200.synth import WORKLOADS, make_level, workload_params
    level = make_level(WORKLOADS[workload])
    p8 = P8_RIPPE if workload == "toy" else workload_params(level)
    orders = [o[:n_frags] if n_frags else o for o in _orders(level.n_frags, 2)]
    n = _host_replay(level, p8, orders, seed=77, refresh_every=refresh_every)
    assert n >= 1   # an acceptance followed by a step: kind 3 predicated on


@pytest.mark.gpu
def test_mode_off_leaves_cycles_unchanged(built):
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    frags = _orders(level.n_frags, 1)[0]
    a = _bombed(level, P8_RIPPE)
    b = _bombed(level, P8_RIPPE)
    a.set_device_nuisance(True)
    a.set_device_nuisance(False)
    ra = a.run_cycle_device(frags, 5, seed=5, cycle=1)
    rb = b.run_cycle_device(frags, 5, seed=5, cycle=1)
    assert np.array_equal(ra, rb)
    assert np.array_equal(a._get_state(), b._get_state())
    a.free_gpu()
    b.free_gpu()


@pytest.mark.gpu
def test_replica_set_with_nuisance_equals_separate_handles(built):
    from instagraal_b200.replicas import ReplicaSet, best_chain
    from instagraal_b200.synth import WORKLOADS, make_level
    from test_gpu_parity import make_sampler
    level = make_level(WORKLOADS["toy"])
    n = 4
    rng = np.random.RandomState(77)
    frags = np.stack([np.concatenate([rng.permutation(level.n_frags) for _ in range(2)]) for _ in range(n)]).astype(np.int32)
    seeds = np.array([11, 12, 13, 14], dtype=np.uint64)
    want, want_nuis, want_state = [], [], []
    for i in range(n):
        s = make_sampler(level)
        s.set_gpu_share(4)
        s.set_param_simu(P8_RIPPE)
        np.random.seed(100 + i)
        s.bomb_the_genome()
        st, nu = s.run_cycle_device(frags[i], 5, seed=int(seeds[i]), cycle=5, nuisance=True)
        want.append(st)
        want_nuis.append(nu)
        want_state.append(s._get_state())
        s.free_gpu()
    first = make_sampler(level)
    first.set_param_simu(P8_RIPPE)
    rs = ReplicaSet(first, n, seeds=seeds)
    rs.bomb(seed0=100)
    got, nuis = rs.run_cycle(frags, 5, cycle=5, nuisance=True)
    for i in range(n):
        assert np.array_equal(got[i], want[i]), i
        assert np.array_equal(nuis[i].view(np.uint8), want_nuis[i].view(np.uint8)), i
        assert np.array_equal(rs.chains[i]._get_state(), want_state[i]), i
    assert sum(int(nu["success"].sum()) for nu in want_nuis) > 0
    best, lik, nc = rs.allgather()
    assert np.array_equal(lik, np.array([got[i][-1]["likelihood"] for i in range(n)]))
    assert best == best_chain(lik)
    rs.free()


@pytest.mark.gpu
def test_checkpoint_resume_with_device_nuisance(built, tmp_path):
    from instagraal_b200.synth import WORKLOADS, make_level
    from test_gpu_parity import make_sampler
    level = make_level(WORKLOADS["toy"])
    o1, o2 = _orders(level.n_frags, 2)
    a = _bombed(level, P8_RIPPE)
    a.run_cycle_device(o1, 5, seed=9, cycle=0, nuisance=True)
    ck = str(tmp_path / "ck.npz")
    a.save_checkpoint(ck)
    sa, na = a.run_cycle_device(o2, 5, seed=9, cycle=1, nuisance=True)
    b = make_sampler(level)
    b.load_checkpoint(ck)
    sb, nb = b.run_cycle_device(o2, 5, seed=9, cycle=1, nuisance=True)
    assert np.array_equal(sa, sb)
    assert np.array_equal(na.view(np.uint8), nb.view(np.uint8))
    assert np.array_equal(a._get_state(), b._get_state())
    assert a.param_simu.tobytes() == b.param_simu.tobytes() and a.likelihood_t == b.likelihood_t
    a.free_gpu()
    b.free_gpu()


@pytest.mark.gpu
def test_invalid_proposals_are_rejected_and_change_nothing(built):
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    p0 = P8_RIPPE.copy()
    p0[3] = np.float32(-1e-4)
    s = _bombed(level, p0)
    steps, nuis = s.run_cycle_device(_orders(level.n_frags, 1)[0], 5, seed=31, cycle=0, nuisance=True)
    cross = (nuis["id_modif"] == 1) & (nuis["p_test"][:, 3] >= 0)
    assert cross.sum() > 0
    assert np.all(nuis["valid"][cross] == 0) and np.all(nuis["accepted"][cross] == 0)
    assert np.all(nuis["accepted"][nuis["valid"] == 0] == 0)
    p = p0.copy()
    for r in nuis:
        if r["accepted"]:
            p = r["p_test"].copy()
        assert (r["fact"], r["d"], r["d_max"], r["d_nuc"], r["slope"]) == (p[6], p[4], p[5], p[7], p[3])
    assert np.array_equal(np.array(list(s.param_simu[0]), dtype=np.float32), p)
    assert np.all(np.isfinite(steps["likelihood"])) and np.all(np.isfinite(nuis["likelihood_t"]))
    s.free_gpu()


@pytest.mark.gpu
def test_refusals(built, monkeypatch):
    from instagraal_b200.synth import WORKLOADS, make_level
    from test_gpu_parity import make_sampler
    level = make_level(WORKLOADS["toy"])
    monkeypatch.setenv("IG_LNZ_CACHE", "0")
    s = make_sampler(level)
    s.set_param_simu(P8_RIPPE)
    with pytest.raises(RuntimeError, match="per-contact likelihood records"):
        s.set_device_nuisance(True)
    s.free_gpu()
    monkeypatch.delenv("IG_LNZ_CACHE")
    s = make_sampler(level)
    with pytest.raises(RuntimeError, match="parameters not set"):
        s.set_device_nuisance(True)
    s.set_param_simu(P8_RIPPE)
    s.set_device_nuisance(True)
    frags = np.arange(level.n_frags, dtype=np.int32)
    with pytest.raises(RuntimeError, match="device nuisance step is on"):
        s.run_cycle(frags[:4], 5)
    s.set_device_nuisance(False)
    s.run_cycle(frags[:4], 5)
    s.free_gpu()
