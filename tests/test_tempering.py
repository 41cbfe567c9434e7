"""Move selection at a chain temperature T > 0 and temperature swaps between replica chains (sampler.set_chain_temperature,
ReplicaSet.set_ladder / swap_temperatures).  CPU: the NumPy restatement of the tempered pick (oracle/tempered.py), its
counters, and the swap decisions.  GPU: T = 0 untouched, the device draws against a host-driven replay, the distribution of
the drawn move, replica sets against separate handles, refusals."""
import ctypes
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy import stats

from oracle import device_nuisance as dn
from oracle import device_rng
from oracle import tempered as tp
from instagraal_b200.replicas import swap_decisions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = np.float32(0.01)


# ------------------------------------------------------------------ CPU: the restated pick
def _scores(rng, n, p_zero=0.3):
    s = -1e4 + rng.normal(0.0, 30.0, n)
    s[rng.random(n) < p_zero] = 0.0
    return s


def test_pick_all_zero_is_index_zero():
    for n in (24, 5 * 24, 12 * 24):
        idx, b, m, lw, nsc = tp.pick(np.zeros(n), 3.0, 0.7, 0.4, wide=n > tp.BATCH)
        assert (idx, b, nsc) == (0, 0, 0) and m == -math.inf


def test_pick_excludes_nan_and_zero():
    rng = np.random.default_rng(1)
    s = _scores(rng, 5 * 24)
    s[rng.random(len(s)) < 0.2] = np.nan
    ok = tp.scored(s)
    for k in range(500):
        idx, *_ = tp.pick(s, 50.0, rng.random(), rng.random(), wide=False)
        assert ok[idx]
    w, m, S, n, last = tp.weights(s, 50.0)
    assert n == ok.sum() and m == np.nanmax(np.where(ok, s, np.nan)) and np.all(w[~ok] == 0)


@pytest.mark.parametrize("n_cands,T", [(12, 5.0), (20, 40.0), (64, 0.5), (9, 1e3)])
def test_two_stage_marginal_equals_weights(n_cands, T):
    rng = np.random.default_rng(n_cands)
    s = _scores(rng, 24 * n_cands)
    s[24 * 8:24 * 9] = 0.0   # a candidate with nothing scored (with 9 candidates: the whole second batch)
    marg = tp.wide_marginal(s, T)
    ok = tp.scored(s)
    m = s[ok].max()
    w = np.where(ok, np.exp((np.where(ok, s, m) - m) / T), 0.0)
    assert np.allclose(marg, w / w.sum(), rtol=1e-12, atol=1e-300)
    assert abs(marg.sum() - 1.0) < 1e-12


def test_two_stage_draw_frequencies():
    """the two-stage pick, fed uniform draws, follows w / sum(w)"""
    rng = np.random.default_rng(5)
    s = _scores(rng, 24 * 12, p_zero=0.6)
    s[s != 0] = -1e4 + rng.normal(0.0, 2.0, int((s != 0).sum()))
    p = tp.wide_marginal(s, 2.0)
    n = 10000
    cnt = np.bincount([tp.pick(s, 2.0, rng.random(), rng.random(), wide=True)[0] for _ in range(n)], minlength=len(s))
    big = p * n >= 5
    f_obs = np.append(cnt[big], cnt[~big].sum())
    f_exp = np.append(p[big] * n, p[~big].sum() * n)
    keep = f_exp > 0
    assert stats.chisquare(f_obs[keep], f_exp[keep] * f_obs[keep].sum() / f_exp[keep].sum()).pvalue > 1e-3


def test_tiny_temperature_is_argmax_and_huge_is_uniform():
    rng = np.random.default_rng(7)
    for wide, n in ((False, 5), (True, 12), (True, 30)):
        s = _scores(rng, 24 * n)
        ok = tp.scored(s)
        best = int(np.flatnonzero(s == s[ok].max())[0])
        for _ in range(50):
            assert tp.pick(s, 1e-9, rng.random(), rng.random(), wide=wide)[0] == best
        w, *_ = tp.weights(s, 1e20)
        assert np.all(w[ok] == 1.0)
        marg = tp.wide_marginal(s, 1e20)
        assert np.allclose(marg[ok], 1.0 / ok.sum(), rtol=1e-12) and np.all(marg[~ok] == 0)


def test_pick_boundaries():
    s = np.zeros(48)
    s[[3, 10, 30]] = [-5.0, -5.0, -5.0]   # three equal weights
    assert tp.pick(s, 1.0, 0.0, 0.0, wide=False)[0] == 3
    assert tp.pick(s, 1.0, 0.34, 0.0, wide=False)[0] == 10
    assert tp.pick(s, 1.0, 0.999999, 0.0, wide=False)[0] == 30


def test_tempered_counters_are_disjoint_from_plan_and_nuisance():
    """k_draw_plan: draw index < IG_MAX_NEIGHBOURS (64) and attempts < 256; nuisance: 0x80000000 / 0x80000001; tempered
    selection: 0x80000002 / 0x80000003, attempt 0"""
    for t, cycle in ((0, 0), (17, 2), (899, 41)):
        cu, cb = tp.counters(t, cycle)
        na, nb = dn.counters(t, cycle)
        assert len({cu[2], cb[2], na[2], nb[2]}) == 4
        for c in (cu, cb):
            assert c[2] >= 0x80000000 and c[3] == 0 and c[:2] == (t, cycle)
        key = (99, 0)
        words = {tuple(device_rng.philox4x32_10(c, key)) for c in (cu, cb, na, nb, (t, cycle, 0, 0))}
        assert len(words) == 5
    u, ub = tp.draws(3, 1, 2024)
    assert 0.0 <= u < 1.0 and 0.0 <= ub < 1.0 and u != ub


# ------------------------------------------------------------------ CPU: swap decisions
def test_swap_decisions_deterministic_and_alternating():
    T = [0.0, 1.0, 3.0, 9.0, 27.0, 81.0]
    lik = np.array([-100.0, -101.0, -99.0, -120.0, -90.0, -95.0])
    lad = np.arange(6)
    for r in range(6):
        a = swap_decisions(T, lad, lik, r, swap_seed=4)
        b = swap_decisions(T, lad.copy(), lik.copy(), r, swap_seed=4)
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2])
        assert [k for k, _ in a[0]] == list(range(r % 2, 5, 2))
        assert set(a[1]) <= set(a[0])
        lad = a[2]
        assert sorted(lad.tolist()) == list(range(6))


def test_swap_zero_temperature_limit():
    # rung 0 at T = 0 takes the other chain only if that does not lower its likelihood (ties accepted)
    for l0, l1, want in ((-10.0, -9.0, True), (-10.0, -10.0, True), (-10.0, -11.0, False)):
        for seed in range(5):
            _, acc, lad = swap_decisions([0.0, 5.0], [0, 1], [l0, l1], 0, seed)
            assert bool(acc) == want and (lad.tolist() == [1, 0]) == want
    # the hot rung is at index 0 and the cold one at index 1
    _, acc, _ = swap_decisions([5.0, 0.0], [0, 1], [-9.0, -10.0], 0, 0)
    assert acc
    _, acc, _ = swap_decisions([5.0, 0.0], [0, 1], [-11.0, -10.0], 0, 0)
    assert not acc


def test_swap_acceptance_frequency_matches_metropolis():
    T0, T1, L0, L1 = 2.0, 5.0, -100.0, -103.0
    want = min(1.0, math.exp((1 / T0 - 1 / T1) * (L1 - L0)))
    n, acc = 4000, 0
    for r in range(0, 2 * n, 2):   # even rounds try the pair (0, 1)
        _, a, _ = swap_decisions([T0, T1], [0, 1], [L0, L1], r, swap_seed=11)
        acc += len(a)
    lo, hi = stats.binom.interval(1 - 1e-4, n, want)
    assert lo <= acc <= hi, (acc, n * want)
    # the uphill direction always swaps
    assert all(swap_decisions([T0, T1], [0, 1], [L1, L0], r, 3)[1] for r in range(0, 40, 2))


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


def _p8(level, workload):
    from test_device_nuisance import P8_RIPPE
    from instagraal_b200.synth import workload_params
    return P8_RIPPE if workload == "toy" else workload_params(level)


@pytest.mark.gpu
@pytest.mark.parametrize("n_neigh", [5, 12])
@pytest.mark.parametrize("nuisance", [False, True])
def test_temperature_back_to_zero_equals_untouched(built, n_neigh, nuisance):
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    p8 = _p8(level, "toy")
    a, b = _bombed(level, p8), _bombed(level, p8)
    o1, o2 = _orders(level.n_frags, 2)
    a.set_chain_temperature(7.5)
    a.run_cycle_device(o1[:20], n_neigh, seed=4, cycle=0, nuisance=nuisance)   # a tempered cycle, then back to T = 0
    a.set_chain_temperature(0.0)
    a._set_state(b._get_state())
    a.set_valid_insert(b.get_valid_insert())
    if nuisance:
        a.set_param_simu(np.array(list(b.param_simu[0]), dtype=np.float32))
    c = _bombed(level, p8)
    for cycle, o in enumerate((o1, o2)):
        ra, rc = a.run_cycle_device(o, n_neigh, seed=9, cycle=cycle, nuisance=nuisance), c.run_cycle_device(o, n_neigh, seed=9, cycle=cycle, nuisance=nuisance)
        if nuisance:
            assert np.array_equal(ra[1].view(np.uint8), rc[1].view(np.uint8)), cycle
            ra, rc = ra[0], rc[0]
        assert np.array_equal(ra, rc), cycle
        assert np.array_equal(a._get_state(), c._get_state()) and np.array_equal(a.get_valid_insert(), c.get_valid_insert())
    for s in (a, b, c):
        s.free_gpu()


def _carried_valid(b, a_frag, cands, k, v0):
    """the validity list get_bounds leaves after candidates 0 .. k-1 of a step started from v0 (quirk Q3)"""
    b.set_valid_insert(v0)
    for j in range(k):
        b.eval_all_sub_likelihood(a_frag, cands[j], flip_eject=1 if j == 0 else 0)
    return b.get_valid_insert()


def _near_boundary(scores, T, u, ub, wide, idx_dev):
    """the device's pick differs from the restatement only where u * S (or u_batch * sum W) lies within 1e-12 relative of a
    cumulative boundary (the device's double exp may differ from NumPy's in the last bit)"""
    s = np.asarray(scores)
    batches = [s[i:i + tp.BATCH] for i in range(0, len(s), tp.BATCH)] if wide else [s]
    def close(w, target):
        c = np.cumsum(w)
        return c.size and np.min(np.abs(c - target)) <= 1e-12 * max(abs(target), c[-1])
    parts = [tp.weights(x, T) for x in batches]
    if wide:
        M = max((p[1] for p in parts if p[3]), default=-math.inf)
        W = np.array([p[2] * math.exp((p[1] - M) / T) if p[3] else 0.0 for p in parts])
        if close(W, ub * W.sum()):
            return True
    b = idx_dev // tp.BATCH if wide else 0
    return bool(close(parts[b][0], u * parts[b][2]))


@pytest.mark.gpu
@pytest.mark.parametrize("workload,n_neigh,T,nuisance,n_steps", [
    ("toy", 5, 2.0, False, 60), ("toy", 12, 30.0, True, 60), ("T", 5, 300.0, False, 40), ("T", 12, 30.0, False, 40),
])
def test_tempered_cycle_equals_host_driven_replay(built, workload, n_neigh, T, nuisance, n_steps):
    """handle a: tempered device cycles; handle b (T = 0): per step the scores of a's plan from the same state (step_sampler,
    then state and validity list restored), the restated pick with the restated draws, the move forced (test_copy_struct).
    Both handles recompute the full likelihood every step (refresh_every=1), so their scores agree bit for bit."""
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS[workload])
    p8 = _p8(level, workload)
    a, b = _bombed(level, p8), _bombed(level, p8)
    a.set_options(refresh_every=1)
    b.set_options(refresh_every=1)
    a.set_chain_temperature(T)
    wide = n_neigh > 8
    seed = 4242
    n_boundary = n_nonargmax = n_acc = 0
    for cycle in range(2):
        frags = _orders(level.n_frags, 1, seed=10 + cycle)[0][:n_steps]
        out = a.run_cycle_device(frags, n_neigh, seed=seed, cycle=cycle, nuisance=nuisance)
        steps, nuis = out if nuisance else (out, None)
        rec = a.last_tempered_records(len(frags))
        plan = a.last_cycle_plan(len(frags), width=max(8, n_neigh))
        for t in range(len(frags)):
            A = int(plan[t, 1])
            cands = plan[t, 2:2 + plan[t, 0]].tolist()
            s0, v0 = b._get_state(), b.get_valid_insert()
            b.step_sampler(A, n_neigh, DT, candidates=cands)
            scores = b.all_scores.copy()
            b._set_state(s0)
            u, ub = tp.draws(t, cycle, seed)
            idx, bt, m, lw, nsc = tp.pick(scores, T, u, ub, wide=wide)
            r = rec[t]
            assert r["u"] == u and r["u_batch"] == (ub if wide else 0.0), (cycle, t)
            assert r["s_max"] == m and r["n_scored"] == nsc, (cycle, t, r["s_max"], m)
            assert abs(r["log_w"] - lw) <= 1e-12 * max(1.0, abs(lw)), (cycle, t, r["log_w"], lw)
            if r["index"] != idx:
                assert _near_boundary(scores, T, u, ub, wide, int(r["index"])), (cycle, t, int(r["index"]), idx)
                idx = int(r["index"])
                n_boundary += 1
            assert r["batch"] == (idx // tp.BATCH if wide else 0)
            assert steps["likelihood"][t] == scores[idx], (cycle, t)
            kc, op = idx // 24, idx % 24
            assert steps["op_sampled"][t] == op and steps["cand_index"][t] == kc and steps["id_f_sampled"][t] == cands[kc]
            n_nonargmax += int(scores[idx] != np.max(scores[tp.scored(scores)]))
            _carried_valid(b, A, cands, kc if op >= 12 else len(cands), v0)
            b._set_state(s0)   # (the evaluations left the scaffold alone; the restore keeps the next step a full refresh)
            b.test_copy_struct(A, cands[kc], op)
            if nuisance:
                nr = nuis[t]
                x = math.exp(min((nr["likelihood_nuis"] - steps["likelihood"][t]) / T, 700.0)) if not np.isnan(nr["likelihood_nuis"]) else float("nan")
                if nr["valid"] and not abs(x - nr["u"]) <= 1e-12:
                    assert bool(nr["accepted"]) == bool(x >= nr["u"]), (cycle, t)
                if nr["accepted"]:
                    b.set_param_simu(nr["p_test"])
                    n_acc += 1
        assert np.array_equal(a._get_state(), b._get_state()), cycle
        assert np.array_equal(a.get_valid_insert(), b.get_valid_insert()), cycle
        if nuisance:
            assert np.array_equal(np.array(list(a.param_simu[0]), dtype=np.float32), np.array(list(b.param_simu[0]), dtype=np.float32))
    assert n_boundary <= 2
    assert n_nonargmax > 0   # the temperatures are hot enough to leave the argmax
    if nuisance:
        assert n_acc > 0
    a.free_gpu()
    b.free_gpu()


@pytest.mark.gpu
def test_drawn_move_follows_the_tempered_weights(built):
    """one fixed state, one fragment whose neighbours are all drawn whatever the seed (so every cycle scores the same
    proposals), 4000 one-step cycles with distinct seeds: the drawn index follows w / sum(w).  Toy with 64 neighbours: every
    fragment of T has more than 64 neighbours, every one of toy at most 64; the fragment is one of at least 33 (a step of at
    least five batches, so the batch draw matters)."""
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    p8 = _p8(level, "toy")
    a, b = _bombed(level, p8), _bombed(level, p8)
    n_neigh = 64
    _ptr, _idx, _cdf, nnz = a.neighbour_weights_csr()
    A = int([f for f in range(level.n_frags) if 33 <= nnz[f] <= n_neigh][0])
    s0, v0 = a._get_state(), a.get_valid_insert()
    a.run_cycle_device(np.array([A], np.int32), n_neigh, seed=1, cycle=0)
    cands = a.last_cycle_plan(1, width=n_neigh)[0]
    cands = cands[2:2 + cands[0]].tolist()
    b.step_sampler(A, n_neigh, DT, candidates=cands)
    scores = b.all_scores.copy()
    ok = tp.scored(scores)
    srt = np.sort(scores[ok])[::-1]
    T = max((srt[0] - srt[min(5, len(srt) - 1)]) / 2.0, 1e-3)
    a.set_chain_temperature(T)
    p = tp.wide_marginal(scores, T)
    n = 4000
    got = np.zeros(len(scores), np.int64)
    for k in range(n):
        a._set_state(s0)
        a.set_valid_insert(v0)
        st = a.run_cycle_device(np.array([A], np.int32), n_neigh, seed=1000 + k, cycle=0)
        r = a.last_tempered_records(1)[0]
        if k < 20:
            pl = a.last_cycle_plan(1, width=n_neigh)[0]
            assert pl[2:2 + pl[0]].tolist() == cands
            assert st["likelihood"][0] == scores[r["index"]]
        got[r["index"]] += 1
    big = p * n >= 5
    f_obs = np.append(got[big], got[~big].sum())
    f_exp = np.append(p[big], p[~big].sum()) * n
    keep = f_exp > 0
    assert got[~ok].sum() == 0 and big.sum() >= 3
    res = stats.chisquare(f_obs[keep], f_exp[keep])
    assert res.pvalue > 1e-3, (res, f_obs, f_exp)
    a.free_gpu()
    b.free_gpu()


@pytest.mark.gpu
def test_replica_set_at_four_temperatures_equals_separate_handles(built):
    from instagraal_b200.replicas import ReplicaSet
    from instagraal_b200.synth import WORKLOADS, make_level
    from test_gpu_parity import make_sampler
    level = make_level(WORKLOADS["toy"])
    p8 = _p8(level, "toy")
    n = 4
    temps = [0.0, 3.0, 30.0, 300.0]
    rng = np.random.RandomState(17)
    f1, f2 = (np.stack([rng.permutation(level.n_frags) for _ in range(n)]).astype(np.int32) for _ in range(2))
    seeds = np.array([21, 22, 23, 24], dtype=np.uint64)
    sep = []
    for i in range(n):
        s = make_sampler(level)
        s.set_gpu_share(4)
        s.set_param_simu(p8)
        np.random.seed(100 + i)
        s.bomb_the_genome()
        s.set_chain_temperature(temps[i])
        sep.append(s)
    first = make_sampler(level)
    first.set_param_simu(p8)
    rs = ReplicaSet(first, n, seeds=seeds)
    rs.bomb(seed0=100)
    rs.set_ladder(temps, swap_seed=3)
    got, nuis = rs.run_cycle(f1, 5, cycle=5, nuisance=True)
    for i in range(n):
        st, nu = sep[i].run_cycle_device(f1[i], 5, seed=int(seeds[i]), cycle=5, nuisance=True)
        assert np.array_equal(got[i], st) and np.array_equal(nuis[i].view(np.uint8), nu.view(np.uint8)), i
        assert np.array_equal(rs.chains[i].last_tempered_records(f1.shape[1]).view(np.uint8),
                              sep[i].last_tempered_records(f1.shape[1]).view(np.uint8)) or temps[i] == 0.0, i
        assert np.array_equal(rs.chains[i]._get_state(), sep[i]._get_state()), i
    tried, accepted, ladder = rs.swap_temperatures()
    live = rs.gathered_live_likelihood()
    assert np.array_equal(live, np.array([nu[-1]["likelihood_t"] for nu in nuis])), (live, [nu[-1]["likelihood_t"] for nu in nuis])
    assert [k for k, _ in tried] == [0, 2] and sorted(ladder.tolist()) == [0, 1, 2, 3]
    assert rs.swap_stats["tried"].tolist() == [1, 0, 1]
    rung = np.empty(n, np.int64)
    rung[ladder] = np.arange(n)
    for i in range(n):
        assert rs.chains[i].chain_temperature == temps[rung[i]]
        sep[i].set_chain_temperature(temps[rung[i]])
    got2 = rs.run_cycle(f2, 5, cycle=6)
    for i in range(n):
        st = sep[i].run_cycle_device(f2[i], 5, seed=int(seeds[i]), cycle=6)
        assert np.array_equal(got2[i], st), i
        assert np.array_equal(rs.chains[i]._get_state(), sep[i]._get_state()), i
    rs.allgather()
    assert np.array_equal(rs.gathered_live_likelihood(), np.array([g[-1]["likelihood"] for g in got2]))
    rs.free()
    for s in sep:
        s.free_gpu()


@pytest.mark.gpu
def test_nccl_ladder_two_gpus(built, tmp_path):
    """2 ranks x 2 chains: after three rounds of swap_temperatures both ranks hold the same ladder"""
    from instagraal_b200 import _lib as L
    if L.lib().ig_device_count() < 2:
        pytest.skip("needs two GPUs")
    worker = os.path.join(ROOT, "tests", "_tempering_worker.py")
    idfile = str(tmp_path / "nccl_id.bin")
    ps = [subprocess.Popen([sys.executable, worker, str(r), "2", idfile], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
          for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in ps]
    for p, o in zip(ps, outs):
        assert p.returncode == 0, o
    res = [json.loads([ln for ln in o.splitlines() if ln.startswith("RESULT ")][-1][7:]) for o in outs]
    assert res[0]["ladders"] == res[1]["ladders"] and len(res[0]["ladders"]) == 3
    assert res[0]["stats"] == res[1]["stats"]
    for r in res:
        assert sorted(r["ladders"][-1]) == [0, 1, 2, 3]


@pytest.mark.gpu
def test_refusals(built):
    from instagraal_b200 import _lib as L
    from instagraal_b200.synth import WORKLOADS, make_level
    level = make_level(WORKLOADS["toy"])
    p8 = _p8(level, "toy")
    s = _bombed(level, p8)
    frags = np.arange(level.n_frags, dtype=np.int32)
    for bad in (-1.0, float("nan"), float("inf"), -float("inf")):
        with pytest.raises(RuntimeError, match="finite and >= 0"):
            s.set_chain_temperature(bad)
    assert s.chain_temperature == 0.0
    s.set_chain_temperature(2.0)
    with pytest.raises(RuntimeError, match="chain temperature is > 0"):
        s.step_sampler(3, 5, DT, candidates=[4, 9])
    with pytest.raises(RuntimeError, match="chain temperature is > 0"):
        s.run_cycle(frags[:4], 5)
    with pytest.raises(RuntimeError, match="chain temperature is > 0"):
        s.step_sampler(3, 12, DT, candidates=list(range(10, 22)))
    s.run_cycle_device(frags[:4], 5, seed=1)   # the production mode runs
    lib = L.lib()
    s._upload_neighbour_weights()
    assert lib.ig_run_cycle_device_async(s._h, 10, frags.ctypes.data_as(ctypes.c_void_p), 5, 7, 1) == 0
    with pytest.raises(RuntimeError, match="asynchronous cycle is still pending"):
        s.set_chain_temperature(0.0)
    out = np.zeros(10, dtype=L.CYCLE_DTYPE)
    L.check(s._h, lib.ig_cycle_wait(s._h, 10, out.ctypes.data_as(ctypes.c_void_p)), "ig_cycle_wait")
    s.set_chain_temperature(0.0)
    s.step_sampler(3, 5, DT, candidates=[4, 9])
    s.free_gpu()
