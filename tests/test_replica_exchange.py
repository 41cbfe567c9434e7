"""Replica exchange: after an all-gather, every local chain restarts from one gathered chain on the device
(ig_adopt_gathered, ReplicaSet.adopt / exchange) with its scaffold, validity list and p(s) parameters.

The oracle is what the host could already do through existing calls: a separate handle given the gathered scaffold
(ig_set_state), the source chain's validity list and parameters, then the adopted chain's seed.  The adopted chain keeps the
source's raw contig labels while the oracle starts from canonical ones; labels are only compared for equality (labels_guard),
so the two runs must agree record for record."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from instagraal_b200.synth import WORKLOADS, make_level, workload_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P8_RIPPE = np.array([50.0, 9.6, np.float32(0.53 * (9.6 / 50.0) ** -1.5 * 50.0 ** -3), -1.5, 2.0, 900.0, 4.0e5, 0.02],
                    dtype=np.float32)
N_CHAINS = 4
SEEDS = np.array([21, 22, 23, 24], dtype=np.uint64)


# ------------------------------------------------------------------ CPU: the binding
def test_adopt_binding():
    from instagraal_b200 import _lib as L
    assert "ig_adopt_gathered" in L.EXPORTS
    hdr = open(os.path.join(ROOT, "include", "instagraal_b200.h")).read()
    assert "int ig_adopt_gathered(ig_handle* lead, ig_handle** local_chains, int32_t n_local, int32_t index" in hdr


def test_adopt_argtypes(built):
    from instagraal_b200 import _lib as L
    f = L.lib().ig_adopt_gathered
    vp, i32 = ctypes.c_void_p, ctypes.c_int32
    assert f.argtypes == [vp, vp, i32, i32, vp, vp, ctypes.POINTER(ctypes.c_double)]
    assert f.restype is ctypes.c_int


# ------------------------------------------------------------------ GPU
def _p8(s):
    return np.array(list(s.param_simu[0]), dtype=np.float32)


def _orders(nf, n_steps, cycle):
    rng = np.random.RandomState(500 + cycle)
    return np.stack([rng.permutation(nf)[:n_steps] for _ in range(N_CHAINS)]).astype(np.int32)


def _replica_set(level, p8, refresh_every=None):
    from instagraal_b200.replicas import ReplicaSet
    from test_gpu_parity import make_sampler
    first = make_sampler(level)
    first.set_param_simu(p8)
    rs = ReplicaSet(first, N_CHAINS, seeds=SEEDS)
    if refresh_every is not None:
        for c in rs.chains:
            c.set_options(refresh_every=refresh_every)
    rs.bomb(seed0=300)
    return rs


def _cycle(rs, frags, n_neighbours, cycle, nuisance):
    out = rs.run_cycle(frags, n_neighbours, cycle=cycle, nuisance=nuisance)
    return out if nuisance else (out, None)


def _level_and_params(workload):
    level = make_level(WORKLOADS[workload])
    return level, (P8_RIPPE if workload == "toy" else workload_params(level)), (None if workload == "toy" else 300)


def _adopt_and_check_against_oracle(workload, n_neighbours=5, nuisance=False, refresh_every=None, pick_best=True):
    """cycle 0 on 4 chains, all-gather, adopt chain `src` (the best, or the worst), cycle 1; every adopted chain's cycle 1 ==
    the oracle's, record for record, and the same final state"""
    from test_gpu_parity import make_sampler
    level, p8, n_steps = _level_and_params(workload)
    n_steps = n_steps or level.n_frags
    rs = _replica_set(level, p8, refresh_every)
    _cycle(rs, _orders(level.n_frags, n_steps, 0), n_neighbours, 0, nuisance)
    best, lik, nc = rs.allgather()
    src = best if pick_best else int(np.argmin(lik))
    if not pick_best:
        assert src != best
    src_state = rs.gathered_state(src)
    src_valid = rs.chains[src].get_valid_insert()
    src_p8 = _p8(rs.chains[src])
    before = [_p8(c) for c in rs.chains]
    p8g, valid_g, lik_g = rs.adopt(src)
    # what the gather carried is what the source chain holds
    assert np.array_equal(p8g.view(np.uint32), src_p8.view(np.uint32))
    assert np.array_equal(valid_g, src_valid) and lik_g == lik[src]
    targets = [c for c in range(N_CHAINS) if c != src]
    for c in targets:
        ch = rs.chains[c]
        assert np.array_equal(ch._get_state(), src_state), c
        assert np.array_equal(ch.get_valid_insert(), src_valid), c
        assert ch.param_simu.tobytes() == rs.chains[src].param_simu.tobytes()
        assert ch.param_simu_test.tobytes() == ch.param_simu.tobytes()
        assert ch.likelihood_t == lik[src] and ch.n_contigs == nc[src]
    if nuisance:   # the case that a host-side scaffold copy could not carry: the targets' parameters differed
        assert any(not np.array_equal(before[c].view(np.uint32), src_p8.view(np.uint32)) for c in targets)
    frags1 = _orders(level.n_frags, n_steps, 1)
    got, got_nuis = _cycle(rs, frags1, n_neighbours, 1, nuisance)
    for c in targets:
        o = make_sampler(level)
        o.set_gpu_share(rs.gpu_share)
        if refresh_every is not None:
            o.set_options(refresh_every=refresh_every)
        o._set_state(src_state)
        o.set_valid_insert(src_valid)
        o.set_param_simu(src_p8)
        want = o.run_cycle_device(frags1[c], n_neighbours, seed=int(SEEDS[c]), cycle=1, nuisance=nuisance)
        want, want_nuis = want if nuisance else (want, None)
        assert want.dtype == got.dtype
        for key in got.dtype.names:
            assert np.array_equal(got[c][key], want[key]), (c, key)
        if nuisance:
            assert np.array_equal(got_nuis[c].view(np.uint8), want_nuis.view(np.uint8)), c
        assert np.array_equal(rs.chains[c]._get_state(), o._get_state()), c
        assert np.array_equal(rs.chains[c].get_valid_insert(), o.get_valid_insert()), c
        assert rs.chains[c].param_simu.tobytes() == o.param_simu.tobytes()
        o.free_gpu()
    if nuisance:
        assert sum(int(got_nuis[c]["success"].sum()) for c in targets) > 0
    rs.free()


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["toy", "T"])
@pytest.mark.parametrize("variant", ["n5", "n12", "nuisance", "refresh1"])
def test_adopted_chain_equals_host_oracle(built, workload, variant):
    kw = {"n5": {}, "n12": {"n_neighbours": 12}, "nuisance": {"nuisance": True}, "refresh1": {"refresh_every": 1}}[variant]
    _adopt_and_check_against_oracle(workload, **kw)


@pytest.mark.gpu
def test_adopt_from_a_chain_other_than_the_best(built):
    _adopt_and_check_against_oracle("toy", nuisance=True, pick_best=False)


@pytest.mark.gpu
def test_source_chain_is_untouched(built):
    """the chain at `best` continues bit-identically to the same chain of a replica set that never adopts"""
    level, p8, _ = _level_and_params("toy")
    runs = []
    for adopt in (True, False):
        rs = _replica_set(level, p8)
        _cycle(rs, _orders(level.n_frags, level.n_frags, 0), 5, 0, True)
        best, lik, _nc = (rs.exchange() if adopt else rs.allgather())
        got, nuis = _cycle(rs, _orders(level.n_frags, level.n_frags, 1), 5, 1, True)
        runs.append((best, got[best].copy(), nuis[best].copy(), rs.chains[best]._get_state(), rs.chains[best].get_valid_insert(),
                     rs.chains[best].param_simu.tobytes()))
        rs.free()
    (b0, g0, n0, s0, v0, p0), (b1, g1, n1, s1, v1, p1) = runs
    assert b0 == b1
    assert np.array_equal(g0, g1) and np.array_equal(n0.view(np.uint8), n1.view(np.uint8))
    assert np.array_equal(s0, s1) and np.array_equal(v0, v1) and p0 == p1


@pytest.mark.gpu
def test_exchange_every_chain_continues_from_the_best(built):
    """exchange() = allgather() + adopt(best): same return values, every chain starts its next cycle from the best state"""
    level, p8, _ = _level_and_params("toy")
    rs = _replica_set(level, p8)
    _cycle(rs, _orders(level.n_frags, level.n_frags, 0), 5, 0, True)
    best, lik, nc = rs.exchange()
    assert rs.n_gathers == 1 and best == int(np.argmax(lik))
    st = rs.gathered_state(best)
    for i, c in enumerate(rs.chains):
        assert np.array_equal(c._get_state(), st) and c.n_contigs == nc[best]
        if i != best:   # (the best chain's own likelihood_t includes its last accepted nuisance step)
            assert c.likelihood_t == lik[best]
    rs.free()


@pytest.mark.gpu
def test_nccl_exchange_two_gpus(built, tmp_path):
    """2 ranks x 2 chains with the nuisance step: after exchange() every chain on both ranks holds the best chain's state,
    validity list and parameters"""
    from instagraal_b200 import _lib as L
    if L.lib().ig_device_count() < 2:
        pytest.skip("needs two GPUs")
    worker = os.path.join(ROOT, "tests", "_exchange_worker.py")
    idfile = str(tmp_path / "nccl_id.bin")
    ps = [subprocess.Popen([sys.executable, worker, str(r), "2", idfile], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
          for r in range(2)]
    res = []
    for p in ps:
        out, _ = p.communicate(timeout=600)
        assert p.returncode == 0, out[-3000:]
        res.append(json.loads([ln for ln in out.splitlines() if ln.startswith("RESULT ")][-1][7:]))
    a, b = sorted(res, key=lambda r: r["rank"])
    assert a["best"] == b["best"] and a["lik"] == b["lik"]
    best = a["best"]
    src = a if best < 2 else b
    want = (src["chains"][best % 2]["crc"], src["chains"][best % 2]["valid"], src["chains"][best % 2]["p8"])
    for r in (a, b):
        assert r["gathered_crc"] == want[0]
        for ch in r["chains"]:
            assert (ch["crc"], ch["valid"], ch["p8"]) == want
    # the chains differed before the exchange (own seeds, own nuisance acceptances)
    assert len({json.dumps(ch["p8_before"]) for r in (a, b) for ch in r["chains"]}) > 1


@pytest.mark.gpu
def test_refusals(built):
    from instagraal_b200 import _lib as L
    from instagraal_b200.replicas import ReplicaSet
    from test_gpu_parity import make_sampler
    level, p8, _ = _level_and_params("toy")
    rs = _replica_set(level, p8)
    with pytest.raises(RuntimeError, match="ig_nccl_init not called"):
        rs.adopt(0)
    rs.init_comm()
    with pytest.raises(RuntimeError, match="no all-gather since ig_nccl_init"):
        rs.adopt(0)
    frags = _orders(level.n_frags, 40, 0)
    rs.run_cycle(frags, 5, cycle=0)
    best, lik, nc = rs.allgather()
    for bad in (-1, N_CHAINS):
        with pytest.raises(RuntimeError, match="no such chain"):
            rs.adopt(bad)
    lead = rs.chains[0]._h
    lib = L.lib()
    rc = lib.ig_adopt_gathered(lead, rs._handles, N_CHAINS - 1, 0, None, None, None)
    assert rc == -1 and b"differs from ig_nccl_init" in lib.ig_last_error(lead)
    other = make_sampler(make_level(WORKLOADS["micro"]))
    other.set_param_simu(p8)
    mixed = (ctypes.c_void_p * N_CHAINS)(*[c._h for c in rs.chains[:-1]], other._h)
    rc = lib.ig_adopt_gathered(lead, mixed, N_CHAINS, 0, None, None, None)
    assert rc == -1 and b"share level and device" in lib.ig_last_error(lead)
    other.free_gpu()
    last = rs.chains[-1]
    assert lib.ig_run_cycle_device_async(last._h, 40, frags[-1].ctypes.data_as(ctypes.c_void_p), 5, 99, 1) == 0
    with pytest.raises(RuntimeError, match="asynchronous cycle is still pending"):
        rs.adopt(best)
    out = np.zeros(40, dtype=L.CYCLE_DTYPE)
    L.check(last._h, lib.ig_cycle_wait(last._h, 40, out.ctypes.data_as(ctypes.c_void_p)), "ig_cycle_wait")
    # after the refusals the set still adopts; every output pointer may be null
    best, lik, nc = rs.allgather()
    assert lib.ig_adopt_gathered(lead, rs._handles, N_CHAINS, best, None, None, None) == 0
    st = rs.gathered_state(best)
    for c in rs.chains:
        assert np.array_equal(c._get_state(), st)
    rs.free()
