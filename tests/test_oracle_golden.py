import os
"""Pins the oracle (oracle/*.py, NumPy restatement) against golden vectors recorded from the
UNMODIFIED reference sampler running on the CPU emulation of its own kernels
(oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden
from instagraal_b200.synth import WORKLOADS, make_level
from oracle import score as sc
from oracle.sampler_oracle import OracleSampler, distance_histogram
from parity_common import FIELDS13, replay


class OracleImpl:
    def __init__(self, level, p8):
        self.o = OracleSampler(level, p8)

    def set_state(self, st):
        self.o.live = {k: st[i].copy() for i, k in enumerate(FIELDS13)}

    def set_valid(self, v):
        self.o.valid = [int(x) for x in v]

    def set_params(self, p8):
        self.o.params = sc.Params(p8)

    def eval_nuisance(self, p8):
        return self.o.eval_likelihood_4_nuisance(np.asarray(p8, dtype=np.float32))

    def get_state(self):
        return np.stack([self.o.live[k] for k in FIELDS13])

    def step(self, a, cands):
        r = self.o.step_sampler(a, 5, candidates=cands)
        return dict(scores=self.o.all_scores, op=r[2], B=r[3], o=r[0], dist=r[1], mean_len=r[4], n_contigs=r[5])


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_replays_reference_trajectory(name):
    g = load_golden(name)
    level = make_level(WORKLOADS[str(g["workload"])])
    max_steps = 120 if name.startswith("toy") else None  # keep the CPU suite short
    res = replay(g, OracleImpl(level, g["params8"]), max_steps=max_steps)
    assert not res.errors, res.errors[:3]
    assert res.same_choice >= 0.9 * res.steps  # the rest are exact ties (see parity_common)
    assert res.max_rel < 1e-7


def test_oracle_rng_stream_matches_reference():
    """Free-running (not teacher-forced) oracle with the same seed draws the same fragments and
    candidates as the reference for as long as no exact tie is broken differently."""
    g = load_golden("micro_bomb_seed1")
    level = make_level(WORKLOADS["micro"])
    np.random.seed(int(g["seed"]))
    o = OracleSampler(level, g["params8"])
    perm_state = o.bomb_the_genome()
    assert np.array_equal(np.stack([o.live[k] for k in FIELDS13]), g["state0"])
    lf = np.arange(level.n_frags)
    np.random.shuffle(lf)
    assert int(lf[0]) == int(g["step_A"][0])
    o.step_sampler(int(lf[0]), 5)
    nc = int(g["step_ncand"][0])
    assert [int(c) for c in o.candidates] == [int(c) for c in g["step_cands"][0][:nc]]
    assert perm_state.shape == (level.n_frags,)


@pytest.mark.parametrize("name", ["micro_seed0", "toy_bomb_seed2"])
def test_oracle_histogram_matches_reference(name):
    g = load_golden(name)
    level = make_level(WORKLOADS[str(g["workload"])])
    max_kb, bin_kb, n_rows = g["hist_args"]
    bins, mean, used = distance_histogram(level.sparse_matrix, level.S_o_A_frags, level.np_sub_frags_2_frags,
                                          int(n_rows), max_kb, bin_kb)
    ref = g["hist_mean"].astype(np.float64)
    # the reference stores float32(mean + mean_value_trans) and NaN for empty bins
    mine = np.where(mean == 0, np.nan, mean + level.mean_value_trans).astype(np.float32)
    assert np.array_equal(np.isnan(mine), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.allclose(mine[ok], ref[ok], rtol=1e-6)


def test_struct_dumps_match_reference():
    """The 24 candidate scaffolds the reference materialised for its first candidate pairs."""
    from oracle import moves as mv
    g = load_golden("micro_seed0")
    o_state = {k: g["state0"][i].copy() for i, k in enumerate(FIELDS13)}
    o_state, n_contigs, _ = mv.renumber_contigs(o_state)  # the dumps are taken after CL:1415
    nc0 = int(g["step_ncand"][0])
    for k in range(min(nc0, len(g["dump_A"]))):
        a, b = int(g["dump_A"][k]), int(g["dump_B"][k])
        max_id = n_contigs - 1
        muts, valid = mv.perform_mutations(o_state, a, b, max_id)
        assert list(valid) == [int(x) for x in g["dump_valid"][k]]
        for m in range(24):
            got = np.stack([muts[m][f] for f in FIELDS13])
            assert np.array_equal(got, g["dump_structs"][k][m]), (k, m)


def test_philox_known_answers():
    """Philox4x32-10 known-answer vectors of Random123 (kat_vectors: philox4x32 10)."""
    from oracle.device_rng import philox4x32_10
    assert philox4x32_10((0, 0, 0, 0), (0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert philox4x32_10((0xffffffff,) * 4, (0xffffffff, 0xffffffff)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert philox4x32_10((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_yeast_toy_config0_oracle_cycle_sample():
    """BASELINE.json configs[0] on the CPU: geometry fixture of the reference's tests/data contigs (75,032
    restriction fragments -> 1015 level-4 fragments), every move of a few steps of one cycle scored by the
    NumPy transcription."""
    import numpy as np
    from instagraal_b200.synth import make_workload
    from oracle.sampler_oracle import OracleSampler
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "yeast_toy_geometry.npz"))
    assert int(z["n_level0"]) == 75032 and len(z["contig_names"]) == 146
    level = make_workload("yeast_toy")
    assert (level.n_frags, level.n_sub_frags) == (1015, 2857)
    assert 1.5e6 < level.sparse_matrix.sum() < 3.5e6      # "~2 M pairs"
    p8 = np.array([50.0, 9.6, np.float32(0.53 * (9.6 / 50.0) ** -1.5 * 50.0 ** -3), -1.5, 2.0, 900.0, 4.0e5, 0.02], dtype=np.float32)
    o = OracleSampler(level, p8)
    np.random.seed(0)
    frs = np.random.permutation(level.n_frags)[:4]
    n_prop = 0
    for f in frs:
        r = o.step_sampler(int(f), 5)
        nz = o.all_scores != 0
        assert nz.any() and np.all(np.isfinite(o.all_scores))
        assert 0 <= int(r[2]) < 24 and 0 <= int(r[3]) < level.n_frags
        n_prop += int(sum(o.n_uniq_list))
    assert n_prop >= 4 * 10


@pytest.mark.parametrize("d_exp", [2.0, 2.37])
def test_contact_terms_return_parts_equal_the_plain_call(d_exp):
    """contact_terms(..., return_parts=True) and zeros_term_raw(..., return_parts=True) return the same terms as the plain
    calls bit for bit, plus float32 expected values the terms are rebuilt from; circular contigs included."""
    from oracle.fuzz import random_state
    level = make_level(WORKLOADS["micro"])
    p8 = np.array([2.2354, 1.4933294, 0.06928191, -0.9384134, d_exp, 386.88467, 65.71848, 0.01698581], dtype=np.float32)
    o = OracleSampler(level, p8)
    from test_gpu_parity import _rebuild_offsets
    st = random_state(level.n_frags, np.random.RandomState(4), p_circ=0.5)
    for k in ("len_bp", "sub_len"):   # the level's fragment lengths, so that coordinates stay meaningful
        st[k] = np.asarray(level.S_o_A_frags[k], dtype=np.int32).copy()
    st = _rebuild_offsets(st)
    assert st["circ"].any()
    for live in (o.live, st):
        v = sc.fill_vect_dist(live, o.sub)
        for len_from in ("row", "col"):
            t0 = sc.contact_terms(v, *o.coo, o.params, o.mbar, len_from=len_from)
            t1, ex, exz = sc.contact_terms(v, *o.coo, o.params, o.mbar, len_from=len_from, return_parts=True)
            assert ex.dtype == np.float32 and exz.dtype == np.float32 and ex.shape == exz.shape == t0.shape
            assert np.array_equal(t0.view(np.int64), t1.view(np.int64))
            t2 = sc.likelihood_pxl(ex, o.coo[2]) + exz.astype(np.float64) * sc.LOG10E_F
            assert np.array_equal(t0.view(np.int64), t2.view(np.int64))
        z0, n0 = sc.zeros_term_raw(v, o.params, o.mbar)
        z1, n1, zt = sc.zeros_term_raw(v, o.params, o.mbar, return_parts=True)
        assert np.isfinite(z0) and (z0, n0) == (z1, n1) and z0 == -float(np.sum(zt)) and zt.size == int((v["pos"] > 0).sum())
