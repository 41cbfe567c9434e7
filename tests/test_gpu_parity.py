"""GPU parity tests proper: the CUDA path, called through the C ABI (ctypes facade), against
(1) golden trajectories recorded from the reference, (2) the oracle on seeded random scaffolds
(incl. circular contigs), (3) size-independent properties at a larger size."""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden
from instagraal_b200.synth import WORKLOADS, SynthSpec, make_level
from parity_common import FIELDS13, replay

pytestmark = pytest.mark.gpu

P8 = np.array([2.2354, 1.4933294, 0.06928191, -0.9384134, 2.0, 386.88467, 65.71848, 0.01698581], dtype=np.float32)
P8_RIPPE = np.array([50.0, 9.6, np.float32(0.53 * (9.6 / 50.0) ** -1.5 * 50.0 ** -3), -1.5, 2.0, 900.0, 4.0e5, 0.02],
                    dtype=np.float32)


def make_sampler(level, **kw):
    from instagraal_b200.cuda_lib_gl_single import sampler
    return sampler(*level.sampler_args(), **kw)


def assert_scoring_path(s, path, rigid=False):
    """the handle scores through `path` (the level's natural one, or IG_SCORING_PATH when it was created): one host step
    from a re-uploaded scaffold launches 4 head kernels (full refresh), the scoring pass -- 10 kernels on the stream path,
    8 on the flat and rows paths -- and 3 tail kernels (2 with rigid pruning).  It moves the scaffold: call it last."""
    s._set_state(s._get_state())
    s.get_stats(reset=True)
    s.step_sampler(0, 3, np.float32(0.01), candidates=[1, 2, 3])
    want = 4 + (10 if path == "stream" else 8) + (2 if rigid else 3)
    assert s.get_stats()["launches"] == want, (path, s.get_stats()["launches"], want)


class GpuImpl:
    def __init__(self, level, **kw):
        self.s = make_sampler(level, **kw)
        self.dt = np.float32(0.01)

    def set_state(self, st):
        self.s._set_state(st)

    def set_valid(self, v):
        self.s.set_valid_insert(v)

    def set_params(self, p8):
        self.s.set_param_simu(p8)

    def get_state(self):
        return self.s._get_state()

    def eval_nuisance(self, p8):
        from instagraal_b200.cuda_lib_gl_single import PARAM_SIMU_RIPPE
        self.s.param_simu_test = np.array([tuple(np.asarray(p8, dtype=np.float32).tolist())], dtype=PARAM_SIMU_RIPPE)
        return self.s.eval_likelihood_4_nuisance()

    def step(self, a, cands):
        r = self.s.step_sampler(a, 5, self.dt, candidates=cands)
        return dict(scores=self.s.all_scores, op=r[2], B=r[3], o=r[0], dist=r[1], mean_len=r[4], n_contigs=r[5])


@pytest.mark.parametrize("split", ["", "24,1"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cuda_replays_reference_trajectory(built, name, split, monkeypatch):
    """the golden levels' natural flat path; `split`: the row-per-warp kernel (rows path) with that forced work split"""
    if split:
        monkeypatch.setenv("IG_SCORING_PATH", "rows")
        monkeypatch.setenv("IG_FORCE_SPLIT", split)
    g = load_golden(name)
    level = make_level(WORKLOADS[str(g["workload"])])
    impl = GpuImpl(level)
    res = replay(g, impl)
    assert not res.errors, res.errors[:4]
    assert res.same_choice >= 0.9 * res.steps
    assert res.nuis_checked > 0
    assert res.max_rel < 1e-7
    assert_scoring_path(impl.s, "rows" if split else "flat")
    impl.s.free_gpu()


def _oracle(level, p8):
    from oracle.sampler_oracle import OracleSampler
    return OracleSampler(level, p8)


@pytest.mark.parametrize("split,d_exp", [("", 2.0), ("24,1", 2.0), ("6,4", 2.0), ("", 2.37), ("24,1", 1.8)])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_cuda_vs_oracle_random_scaffolds_with_circular_contigs(built, seed, split, d_exp, monkeypatch):
    """eval (score) + apply on random scaffolds the trajectories never reach (circular contigs,
    reversed fragments), every op forced once through ig_apply.  `split` scores through the row-per-warp kernel
    (rows path) with a forced work split (all 24 mutations per item = the large-assembly path with one evaluation per
    group of identical motions; 6 mutations x 4 row parts = the small-assembly path), which small test levels would not
    reach; `d_exp` = the exponent-cutoff parameter d of the p(s) model."""
    from oracle import moves as mv
    from oracle.fuzz import random_state
    if split:
        monkeypatch.setenv("IG_SCORING_PATH", "rows")
        monkeypatch.setenv("IG_FORCE_SPLIT", split)
    level = make_level(WORKLOADS["micro"])
    rng = np.random.RandomState(seed)
    s = make_sampler(level)
    p8 = P8.copy()
    p8[4] = d_exp   # d != 2 takes the expf branch of rippe_contacts (KA:153-163), the usual case after the p(s) fit
    s.set_param_simu(p8)
    o = _oracle(level, p8)
    nf = level.n_frags
    for it in range(12):
        st = random_state(nf, rng, p_circ=0.4)
        # keep the real fragment lengths so coordinates stay meaningful
        for k in ("len_bp", "sub_len"):
            st[k] = np.asarray(level.S_o_A_frags[k], dtype=np.int32).copy()
        st = _rebuild_offsets(st)
        st13 = np.stack([st[k] for k in FIELDS13]).astype(np.int32)
        a, b = [int(x) for x in rng.choice(nf, 2, replace=False)]
        valid0 = rng.choice([-1, 1], 12).astype(np.int32)
        s._set_state(st13)
        s.set_valid_insert(valid0)
        got = s.eval_all_sub_likelihood(a, b, 1)
        o.live = {k: st[k].copy() for k in FIELDS13}
        o.valid = valid0.tolist()
        import oracle.score as sc
        o.v_cur = sc.fill_vect_dist(o.live, o.sub)
        lnz = sc.full_likelihood_nz(o.v_cur, o.coo, o.params, o.mbar)
        id_host = o.live["id_c"].copy()
        max_id = int(o.live["id_c"].max())
        want, uniq, n_sub = o.score_candidate(a, b, max_id, 1, id_host, lnz)
        assert np.array_equal(want != 0, got != 0), (it, a, b)
        nz = want != 0
        assert s.n_sub_vals[0] == n_sub
        tol = 1e-5 * np.abs(want[nz] - want[nz].max()) + 2e-8 * np.abs(want[nz]) + 1e-9
        assert np.all(np.abs(got[nz] - want[nz]) <= tol), (it, a, b, np.max(np.abs(got[nz] - want[nz])))
        assert np.array_equal(s.get_valid_insert(), np.array(o.valid, dtype=np.int32))
        # apply one op (cycling through all 24) and compare the whole integer state
        op = (it * 2 + seed) % 24
        s._set_state(st13)
        s.set_valid_insert(valid0)
        s.test_copy_struct(a, b, op)
        new, _ = mv.apply_family({k: st[k].copy() for k in FIELDS13}, a, b, op, max_id)
        new, _, _ = mv.renumber_contigs(new)
        got_state = s._get_state()
        for i, k in enumerate(FIELDS13):
            assert np.array_equal(got_state[i], new[k]), (it, op, k)
    assert_scoring_path(s, "rows" if split else "flat")
    s.free_gpu()


def _rebuild_offsets(st):
    """recompute start_bp / sub_pos / contig totals after swapping in real fragment lengths"""
    for c in np.unique(st["id_c"]):
        mem = np.flatnonzero(st["id_c"] == c)
        mem = mem[np.argsort(st["pos"][mem])]
        bp = np.cumsum(st["len_bp"][mem]) - st["len_bp"][mem]
        sp = np.cumsum(st["sub_len"][mem]) - st["sub_len"][mem]
        st["start_bp"][mem] = bp
        st["sub_pos"][mem] = sp
        st["l_cont_bp"][mem] = st["len_bp"][mem].sum()
        st["sub_l_cont"][mem] = st["sub_len"][mem].sum()
    return st


def test_cuda_histogram_matches_oracle(built):
    from oracle.sampler_oracle import distance_histogram
    level = make_level(WORKLOADS["toy"])
    s = make_sampler(level)
    id_start = np.nonzero(level.S_o_A_frags["start_bp"] == 0)[0]
    max_kb = level.S_o_A_frags["l_cont_bp"][id_start].max() / 1000.0
    bin_kb = level.S_o_A_sub_frags["len_bp"].mean() / 1000.0 / 2.0
    n_rows = level.n_frags // 10
    bins, hist, used = s.distance_histogram(max_kb, bin_kb, n_rows)
    obins, omean, oused = distance_histogram(level.sparse_matrix, level.S_o_A_frags, level.np_sub_frags_2_frags,
                                             n_rows, max_kb, bin_kb)
    assert used == oused and len(bins) == len(obins)
    assert np.array_equal(hist, np.round(omean * oused).astype(np.int64))  # integer-exact sums
    s.free_gpu()


def test_full_fit_path_runs_like_the_reference(built):
    """estimate_parameters_rippe -> param_simu identical to the reference's fit on the same data."""
    g = load_golden("toy_bomb_seed2")
    level = make_level(WORKLOADS["toy"])
    s = make_sampler(level)
    max_kb, bin_kb, _ = g["hist_args"]
    s.estimate_parameters_rippe(max_kb, bin_kb, False)
    got = np.array(list(s.param_simu[0]), dtype=np.float32)
    assert np.allclose(got, g["params8"], rtol=1e-5), (got, g["params8"])
    s.free_gpu()


def test_free_running_chain_determinism_and_invariants(built):
    """Size-independent properties on a yeast-like level (config T): two chains with the same seed
    produce bit-identical trajectories (deterministic reductions), scaffold invariants (SURVEY A.3)
    hold after every cycle, the incremental bookkeeping (n_contigs) matches a recount."""
    level = make_level(WORKLOADS["T"])
    outs = []
    for rep in range(2):
        s = make_sampler(level)
        s.set_param_simu(P8_RIPPE)
        np.random.seed(5)
        s.bomb_the_genome()
        traj = []
        frs = np.arange(level.n_frags)
        np.random.shuffle(frs)
        for f in frs[:300]:
            r = s.step_sampler(int(f), 5, np.float32(0.01))
            traj.append((float(r[0]), int(r[2]), int(r[3]), int(r[5])))
        st = s._get_state()
        outs.append((traj, st))
        d = {k: st[i] for i, k in enumerate(FIELDS13)}
        assert (d["pos"] >= 0).all() and (d["l_cont"] > 0).all()
        assert ((d["start_bp"] == 0) == (d["pos"] == 0)).all()
        assert (d["l_cont_bp"] > d["start_bp"]).all()
        assert int((d["pos"] == 0).sum()) == int(s.n_contigs)
        for c in np.unique(d["id_c"])[:50]:
            mem = np.flatnonzero(d["id_c"] == c)
            assert sorted(d["pos"][mem].tolist()) == list(range(len(mem)))
            o = mem[np.argsort(d["pos"][mem])]
            assert np.array_equal(d["start_bp"][o], np.cumsum(d["len_bp"][o]) - d["len_bp"][o])
        assert s.q4_hits == 0
        s.free_gpu()
    assert outs[0][0] == outs[1][0]
    assert np.array_equal(outs[0][1], outs[1][1])
    # the chain must actually assemble something
    assert outs[0][0][-1][3] < level.n_frags


def test_last_block_quirk_switch(built):
    """compat_last_block=False sums every contact: scores may only differ for uniq slots >= n_sub % 64."""
    level = make_level(WORKLOADS["micro"])
    a, b = 3, 4
    res = []
    for compat in (True, False):
        s = make_sampler(level, compat_last_block=compat)
        s.set_param_simu(P8)
        res.append((s.eval_all_sub_likelihood(a, b, 1), s.n_sub_vals[0]))
        s.free_gpu()
    (s1, n1), (s0, n0) = res
    assert n1 == n0
    t = n1 % 64
    order = [m for m in range(24) if s1[m] != 0]
    for k, m in enumerate(order):
        if k < t or t == 0:
            assert s1[m] == s0[m]
        else:
            assert s1[m] >= s0[m]  # the quirk drops (negative) terms


def test_incremental_likelihood_equals_full_recompute(built):
    """Default mode maintains coordinates / lnz_full / zero terms incrementally between full refreshes;
    refresh_every=1 recomputes them over every contact each step like the reference (CL:1407-1409).
    Both must give the same trajectory and the same likelihoods (f64 summation-order noise only);
    a divergence is only allowed at an exact tie."""
    level = make_level(WORKLOADS["T"])
    runs = []
    for refresh, graph in ((1, False), (0, True)):
        s = make_sampler(level)
        s.set_options(refresh_every=refresh, use_graph=graph)
        s.set_param_simu(P8_RIPPE)
        np.random.seed(11)
        s.bomb_the_genome()
        frs = np.arange(level.n_frags)
        np.random.shuffle(frs)
        out = []
        for f in list(frs) + list(frs[:300]):
            r = s.step_sampler(int(f), 5, np.float32(0.01))
            out.append((float(r[0]), int(r[2]), int(r[3]), int(r[5]), np.sort(s.all_scores[s.all_scores != 0])[-2:].copy()))
        runs.append(out)
        st = s.get_stats()
        if refresh == 0:
            assert st["full_refreshes"] <= 1
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


def test_run_cycle_equals_stepwise(built):
    """ig_run_cycle (whole run enqueued without host synchronisation) == the same steps through ig_step."""
    from oracle.sampler_oracle import return_neighbours, setup_distri_frags
    level = make_level(WORKLOADS["toy"])
    distri = setup_distri_frags(level.sub_sampled_sparse_matrix, level.n_frags)
    np.random.seed(21)
    perm = np.random.permutation(level.n_frags).astype(np.int32)
    frs = np.concatenate([np.random.permutation(level.n_frags) for _ in range(3)])
    cands = [sorted(return_neighbours(distri, level.n_frags, int(f), 5)) for f in frs]
    res = []
    for mode in ("step", "cycle"):
        s = make_sampler(level)
        s.set_param_simu(P8)
        import ctypes as C
        from instagraal_b200 import _lib as L
        L.check(s._h, L.lib().ig_bomb(s._h, perm.ctypes.data_as(C.c_void_p)), "ig_bomb")
        if mode == "step":
            out = [s.step_sampler(int(f), 5, np.float32(0.01), candidates=c) for f, c in zip(frs, cands)]
            rec = [(float(o[0]), float(o[1]), int(o[2]), int(o[3]), int(o[5])) for o in out]
        else:
            out = s.run_cycle(frs, 5, candidates=cands)
            rec = [(float(r["likelihood"]), float(r["dist"]), int(r["op_sampled"]), int(r["id_f_sampled"]), int(r["n_contigs"]))
                   for r in out]
        res.append((rec, s._get_state(), s.get_valid_insert()))
        s.free_gpu()
    assert res[0][0] == res[1][0]
    assert np.array_equal(res[0][1], res[1][1])
    assert np.array_equal(res[0][2], res[1][2])


def _lockstep(level, p8, n_steps, seed, bomb=False, n_neigh=5, path=None):
    """product and oracle advance together; after every step the oracle is resynchronised to the
    product's state (so an exact tie broken differently cannot cascade).  path: the scoring path the product must
    have taken (assert_scoring_path)."""
    import oracle.score as sc
    s = make_sampler(level)
    s.set_param_simu(p8)
    o = _oracle(level, p8)
    np.random.seed(seed)
    if bomb:
        s.bomb_the_genome()
    o.live = {k: s._get_state()[i].copy() for i, k in enumerate(FIELDS13)}
    o.valid = [int(x) for x in s.get_valid_insert()]
    frs = np.concatenate([np.random.permutation(level.n_frags) for _ in range(1 + n_steps // level.n_frags)])[:n_steps]
    ties = 0
    for f in frs:
        cands = sorted(int(c) for c in s.return_neighbours(int(f), n_neigh) if int(c) != int(f))
        if not cands:
            continue
        r = s.step_sampler(int(f), n_neigh, np.float32(0.01), candidates=cands)
        ro = o.step_sampler(int(f), n_neigh, candidates=cands)
        want, got = o.all_scores, s.all_scores
        assert np.array_equal(want != 0, got != 0), (f, cands)
        nz = want != 0
        tol = 1e-5 * np.abs(want[nz] - want[nz].max()) + 2e-8 * np.abs(want[nz]) + 1e-9
        assert np.all(np.abs(got[nz] - want[nz]) <= tol), (f, cands, float(np.max(np.abs(got[nz] - want[nz]))))
        st = s._get_state()
        if (int(r[2]), int(r[3])) == (int(ro[2]), int(ro[3])):
            for i, k in enumerate(FIELDS13):
                assert np.array_equal(st[i], o.live[k]), (f, k)
            assert float(r[1]) == float(ro[1]) and int(r[5]) == int(ro[5])
        else:
            gid_s = cands.index(int(r[3])) * 24 + int(r[2])
            gid_o = cands.index(int(ro[3])) * 24 + int(ro[2])
            assert abs(want[gid_s] - want[gid_o]) <= 2e-8 * abs(want[gid_o]) + 1e-9, "diverged without a tie"
            ties += 1
            o.live = {k: st[i].copy() for i, k in enumerate(FIELDS13)}
        o.valid = [int(x) for x in s.get_valid_insert()]
    if path:
        assert_scoring_path(s, path)
    s.free_gpu()
    return ties


def test_edge_tiny_level_down_to_one_contig(built):
    """12 fragments / 34 sub-fragments: ragged sub-fragment counts, windowed same-contig slices, slices
    shorter than one 64-contact block, everything merging into a single contig."""
    level = make_level(SynthSpec(n_frags=12, n_contigs=3, n_chrom=1, max_offset=10, lambda1=5.0, trans_per_row=0.5, seed=3))
    ties = _lockstep(level, P8, 60, seed=0)
    assert ties <= 30


def test_edge_isolated_fragments_and_single_candidate(built):
    """fragments without any contact (empty CSR rows, no level-L neighbour => uniform candidate draw) and
    steps with a single candidate."""
    import scipy.sparse as sp
    level = make_level(SynthSpec(n_frags=30, n_contigs=4, n_chrom=2, max_offset=30, lambda1=8.0, trans_per_row=1.0, seed=9))
    # wipe every contact of fragments 0 and 7 (their sub-fragment rows and columns)
    parent = level.np_sub_frags_2_frags["x"].astype(np.int64)
    kill = np.isin(parent, [0, 7])
    m = level.sparse_matrix.tocoo()
    keep = ~(kill[m.row] | kill[m.col])
    level.sparse_matrix = sp.csr_matrix((m.data[keep], (m.row[keep], m.col[keep])), shape=m.shape, dtype=np.int32)
    mm = level.sub_sampled_sparse_matrix.tocoo()
    keep2 = ~(np.isin(mm.row, [0, 7]) | np.isin(mm.col, [0, 7]))
    level.sub_sampled_sparse_matrix = sp.csr_matrix((mm.data[keep2], (mm.row[keep2], mm.col[keep2])), shape=mm.shape, dtype=np.int32)
    ties = _lockstep(level, P8, 70, seed=4, bomb=True)
    assert ties <= 35
    ties = _lockstep(level, P8, 40, seed=5, n_neigh=1)
    assert ties <= 20


def test_checkpoint_resume_is_bit_identical(built, tmp_path):
    """N3 (SURVEY 8f): stop after 150 steps, resume in a NEW sampler, and the next 150 steps (incl. the
    host RNG draws) equal the uninterrupted run's."""
    level = make_level(WORKLOADS["toy"])

    def steps(s, n):
        out = []
        frs = np.arange(level.n_frags)
        while len(out) < n:
            np.random.shuffle(frs)
            for f in frs:
                r = s.step_sampler(int(f), 5, np.float32(0.01))
                out.append((float(r[0]), float(r[1]), int(r[2]), int(r[3]), int(r[5])))
                if len(out) == n:
                    break
        return out

    a = make_sampler(level)
    a.set_param_simu(P8)
    np.random.seed(33)
    a.bomb_the_genome()
    steps(a, 150)
    ck = str(tmp_path / "chain.npz")
    a.save_checkpoint(ck)
    cont = steps(a, 150)
    final_a = a._get_state()
    a.free_gpu()
    b = make_sampler(level)
    np.random.seed(999)  # must be overwritten by the checkpoint
    b.load_checkpoint(ck)
    res = steps(b, 150)
    assert res == cont
    assert np.array_equal(b._get_state(), final_a)
    b.free_gpu()


def test_contact_thumbnail_matches_numpy_binning(built, tmp_path):
    """N1 (SURVEY 8f): GPU-binned K x K contact map in the current scaffold order == NumPy binning."""
    from oracle.sampler_oracle import upper_coo
    level = make_level(WORKLOADS["toy"])
    s = make_sampler(level)
    s.set_param_simu(P8)
    np.random.seed(2)
    s.bomb_the_genome()
    for f in np.random.permutation(level.n_frags)[:120]:
        s.step_sampler(int(f), 5, np.float32(0.01))
    K = 64
    img = s.contact_thumbnail(K)
    _fo, _dc, high = s.display_order()
    assert sorted(high) == list(range(level.n_sub_frags))
    rank = np.empty(level.n_sub_frags, dtype=np.int64)
    rank[np.asarray(high)] = np.arange(len(high))
    rows, cols, dat = upper_coo(level.sparse_matrix)
    pi, pj = rank[rows] * K // level.n_sub_frags, rank[cols] * K // level.n_sub_frags
    want = np.zeros((K, K), dtype=np.int64)
    np.add.at(want, (pi, pj), dat)
    off = pi != pj
    np.add.at(want, (pj[off], pi[off]), dat[off])
    assert np.array_equal(img.astype(np.int64), want)
    out = s.display_current_matrix(str(tmp_path / "m.pgm"), size=K)
    assert len(out[0]) == level.n_frags and (tmp_path / "m.pgm").stat().st_size > K * K
    s.free_gpu()


def test_rigid_pruning_mode_differs_only_by_coordinate_rounding_noise(built):
    """rigid_pruning=True skips contacts whose two ends undergo the same rigid motion (their term cannot
    change mathematically); the default re-evaluates them like the reference and picks up the float32
    re-rounding of shifted coordinates (an ulp of the COORDINATE, i.e. ~1e-5 relative on short distances).
    The two modes must agree up to that noise and choose the same move unless two scores are that close."""
    level = make_level(WORKLOADS["T"])
    ss = [make_sampler(level, rigid_pruning=e) for e in (True, False)]
    for s in ss:
        s.set_param_simu(P8_RIPPE)
        np.random.seed(5)
        s.bomb_the_genome()
    rng = np.random.RandomState(9)
    worst_rel, n_div = 0.0, 0
    for t in range(1500):
        a = int(rng.randint(level.n_frags))
        cands = [int(c) for c in rng.choice(level.n_frags, 5, replace=False) if c != a]
        outs = [s.step_sampler(a, 5, np.float32(0.01), candidates=cands) for s in ss]
        f, e = ss[0].all_scores.copy(), ss[1].all_scores.copy()
        assert np.array_equal(f != 0, e != 0)
        nz = e != 0
        rel = float(np.max(np.abs(f[nz] - e[nz]) / np.abs(e[nz])))
        worst_rel = max(worst_rel, rel)
        assert rel < 2e-6, (t, rel)
        if (outs[0][2], outs[0][3]) != (outs[1][2], outs[1][3]):
            top = np.sort(e[nz])[-2:]
            assert abs(top[1] - top[0]) <= 4e-6 * abs(top[1]), "diverged without a near-tie"
            n_div += 1
            ss[0]._set_state(ss[1]._get_state())
            ss[0].set_valid_insert(ss[1].get_valid_insert())
    print("rigid pruning vs default: worst relative score difference", worst_rel, "divergences", n_div)
    for s in ss:
        s.free_gpu()


def test_device_rng_cycle_matches_oracle_plan_and_host_plan_run(built):
    """Production RNG mode: the candidates drawn on the device (Philox4x32-10) equal the NumPy restatement
    (oracle/device_rng.py) draw for draw, and the chain they drive is bit-identical to run_cycle fed with
    that plan from the host."""
    from oracle.device_rng import draw_plan
    level = make_level(WORKLOADS["toy"])
    a, b = make_sampler(level), make_sampler(level)
    for s in (a, b):
        s.set_param_simu(P8_RIPPE)
        np.random.seed(4)
        s.bomb_the_genome()
    rng = np.random.RandomState(21)
    seed = 0x1234_5678_9ABC_DEF0
    for cyc in range(2):
        frags = rng.permutation(level.n_frags).astype(np.int32)
        out_dev = a.run_cycle_device(frags, 5, seed=seed, cycle=cyc)
        plan = a.last_cycle_plan(len(frags))
        ptr, idx, cdf, nnz = a.neighbour_weights_csr()
        want = draw_plan(frags, 5, level.n_frags, ptr, idx, cdf, nnz, seed, cyc)
        assert np.array_equal(plan, want)
        assert plan[:, 0].min() >= 1 and plan[:, 0].max() <= 5
        cands = [plan[t, 2:2 + plan[t, 0]].tolist() for t in range(len(frags))]
        out_host = b.run_cycle(frags, 5, candidates=cands)
        for f in ("op_sampled", "id_f_sampled", "n_contigs", "sum_l_cont", "n_proposals", "likelihood", "dist"):
            assert np.array_equal(out_dev[f], out_host[f]), f
        assert np.array_equal(a._get_state(), b._get_state())
    # a different seed gives a different plan; draws are proportional to the weights
    a.run_cycle_device(frags, 5, seed=seed + 1, cycle=0)
    assert not np.array_equal(a.last_cycle_plan(len(frags)), plan)
    for s in (a, b):
        s.free_gpu()


def test_yeast_toy_config0_lockstep(built):
    """BASELINE.json configs[0]: the reference's tests/data contigs digested (DpnII + HinfI) and binned to
    level 4 (1015 fragments / 2857 sub-fragments, 146 contigs incl. single-fragment ones with 1-2
    sub-fragments), simulated contacts; product and oracle in lockstep from the contig-order start."""
    from instagraal_b200.synth import make_workload
    level = make_workload("yeast_toy")
    assert (level.n_frags, level.n_sub_frags) == (1015, 2857)
    ties = _lockstep(level, P8_RIPPE, 40, seed=2)
    assert ties <= 8


@pytest.mark.parametrize("env", [{"IG_SCORING_PATH": "stream"}, {"IG_SCORING_PATH": "rows"},
                                 {"IG_SCORING_PATH": "rows", "IG_FORCE_SPLIT": "24,1"}])
def test_large_level_code_paths_on_a_small_level(built, env, monkeypatch):
    """The two-pass affected-row list (levels above 16 Ki sub-fragments) with the streaming path, with the row-per-warp
    kernel, and with its whole-row work split only run on large levels by default; forced here on the toy level, in
    lockstep with the oracle."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    level = make_level(WORKLOADS["toy"])
    ties = _lockstep(level, P8_RIPPE, 80, seed=6, bomb=True, path=env["IG_SCORING_PATH"])
    assert ties <= 40


def test_medium_level_with_long_contigs_takes_the_large_level_paths_naturally(built):
    """6000 fragments / 18k sub-fragments in 12 long contigs: above 16 Ki sub-fragments the affected-row list is
    built in two passes, candidates have > 1000 affected rows so each work item covers all 24 mutations of a
    whole row (chunk-ahead fetch), and most contacts of a 500-fragment contig do not change under a mutation, so
    the (contact, mutation) pairs are dealt sparsely to the lanes -- the operating point of the 1 Gb workload,
    at a size the oracle still finishes in seconds per step.  Lockstep with the oracle."""
    level = make_level(SynthSpec(n_frags=6000, n_contigs=12, n_chrom=2, max_offset=300, lambda1=30.0, trans_per_row=2.0, seed=11))
    assert level.n_sub_frags > 16 * 1024
    ties = _lockstep(level, P8_RIPPE, 30, seed=3, path="stream")
    assert ties <= 6


@pytest.mark.parametrize("rigid", [True, False])
@pytest.mark.parametrize("workload,steps", [("T", 1200), ("toy", 400)])
def test_streaming_path_equals_row_per_warp_rigid_path(built, workload, steps, rigid, monkeypatch):
    """The streaming scoring path of large levels (k_stream + k_eval_flat<true>, rigid_pruning=1) forced on small levels
    against the row-per-warp kernel k_score (rows path): same selected-contact counts, scores equal up to the 2^-32
    fixed-point rounding of the streaming path's order-independent sums, same trajectory (unless two scores are that
    close), and two runs of the streaming path are bit-identical although its pick list is appended in arbitrary order.
    rigid = False: the same in the reference-faithful mode, where large levels send their small candidates (mid-assembly
    contigs) down this path."""
    level = make_level(WORKLOADS[workload])
    p8 = P8_RIPPE if workload == "T" else P8
    monkeypatch.setenv("IG_SCORING_PATH", "rows")
    ref = make_sampler(level, rigid_pruning=rigid)        # k_score (rigid: with the rigid class-pair table)
    monkeypatch.setenv("IG_SCORING_PATH", "stream")
    st1 = make_sampler(level, rigid_pruning=rigid)
    st2 = make_sampler(level, rigid_pruning=rigid)
    ss = [ref, st1, st2]
    for s in ss:
        s.set_param_simu(p8)
        np.random.seed(5)
        s.bomb_the_genome()
    rng = np.random.RandomState(10)
    n_div = 0
    worst = 0.0
    for t in range(steps):
        a = int(rng.randint(level.n_frags))
        cands = sorted(int(c) for c in rng.choice(level.n_frags, 5, replace=False) if c != a)
        outs = [s.step_sampler(a, 5, np.float32(0.01), candidates=cands) for s in ss]
        r, x, y = (s.all_scores.copy() for s in ss)
        assert np.array_equal(x, y), ("streaming path not deterministic", t)
        assert outs[1] == outs[2]
        assert ss[0].n_sub_vals == ss[1].n_sub_vals, (t, ss[0].n_sub_vals, ss[1].n_sub_vals)
        assert np.array_equal(r != 0, x != 0)
        nz = r != 0
        d = float(np.max(np.abs(r[nz] - x[nz])))
        worst = max(worst, d)
        assert d < 1e-6, (t, d)
        if (outs[0][2], outs[0][3]) != (outs[1][2], outs[1][3]):
            top = np.sort(r[nz])[-2:]
            assert abs(top[1] - top[0]) <= 2e-6, "diverged without a tie"
            n_div += 1
            for s in ss[1:]:
                s._set_state(ss[0]._get_state())
                s.set_valid_insert(ss[0].get_valid_insert())
    assert np.array_equal(ss[0]._get_state(), ss[1]._get_state()) or n_div > 0
    print("streaming vs row-per-warp (rigid): worst |score difference|", worst, "tie divergences", n_div)
    for s, path in zip(ss, ("rows", "stream", "stream")):
        assert_scoring_path(s, path, rigid)
        s.free_gpu()


@pytest.mark.parametrize("rigid", [True, False])
def test_streaming_path_random_scaffolds_with_circular_contigs(built, rigid, monkeypatch):
    """eval on random scaffolds incl. circular contigs (left to k_score inside a streaming-mode step) and reversed
    fragments: the streaming path == the row-per-warp kernel (rows path)."""
    from oracle.fuzz import random_state
    level = make_level(WORKLOADS["micro"])
    monkeypatch.setenv("IG_SCORING_PATH", "rows")
    ref = make_sampler(level, rigid_pruning=rigid)
    monkeypatch.setenv("IG_SCORING_PATH", "stream")
    st = make_sampler(level, rigid_pruning=rigid)
    for s in (ref, st):
        s.set_param_simu(P8)
    rng = np.random.RandomState(3)
    nf = level.n_frags
    for it in range(40):
        state = random_state(nf, rng, p_circ=0.4)
        for k in ("len_bp", "sub_len"):
            state[k] = np.asarray(level.S_o_A_frags[k], dtype=np.int32).copy()
        state = _rebuild_offsets(state)
        st13 = np.stack([state[k] for k in FIELDS13]).astype(np.int32)
        a, b = [int(x) for x in rng.choice(nf, 2, replace=False)]
        valid0 = rng.choice([-1, 1], 12).astype(np.int32)
        res = []
        for s in (ref, st):
            s._set_state(st13)
            s.set_valid_insert(valid0)
            res.append((s.eval_all_sub_likelihood(a, b, 1), s.n_sub_vals[0]))
        assert res[0][1] == res[1][1], (it, a, b)
        assert np.array_equal(res[0][0] != 0, res[1][0] != 0)
        assert np.max(np.abs(res[0][0] - res[1][0])) < 1e-6, (it, a, b, np.max(np.abs(res[0][0] - res[1][0])))
    assert_scoring_path(ref, "rows", rigid)
    assert_scoring_path(st, "stream", rigid)
    ref.free_gpu(); st.free_gpu()


def _nuis_params(p8, i):
    q = np.array(p8, dtype=np.float32).copy()
    q[3] += np.float32(0.002 * (i % 5))        # slope
    q[5] *= np.float32(1.0 + 0.05 * (i % 3))   # d_max: moves contacts between the queued and the floor class
    q[6] *= np.float32(1.0 + 0.01 * i)         # fact
    return q


@pytest.mark.parametrize("workload,steps", [("toy", 150), ("T", 300)])
def test_cached_likelihood_records_equal_the_gather_kernel(built, workload, steps, monkeypatch):
    """The nuisance likelihood from the cached per-contact records (k_lnz_refresh + k_lnz_stream, the default) against the
    row-by-row gather kernel (k_full_lnz, IG_LNZ_CACHE=0) along one trajectory: after every step (only the rows of the
    contigs the last move touched are rebuilt; the coordinates are the STALE ones of quirk Q5 in both), for several test
    parameter sets per step (the second and third run on a clean cache), after a bomb and after a state upload.  Every
    tenth step follows a parameter change: the default then recomputes lnz_full from the records too (step kind 2)."""
    from instagraal_b200.synth import make_workload
    level = make_workload(workload) if workload == "T" else make_level(WORKLOADS[workload])
    a = GpuImpl(level)
    monkeypatch.setenv("IG_LNZ_CACHE", "0")
    b = GpuImpl(level)
    monkeypatch.delenv("IG_LNZ_CACHE")
    for impl in (a, b):
        impl.set_params(P8_RIPPE)
        np.random.seed(5)
        impl.s.bomb_the_genome()
    rng = np.random.RandomState(9)
    worst = 0.0
    t = 0
    for f in rng.permutation(level.n_frags)[:steps]:
        f = int(f)
        cands = sorted(int(c) for c in rng.choice(level.n_frags, 4, replace=False) if c != f)
        if t % 10 == 5:   # an accepted nuisance proposal: the next step recomputes the likelihood sums under the new parameters
            q = _nuis_params(P8_RIPPE, t)   # (a: from the records, coordinates through the incremental commit; b: from scratch)
            a.set_params(q); b.set_params(q)
        ra, rb = a.step(f, cands), b.step(f, cands)
        assert (int(ra["op"]), int(ra["B"])) == (int(rb["op"]), int(rb["B"])), (t, ra["op"], rb["op"])
        assert abs(float(ra["o"]) - float(rb["o"])) <= 1e-11 * abs(float(rb["o"])), (t, ra["o"], rb["o"])
        assert np.allclose(ra["scores"], rb["scores"], rtol=1e-11, atol=0)
        for i in range(3 if t % 7 == 0 else 1):
            q = _nuis_params(P8_RIPPE, t + i)
            va, vb = a.eval_nuisance(q), b.eval_nuisance(q)
            worst = max(worst, abs(va - vb) / abs(vb))
            assert abs(va - vb) <= 1e-11 * abs(vb), (t, i, va, vb)
        if t == steps // 2:   # state upload in mid-run: every record is rebuilt from fresh coordinates
            st = a.get_state()
            for impl in (a, b):
                impl.set_state(st)
        t += 1
    a.s.free_gpu(); b.s.free_gpu()


def test_cached_likelihood_records_with_circular_contigs(built, monkeypatch):
    """rows of circular contigs never enter the record stream: k_lnz_refresh evaluates them with the generic routine on
    every call.  Random scaffolds with circular contigs, fresh and repeated evaluations, d == 2 and d != 2."""
    from oracle.fuzz import random_state
    level = make_level(WORKLOADS["micro"])
    a = GpuImpl(level)
    monkeypatch.setenv("IG_LNZ_CACHE", "0")
    b = GpuImpl(level)
    monkeypatch.delenv("IG_LNZ_CACHE")
    rng = np.random.RandomState(3)
    for it in range(10):
        p8 = P8.copy()
        if it % 2:
            p8[4] = 2.37
        st = random_state(level.n_frags, rng, p_circ=0.5)
        for k in ("len_bp", "sub_len"):
            st[k] = np.asarray(level.S_o_A_frags[k], dtype=np.int32).copy()
        st = _rebuild_offsets(st)
        st13 = np.stack([st[k] for k in FIELDS13]).astype(np.int32)
        for impl in (a, b):
            impl.set_params(p8)
            impl.set_state(st13)
        for i in range(3):
            q = _nuis_params(p8, it + i)
            va, vb = a.eval_nuisance(q), b.eval_nuisance(q)
            assert abs(va - vb) <= 1e-11 * abs(vb), (it, i, va, vb)
    a.s.free_gpu(); b.s.free_gpu()
