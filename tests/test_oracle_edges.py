"""The large-level kernels against the NumPy oracle (oracle/score.py, oracle/sampler_oracle.py) at the edges where a kernel
can be wrong while two GPU paths still agree with each other:

A. the full likelihood (ig_full_likelihood: k_exz_table, k_coords + k_reduce, k_lnz_refresh + k_lnz_stream or k_full_lnz)
   and the facade's eval_likelihood_4_nuisance, over scaffolds with circular and long contigs, a parameter grid that puts
   d_max, v_inter and the counts on their switch points, both likelihood paths, stale and fresh coordinates, graphed and not;
   the error bound is derived per contact from the float32 expected values, not fitted;
B. scores and apply of one candidate pair on levels above 16 Ki sub-fragments (two-pass row list, whole-row splits, sparse
   pair dealing, the streaming path) with circular contigs and reversed fragments;
C. the distance histogram of the p(s) fit, integer-exact.

The wrap level holds >= 46 342 sub-fragments in one contig, so the int32 products of quirk Q8 (n_pixl_sub_mat) and of
intra_pairs wrap (KA:3950-3953) -- the regime of every human-scale level of the reference.

IG_TEST_G_LIKELIHOOD=1 also runs part A on one scaffold of the 1 Gb level G (about 10 GB of host memory for the oracle)."""
import contextlib
import math
import os

import numpy as np
import pytest

import oracle.score as sc
from instagraal_b200 import _lib as L
from instagraal_b200.cuda_lib_gl_single import PARAM_SIMU_RIPPE, _ptr
from instagraal_b200.synth import WORKLOADS, SynthSpec, make_level, make_workload
from oracle import moves as mv
from oracle.fuzz import random_state
from oracle.sampler_oracle import OracleSampler, distance_histogram
from parity_common import FIELDS13
from test_gpu_parity import P8, P8_RIPPE, _rebuild_offsets, assert_scoring_path, make_sampler

pytestmark = pytest.mark.gpu

LOG10E = 0.43429448190325182
ULP8 = 2.0 ** -20          # ~8 float32 ulp: libm vs libdevice powf / expf on an expected value, with margin
INT32_PAIRS_WRAP = 46342   # smallest n with n * (n - 1) > 2^31 - 1

MEDIUM = SynthSpec(n_frags=6000, n_contigs=12, n_chrom=2, max_offset=300, lambda1=30.0, trans_per_row=2.0, seed=11)
# ~16.5k fragments of <= 3 sub-fragments, short-range contacts only: ~50k sub-fragments, ~250k contacts
WRAP = SynthSpec(n_frags=16500, n_contigs=4, n_chrom=1, max_offset=30, lambda1=4.0, trans_per_row=0.2, seed=5)
COUNT_VALUES = np.array(list(range(1, 17)) + [1000, 4096, 65535], dtype=np.int32)   # every count around ob_const's switch


@contextlib.contextmanager
def _env(**kw):
    """environment variables read by ig_create, set while a handle is created"""
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


_LEVELS = {}


def _level(name):
    if name not in _LEVELS:
        if name == "micro_counts":
            lv = make_level(WORKLOADS["micro"])
            m = lv.sparse_matrix
            m.data[:] = COUNT_VALUES[np.arange(m.nnz) % COUNT_VALUES.size]
        elif name == "medium":
            lv = make_level(MEDIUM)
        elif name == "wrap":
            lv = make_level(WRAP)
        else:
            lv = make_workload(name)
        _LEVELS[name] = lv
    return _LEVELS[name]


def _check_level_size(name, level):
    ns = level.n_sub_frags
    if name == "T":
        assert (level.n_frags, ns) == (900, 2549)
    elif name == "medium":
        assert level.n_frags == 6000 and ns > 16 * 1024
    elif name == "wrap":
        assert ns >= INT32_PAIRS_WRAP and ns * (ns - 1) < 2 ** 32, ns   # the int32 pair counts wrap to negative values
        assert level.sparse_matrix.nnz < 5_000_000
    elif name == "micro_counts":
        assert set(np.unique(level.sparse_matrix.data)) == set(COUNT_VALUES.tolist())


def _dp_bits(ns):
    """the width of the table index in a packed likelihood record, as ig_create computes it"""
    b = 1
    while (1 << b) < ns + 3:
        b += 1
    return b


def _full_likelihood(s, p8, stale):
    out = np.zeros(3, dtype=np.float64)
    p = np.ascontiguousarray(np.asarray(p8, dtype=np.float32))
    L.check(s._h, L.lib().ig_full_likelihood(s._h, _ptr(p), int(stale), _ptr(out)), "ig_full_likelihood")
    return out


def _facade_nuisance(s, p8):
    s.param_simu_test = np.array([tuple(np.asarray(p8, dtype=np.float32).tolist())], dtype=PARAM_SIMU_RIPPE)
    return s.eval_likelihood_4_nuisance()


def _as13(st):
    return np.stack([np.asarray(st[k], dtype=np.int32) for k in FIELDS13])


def _as_dict(st13):
    return {k: np.array(st13[i], dtype=np.int32) for i, k in enumerate(FIELDS13)}


def _real_lengths(level, st):
    for k in ("len_bp", "sub_len"):
        st[k] = np.asarray(level.S_o_A_frags[k], dtype=np.int32).copy()
    return _rebuild_offsets(st)


# ------------------------------------------------------------------------------------------------------------------
# A. full likelihood
class Reference:
    """the oracle's likelihood parts for one scaffold and one parameter set, with the error bound of each:
    per contact b = 2^-20 (log10(e) ob + ex + log10(e) exz) -- a relative error of 2^-20 on the float32 expected value ex
    moves ob log10(ex) by log10(e) ob 2^-20 and ex by ex 2^-20 -- plus 1e-13 of the sum of |term| for the summation
    order; the zero term Z likewise with ex (len - pos)."""

    def __init__(self, o, v, p8):
        p = sc.Params(p8)
        rows, cols, dat = o.coo
        with np.errstate(all="ignore"):
            t, ex, exz = sc.contact_terms(v, rows, cols, dat, p, o.mbar, len_from="row", return_parts=True)
        assert np.all(np.isfinite(t))
        ob = dat.astype(np.float64)
        b = ULP8 * (LOG10E * ob + np.abs(ex.astype(np.float64)) + LOG10E * np.abs(exz.astype(np.float64)))
        self.lnz = math.fsum(t)
        self.lnz_bound = math.fsum(b) + 1e-13 * math.fsum(np.abs(t))
        with np.errstate(all="ignore"):
            _, self.n_intra, zt = sc.zeros_term_raw(v, p, o.mbar, return_parts=True)
        self.z = -math.fsum(zt)
        self.z_bound = (ULP8 + 1e-13) * math.fsum(np.abs(zt))
        self.ex, self.dat = ex, dat
        self.p8 = np.asarray(p8, dtype=np.float32)

    def check(self, out3, what):
        """-> worst error / bound ratio of Lnz and Z; n_intra exactly"""
        assert int(out3[2]) == self.n_intra, (what, int(out3[2]), self.n_intra)
        e_l, e_z = abs(out3[0] - self.lnz), abs(out3[1] - self.z)
        assert e_l <= self.lnz_bound, (what, out3[0], self.lnz, e_l, self.lnz_bound)
        assert e_z <= self.z_bound, (what, out3[1], self.z, e_z, self.z_bound)
        return max(e_l / max(self.lnz_bound, 1e-300), e_z / max(self.z_bound, 1e-300))


def _param_grid(base, o, v, single_linear):
    """(name, p8) around ``base`` for the scaffold with coordinates ``v``"""
    base = np.asarray(base, dtype=np.float32)
    grid = [("base", base.copy())]

    def var(name, **kw):
        q = base.copy()
        for k, x in kw.items():
            q[("kuhn", "lm", "c1", "slope", "d", "d_max", "fact", "v_inter").index(k)] = np.float32(x)
        grid.append((name, q))

    for d in (1.8, 2.37, 3.0):
        var("d=%g" % d, d=d)
    for sl in (-0.5, -2.5):
        var("slope=%g" % sl, slope=sl)
    for f in (1e-3, 1e3):
        var("fact*%g" % f, fact=base[6] * np.float32(f))
    rows, cols, _ = o.coo
    same = v["id_c"][rows] == v["id_c"][cols]
    s = np.abs(v["dist"][rows] - v["dist"][cols]).astype(np.float32)
    s_in = np.sort(s[same & (s > 0)])
    assert s_in.size > 0
    var("d_max below every separation", d_max=s_in[0] * np.float32(0.5))
    var("d_max above every contig", d_max=np.float32(2e-3) * np.float32(np.max(o.live["l_cont_bp"])) + np.float32(1.0))
    s_k = s_in[s_in.size // 2]   # a contact's separation: d_max on it, one ulp below and one above (strict s < d_max)
    for nm, x in (("d_max = s", s_k), ("d_max = s-", np.nextafter(s_k, np.float32(0))), ("d_max = s+", np.nextafter(s_k, np.float32(np.inf)))):
        var(nm, d_max=x)
    dp = np.abs(v["pos"][rows] - v["pos"][cols])[same]
    dp_k = int(np.bincount(dp).argmax())   # the most frequent separation: as many contacts as possible on the boundary
    s_z = np.float32(dp_k) * o.mbar   # a contact's zero-term separation (the expected-contact table's s_z < d_max)
    var("d_max = s_z", d_max=s_z)
    with np.errstate(all="ignore"):
        _, ex0, exz0 = sc.contact_terms(v, rows, cols, o.coo[2], sc.Params(base), o.mbar, len_from="row", return_parts=True)
    var("v_inter tiny", v_inter=1e-12)
    var("v_inter above every expected value", v_inter=np.float32(2.0) * max(float(ex0.max()), float(exz0.max())))
    lin_in = same & (v["s_tot"][rows] == 0) & (s > 0) & (s < base[5]) & (ex0 > base[7])
    if lin_in.any():   # (linear contigs only: a circular contig's expected value is floored at d_max, not v_inter)
        var("v_inter = ex of a contact", v_inter=ex0[np.flatnonzero(lin_in)[int(lin_in.sum()) // 3]])
    var("v_inter = 0", v_inter=0.0)
    if single_linear:
        # one linear contig: no contact sits on the floor, so a negative v_inter keeps every term finite; then the table entry
        # at s_z == d_max (v_inter) differs from rippe_contacts(d_max) (max(0, v_inter)) -- the only case where it does
        var("v_inter < 0, d_max = s_z", v_inter=-0.25, d_max=s_z)
    return grid


def _scaffolds(name, level, s0):
    """(label, int32[13, NF]) of part A for one level"""
    nf = level.n_frags
    out = [("initial", s0._get_state())]
    rng = np.random.RandomState(17)
    if name == "wrap":
        for circ in (0, 1):
            st = _real_lengths(level, random_state(nf, rng, p_circ=circ, max_contigs=1))
            assert int(st["circ"][0]) == circ and int(st["l_cont"][0]) == nf
            out.append(("one %s contig" % ("circular" if circ else "linear"), _as13(st)))
        return out
    np.random.seed(3)
    s0.bomb_the_genome()
    out.append(("bombed", s0._get_state()))
    for i in range(2):
        st = _real_lengths(level, random_state(nf, rng, p_circ=0.4, max_contigs=20))
        out.append(("random %d (%d circular fragments)" % (i, int(st["circ"].sum())), _as13(st)))
    out.append(("initial contigs joined into one", _joined(level, out[0][1])))
    return out


def _joined(level, st13):
    """one linear contig holding every fragment in the order of ``st13``'s contigs: near-diagonal contacts stay close, so
    many of them share a sub-fragment separation"""
    st = _as_dict(st13)
    order = np.lexsort((st["pos"], st["id_c"]))
    nf = order.size
    st["pos"][order] = np.arange(nf)
    st["id_c"][:] = 0
    st["circ"][:] = 0
    st["l_cont"][:] = nf
    st["prev"][order] = np.r_[-1, order[:-1]]
    st["next"][order] = np.r_[order[1:], -1]
    return _as13(_real_lengths(level, st))


def _likelihood_grid(name, base):
    level = _level(name)
    _check_level_size(name, level)
    rec = make_sampler(level)
    with _env(IG_LNZ_CACHE=0):
        gat = make_sampler(level)
    o = OracleSampler(level, base)
    worst = {}
    try:
        for s in (rec, gat):
            s.set_param_simu(base)
        if name == "wrap":   # quirk Q8: the product's n_pixl_sub_mat (int32 arithmetic) wraps to a negative value
            ns = level.n_sub_frags
            assert rec.n_pixl_sub_mat == o.n_pix < 0 and o.n_pix != ns * (ns - 1) / 2
        for label, st13 in _scaffolds(name, level, rec):
            live = _as_dict(st13)
            v = sc.fill_vect_dist(live, o.sub)
            o.live, o.v_cur = live, v
            single_linear = int(live["l_cont"][0]) == level.n_frags and int(live["circ"][0]) == 0
            if name == "wrap" and int(live["l_cont"][0]) == level.n_frags:
                ref0 = Reference(o, v, base)
                assert ref0.n_intra < 0, ref0.n_intra   # the int32 pair count of the one contig wrapped
            for s in (rec, gat):
                s._set_state(st13)
                _full_likelihood(s, base, 0)   # fresh coordinates of this scaffold (stale = 1 reuses them)
            for pname, p8 in _param_grid(base, o, v, single_linear):
                ref = Reference(o, v, p8)
                if p8[7] == 0:
                    # gather path only (records need v_inter > 0); a zero or subnormal ex would make log10 ill-posed
                    eval_ex = ref.ex[ref.ex != 0]
                    assert np.all(np.abs(eval_ex) >= np.finfo(np.float32).tiny), pname
                runs = [("gather", gat, 0, False), ("gather", gat, 1, False)]
                for graph in (False, True):
                    runs += [("records", rec, 0, graph), ("records", rec, 1, graph)]
                for path, s, stale, graph in runs:
                    s.set_options(refresh_every=4096, use_graph=graph)
                    what = (label, pname, path, "stale" if stale else "fresh", "graph" if graph else "no graph")
                    worst[path] = max(worst.get(path, 0.0), ref.check(_full_likelihood(s, p8, stale), what))
                # the facade's nuisance likelihood (stale coordinates + the Q8 inter-contig zero term) against the oracle's
                got = _facade_nuisance(rec, p8)
                want = o.eval_likelihood_4_nuisance(p8)
                bound = ref.lnz_bound + LOG10E * ref.z_bound + 1e-13 * abs(want)
                assert abs(got - want) <= bound, (label, pname, got, want, bound)
                worst["facade"] = max(worst.get("facade", 0.0), abs(got - want) / bound)
    finally:
        rec.free_gpu()
        gat.free_gpu()
    print("%s: worst |error| / bound" % name, {k: "%.3g" % x for k, x in worst.items()})
    return worst


@pytest.mark.parametrize("name,base", [("micro_counts", P8), ("T", P8_RIPPE), ("medium", P8_RIPPE), ("wrap", P8_RIPPE)],
                         ids=["micro_counts", "T", "medium", "wrap"])
def test_full_likelihood_matches_oracle_within_derived_bound(built, name, base):
    """Lnz, raw Z and n_intra of ig_full_likelihood, and the facade's eval_likelihood_4_nuisance, against the oracle:
    initial / bombed / random scaffolds with circular and long contigs (the wrap level: all fragments in one linear or
    circular contig), d != 2, extreme slopes and scale factors, d_max below / above / on a contact's separation and on a
    table entry, v_inter tiny / above every expected value / equal to one / zero; records and gather path, stale and fresh
    coordinates, graphed and not.  micro_counts: counts 1..16 (the ob >= 15 switch of ob_const) and >= 1000."""
    _likelihood_grid(name, base)


@pytest.mark.skipif(os.environ.get("IG_TEST_G_LIKELIHOOD") != "1", reason="opt-in: IG_TEST_G_LIKELIHOOD=1 (~10 GB host memory)")
def test_full_likelihood_matches_oracle_on_G(built):
    level = make_workload("G")
    _LEVELS["G"] = level
    try:
        _likelihood_grid("G", P8_RIPPE)
    finally:
        _LEVELS.pop("G", None)


@pytest.mark.parametrize("over", [0, 1])
def test_likelihood_record_packing_limit(built, over):
    """A count of 2^(32 - dp_bits) - 1 still fits a packed likelihood record (records used), 2^(32 - dp_bits) does not
    (records refused: the gather path); both likelihoods equal the oracle's.  An overflowing pack or a guard off by one
    shows up as an error of the size of the count."""
    level = make_level(WORKLOADS["micro"])
    limit = 1 << (32 - _dp_bits(level.n_sub_frags))
    m = level.sparse_matrix
    row = np.repeat(np.arange(m.shape[0]), np.diff(m.indptr))
    parent = level.np_sub_frags_2_frags["x"].astype(np.int64)
    cid = level.S_o_A_frags["id_c"][parent]
    near = (m.indices > row) & (m.indices - row <= 2) & (cid[row] == cid[m.indices])
    k = int(np.flatnonzero(near)[7])   # an intra-contig contact a few sub-fragments apart: queued, not a floor term
    m.data[k] = limit - 1 + over
    s = make_sampler(level)
    try:
        s.set_param_simu(P8)
        o = OracleSampler(level, P8)
        assert int(o.coo[2].max()) == limit - 1 + over
        rc = L.lib().ig_set_device_nuisance(s._h, 1)   # needs the records: refused exactly when the count does not fit
        if over:
            assert rc != 0 and b"records" in L.lib().ig_last_error(s._h)
        else:
            assert rc == 0
            L.check(s._h, L.lib().ig_set_device_nuisance(s._h, 0), "ig_set_device_nuisance")
        o.live = _as_dict(s._get_state())
        o.v_cur = sc.fill_vect_dist(o.live, o.sub)
        _full_likelihood(s, P8, 0)
        for d in (2.0, 2.37):
            p8 = P8.copy()
            p8[4] = d
            ref = Reference(o, o.v_cur, p8)
            for stale in (0, 1):
                ref.check(_full_likelihood(s, p8, stale), ("packing", over, d, stale))
            got, want = _facade_nuisance(s, p8), o.eval_likelihood_4_nuisance(p8)
            assert abs(got - want) <= ref.lnz_bound + LOG10E * ref.z_bound + 1e-13 * abs(want), (got, want)
    finally:
        s.free_gpu()


# ------------------------------------------------------------------------------------------------------------------
# B. scores and apply on large-level paths
def _score_pairs(name, rng, n):
    """(scaffold dict, a, b) for part B"""
    level = _level(name)
    nf = level.n_frags
    out = []
    if name == "wrap":   # all fragments in one contig: linear, then circular
        for circ in (0, 1):
            st = _real_lengths(level, random_state(nf, rng, p_circ=circ, max_contigs=1))
            for _ in range(n):
                a, b = [int(x) for x in rng.choice(nf, 2, replace=False)]
                out.append((st, a, b))
        return out
    while len(out) < n:
        st = _real_lengths(level, random_state(nf, rng, p_circ=0.4, max_contigs=20))
        if not st["circ"].any():
            continue
        a, b = [int(x) for x in rng.choice(nf, 2, replace=False)]
        out.append((st, a, b))
    return out


@pytest.mark.parametrize("d_exp", [2.0, 2.37])
@pytest.mark.parametrize("name", ["medium", "wrap"])
def test_large_level_scores_and_apply_match_oracle(built, name, d_exp):
    """eval_all_sub_likelihood (scores, scored set, n_sub_vals, validity list) and test_copy_struct (whole 13 x NF state)
    against the oracle on random scaffolds with long circular contigs and reversed fragments, through the level's natural
    path (the streaming path, in the reference-faithful mode), the row-per-warp kernel (IG_SCORING_PATH=rows) and its
    whole-row split (IG_FORCE_SPLIT=24,1).
    The wrap level's zero terms count intra pairs with a wrapping int32 (k_precompute / k_finalize) against a wrapped n_pix."""
    level = _level(name)
    _check_level_size(name, level)
    p8 = P8_RIPPE.copy()
    p8[4] = d_exp
    handles = [("stream", make_sampler(level))]
    with _env(IG_SCORING_PATH="rows"):
        handles.append(("rows", make_sampler(level)))
    with _env(IG_SCORING_PATH="rows", IG_FORCE_SPLIT="24,1"):
        handles.append(("rows split 24,1", make_sampler(level)))
    o = OracleSampler(level, p8)
    di = int(d_exp != 2.0)
    rng = np.random.RandomState(100 + di)
    pairs = _score_pairs(name, rng, 2 if name == "wrap" else 12)
    try:
        for _, s in handles:
            s.set_param_simu(p8)
        for it, (st, a, b) in enumerate(pairs):
            st13 = _as13(st)
            valid0 = rng.choice([-1, 1], 12).astype(np.int32)
            o.live = {k: st[k].copy() for k in FIELDS13}
            o.valid = valid0.tolist()
            o.v_cur = sc.fill_vect_dist(o.live, o.sub)
            lnz = sc.full_likelihood_nz(o.v_cur, o.coo, o.params, o.mbar)
            id_host = o.live["id_c"].copy()
            max_id = int(id_host.max())
            want, _, n_sub = o.score_candidate(a, b, max_id, 1, id_host, lnz)
            valid_want = np.array(o.valid, dtype=np.int32)
            nz = want != 0
            tol = 1e-5 * np.abs(want[nz] - want[nz].max()) + 2e-8 * np.abs(want[nz]) + 1e-9
            op = (it * 2 + di) % 24 if name != "wrap" else (it * 5 + 3 * di) % 24
            new, _ = mv.apply_family({k: st[k].copy() for k in FIELDS13}, a, b, op, max_id)
            new, _, _ = mv.renumber_contigs(new)
            for path, s in handles:
                s._set_state(st13)
                s.set_valid_insert(valid0)
                got = s.eval_all_sub_likelihood(a, b, 1)
                where = (path, it, a, b)
                assert np.array_equal(want != 0, got != 0), where
                assert s.n_sub_vals[0] == n_sub, (where, s.n_sub_vals[0], n_sub)
                assert np.all(np.abs(got[nz] - want[nz]) <= tol), (where, float(np.max(np.abs(got[nz] - want[nz]))))
                assert np.array_equal(s.get_valid_insert(), valid_want), where
                s._set_state(st13)
                s.set_valid_insert(valid0)
                s.test_copy_struct(a, b, op)
                got_state = s._get_state()
                for i, k in enumerate(FIELDS13):
                    assert np.array_equal(got_state[i], new[k]), (where, op, k)
        for label, s in handles:
            assert_scoring_path(s, label.split()[0])
    finally:
        for _, s in handles:
            s.free_gpu()


# ------------------------------------------------------------------------------------------------------------------
# C. histogram of the p(s) fit
def _a_separation(level, n_rows):
    """the separation (kb, float64 exactly as the oracle computes it) of an intra-contig contact of one of the first
    n_rows rows"""
    soa, s2f = level.S_o_A_frags, level.np_sub_frags_2_frags
    m = level.sparse_matrix.tocoo()
    parent = s2f["x"].astype(np.int64)
    fi, fj = parent[m.row], parent[m.col]
    ok = (soa["id_c"][fi] == soa["id_c"][fj]) & (m.row != m.col) & (m.row < n_rows)
    d = np.abs((soa["start_bp"][fi] / 1000.0 + s2f["y"][m.row].astype(np.float64))
               - (soa["start_bp"][fj] / 1000.0 + s2f["y"][m.col].astype(np.float64)))[ok]
    return float(np.sort(d)[d.size // 2])


@pytest.mark.parametrize("name", ["T", "Y3", "medium"])
def test_histogram_matches_oracle_exactly(built, name):
    """distance_histogram: per-bin sums and rows_used integer-equal to the oracle's for n_rows = NS/10, NS and NS + 7 (rows
    past the level's last do not exist), the reference's bin width and a dyadic one, max_kb = the longest contig and
    max_kb = the separation of an actual contact (excluded: the test is strict)."""
    level = _level(name)
    s = make_sampler(level)
    try:
        ns = level.n_sub_frags
        id_start = np.nonzero(level.S_o_A_frags["start_bp"] == 0)[0]
        max_ref = level.S_o_A_frags["l_cont_bp"][id_start].max() / 1000.0
        bin_ref = level.S_o_A_sub_frags["len_bp"].mean() / 1000.0 / 2.0
        sep = _a_separation(level, ns // 10)
        for n_rows in (ns // 10, ns, ns + 7):
            for bin_kb in (bin_ref, 0.5):
                for max_kb in (max_ref, sep):
                    bins, hist, used = s.distance_histogram(max_kb, bin_kb, n_rows)
                    obins, omean, oused = distance_histogram(level.sparse_matrix, level.S_o_A_frags,
                                                             level.np_sub_frags_2_frags, n_rows, max_kb, bin_kb)
                    where = (n_rows, bin_kb, max_kb)
                    assert used == oused and len(bins) == len(obins), where
                    assert np.array_equal(hist, np.round(omean * oused).astype(np.int64)), where
                    assert hist.sum() > 0, where
    finally:
        s.free_gpu()
