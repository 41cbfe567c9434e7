"""ORACLE (test infrastructure only -- never imported by the product path).

NumPy restatement of the reference ``sampler`` orchestration for the hot path
(/root/reference/src/instagraal/cuda_lib_gl_single.py, CL): step_sampler CL:1401-1465,
modify_gl_cuda_buffer CL:2715-2881, dist_inter_genome CL:665-716, return_neighbours CL:3103-3141,
setup_distri_frags CL:3053-3101, step_nuisance_parameters CL:2961-3051,
estimate_parameters_rippe (histogram part) CL:2239-2318, bomb_the_genome CL:1925-1948.
Kernels are the restatements in oracle/moves.py and oracle/score.py.

Host RNG contract (SURVEY F.3): this class makes the SAME ``np.random`` calls in the same order
as the reference, so seeding ``np.random.seed(k)`` before a run reproduces its draws.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from . import moves as mv
from . import score as sc


def upper_coo(sparse_matrix):
    """sparse_data_2_gpu CL:551-609: (M + M^T), strict upper triangle, canonical row-major COO."""
    sym = (sparse_matrix + sparse_matrix.transpose()).tocsr()
    sym.sort_indices()
    coo = sp.triu(sym.tocoo(), k=1, format="coo")
    o = np.lexsort((coo.col, coo.row))
    return (coo.row[o].astype(np.int32), coo.col[o].astype(np.int32), coo.data[o].astype(np.int32))


def setup_distri_frags(sub_sampled_sparse_matrix, n_frags):
    """CL:3053-3101."""
    sym = (sub_sampled_sparse_matrix + sub_sampled_sparse_matrix.T).tocsr()
    out = {}
    for i in range(n_frags):
        st, en = sym.indptr[i], sym.indptr[i + 1]
        vk, yk = sym.data[st:en], sym.indices[st:en]
        het = np.nonzero(yk != i)[0]
        xk = np.copy(yk)[het]
        dat = np.float32(np.copy(vk)[het]) * 3.0
        if dat.sum() > 0:
            pk = dat / np.linalg.norm(dat, 1)
        else:
            tmp = np.ones_like(dat, dtype=np.float32)
            pk = tmp / tmp.sum()
        out[i] = (xk, pk) if len(xk) > 0 else None
    return out


def return_neighbours(distri, n_frags, id_fa, delta):
    """CL:3103-3141 (repeat/blacklist machinery inert)."""
    d = distri[id_fa]
    if d is not None:
        xk, pk = d
        n_max = min(delta, np.nonzero(pk != 0)[0].shape[0])
        init_id = np.random.choice(xk, n_max, p=pk, replace=False)
    else:
        init_id = np.random.choice(n_frags, delta, replace=False)
    return [np.int32(x) for x in init_id]


def dist_inter_genome(live, init_prev, init_next, orientable):
    """CL:665-716 (blacklist empty, init_ori == +1)."""
    n = len(init_prev)
    d = 3.0 * n
    p1, n1, o1 = live["prev"], live["next"], live["ori"]
    for f in range(n):
        p0, n0 = init_prev[f], init_next[f]
        pt, nt = p1[f], n1[f]
        swap = 1
        if (pt == p0 and nt == n0) or (pt == n0 and nt == p0):
            d -= 1
        if orientable[f]:
            if 1 != o1[f]:
                pt, nt = nt, pt
                swap = -1
            if p0 == pt:
                if p0 == -1 or not orientable[pt]:
                    d -= 1
                else:
                    d -= 0.5
                    if 1 == swap * o1[pt]:
                        d -= 0.5
            if n0 == nt:
                if n0 == -1 or not orientable[nt]:
                    d -= 1
                else:
                    d -= 0.5
                    if 1 == swap * o1[nt]:
                        d -= 0.5
        else:
            if pt == p0 or pt == n0:
                d -= 1
            if nt == n0 or nt == p0:
                d -= 1
    return d / (3.0 * n)


def distance_histogram(sparse_matrix, soa, s2f, n_rows, max_dist_kb, size_bin_kb):
    """Histogram part of estimate_parameters_rippe CL:2247-2297: for the first ``n_rows`` rows of the
    SYMMETRIC level L-1 matrix, per-row contact sums per distance bin (intra-contig only), then the
    mean over rows.  Returns (bins, mean_contacts float64, n_rows_used).  Rows past the level's last do not exist: n_rows
    is clamped to the number of sub-fragments."""
    sym = (sparse_matrix + sparse_matrix.transpose()).tocsr()
    n_rows = min(int(n_rows), sym.shape[0])
    bins = np.arange(size_bin_kb, max_dist_kb + size_bin_kb, size_bin_kb)
    acc = np.zeros(len(bins), dtype=np.int64)
    used = 0
    parent = s2f["x"].astype(np.int64)
    for i in range(n_rows):
        fi = parent[i]
        len_kb_c_i = soa["l_cont_bp"][fi] / 1000
        if not (size_bin_kb < len_kb_c_i):
            continue
        used += 1
        st, en = sym.indptr[i], sym.indptr[i + 1]
        jj, dd = sym.indices[st:en], sym.data[st:en]
        s_i = soa["start_bp"][fi] / 1000.0 + s2f[i][1]
        fj = parent[jj]
        ok = soa["id_c"][fj] == soa["id_c"][fi]
        s_j = soa["start_bp"][fj] / 1000.0 + s2f["y"][jj]
        dist = np.abs(s_i - s_j)
        ok &= dist < max_dist_kb
        idb = (dist[ok] / size_bin_kb).astype(np.int64)
        np.add.at(acc, idb, dd[ok].astype(np.int64))
    mean = acc / max(used, 1)
    return bins, mean, used


class OracleSampler:
    def __init__(self, level, params8=None, compat_int32_wrap=True):
        self.level = level
        self.nf = level.n_frags
        self.ns = level.n_sub_frags
        self.coo = upper_coo(level.sparse_matrix)
        self.sub = sc.sub_tables(level.np_sub_frags_2_frags)
        self.live = mv.state_from_soa(level.S_o_A_frags)
        self.init_prev = np.copy(level.S_o_A_frags["prev"])
        self.init_next = np.copy(level.S_o_A_frags["next"])
        self.orientable = (level.np_sub_frags_id["w"] > 1).astype(np.int32)
        self.mbar = np.float32(level.S_o_A_sub_frags["len_bp"].mean() / 1000.0)
        with np.errstate(over="ignore"):
            ns32 = np.int32(self.ns)
            self.n_pix = float(ns32 * (ns32 - np.int32(1)) / 2) if compat_int32_wrap else self.ns * (self.ns - 1) / 2
        self.max_bounds_insert = int(50 * np.int32(np.round(level.S_o_A_frags["sub_len"].mean()) + 1))
        self.valid = [0] * 12  # ga.zeros at construction: "all valid" until the first get_bounds
        self.distri = setup_distri_frags(level.sub_sampled_sparse_matrix, self.nf)
        self.params = None if params8 is None else sc.Params(params8)
        self.params8 = None if params8 is None else np.asarray(params8, dtype=np.float32).copy()
        self.likelihood_t = None
        self.v_cur = None
        self.n_contigs = None
        self.mean_length_contigs = None

    # -- contig bookkeeping
    def _renumber(self):
        self.live, nc, lens = mv.renumber_contigs(self.live)
        self.n_contigs = np.int32(nc)
        self.mean_length_contigs = np.float32(lens).mean()
        return nc - 1

    def bomb_the_genome(self):
        a = np.arange(0, self.nf, dtype=np.int32)
        np.random.shuffle(a)
        self.live = mv.explode_genome(self.live, a)
        self._renumber()
        return a

    # -- scoring of one candidate pair (also the unit the C-ABI ig_eval_scores exposes)
    def score_candidate(self, a, b, max_id, flip_eject, id_c_host, lnz_full):
        p, mbar = self.params, self.mbar
        uniq = mv.extract_uniq_mutations(self.live, a, b, self.valid, flip_eject)
        muts, self.valid = mv.perform_mutations(self.live, a, b, max_id)
        w = sc.slice_windows(self.live, a, b, self.max_bounds_insert)
        mask = sc.slice_mask(self.v_cur, self.coo, int(id_c_host[a]), int(id_c_host[b]), w)
        sub = tuple(x[mask] for x in self.coo)
        lsub_cur = float(np.sum(sc.contact_terms(self.v_cur, *sub, p, mbar, len_from="col")))
        vm = {m: sc.fill_vect_dist(muts[m], self.sub) for m in uniq}
        lz = {m: sc.zeros_term(vm[m], p, mbar, self.n_pix) for m in uniq}
        lsub = sc.sub_likelihoods(vm, uniq, sub, p, mbar)
        scores = np.zeros(24, dtype=np.float64)
        for m in uniq:
            scores[m] = lsub[m] + lz[m] + lnz_full - lsub_cur
        return scores, uniq, int(mask.sum())

    def step_sampler(self, id_frag, n_neighbours=5, candidates=None):
        if candidates is None:
            candidates = return_neighbours(self.distri, self.nf, id_frag, n_neighbours)
        candidates = sorted(c for c in candidates if int(c) != int(id_frag))  # B == A dropped (DESIGN.md, D1)
        self.candidates = candidates
        self.v_cur = sc.fill_vect_dist(self.live, self.sub)
        lnz_full = sc.full_likelihood_nz(self.v_cur, self.coo, self.params, self.mbar)
        id_c_host = self.live["id_c"].copy()
        max_id = self._renumber()
        n = len(candidates)
        all_scores = np.zeros(24 * n, dtype=np.float64)
        self.n_uniq_list = []
        for k, b in enumerate(candidates):
            s24, uniq, _ = self.score_candidate(id_frag, int(b), max_id, 1 if k == 0 else 0, id_c_host, lnz_full)
            all_scores[24 * k:24 * (k + 1)] = s24
            self.n_uniq_list.append(len(uniq))
        self.all_scores = all_scores
        ok = np.copy(all_scores)
        ok[ok == 0] = -np.inf
        filt = ok - (ok.max() - 30)
        filt[filt < 0] = 0
        gid = int(np.argmax(filt))
        id_f_sampled = candidates[gid // 24]
        op = gid % 24
        self.live, valid = mv.apply_family(self.live, id_frag, int(id_f_sampled), op, max_id)
        if valid is not None:
            self.valid = valid
        self._renumber()
        o = all_scores[gid]
        dist = dist_inter_genome(self.live, self.init_prev, self.init_next, self.orientable)
        self.likelihood_t = o
        return (o, dist, op, id_f_sampled, self.mean_length_contigs, self.n_contigs)

    # -- nuisance parameters
    def eval_likelihood_4_nuisance(self, p8_test):
        """CL:1296-1344 + 762-801 on the coordinates of the LAST fill_dist_single (quirk Q5)."""
        p = sc.Params(p8_test)
        z, n_intra = sc.zeros_term_raw(self.v_cur, p, self.mbar)
        log_e = 0.43429448190325182
        on_z = z * log_e + log_e * (np.float64(self.n_pix) - n_intra) * -1.0 * np.float32(p8_test[7])
        return sc.full_likelihood_nz(self.v_cur, self.coo, p, self.mbar) + on_z
