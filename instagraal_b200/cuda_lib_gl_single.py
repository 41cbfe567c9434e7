"""Drop-in replacement for the reference module ``instagraal/cuda_lib_gl_single.py`` ("CL"):
the ``sampler`` class with the same constructor arguments, method names, return tuples and public
attributes, implemented over the C ABI of ``libinstagraal_b200.so`` through ctypes.

Mirrors (reference file:line):
  sampler.__init__            CL:92-319    -> ig_create (+ host-side neighbour pmfs, CL:3053-3101)
  step_sampler                CL:1401-1465 -> ig_step_wide
  step_nuisance_parameters    CL:2961-3051 -> ig_full_likelihood (+ host RNG / fsolve as in the reference);
                              production RNG mode: run_cycle_device(nuisance=True) -> ig_set_device_nuisance (on the device)
  bomb_the_genome             CL:1925-1948 -> ig_bomb
  estimate_parameters_rippe   CL:2239-2372 -> ig_distance_histogram (+ scipy fit as in the reference)
  eval_likelihood / eval_all_sub_likelihood / test_copy_struct (step / eval / apply entry points)
  gpu_vect_frags.copy_from_gpu  gpustruct.py:157-186 -> ig_get_state
  free_gpu                    CL:3167-3177 -> ig_destroy

Host RNG contract: every ``np.random`` call of the reference is made here, in the same order
(shuffle in bomb_the_genome; choice in return_neighbours; choice(4)/normal/rand in
step_nuisance_parameters), so a seeded legacy NumPy stream reproduces the reference's draws.
No PyTorch, pycuda, OpenGL or CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from . import host_rng
try:   # inside the reference's tree: its own host-side p(s) fitting module (scipy leastsq / fsolve), untouched
    from instagraal import optim_rippe_curve_update as opti
except ImportError:   # stand-alone: the restatement of the same functions
    from . import rippe_fit as opti

FIELDS13 = L.FIELDS13
ALL17 = ("pos", "sub_pos", "id_c", "start_bp", "len_bp", "sub_len", "circ", "id", "prev", "next",
         "l_cont", "sub_l_cont", "l_cont_bp", "ori", "rep", "activ", "id_d")

PARAM_SIMU_RIPPE = np.dtype([("kuhn", np.float32), ("lm", np.float32), ("c1", np.float32), ("slope", np.float32),
                             ("d", np.float32), ("d_max", np.float32), ("fact", np.float32), ("v_inter", np.float32)],
                            align=True)  # CL:235-247
# run_cycle_device(nuisance=True): the device record of every nuisance step, followed by the tuple step_nuisance_parameters
# returns (IG:252; the list_* feeds of IG:291-330): the live parameters after the step, likelihood_t and success
NUIS_STEP_DTYPE = np.dtype(L.NUIS_DTYPE[:-1] + [("fact", np.float32), ("d", np.float32), ("d_max", np.float32),
                                                ("d_nuc", np.float32), ("slope", np.float32), ("likelihood_t", np.float64),
                                                ("success", np.int32)])


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class _VectFrags:
    """Stand-in for the reference's GPUStruct (gpustruct.py): the 17 arrays as NumPy attributes,
    refreshed by copy_from_gpu()."""

    def __init__(self, owner, soa):
        self._owner = owner
        n = owner.n_new_frags
        for k in ALL17:
            if k == "ori":
                setattr(self, k, np.ones(n, dtype=np.int32))
            elif k in soa:
                setattr(self, k, np.array(soa[k], dtype=np.int32))
        self.__next__ = self.next  # the reference (2to3 artefact) reads both spellings

    def copy_from_gpu(self, skip=None):
        st = self._owner._get_state()
        for i, k in enumerate(FIELDS13):
            setattr(self, k, st[i].copy())
        self.__next__ = self.next
        self.id = np.arange(self._owner.n_new_frags, dtype=np.int32)

    def copy_to_gpu(self, skip=None):
        st = np.ascontiguousarray(np.stack([np.asarray(getattr(self, k), dtype=np.int32) for k in FIELDS13]))
        self._owner._set_state(st)

    def __del__(self):
        pass


class sampler:
    def __init__(self, use_rippe, S_o_A_frags, collector_id_repeats, frag_dispatcher, id_frag_duplicated,
                 id_frags_blacklisted, n_frags, n_new_frags, init_n_sub_frags, n_new_sub_frags, np_rep_sub_frags_id,
                 sub_sampled_sparse_matrix, np_sub_frags_len_bp, np_sub_frags_id, np_sub_frags_accu,
                 np_sub_frags_2_frags, mean_squared_frags_per_bin, norm_vect_accu, sub_candidates_dup,
                 sub_candidates_output_data, S_o_A_sub_frags, sub_collector_id_repeats, sub_frag_dispatcher,
                 sparse_matrix, mean_value_trans, n_iterations, is_simu, vel, pos, device=0,
                 compat_last_block=True, compat_int32_wrap=True, rigid_pruning=False):
        if not use_rippe:
            raise NotImplementedError("only the Rippe p(s) model is on the live path (IG:564 use_rippe=True)")
        if len(id_frag_duplicated) or len(sub_candidates_dup) or len(id_frags_blacklisted):
            raise NotImplementedError("repeat / blacklist machinery is inert in the reference (SS:513) and not supported")
        self._h = None
        self.o = 0
        self.log_e = 0.43429448190325182
        self.use_rippe = use_rippe
        self.n_frags = np.int32(n_frags)
        self.n_new_frags = np.int32(n_new_frags)
        self.init_n_sub_frags = np.int32(init_n_sub_frags)
        self.n_new_sub_frags = np.int32(n_new_sub_frags)
        self.S_o_A_frags = S_o_A_frags
        self.S_o_A_sub_frags = S_o_A_sub_frags
        self.np_sub_frags_2_frags = np_sub_frags_2_frags
        self.np_sub_frags_id = np_sub_frags_id
        self.np_sub_frags_len_bp = np_sub_frags_len_bp
        self.np_sub_frags_accu = np_sub_frags_accu
        self.sub_sampled_sparse_matrix = sub_sampled_sparse_matrix
        self.id_frags_blacklisted = id_frags_blacklisted
        self.id_frag_duplicated = id_frag_duplicated
        self.frag_dispatcher = frag_dispatcher
        self.collector_id_repeats = collector_id_repeats
        self.n_iterations = n_iterations
        self.is_simu = is_simu
        self.mean_value_trans = mean_value_trans
        self.n_insert_blocks = 6
        self.n_tmp_struct = 12 + self.n_insert_blocks * 2
        self.dt = np.float32(0.01)
        self.mean_len_bp_frags = self.S_o_A_sub_frags["len_bp"].mean()  # CL:231
        self.sparse_matrix = (sparse_matrix + sparse_matrix.transpose()).tocsr()  # CL:129
        self.sparse_matrix.sort_indices()

        nf, ns = int(n_new_frags), int(init_n_sub_frags)
        # ---- contacts: strict upper triangle of the symmetrised level L-1 matrix (CL:592-609) as CSR
        import scipy.sparse as sp
        up = sp.triu(self.sparse_matrix, k=1, format="csr")
        up.sort_indices()
        self._row_ptr = np.ascontiguousarray(up.indptr, dtype=np.int64)
        self._col = np.ascontiguousarray(up.indices, dtype=np.int32)
        self._val = np.ascontiguousarray(up.data, dtype=np.int32)
        self.n_non_zero = int(self._val.shape[0])
        self._sym_diag = np.ascontiguousarray(self.sparse_matrix.diagonal(), dtype=np.int32)
        # ---- scaffold (CL:521-549: ori starts at +1)
        st = np.zeros((13, nf), dtype=np.int32)
        for i, k in enumerate(FIELDS13):
            st[i] = 1 if k == "ori" else np.asarray(S_o_A_frags[k], dtype=np.int32)
        self._state0 = np.ascontiguousarray(st)
        s2f = np_sub_frags_2_frags
        self._sub_parent = np.ascontiguousarray(s2f["x"].astype(np.int32))
        self._sub_watson = np.ascontiguousarray(s2f["y"], dtype=np.float32)
        self._sub_crick = np.ascontiguousarray(s2f["z"], dtype=np.float32)
        self._sub_j = np.ascontiguousarray(s2f["w"].astype(np.int32))
        self.np_init_prev = np.copy(S_o_A_frags["prev"]).astype(np.int32)
        self.np_init_next = np.copy(S_o_A_frags["next"]).astype(np.int32)
        id_d = np.asarray(S_o_A_frags["id_d"])
        self.np_init_orientable = np.ascontiguousarray((np_sub_frags_id["w"][id_d] > 1).astype(np.int32))  # CL:271-275
        self.np_init_ori = np.ones((nf,), dtype=np.int32)
        # ---- scalars
        with np.errstate(over="ignore"):
            if compat_int32_wrap:  # quirk Q8: np.int32 scalar arithmetic (CL:366)
                self.n_pixl_sub_mat = self.init_n_sub_frags * (self.init_n_sub_frags - np.int32(1)) / 2
            else:
                self.n_pixl_sub_mat = np.float64(ns) * (ns - 1) / 2
        list_size = np.array([1, 3, 5, 10, 20, 50, 200, 200], dtype=np.int32)
        self.max_bounds_insert = list_size[:self.n_insert_blocks].max() * np.int32(
            np.round(self.S_o_A_frags["sub_len"].mean()) + 1)  # CL:417-420
        self._mbar = np.float32(self.mean_len_bp_frags / 1000.0)

        cfg = L.ig_config(device=int(device), n_frags=nf, n_sub_frags=ns, nnz=self.n_non_zero,
                          max_bounds_insert=int(self.max_bounds_insert), mean_sub_len_kb=float(self._mbar),
                          n_pix=float(self.n_pixl_sub_mat), compat_last_block=int(bool(compat_last_block)), rigid_pruning=int(bool(rigid_pruning)))
        data = L.ig_level_data(
            frags13=_ptr(self._state0), sub_parent=_ptr(self._sub_parent), sub_watson=_ptr(self._sub_watson),
            sub_crick=_ptr(self._sub_crick), sub_j=_ptr(self._sub_j), row_ptr=_ptr(self._row_ptr), col=_ptr(self._col),
            val=_ptr(self._val), init_prev=_ptr(self.np_init_prev), init_next=_ptr(self.np_init_next),
            orientable=_ptr(self.np_init_orientable))
        h = C.c_void_p()
        rc = L.lib().ig_create(C.byref(cfg), C.byref(data), C.byref(h))
        L.check(None, rc, "ig_create")
        self._h = h
        L.check(self._h, L.lib().ig_set_sym_diag(self._h, _ptr(self._sym_diag)), "ig_set_sym_diag")

        self.gpu_vect_frags = _VectFrags(self, S_o_A_frags)
        self.param_simu = None
        self.param_simu_test = None
        self.likelihood_t = None
        self.candidates = []
        self.all_scores = np.zeros(0)
        self.n_contigs = None
        self.mean_length_contigs = None
        self.n_proposals_scored = 0
        self._last_dist = 1.0
        # step_nuisance_parameters' proposal (host RNG draws + scipy fsolve, ~0.35 ms) is prepared while the GPU scores the
        # step before it, on a private copy of the generator; results and RNG stream are unchanged (see _speculate_nuisance).
        self.overlap_nuisance_proposal = True
        self._nuis_follows = False
        self._spec = None
        self._spec_pool = None
        self._twin = None
        self._twin_synced = False
        self.n_nuis_overlapped = 0
        self._nuis_device = False   # ig_set_device_nuisance state of the handle
        self.chain_temperature = 0.0   # set_chain_temperature (not the reference's temperature(t, n_step))
        self.modification_str = [  # CL:1601-1620
            "eject frag", "flip frag", "pop out split insert @ left or 1", "pop out split insert @ left or -1",
            "pop out split insert @ right or 1", "pop out split insert @ right or -1", "pop out insert @ right or 1",
            "pop out insert @ right or -1", "transloc_1", "transloc_2", "transloc_3", "transloc_4",
            "local_scramble d1", "local_scramble d2", "local_scramble d3", "local_scramble d4"]
        self.setup_distri_frags()
        self._nb_state = {}   # shared (by reference) with the clones of this chain: neighbour weights uploaded once per level
        self._bind_step_buffers()

    def _bind_step_buffers(self):
        """this chain's host buffers of ig_step_wide (a result record, candidates, scores, n_uniq, n_sub of up to
        IG_MAX_NEIGHBOURS candidates), bound once with the ctypes function: no per-step ctypes conversions"""
        self._res = L.ig_step_result()
        self._cand_buf = np.zeros(L.IG_MAX_NEIGHBOURS, dtype=np.int32)
        self._scores_buf = np.zeros(L.IG_MAX_NEIGHBOURS * L.IG_N_OPS, dtype=np.float64)
        self._nuniq_buf = np.zeros(L.IG_MAX_NEIGHBOURS, dtype=np.int32)
        self._nsub_buf = np.zeros(L.IG_MAX_NEIGHBOURS, dtype=np.int32)
        self._step_args = (_ptr(self._cand_buf), C.byref(self._res), _ptr(self._scores_buf), _ptr(self._nuniq_buf),
                           _ptr(self._nsub_buf))
        self._ig_step_wide = L.lib().ig_step_wide

    @classmethod
    def clone_of(cls, other):
        """A further chain on the same level and GPU (ig_clone): shares the contacts / sub-fragment table / neighbour
        weights of ``other`` in device memory; own scaffold (starting from the level's initial one), own RNG-free state.
        Parameters are copied from ``other``."""
        import copy
        s = copy.copy(other)   # host-side attributes (level arrays, neighbour pmfs) are shared read-only
        h = C.c_void_p()
        L.check(other._h, L.lib().ig_clone(other._h, C.byref(h)), "ig_clone")
        s._h = h
        s.gpu_vect_frags = _VectFrags(s, other.S_o_A_frags)
        s.candidates = []
        s.all_scores = np.zeros(0)
        s.n_proposals_scored = 0
        s.likelihood_t = None
        s._nuis_follows, s._spec, s._spec_pool, s._twin, s._twin_synced = False, None, None, None, False
        s._nuis_device = False
        s.chain_temperature = 0.0   # a new handle starts at T = 0
        s._bind_step_buffers()
        if other.param_simu is not None:
            s.set_param_simu(np.array(list(other.param_simu[0]), dtype=np.float32))
            s.param_simu_test = s.param_simu
        return s

    # ------------------------------------------------------------------ state plumbing
    def _get_state(self):
        out = np.zeros((13, int(self.n_new_frags)), dtype=np.int32)
        L.check(self._h, L.lib().ig_get_state(self._h, _ptr(out)), "ig_get_state")
        return out

    def _set_state(self, st13):
        st13 = np.ascontiguousarray(st13, dtype=np.int32)
        L.check(self._h, L.lib().ig_set_state(self._h, _ptr(st13)), "ig_set_state")

    def get_valid_insert(self):
        out = np.zeros(12, dtype=np.int32)
        L.check(self._h, L.lib().ig_get_valid_insert(self._h, _ptr(out)), "ig_get_valid_insert")
        return out

    def set_valid_insert(self, v):
        v = np.ascontiguousarray(v, dtype=np.int32)
        L.check(self._h, L.lib().ig_set_valid_insert(self._h, _ptr(v)), "ig_set_valid_insert")

    def set_param_simu(self, p8):
        """memcpy_htod(gpu_param_simu, param_simu) (CL:2348, 3033)."""
        p = np.ascontiguousarray(np.asarray(p8, dtype=np.float32).ravel())
        L.check(self._h, L.lib().ig_set_params(self._h, _ptr(p)), "ig_set_params")
        self.param_simu = np.array([tuple(p.tolist())], dtype=PARAM_SIMU_RIPPE)

    def device_state(self):
        """(device pointer, n_bytes) of the live scaffold records (64 B per fragment) for replica exchange."""
        ptr, n = C.c_void_p(), C.c_int64(0)
        L.check(self._h, L.lib().ig_device_state_ptr(self._h, C.byref(ptr), C.byref(n)), "ig_device_state_ptr")
        return int(ptr.value), int(n.value)

    def set_profiling(self, on):
        L.check(self._h, L.lib().ig_set_profiling(self._h, int(bool(on))), "ig_set_profiling")

    KERNEL_ORDER = ("k_cand_setup", "k_find_cuts", "k_rows_count", "k_rows_write", "k_precompute", "k_score",
                    "k_finalize", "k_select_step", "k_lnz_outside", "k_apply", "k_post")

    def get_kernel_times(self, reset=False):
        out = np.zeros(11, dtype=np.float64)
        L.check(self._h, L.lib().ig_get_kernel_times(self._h, _ptr(out), int(bool(reset))), "ig_get_kernel_times")
        return dict(zip(self.KERNEL_ORDER, out.tolist()))

    def set_options(self, refresh_every=4096, use_graph=True):
        """refresh_every=1 reproduces the reference's schedule (full likelihood over every contact each
        step); larger values maintain it incrementally between full refreshes (same values up to f64
        summation order)."""
        L.check(self._h, L.lib().ig_set_options(self._h, int(refresh_every), int(bool(use_graph))), "ig_set_options")

    def set_gpu_share(self, share):
        """this chain's scoring grids use 1/share of the GPU (several chains per GPU, see ReplicaSet)"""
        L.check(self._h, L.lib().ig_set_gpu_share(self._h, int(share)), "ig_set_gpu_share")

    def get_stats(self, reset=False):
        out = np.zeros(10, dtype=np.float64)
        L.check(self._h, L.lib().ig_get_stats(self._h, _ptr(out), int(bool(reset))), "ig_get_stats")
        keys = ("ms_step", "ms_score", "ms_full", "launches", "steps", "contacts_read", "rows", "frags",
                "contacts_selected", "proposals")
        d = dict(zip(keys, out.tolist()))
        nf = C.c_int64(0)
        L.lib().ig_get_full_refresh_count(self._h, C.byref(nf))
        d["full_refreshes"] = int(nf.value)
        return d

    # ------------------------------------------------------------------ checkpoint / resume (SURVEY 8f, N3)
    def save_checkpoint(self, path):
        """Everything an MCMC run needs to continue bit-identically: the 13 live scaffold arrays, the
        carried list_valid_insert (quirk Q3), the parameters, likelihood_t and the host RNG state.  The
        reference cannot resume a run (SURVEY section 5).  Saving re-synchronises the incremental
        likelihood state (one full refresh on the next step) so that the continued and the resumed run
        perform identical arithmetic.  The chain temperature (set_chain_temperature) is a run setting like the seed and is
        not saved."""
        st = self._get_state()
        valid = self.get_valid_insert()
        self._set_state(st)
        self.set_valid_insert(valid)
        rs = np.random.get_state()
        np.savez(path, state13=st, valid=valid,
                 params8=np.array(list(self.param_simu[0]), dtype=np.float32) if self.param_simu is not None else np.zeros(0, np.float32),
                 likelihood_t=np.float64(self.likelihood_t if self.likelihood_t is not None else np.nan),
                 mean_value_trans=np.float64(self.mean_value_trans), n_proposals_scored=np.int64(self.n_proposals_scored),
                 rng_name=np.array(rs[0]), rng_keys=rs[1], rng_pos=np.int64(rs[2]), rng_has_gauss=np.int64(rs[3]),
                 rng_cached=np.float64(rs[4]))

    def load_checkpoint(self, path):
        z = np.load(path if str(path).endswith(".npz") else str(path) + ".npz", allow_pickle=False)
        self._set_state(z["state13"])
        self.set_valid_insert(z["valid"])
        if z["params8"].size == 8:
            self.set_param_simu(z["params8"])
            self.param_simu_test = self.param_simu
        lt = float(z["likelihood_t"])
        self.likelihood_t = None if np.isnan(lt) else np.float64(lt)
        self.mean_value_trans = float(z["mean_value_trans"])
        self.n_proposals_scored = int(z["n_proposals_scored"])
        np.random.set_state((str(z["rng_name"]), z["rng_keys"], int(z["rng_pos"]), int(z["rng_has_gauss"]), float(z["rng_cached"])))
        self.gpu_vect_frags.copy_from_gpu()

    def free_gpu(self):
        if getattr(self, "_spec_pool", None) is not None:
            self._spec_pool.shutdown(wait=True)
            self._spec_pool = None
        if self._h is not None:
            L.lib().ig_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free_gpu()
        except Exception:
            pass

    # ------------------------------------------------------------------ neighbours (host, CL:3053-3141)
    def setup_distri_frags(self):
        self.distri_frags = dict()
        fact = 3.0
        self.sym_sub_sampled_sparse_matrix = (self.sub_sampled_sparse_matrix + self.sub_sampled_sparse_matrix.T).tocsr()
        sym = self.sym_sub_sampled_sparse_matrix
        for i in range(0, int(self.n_frags)):
            start, end = sym.indptr[i], sym.indptr[i + 1]
            vk, yk = sym.data[start:end], sym.indices[start:end]
            het = np.nonzero(yk != i)[0]
            xk = np.copy(yk)[het]
            dat = np.float32(np.copy(vk)[het]) * fact
            if dat.sum() > 0:
                pk = dat / np.linalg.norm(dat, 1)
            else:
                tmp = np.ones_like(dat, dtype=np.float32)
                pk = tmp / tmp.sum()
            if len(xk) > 0:
                p64, cdf0 = host_rng.prepare(pk)
                self.distri_frags[i] = {"distri": "ok", "xk": xk, "pk": pk, "p64": p64, "cdf0": cdf0,
                                        "nnz": int(np.nonzero(pk != 0)[0].shape[0])}
            else:
                self.distri_frags[i] = {"distri": None}

    def return_neighbours(self, id_fA, delta0):
        ori_id = self.gpu_vect_frags.id_d[id_fA]
        delta = delta0
        d = self.distri_frags[ori_id]
        if d["distri"] is not None:
            # = np.random.choice(xk, min(delta, #non-zero pk), p=pk, replace=False) (CL:3113-3122): same values, same
            # generator state afterwards, without NumPy's per-call validation of p (host_rng.py)
            init_id = host_rng.weighted_choice_no_replace(d["xk"], d["p64"], d["cdf0"], min(delta, d["nnz"]))
        else:
            init_id = np.random.choice(self.n_frags, delta, replace=False)
        out = []
        for id_fB in init_id:
            d = self.frag_dispatcher[id_fB]
            out.extend(self.collector_id_repeats[d["x"]:d["y"]])
        return out

    # ------------------------------------------------------------------ the hot path
    def _usable_candidates(self, id_frag, candidates):
        """Sorted candidate list of one step: deviation D1 (B == A dropped, see step_sampler) and the library's limit of
        IG_MAX_NEIGHBOURS candidates per step (the reference has no limit; its CLI default is 5)."""
        cs = sorted(int(c) for c in candidates if int(c) != int(id_frag))
        if len(cs) > L.IG_MAX_NEIGHBOURS:
            raise ValueError("instagraal_b200 scores at most %d candidate neighbours per step (got %d: lower "
                             "--neighborhood / n_neighbours)" % (L.IG_MAX_NEIGHBOURS, len(cs)))
        return cs

    def step_sampler(self, id_frag, n_neighbours, dt, candidates=None):
        """CL:1401-1465.  ``candidates`` (optional) bypasses the host RNG draw (replay / parity)."""
        if candidates is None:
            candidates = self.return_neighbours(id_frag, n_neighbours)
        # Deviation D1 (DESIGN.md): a fragment without level-L neighbours gets a uniform draw over ALL
        # fragments (CL:3124), which can contain the fragment itself; for B == A the reference's
        # paste_contigs writes nothing (quirk Q4) and stale candidate structs get scored and possibly
        # applied.  The draw is made as in the reference (same RNG consumption) but B == A is dropped.
        self.candidates = self._usable_candidates(id_frag, candidates)
        n = len(self.candidates)
        if n == 0:
            # only reachable through D1 (the uniform fallback draw returned nothing but the visited fragment): nothing
            # to score, the scaffold stays as it is and the previous step's outputs are returned with op_sampled = -1
            self.all_scores = np.zeros(0)
            self.n_uniq, self.n_sub_vals = [], []
            return (self.likelihood_t, self._last_dist, -1, int(id_frag), self.mean_length_contigs, self.n_contigs)
        self._cand_buf[:n] = self.candidates
        res = self._res
        fut = None
        if self._nuis_follows and self.param_simu is not None:   # the previous call was a nuisance step: expect the next one
            if self._spec_pool is None:
                from concurrent.futures import ThreadPoolExecutor
                self._spec_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="ig-nuisance")
            fut = self._spec_pool.submit(self._speculate_nuisance)
        self._nuis_follows = False
        cands, res_ref, scores, n_uniq, n_sub = self._step_args
        rc = self._ig_step_wide(self._h, int(id_frag), cands, n, res_ref, scores, n_uniq, n_sub)   # (batches of IG_MAX_CANDS beyond)
        self._spec = fut.result() if fut is not None else None
        if rc != 0:
            L.check(self._h, rc, "ig_step")
        self.all_scores = self._scores_buf[:self.n_tmp_struct * n].copy()
        self.n_uniq = self._nuniq_buf[:n].tolist()
        self.n_sub_vals = self._nsub_buf[:n].tolist()
        self.n_proposals_scored += sum(self.n_uniq)
        self.q4_hits = res.q4_hits
        global_id = np.int64(res.cand_index * self.n_tmp_struct + res.op_sampled)
        id_f_sampled = self.candidates[int(global_id / self.n_tmp_struct)]
        op_sampled = global_id % self.n_tmp_struct
        self.n_contigs = np.int32(res.n_contigs)
        self.mean_length_contigs = np.float32(res.sum_l_cont) / np.float32(res.n_contigs)  # CL:2741-2742
        o = self.all_scores[global_id]
        self.o = o
        self.likelihood_t = o
        self.curr_likelihood_on_nz = res.lnz_full
        self._last_dist = res.dist
        return (o, res.dist, op_sampled, id_f_sampled, self.mean_length_contigs, self.n_contigs)

    def run_cycle(self, list_frags, n_neighbours=5, candidates=None):
        """The inner loop of full_em (IG:217-241) for the fragments in ``list_frags`` as ONE library call:
        candidates are drawn here with the reference's own RNG calls in the reference's order (they do not
        depend on the chain state), the whole run is enqueued on the GPU without host synchronisation, and
        the per-step tuples of step_sampler come back as a structured array
        (likelihood, dist, op_sampled, id_f_sampled, sum_l_cont, n_contigs, n_proposals)."""
        n = len(list_frags)
        frags = np.ascontiguousarray(list_frags, dtype=np.int32)
        lists = []
        for t in range(n):
            cs = candidates[t] if candidates is not None else self.return_neighbours(int(frags[t]), n_neighbours)
            cs = self._usable_candidates(frags[t], cs)  # deviation D1, see step_sampler
            if not cs:
                raise ValueError("run_cycle: step %d (fragment %d) has no candidate but the visited fragment itself; "
                                 "use step_sampler (which skips such a step) or n_neighbours >= 2" % (t, int(frags[t])))
            lists.append(cs)
        # candidate array of IG_MAX_CANDS columns, or as wide as the longest list (ig_run_cycle_wide)
        width = max([L.IG_MAX_CANDS] + [len(cs) for cs in lists])
        c8 = np.zeros((n, width), dtype=np.int32)
        nc = np.zeros(n, dtype=np.int32)
        for t, cs in enumerate(lists):
            nc[t] = len(cs)
            c8[t, :len(cs)] = cs
        out = np.zeros(n, dtype=L.CYCLE_DTYPE)
        assert out.dtype.itemsize == C.sizeof(L.ig_cycle_step)
        L.check(self._h, L.lib().ig_run_cycle_wide(self._h, n, _ptr(frags), _ptr(c8), int(width), _ptr(nc), _ptr(out)), "ig_run_cycle")
        self._after_cycle(out, width)
        if n:
            self.candidates = c8[-1, :nc[-1]].tolist()
        return out

    def neighbour_weights_csr(self):
        """setup_distri_frags (CL:3053-3101) as the CSR ig_set_neighbour_weights takes: (ptr int64[NF+1], idx int32,
        cdf float64 = running sum of pk per fragment, n_nonzero int32[NF])."""
        nf = int(self.n_frags)
        ptr = np.zeros(nf + 1, dtype=np.int64)
        idx, cdf = [], []
        nnz = np.zeros(nf, dtype=np.int32)
        for i in range(nf):
            d = self.distri_frags[i]
            if d["distri"] is not None:
                pk = np.asarray(d["pk"], dtype=np.float64)
                idx.append(np.asarray(d["xk"], dtype=np.int32))
                cdf.append(np.cumsum(pk))
                nnz[i] = int(np.count_nonzero(pk))
                ptr[i + 1] = ptr[i] + len(pk)
            else:
                ptr[i + 1] = ptr[i]
        idx = np.ascontiguousarray(np.concatenate(idx) if idx else np.zeros(0, np.int32), dtype=np.int32)
        cdf = np.ascontiguousarray(np.concatenate(cdf) if cdf else np.zeros(0, np.float64), dtype=np.float64)
        return ptr, idx, cdf, nnz

    def run_cycle_device(self, list_frags, n_neighbours=5, seed=0, cycle=0, nuisance=False):
        """Production RNG mode: like run_cycle, but every step's neighbours are drawn ON THE DEVICE (Philox4x32-10
        keyed by (seed, cycle, step, draw); same distribution as return_neighbours, a different random stream than
        NumPy's).  The host only provides the visiting order (np.random.shuffle in full_em, IG:213).

        nuisance=True: every step is followed by step_nuisance_parameters (full_em from cycle 5 on, IG:242-252), also on
        the device (ig_set_device_nuisance: Philox draws with the same seed, d_max by root finding, DESIGN.md D3).  Returns
        (steps, nuis) with nuis a NUIS_STEP_DTYPE record per step; param_simu, param_simu_test and likelihood_t are left
        where the device left them."""
        self._upload_neighbour_weights()
        self.set_device_nuisance(nuisance)
        n = len(list_frags)
        frags = np.ascontiguousarray(list_frags, dtype=np.int32)
        out = np.zeros(n, dtype=L.CYCLE_DTYPE)
        L.check(self._h, L.lib().ig_run_cycle_device(self._h, n, _ptr(frags), int(n_neighbours), int(seed), int(cycle), _ptr(out)),
                "ig_run_cycle_device")
        self._after_cycle(out, max(L.IG_MAX_CANDS, int(n_neighbours)))
        if not nuisance:
            return out
        return out, self._after_nuisance(n)

    def set_device_nuisance(self, on):
        """ig_set_device_nuisance: run the nuisance step on the device after every step of run_cycle_device (and of
        ReplicaSet.run_cycle)."""
        on = bool(on)
        if on != self._nuis_device:
            L.check(self._h, L.lib().ig_set_device_nuisance(self._h, int(on)), "ig_set_device_nuisance")
            self._nuis_device = on

    def set_chain_temperature(self, T):
        """ig_set_temperature: the temperature T >= 0 at which this chain selects its moves in the production RNG mode
        (run_cycle_device, ReplicaSet.run_cycle).  T = 0 (the default) is the reference's argmax.  At T > 0 a step draws its
        move among the scored proposals with probability exp((s_i - max s) / T) / sum, and the device nuisance step accepts
        when exp((L_nuis - likelihood_t) / T) >= u (DESIGN.md 4e).  step_sampler and run_cycle (the host-RNG,
        reference-parity entry points) refuse to run at T > 0.  Like the seed, the temperature is a run setting: checkpoints
        do not hold it."""
        T = float(T)
        L.check(self._h, L.lib().ig_set_temperature(self._h, C.c_double(T)), "ig_set_temperature")
        self.chain_temperature = T

    def last_tempered_records(self, n_steps):
        """the ig_tempered_step records of the last production-mode cycle run at T > 0 (L.TEMPERED_DTYPE)"""
        rec = np.zeros(int(n_steps), dtype=L.TEMPERED_DTYPE)
        assert rec.dtype.itemsize == 48
        L.check(self._h, L.lib().ig_get_tempered_records(self._h, int(n_steps), _ptr(rec)), "ig_get_tempered_records")
        return rec

    def last_nuisance_records(self, n_steps):
        """the raw ig_nuisance_step records of the last production-mode cycle (L.NUIS_DTYPE)"""
        rec = np.zeros(int(n_steps), dtype=L.NUIS_DTYPE)
        assert rec.dtype.itemsize == 80
        L.check(self._h, L.lib().ig_get_nuisance_records(self._h, int(n_steps), _ptr(rec)), "ig_get_nuisance_records")
        return rec

    def _after_nuisance(self, n_steps):
        """the records of the last cycle's device nuisance steps + the per-step tuple of step_nuisance_parameters; the host
        copies of the parameters follow the device (no upload: the device already holds them)"""
        rec = self.last_nuisance_records(n_steps)
        out = np.zeros(len(rec), dtype=NUIS_STEP_DTYPE)
        for k in rec.dtype.names[:-1]:
            out[k] = rec[k]
        p0 = np.array(list(self.param_simu[0]), dtype=np.float32)
        acc = rec["accepted"] != 0
        last = np.maximum.accumulate(np.where(acc, np.arange(len(rec)), -1))
        live = np.where((last >= 0)[:, None], rec["p_test"][np.maximum(last, 0)], p0[None, :])
        for k, i in (("fact", 6), ("d", 4), ("d_max", 5), ("d_nuc", 7), ("slope", 3)):
            out[k] = live[:, i]
        out["likelihood_t"] = rec["likelihood_t_after"]
        out["success"] = rec["accepted"]
        if len(rec):
            self.param_simu = np.array([tuple(live[-1].tolist())], dtype=PARAM_SIMU_RIPPE)
            self.param_simu_test = np.array([tuple(rec["p_test"][-1].tolist())], dtype=PARAM_SIMU_RIPPE)
            self.likelihood_t = self.o = np.float64(rec["likelihood_t_after"][-1])
        return out

    def _upload_neighbour_weights(self):
        """setup_distri_frags (CL:3053-3101) to the device once per level (shared by the chains cloned from this one)"""
        if not self._nb_state.get("uploaded", False):
            ptr, idx, cdf, nnz = self.neighbour_weights_csr()
            L.check(self._h, L.lib().ig_set_neighbour_weights(self._h, _ptr(ptr), _ptr(idx), _ptr(cdf), _ptr(nnz)),
                    "ig_set_neighbour_weights")
            self._nb_state["uploaded"] = True

    def _after_cycle(self, out, plan_width):
        """the host copies of the last step's outputs after a cycle, and the candidate slots of its plan (last_cycle_plan)"""
        self._plan_width = plan_width
        if len(out):
            last = out[-1]
            self.n_contigs = np.int32(last["n_contigs"])
            self.mean_length_contigs = np.float32(last["sum_l_cont"]) / np.float32(last["n_contigs"])
            self.likelihood_t = self.o = np.float64(last["likelihood"])
            self.n_proposals_scored += int(out["n_proposals"].sum())

    def last_cycle_plan(self, n_steps, width=None):
        """(n_cands, fragment, candidates[width]) per step of the last run_cycle / run_cycle_device call; width defaults to
        that call's (IG_MAX_CANDS, or its number of neighbours / longest candidate list when larger)."""
        width = int(width if width is not None else getattr(self, "_plan_width", L.IG_MAX_CANDS))
        plan = np.zeros((int(n_steps), 2 + width), dtype=np.int32)
        L.check(self._h, L.lib().ig_get_cycle_plan_wide(self._h, int(n_steps), width, _ptr(plan)), "ig_get_cycle_plan")
        return plan

    def eval_likelihood(self):
        """CL:1245-1294: refresh the coordinates and the full non-zero likelihood of the live scaffold."""
        out = np.zeros(3, dtype=np.float64)
        p = np.ascontiguousarray(np.array(list(self.param_simu[0]), dtype=np.float32))
        L.check(self._h, L.lib().ig_full_likelihood(self._h, _ptr(p), 0, _ptr(out)), "ig_full_likelihood")
        self.curr_likelihood_on_nz = out[0]
        return out[0]

    def eval_all_sub_likelihood(self, id_fA, id_fB, flip_eject=1):
        """eval entry point: score the <=24 mutations of one (A,B) pair without applying
        (CL:1417-1431 for a single candidate).  Returns float64[24], 0.0 = not evaluated."""
        out = np.zeros(24, dtype=np.float64)
        nu, nsub = C.c_int32(0), C.c_int32(0)
        L.check(self._h, L.lib().ig_eval_scores(self._h, int(id_fA), int(id_fB), int(flip_eject), _ptr(out),
                                               C.byref(nu), C.byref(nsub)), "ig_eval_scores")
        self.n_sub_vals = [int(nsub.value)]
        return out

    def test_copy_struct(self, id_fA, id_f_sampled, mode, max_id=None):
        """apply entry point (CL:2094-2151) followed by the contig bookkeeping of CL:1453."""
        res = L.ig_step_result()
        L.check(self._h, L.lib().ig_apply(self._h, int(id_fA), int(id_f_sampled), int(mode), C.byref(res)), "ig_apply")
        self.n_contigs = np.int32(res.n_contigs)
        self.mean_length_contigs = np.float32(res.sum_l_cont) / np.float32(res.n_contigs)
        return res.dist

    def modify_gl_cuda_buffer(self, id_fi, dt):
        """CL:2715-2881: contig ids are canonical whenever they are read back, so this only refreshes
        n_contigs / mean_length_contigs and returns max_id."""
        st = self._get_state()
        heads = st[0] == 0
        self.n_contigs = np.int32(heads.sum())
        self.mean_length_contigs = np.float32(st[9][heads]).mean()
        return np.int32(self.n_contigs - 1)

    def bomb_the_genome(self):
        a = np.arange(0, self.n_new_frags, dtype=np.int32)
        np.random.shuffle(a)
        L.check(self._h, L.lib().ig_bomb(self._h, _ptr(a)), "ig_bomb")
        self.modify_gl_cuda_buffer(0, self.dt)

    # ------------------------------------------------------------------ p(s) model
    def setup_rippe_parameters(self, param, d_max):
        """CL:2206-2221."""
        kuhn, lm, slope, d, fact = param
        fact = np.float32(np.abs(fact))
        kuhn = np.float32(np.abs(kuhn))
        lm = np.float32(np.abs(lm))
        c1 = np.float32((0.53 * np.power(lm / kuhn, slope)) * np.power(kuhn, -3))
        return np.array([(kuhn, lm, c1, np.float32(slope), np.float32(d), np.float32(d_max), np.float32(fact),
                          self.mean_value_trans)], dtype=PARAM_SIMU_RIPPE)

    def distance_histogram(self, max_dist_kb, size_bin_kb, n_rows):
        bins = np.arange(size_bin_kb, max_dist_kb + size_bin_kb, size_bin_kb)
        hist = np.zeros(len(bins), dtype=np.int64)
        used = C.c_int64(0)
        L.check(self._h, L.lib().ig_distance_histogram(self._h, float(size_bin_kb), float(max_dist_kb), int(n_rows),
                                                      len(bins), _ptr(hist), C.byref(used)), "ig_distance_histogram")
        return bins, hist, int(used.value)

    def estimate_parameters_rippe(self, max_dist_kb, size_bin_kb, display_graph):
        """CL:2239-2372 with the Python double loop over contacts (CL:2253-2293) replaced by a GPU histogram."""
        self.bins, hist, used = self.distance_histogram(max_dist_kb, size_bin_kb, int(self.n_frags) // 10)
        epsi = self.mean_value_trans
        with np.errstate(invalid="ignore", divide="ignore"):
            means = hist / np.float64(used) if used > 0 else np.full(len(hist), np.nan)
        self.mean_contacts = np.zeros_like(self.bins, dtype=np.float32)
        for id_bin in range(len(self.bins)):
            tmp = means[id_bin]
            self.mean_contacts[id_bin] = np.nan if (np.isnan(tmp) or tmp == 0) else tmp + epsi
        keep = ~np.isnan(self.mean_contacts)
        self.bins_upd = np.array(self.bins)[keep]
        self.mean_contacts_upd = np.array(self.mean_contacts[keep])
        p, self.y_estim = opti.estimate_param_rippe(self.mean_contacts_upd, self.bins_upd)
        self.mean_value_trans = self.mean_value_trans / 10.0  # "BEWARE" CL:2337-2338 (quirk Q12)
        estim_max_dist = opti.estimate_max_dist_intra(p, self.mean_value_trans)
        self.param_simu = self.setup_rippe_parameters(p, estim_max_dist)
        self.param_simu_test = self.param_simu
        self.set_param_simu(np.array(list(self.param_simu[0]), dtype=np.float32))
        self.eval_likelihood()

    def eval_likelihood_4_nuisance(self):
        """CL:1296-1344 + 762-801, on the coordinates of the last fill_dist_single (quirk Q5)."""
        out = np.zeros(3, dtype=np.float64)
        p = np.ascontiguousarray(np.array(list(self.param_simu_test[0]), dtype=np.float32))
        L.check(self._h, L.lib().ig_full_likelihood(self._h, _ptr(p), 1, _ptr(out)), "ig_full_likelihood")
        self.val_on_zero_intra_nuis = out[1] * self.log_e
        self.n_vals_intra = np.int32(out[2])
        self.val_on_zero_inter_nuis = (self.log_e * (np.float64(self.n_pixl_sub_mat) - self.n_vals_intra) * -1.0
                                       * self.param_simu_test["v_inter"][0])
        self.curr_likelihood_on_z_nuis = self.val_on_zero_intra_nuis + self.val_on_zero_inter_nuis
        self.curr_likelihood_nuis = out[0] + self.curr_likelihood_on_z_nuis
        return self.curr_likelihood_nuis

    def temperature(self, t, n_step):
        return 1.0

    def _nuisance_draws(self, rng):
        """The random part of a nuisance proposal (CL:2961-3032): which of the four parameters moves (``choice(4)``) and by how
        much (one ``normal`` draw).  ``rng`` = the ``np.random`` module (the reference's global stream) or a RandomState."""
        kuhn, lm, c1, slope, d, d_max, fact, d_nuc = self.param_simu[0]
        self.sigma_fact = 10 ** (np.log10(fact) - 2)
        self.sigma_slope = 0.005
        self.sigma_d_max = 100
        self.sigma_d_nuc = 10 ** (np.log10(d_nuc) - 2)
        self.sigma_d = 10
        id_modif = rng.choice(4)
        if id_modif == 0:
            draw = rng.normal(loc=0.0, scale=self.sigma_fact)
        elif id_modif == 1:
            draw = rng.normal(loc=0.0, scale=self.sigma_slope)
        elif id_modif == 2:
            draw = rng.normal(loc=0.0, scale=self.sigma_d_max)
        else:
            draw = None if self.sigma_d_nuc <= 0 else rng.normal(loc=0.0, scale=self.sigma_d_nuc)
        return int(id_modif), draw

    def _nuisance_finish(self, id_modif, draw):
        """The deterministic part: the test parameter set for these draws, incl. the d_max that goes with it (scipy fsolve)."""
        curr_param = np.copy(self.param_simu)
        kuhn, lm, c1, slope, d, d_max, fact, d_nuc = curr_param[0]
        if id_modif == 0:
            new_fact = fact + draw
            test_param = [kuhn, lm, slope, d, new_fact]
            new_d_max = opti.estimate_max_dist_intra_nuis(test_param, d_nuc, d_max)
            c1 = np.float32((0.53 * np.power(lm / kuhn, slope)) * np.power(kuhn, -3))
            out_test_param = [(kuhn, lm, c1, slope, d, new_d_max, new_fact, d_nuc)]
        elif id_modif == 1:
            new_slope = slope + draw
            test_param = [kuhn, lm, new_slope, d, fact]
            new_d_max = opti.estimate_max_dist_intra_nuis(test_param, d_nuc, d_max)
            c1 = np.float32((0.53 * np.power(lm / kuhn, new_slope)) * np.power(kuhn, -3))
            out_test_param = [(kuhn, lm, c1, new_slope, d, new_d_max, fact, d_nuc)]
        elif id_modif == 2:
            new_d_max = d_max + draw
            test_param = [kuhn, lm, slope, d, fact]
            new_d_nuc = opti.peval(new_d_max, test_param)  # sic: 5-vector, param[3] = d (quirk Q7)
            c1 = np.float32((0.53 * np.power(lm / kuhn, slope)) * np.power(kuhn, -3))
            out_test_param = [(kuhn, lm, c1, slope, d, new_d_max, fact, new_d_nuc)]
        else:
            new_d_nuc = d_nuc if draw is None else d_nuc + draw
            test_param = [kuhn, lm, slope, d, fact]
            new_d_max = opti.estimate_max_dist_intra_nuis(test_param, new_d_nuc, d_max)
            c1 = np.float32((0.53 * np.power(lm / kuhn, slope)) * np.power(kuhn, -3))
            out_test_param = [(kuhn, lm, c1, slope, d, new_d_max, fact, new_d_nuc)]
        return np.array(out_test_param, dtype=PARAM_SIMU_RIPPE)

    # -- the proposal of the NEXT step_nuisance_parameters call, PREDICTED on a worker thread while ig_step blocks (the ctypes
    #    call releases the GIL).  The reference's RNG order is: neighbours of step t, proposal draws of the nuisance step t,
    #    its acceptance draw, neighbours of step t + 1 ...  The worker copies the global generator's state (as the neighbour
    #    draw left it) into a private twin, makes the two proposal draws THERE and runs the expensive deterministic part
    #    (fsolve) for them.  The global stream is never touched: the nuisance step makes its own draws on it as always and
    #    takes the prepared parameter set only if its draws and the live parameters are the predicted ones, bit for bit --
    #    anything else (the caller drew numbers in between, parameters changed) just means the prediction is not used.
    def _speculate_nuisance(self):
        try:
            if self._twin is None:
                self._twin = np.random.RandomState()
                self._twin_addr = self._twin._bit_generator.ctypes.state_address
                self._glob_addr = np.random.mtrand._rand._bit_generator.ctypes.state_address
                self._twin_synced = False
            if self._twin_synced:
                # the Mersenne-Twister words + position (624 x 4 + 4 bytes) straight from the global generator; the cached
                # second Gaussian of the legacy stream is already the same in both: since the last full copy every normal()
                # the global made was made by the twin first, from the same state (checked when the prediction is adopted)
                C.memmove(self._twin_addr, self._glob_addr, 624 * 4 + 4)
            else:
                self._twin.set_state(np.random.get_state())   # full copy, ~0.1 ms (first use, or after a missed prediction)
                self._twin_synced = True
            key = self.param_simu.tobytes()
            id_modif, draw = self._nuisance_draws(self._twin)
            return (key, id_modif, draw, self._nuisance_finish(id_modif, draw))
        except Exception:
            self._twin_synced = False
            return None

    def step_nuisance_parameters(self, dt, t, n_step):
        """CL:2961-3051 (same host RNG calls, same scipy fsolve)."""
        spec, self._spec = self._spec, None
        self._nuis_follows = self.overlap_nuisance_proposal
        id_modif, draw = self._nuisance_draws(np.random)
        if (spec is not None and spec[0] == self.param_simu.tobytes() and spec[1] == id_modif
                and ((draw is None and spec[2] is None) or (draw is not None and spec[2] is not None and float(draw) == float(spec[2])))):
            out_test_param = spec[3]
            self.n_nuis_overlapped += 1
        else:
            self._twin_synced = False   # the twin's Gaussian cache may have parted from the global one: full copy next time
            out_test_param = self._nuisance_finish(id_modif, draw)
        self.param_simu_test = out_test_param
        self.likelihood_nuis = self.eval_likelihood_4_nuisance()
        F_t = self.temperature(t, n_step)
        with np.errstate(over="ignore"):
            ratio = np.exp((self.likelihood_nuis - self.likelihood_t) / F_t)
        u = np.random.rand()
        success = 0
        if ratio >= u:
            success = 1
            self.set_param_simu(np.array(list(out_test_param[0]), dtype=np.float32))
            self.param_simu = out_test_param
            self.likelihood_t = self.likelihood_nuis
        kuhn, lm, c1, slope, d, d_max, fact, d_nuc = self.param_simu[0]
        p0 = [kuhn, lm, slope, d, fact]
        y_rippe = opti.peval(self.bins, p0) if hasattr(self, "bins") else None
        return (fact, d, d_max, d_nuc, slope, self.likelihood_t, success, y_rippe)

    # ------------------------------------------------------------------ host-side helpers kept from the reference
    def dist_inter_genome(self, tmp_gpu_vect_frags=None):
        """CL:665-716 is computed on the device inside every step; this returns it for the live state."""
        raise NotImplementedError("dist is returned by step_sampler / test_copy_struct")

    def display_order(self):
        """CL:2556-2585: (full_order, dict_contig, full_order_high) -- fragments / sub-fragments in displayed
        order: contigs by ascending id, fragments by position, sub-fragments reversed when ori == -1."""
        self.gpu_vect_frags.copy_from_gpu()
        c = self.gpu_vect_frags
        order = np.lexsort((c.pos, c.id_c))                       # by contig id, then position
        full_order = c.id_d[order]
        dict_contig = {int(k): full_order[c.id_c[order] == k].tolist() for k in np.unique(c.id_c)}
        ids = self.np_sub_frags_id
        high = []
        for i in full_order:
            v = [int(ids[i]["x"]), int(ids[i]["y"]), int(ids[i]["z"])][: int(ids[i]["w"])]
            if c.ori[i] == -1:
                v.reverse()
            high.extend(v)
        return full_order.tolist(), dict_contig, high

    def contact_thumbnail(self, size=1024):
        """K x K binned contact map in the current scaffold order, computed on the GPU (SURVEY 8f, N1)."""
        _fo, _dc, high = self.display_order()
        rank = np.empty(int(self.init_n_sub_frags), dtype=np.int32)
        rank[np.asarray(high, dtype=np.int64)] = np.arange(len(high), dtype=np.int32)
        img = np.zeros((size, size), dtype=np.uint32)
        L.check(self._h, L.lib().ig_contact_thumbnail(self._h, _ptr(rank), int(size), _ptr(img)), "ig_contact_thumbnail")
        return img

    def display_current_matrix(self, filename, size=1024):
        """CL:2555-2606.  The reference densifies the NS x NS matrix on the host (impossible at 1 Gb scale);
        here a size x size thumbnail is binned on the GPU and written as PNG when matplotlib is available,
        else as a binary PGM (8-bit, 99th-percentile scaling like the reference's vmax)."""
        full_order, dict_contig, full_order_high = self.display_order()
        img = self.contact_thumbnail(size).astype(np.float64)
        vmax = max(np.percentile(img, 99), 1.0)
        try:
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt
            fig, ax = plt.subplots(figsize=(14, 14))
            ax.imshow(img, vmax=vmax, interpolation="nearest")
            ax.axis("off")
            fig.savefig(filename, dpi=200, bbox_inches="tight")
            plt.close(fig)
        except ImportError:
            g = np.clip(img / vmax * 255.0, 0, 255).astype(np.uint8)
            with open(filename, "wb") as fh:
                fh.write(b"P5\n%d %d\n255\n" % (size, size))
                fh.write(g.tobytes())
        return full_order, dict_contig, full_order_high
