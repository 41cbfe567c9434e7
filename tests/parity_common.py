"""Shared parity checker: replays a golden trajectory recorded from the reference
(oracle/make_golden.py) against any implementation of the hot path, teacher-forced per step.

Why teacher-forced: many candidate moves are *exactly* tied by construction (different ops that
produce the same scaffold), so which one the reference's argmax picks depends on floating-point
summation order at the 1e-13 level (on a real GPU: on atomicAdd ordering, i.e. it is not even
reproducible run to run).  north_star permits divergence only there.  So each step starts from the
reference's recorded pre-step state; scores must agree within tolerance for every scored proposal,
the set of scored proposals must be identical, and the chosen move must either be identical (then
the post-step integer state must be bit-identical) or be tied with the reference's choice.

Tolerance (floating point): |s - s_ref| <= 1e-5 * |s_ref - best_ref| + 2e-8 * |s_ref|, i.e. 1e-5
relative on the delta to the step's best proposal plus a floor for the few-ulp libm/libdevice
powf differences accumulated over the slice.  Integer state: bit-exact.
"""
from __future__ import annotations

import numpy as np

FIELDS13 = ("pos", "sub_pos", "id_c", "start_bp", "len_bp", "sub_len", "circ", "prev", "next",
            "l_cont", "sub_l_cont", "l_cont_bp", "ori")


class Result:
    def __init__(self):
        self.steps = 0
        self.same_choice = 0
        self.tied_choice = 0
        self.max_rel = 0.0
        self.errors = []
        self.nuis_checked = 0


def score_tol(s_ref):
    best = s_ref.max()
    return 1e-5 * np.abs(s_ref - best) + 2e-8 * np.abs(s_ref) + 1e-9


def replay(golden, impl, max_steps=None, check_state=True, check_nuis=True):
    """``impl`` must provide: set_state(int32[13,NF]), set_valid(int32[12]), set_params(f32[8]),
    eval_nuisance(f32[8]) -> float (full likelihood under test params on the stale coordinates),
    step(A, cands:list[int]) -> dict(scores f64[24*n], op, B, o, dist, mean_len, n_contigs),
    get_state() -> int32[13,NF]."""
    g = golden
    res = Result()
    n = len(g["step_A"])
    if max_steps:
        n = min(n, max_steps)
    prev_state = g["state0"]
    nuis_at = {int(s): k for k, s in enumerate(g.get("step_nuis_step", []))}
    for t in range(n):
        nc = int(g["step_ncand"][t])
        cands = [int(c) for c in g["step_cands"][t][:nc]]
        impl.set_state(prev_state)
        impl.set_valid(g["step_valid_before"][t])
        impl.set_params(g["step_params_before"][t])
        out = impl.step(int(g["step_A"][t]), cands)
        s_ref = g["step_scores"][t][:24 * nc]
        s = np.asarray(out["scores"], dtype=np.float64)
        if s.shape != s_ref.shape:
            res.errors.append((t, "score vector shape", s.shape, s_ref.shape))
            break
        zr, zs = s_ref == 0, s == 0
        if not np.array_equal(zr, zs):
            res.errors.append((t, "scored-proposal set differs", np.flatnonzero(zr != zs).tolist()))
        else:
            ok = ~zr
            tol = score_tol(s_ref[ok])
            diff = np.abs(s[ok] - s_ref[ok])
            if np.any(diff > tol):
                w = int(np.argmax(diff - tol))
                res.errors.append((t, "score out of tolerance", float(diff[w]), float(tol[w]), float(s_ref[ok][w])))
            res.max_rel = max(res.max_rel, float(np.max(diff / np.maximum(np.abs(s_ref[ok]), 1e-300))))
        gid_ref = (cands.index(int(g["step_Bs"][t]))) * 24 + int(g["step_op"][t])
        gid = cands.index(int(out["B"])) * 24 + int(out["op"])
        if gid == gid_ref:
            res.same_choice += 1
            if check_state:
                st = impl.get_state()
                want = g["step_states"][t]
                if not np.array_equal(st, want):
                    bad = [FIELDS13[i] for i in range(13) if not np.array_equal(st[i], want[i])]
                    res.errors.append((t, "post-step state differs", bad))
            for key, want in (("dist", g["step_dist"][t]), ("n_contigs", g["step_n_contigs"][t]),
                              ("mean_len", g["step_mean_len"][t])):
                if not (float(out[key]) == float(want)):
                    res.errors.append((t, key, float(out[key]), float(want)))
            if abs(float(out["o"]) - float(g["step_o"][t])) > 2e-8 * abs(float(g["step_o"][t])) + 1e-9:
                res.errors.append((t, "o", float(out["o"]), float(g["step_o"][t])))
        else:
            gap = abs(s_ref[gid] - s_ref[gid_ref])
            if gap <= 2e-8 * abs(s_ref[gid_ref]) + 1e-9 and not zr[gid]:
                res.tied_choice += 1
            else:
                res.errors.append((t, "different move chosen", gid, gid_ref, float(gap)))
        # nuisance-parameter likelihood (evaluated on the coordinates of THIS step's start, quirk Q5)
        if check_nuis and "step_nuis_step" in g and t in nuis_at and gid == gid_ref:
            k = nuis_at[t]
            want = float(g["step_nuis"][k][7])
            got = float(impl.eval_nuisance(g["step_params"][k]))
            if abs(got - want) > 2e-8 * abs(want) + 1e-9:
                res.errors.append((t, "nuisance likelihood", got, want))
            res.nuis_checked += 1
        prev_state = g["step_states"][t]
        res.steps += 1
        if len(res.errors) > 5:
            break
    return res


class OracleTeacher:
    """The NumPy port of the reference (oracle/sampler_oracle.py, held to the reference's recorded trajectories by
    tests/test_oracle_golden.py) behind the interface of oracle.ref_replay.RefReplaySampler.  Lockstep tests whose teacher is
    the reference's own compiled kernels (oracle/_ref/, built from a checkout of the reference) use it where those are not
    built.  Its scores follow the host's powf / log10, so they are compared within score_tol and ties at 2e-8 relative,
    not at the 1e-9 that holds between the reference's kernels and the product (same libdevice code on the GPU)."""

    def __init__(self, level, p8):
        from oracle.sampler_oracle import OracleSampler
        self.o = OracleSampler(level, p8)
        self.valid_insert = self   # RefReplaySampler.valid_insert.get()

    def get(self):
        return np.asarray(self.o.valid, dtype=np.int32)

    def set_state(self, st):
        self.o.live = {k: np.array(st[i], dtype=np.int32) for i, k in enumerate(FIELDS13)}

    def get_state(self):
        return np.stack([self.o.live[k] for k in FIELDS13]).astype(np.int32)

    def set_valid(self, v):
        self.o.valid = [int(x) for x in v]

    def set_params(self, p8):
        from oracle import score as sc
        self.o.params8 = np.asarray(p8, dtype=np.float32).copy()
        self.o.params = sc.Params(self.o.params8)

    def step_sampler(self, a, cands):
        return self.o.step_sampler(int(a), candidates=[int(c) for c in cands])

    @property
    def all_scores(self):
        return self.o.all_scores


def state_mismatch_modulo_length_ties(got, want):
    """Fields that differ between two [13, NF] scaffolds, with contig labels compared the way BASELINE.md prescribes:
    modulo relabelling among contigs of EQUAL length.  The reference numbers contigs by descending length through a
    list that select_uniq_id_c fills with an atomic counter (KA:357-406), so on a real GPU the order inside a group of
    equal-length contigs is arbitrary (it is sequential, hence reproducible, only on the CPU emulation the golden vectors
    were recorded with).  Checked instead: same partition of the fragments into contigs, and in both states a larger
    label never belongs to a shorter contig (id = NC - 1 - rank by descending length, CL:2747-2806)."""
    bad = [FIELDS13[i] for i in range(13) if i != 2 and not np.array_equal(got[i], want[i])]
    a, b = np.asarray(got[2]), np.asarray(want[2])
    # same partition: the map label_a -> label_b must be a bijection
    pairs = np.unique(np.stack([a, b]), axis=1)
    if len(np.unique(pairs[0])) != pairs.shape[1] or len(np.unique(pairs[1])) != pairs.shape[1]:
        bad.append("id_c (partition)")
    for st in (got, want):
        lab, first = np.unique(st[2], return_index=True)
        ln = np.asarray(st[9])[first]          # l_cont per contig, labels ascending
        if np.any(np.diff(ln) < 0) or lab[0] != 0 or lab[-1] != len(lab) - 1:
            bad.append("id_c (labels not ordered by length)")
            break
    return bad
