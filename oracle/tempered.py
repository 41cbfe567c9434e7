"""TEST INFRASTRUCTURE ONLY -- restatement of the product's tempered move selection (instagraal_b200/csrc/ig_k_temper.cuh,
k_wide_stash / k_wide_pick in ig_k_wide.cuh) in NumPy/Python.

At a chain temperature T > 0 a step draws proposal i among the scored ones (score non-zero and not NaN) with probability
w_i / sum(w), w_i = exp((s_i - m) / T), m = the maximum score.  A step of more than 8 candidates draws its batch of 8
candidates b from W_b = S_b exp((m_b - M) / T) with u_batch, then the proposal inside it with u.  Sums are sequential in
ascending index; the pick is the first index whose running sum exceeds u * S, the last scored index when rounding leaves
none, index 0 when nothing is scored.  Only tests import this module."""
import math

import numpy as np

from oracle import device_rng

U_DOMAIN = 0x80000002         # draw index of u in the Philox counter (t, cycle, draw, 0)
U_BATCH_DOMAIN = 0x80000003   # ... of u_batch
BATCH = 8 * 24                # proposals of one batch of IG_MAX_CANDS candidates


def counters(t, cycle):
    return (t, cycle, U_DOMAIN, 0), (t, cycle, U_BATCH_DOMAIN, 0)


def draws(t, cycle, seed):
    """(u, u_batch) of plan step t of `cycle` for a chain keyed by `seed`"""
    return device_rng.uniform(t, cycle, U_DOMAIN, 0, seed), device_rng.uniform(t, cycle, U_BATCH_DOMAIN, 0, seed)


def scored(scores):
    s = np.asarray(scores, dtype=np.float64)
    return (s != 0.0) & ~np.isnan(s)


def weights(scores, T):
    """(w, m, S, n_scored, last scored index) of one batch (or narrow step), in the kernel's order of operations"""
    s = np.asarray(scores, dtype=np.float64)
    ok = scored(s)
    m = float(s[ok].max()) if ok.any() else -math.inf
    w = np.zeros(len(s))
    for i in np.flatnonzero(ok):
        w[i] = math.exp((float(s[i]) - m) / T)
    S = 0.0
    for x in w:
        S += float(x)
    last = int(np.flatnonzero(ok)[-1]) if ok.any() else -1
    return w, m, S, int(ok.sum()), last


def _pick(w, target, last):
    cum = 0.0
    for i, x in enumerate(w):
        cum += float(x)
        if cum > target:
            return i
    return last


def pick_narrow(scores, T, u):
    """-> (index, s_max, log_w, n_scored) of a step of up to 8 candidates"""
    w, m, S, n, last = weights(scores, T)
    idx = _pick(w, u * S, last) if n else 0
    return idx, m, (math.log(S) if S > 0 else -math.inf), n


def pick_wide(scores, T, u, u_batch):
    """-> (index over the whole step, batch, s_max, log_w, n_scored) of a step of more than 8 candidates"""
    s = np.asarray(scores, dtype=np.float64)
    parts = [weights(s[b:b + BATCH], T) for b in range(0, len(s), BATCH)]
    have = [p[3] > 0 for p in parts]
    M = max((p[1] for p, h in zip(parts, have) if h), default=-math.inf)
    W = [p[2] * math.exp((p[1] - M) / T) if h else 0.0 for p, h in zip(parts, have)]
    tot = 0.0
    for x in W:
        tot += x
    n = sum(p[3] for p in parts)
    last_b = max((b for b, h in enumerate(have) if h), default=-1)
    b = _pick(W, u_batch * tot, last_b) if last_b >= 0 else 0
    w, _m, S, nb, last = parts[b] if parts else (np.zeros(0), 0.0, 0.0, 0, -1)
    i = _pick(w, u * S, last) if nb else 0
    return b * BATCH + i, b, M, (math.log(tot) if tot > 0 else -math.inf), n


def pick(scores, T, u, u_batch, wide):
    """the product's choice for a step whose proposals (flattened, candidate * 24 + op) are `scores`: (index, batch, s_max,
    log_w, n_scored).  wide = the step runs in batches (its grid holds more than 8 candidate slots, even when the plan drew
    fewer); a narrow step records batch 0"""
    if wide:
        return pick_wide(scores, T, u, u_batch)
    idx, m, lw, n = pick_narrow(scores, T, u)
    return idx, 0, m, lw, n


def wide_marginal(scores, T):
    """P(b) P(i | b) of the two-stage draw for every proposal (exact arithmetic of the intended distribution, not of the
    draw): what the tests compare with w_i / sum(w)"""
    s = np.asarray(scores, dtype=np.float64)
    out = np.zeros(len(s))
    parts = [(b, weights(s[b:b + BATCH], T)) for b in range(0, len(s), BATCH)]
    M = max((p[1] for _b, p in parts if p[3] > 0), default=-math.inf)
    W = {b: (p[2] * math.exp((p[1] - M) / T) if p[3] > 0 else 0.0) for b, p in parts}
    tot = sum(W.values())
    for b, p in parts:
        if p[3] == 0:
            continue
        out[b:b + len(p[0])] = (W[b] / tot) * (p[0] / p[2])
    return out
