"""ORACLE (test infrastructure only -- never imported by the product path).

NumPy restatement of the reference's scoring kernels (float32 expected contacts, float64
accumulation), following /root/reference/src/instagraal/kernels/kernel_sparse_adapt.cu (KA) and the
launch sites in cuda_lib_gl_single.py (CL).  libm (here) and libdevice (reference on a GPU) differ
by a few ulp in powf/expf, so float results are compared with a tolerance; every integer output
(slice membership, uniq lists, pixel counts) is exact.
"""
from __future__ import annotations

import math

import numpy as np

F32 = np.float32
LOG10E_F = np.float64(np.float32(0.43429448190325182))  # float literal promoted to double (KA:4353)


class Params:
    """param_simu (KA:91-100): 8 packed float32."""

    def __init__(self, p8):
        p8 = np.asarray(p8, dtype=np.float32).ravel()
        (self.kuhn, self.lm, self.c1, self.slope, self.d, self.d_max, self.fact, self.v_inter) = [F32(x) for x in p8]


def factorial_f32(n):
    """KA:111-124 (float)."""
    n = F32(math.floor(float(n)))
    if n < 10:
        r = F32(1)
        c = 1
        while c <= n:
            r = F32(r * F32(c))
            c += 1
        return r
    return F32(F32(F32(np.power(n, n)) * F32(np.exp(-n))) * F32(math.sqrt(F32(2 * math.pi * float(n)))))


_LOG10_FACT = np.array([0.0] + [math.log10(float(factorial_f32(k))) for k in range(1, 15)])


def rippe_contacts(s, p: Params):
    """KA:153-163, float32 throughout."""
    s = np.asarray(s, dtype=np.float32)
    with np.errstate(all="ignore"):
        t = (s * p.lm) / p.kuhn
        e = np.exp((p.d - F32(2)) / (np.power(t, F32(2.0)) + p.d))
        r = ((p.c1 * np.power(s, p.slope)) * e) * p.fact
    r = np.where((s > 0) & (s < p.d_max), r, F32(0)).astype(np.float32)
    return np.maximum(r, p.v_inter).astype(np.float32)


def rippe_contacts_circ(s, s_tot, p: Params):
    """KA:200-225 (note: floored at d_max, quirk Q6)."""
    s = np.asarray(s, dtype=np.float32)
    s_tot = np.asarray(s_tot, dtype=np.float32)
    with np.errstate(all="ignore"):
        K = p.lm / p.kuhn
        n = ((K * s) * (s_tot - s)) / s_tot
        e = np.exp((p.d - F32(2.0)) / (np.power(n, F32(2.0)) + p.d))
        r = ((np.power(p.kuhn, F32(-3.0)) * np.power(n, p.slope)) * e) * p.fact
    r = np.where((s > 0) & (s < p.d_max), r, F32(0)).astype(np.float32)
    return np.maximum(r, p.d_max).astype(np.float32)


def likelihood_pxl(ex, ob):
    """KA:251-270 in float64 (ex: float32 promoted; ob: counts)."""
    ex = np.asarray(ex, dtype=np.float64)
    ob = np.asarray(ob, dtype=np.float64)
    with np.errstate(all="ignore"):
        big = ob * np.log10(ex) - ex - (ob * np.log10(ob) - ob + np.log10(np.sqrt(ob * 2.0 * math.pi)))
        small = ob * np.log10(ex) - ex - _LOG10_FACT[np.clip(ob, 0, 14).astype(np.int64)]
    res = np.where(ob >= 15, big, np.where(ob > 0, small, -ex))
    return np.where(ex != 0, res, 0.0)


def fill_vect_dist(s, sub):
    """KA:3699-3822: per sub-fragment coordinates of a scaffold state.
    ``sub`` = dict(parent int64[NS], watson f32, crick f32, j int64)."""
    f = sub["parent"]
    ori = s["ori"][f]
    start = s["start_bp"][f].astype(np.float32)
    d = np.where(ori == 1, sub["watson"], sub["crick"]).astype(np.float32)
    dist = (start / F32(1000.0) + d).astype(np.float32)
    circ = s["circ"][f].astype(np.float32)
    st = (circ * s["l_cont_bp"][f].astype(np.float32)) / F32(1000.0)
    s_tot = np.trunc(st).astype(np.int32).astype(np.float32)  # local declared int (KA:3715)
    pos = s["sub_pos"][f] + np.where(ori == 1, sub["j"], s["sub_len"][f] - (sub["j"] + 1))
    return dict(dist=dist, id_c=s["id_c"][f].astype(np.int32), s_tot=s_tot, pos=pos.astype(np.int32),
                len=s["sub_l_cont"][f].astype(np.int32))


def sub_tables(np_sub_frags_2_frags):
    a = np_sub_frags_2_frags
    return dict(parent=a["x"].astype(np.int64), watson=a["y"].astype(np.float32),
                crick=a["z"].astype(np.float32), j=a["w"].astype(np.int64))


def contact_terms(v, rows, cols, dat, p: Params, mbar, len_from="col", return_parts=False):
    """Per-contact term of KA:4296-4354 / 4155-4208 / 4409-4464 for coordinates ``v``.
    return_parts=True: (terms, ex, exz), the float32 expected contacts of each contact and of its zero term
    (error bounds on a device sum are built from them)."""
    ci, cj = v["id_c"][rows], v["id_c"][cols]
    si, sj = v["dist"][rows], v["dist"][cols]
    s = np.abs((si - sj).astype(np.float32))
    pi, pj = v["pos"][rows].astype(np.float32), v["pos"][cols].astype(np.float32)
    s_z = (np.abs((pi - pj).astype(np.float32)) * mbar).astype(np.float32)
    s_tot = v["s_tot"][rows]
    ln = v["len"][cols if len_from == "col" else rows].astype(np.float32)
    s_tot_z = (ln * mbar).astype(np.float32)
    same = ci == cj
    lin = s_tot == 0
    ex_lin = rippe_contacts(s, p)
    exz_lin = np.where(s_z < p.d_max, rippe_contacts(s_z, p), p.v_inter)
    if np.any(same & ~lin):
        ex_c = rippe_contacts_circ(s, s_tot, p)
        exz_c = np.where(s_z < p.d_max, rippe_contacts_circ(s_z, s_tot_z, p), p.v_inter)
    else:
        ex_c, exz_c = ex_lin, exz_lin
    ex = np.where(same, np.where(lin, ex_lin, ex_c), p.v_inter).astype(np.float32)
    exz = np.where(same, np.where(lin, exz_lin, exz_c), p.v_inter).astype(np.float32)
    terms = likelihood_pxl(ex, dat) + exz.astype(np.float64) * LOG10E_F
    return (terms, ex, exz) if return_parts else terms


def full_likelihood_nz(v, coo, p, mbar):
    """evaluate_likelihood_sparse KA:4374-4488 (s_tot_z uses the ROW's len, KA:4428)."""
    rows, cols, dat = coo
    return float(np.sum(contact_terms(v, rows, cols, dat, p, mbar, len_from="row")))


def zeros_term_raw(v, p, mbar, return_parts=False):
    """eval_likelihood_on_zero / eval_all_likelihood_on_zero_1st (KA:3850-4002):
    returns (Z = -sum ex*(len-pos), n_intra as wrapped int32); return_parts=True appends the float64 terms
    ex*(len-pos) of the sub-fragments that have one (pos > 0)."""
    pos, ln, s_tot = v["pos"], v["len"], v["s_tot"]
    heads = pos == 0
    lh = ln[heads].astype(np.int64)
    t = np.array([_wrap32(int(x)) for x in lh * (lh - 1)], dtype=np.int64)  # int32 product wraps
    half = np.where(t >= 0, t // 2, -((-t) // 2))                          # C division truncates
    n_intra = _wrap32(int(np.sum(half)))                                   # int32 atomicAdd wraps
    m = pos > 0
    s = (pos[m].astype(np.float32) * mbar).astype(np.float32)
    s_tot_z = (ln[m].astype(np.float32) * mbar).astype(np.float32)
    lin = s_tot[m] == 0
    ex = np.where(lin, rippe_contacts(s, p), rippe_contacts_circ(s, s_tot_z, p) if np.any(~lin) else F32(0))
    ex = np.where(s < p.d_max, ex, p.v_inter).astype(np.float64)
    terms = ex * (ln[m] - pos[m]).astype(np.float64)
    z = -float(np.sum(terms))
    return (z, n_intra, terms) if return_parts else (z, n_intra)


def _wrap32(x):
    x &= 0xFFFFFFFF
    return x - (1 << 32) if x >= (1 << 31) else x


def zeros_term(v, p, mbar, n_pix):
    """eval_all_likelihood_on_zero_2nd KA:4005-4027."""
    z, n_intra = zeros_term_raw(v, p, mbar)
    val_inter = -1.0 * LOG10E_F * (np.float64(n_pix) - np.float64(n_intra)) * np.float64(p.v_inter)
    return float(z * LOG10E_F + val_inter)


def slice_windows(live, a, b, n_bounds):
    """slice_sp_mat thread-0 prologue KA:526-551 (sub-fragment units of the live scaffold)."""
    def head(f):
        sp, sl, ori = int(live["sub_pos"][f]), int(live["sub_len"][f]), int(live["ori"][f])
        return max(0, sp * (ori == 1) + (sp - sl) * (ori == -1)), sl
    pfa, sla = head(a)
    pfb, slb = head(b)
    la, lb = int(live["sub_l_cont"][a]), int(live["sub_l_cont"][b])
    return dict(pos_fa=pfa, pos_fb=pfb, is_circ=int(live["circ"][a]),
                up_a=max(0, pfa - n_bounds - sla), down_a=min(la - 1, pfa + n_bounds + sla),
                up_b=max(0, pfb - slb), down_b=min(lb - 1, pfb + slb))


def slice_mask(vcur, coo, id_ctg1, id_ctg2, w):
    """slice_sp_mat body KA:557-606 -> boolean mask over the canonical COO (incl. the C operator
    precedence of KA:587, quirk Q11, and the dat>0 filter of KA:602)."""
    rows, cols, dat = coo
    c1 = vcur["id_c"][rows]
    c2 = vcur["id_c"][cols]
    same = id_ctg1 == id_ctg2
    first = (c1 == id_ctg1) | (c1 == id_ctg2)
    smart = (c2 == c1) & same & (w["is_circ"] == 0)
    pi, pj = vcur["pos"][rows], vcur["pos"][cols]
    x, y = np.minimum(pi, pj), np.maximum(pi, pj)
    cond = ((x <= w["down_a"]) & (y >= w["up_a"])) | ((y >= w["up_b"]) & (x <= w["down_b"]))
    other = ((not same) & (c2 == id_ctg1)) | (c2 == id_ctg2)
    return first & np.where(smart, cond, other) & (dat > 0)


def sub_likelihoods(vmuts, uniq, sub_coo, p, mbar, block=64):
    """eval_sub_likelihood KA:4236-4370 over the (row-sorted) sliced contacts, including the
    reference's last-block quirk: in the final 64-thread block only threads tid < #valid contacts
    perform the per-mutation block sum, so uniq-list positions k >= (n_sub % 64) lose that block's
    contributions (KA:4362)."""
    rows, cols, dat = sub_coo
    n = len(rows)
    out = np.zeros(24, dtype=np.float64)
    t = n % block
    last0 = n - t
    for k, m in enumerate(uniq):
        terms = contact_terms(vmuts[m], rows, cols, dat, p, mbar, len_from="col")
        if k >= t:
            out[m] = float(np.sum(terms[:last0]))
        else:
            out[m] = float(np.sum(terms))
    return out
