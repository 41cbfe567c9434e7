// instagraal_b200 -- finalisation, move selection, incremental maintenance, apply, contig bookkeeping, histogram, thumbnail.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// K9: per-candidate finalisation: fixed-order parallel reduction of the block partials, the
//     reference's last-block quirk (KA:4362), zero terms (eval_all_likelihood_on_zero_2nd
//     KA:4005-4027) and score assembly (eval_all_scores KA:4029-4046).  One block per candidate.
__global__ void __launch_bounds__(1024)
k_finalize(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const CoordRec* __restrict__ coord,
           DevScalars* sc, const IgDescriptor* __restrict__ desc_g, const int* __restrict__ rows, const int* __restrict__ rowidx,
           int ns, const int* __restrict__ row_cnt, const RowMut* __restrict__ table, const int* __restrict__ table_len,
           float mbar, const float* __restrict__ exz_tab, const double* __restrict__ part_nz, const int* __restrict__ part_c,
           int n_part, const double* __restrict__ part_z, const int* __restrict__ part_i, int n_part_z, double n_pix,
           int compat_last_block, int* __restrict__ n_uniq_out, int* __restrict__ n_sub_out, int do_select, int n_part_c, int flat) {
    TL(7);
    TLP_DECL();
    const int k = blockIdx.x;
    if (k >= sc->n_cands) return;
    __shared__ double s_nz[25], s_z[25], s_corr[IG_N_OPS];
    __shared__ int s_i[25], s_c[2];
    __shared__ double t_val[IG_N_OPS][64];
    __shared__ int2 t_cv[64];
    __shared__ int t_ri[64];
    __shared__ int t_cnt, t_need, tr_n;
    __shared__ int tr_ri[64], tr_skip[64], tr_off[64];
    __shared__ int t_wsum[32];
    const IgDescriptor& d = desc_g[k];
    const Params p = sc->p;
    const double l10v = sc->log10_vinter;
    const CandInfo ci_k = sc->ci[k];
    const int n_uniq = d.n_uniq;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    // 25 + 25 + 25 + 2 slots, one warp per slot, lanes stride the partial blocks, fixed shuffle tree
    // 32 warps, one slot each per round; every lane first issues all of its loads (independent, in
    // flight together), then adds them in index order; fixed shuffle tree => deterministic
    // (k_precompute's block b owns the row tiles b, b + grid, ...: blocks beyond the candidate's tile count wrote zeros)
    const int n_z_eff = min(n_part_z, max(1, (ci_k.n_rows + 31) >> 5));
    int nz_first = 0, nz_count = n_part;
    const bool fixed = sc->use_stream[k] != 0;   // streaming path: int64 fixed-point partials from k_eval_flat<true>
    if (flat || fixed) { int t_, c_; flat_block_range(sc, sc->n_cands, n_part, k, 0, &nz_first, &nz_count, &t_, &c_); }   // k_eval_flat's blocks for k
    for (int slot = w; slot < 77; slot += nwarp) {
        if (slot < 25 && fixed) {
            const long long* src = reinterpret_cast<const long long*>(&part_nz[PART_IDX(k, 25, slot, n_part, nz_first)]);
            long long v = 0;
            for (int i = lane; i < nz_count; i += 32) v += src[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) s_nz[slot] = (double)v * (1.0 / IG_FIX_SCALE);   // exact integer total, whatever the order
        } else if (slot < 50) {
            const double* src = slot < 25 ? &part_nz[PART_IDX(k, 25, slot, n_part, nz_first)] : &part_z[PART_IDX(k, 25, slot - 25, n_part_z, 0)];
            const int n = slot < 25 ? nz_count : n_z_eff;
            double v = 0.0;
            for (int i0 = 0; i0 < n; i0 += 32 * 16) {
                double x[16];
#pragma unroll
                for (int j = 0; j < 16; j++) { const int i = i0 + j * 32 + lane; x[j] = i < n ? src[i] : 0.0; }
#pragma unroll
                for (int j = 0; j < 16; j++) v += x[j];
            }
            v = warp_sum(v);
            if (lane == 0) { if (slot < 25) s_nz[slot] = v; else s_z[slot - 25] = v; }
        } else {
            // (the selection counters may come from another kernel than the likelihood partials: own block count)
            const int* src = slot < 75 ? &part_i[PART_IDX(k, 25, slot - 50, n_part_z, 0)] : &part_c[PART_IDX(k, 2, slot - 75, n_part_c, 0)];
            const int n = slot < 75 ? n_z_eff : n_part_c;
            int v = 0;
            for (int i0 = 0; i0 < n; i0 += 32 * 16) {
                int x[16];
#pragma unroll
                for (int j = 0; j < 16; j++) { const int i = i0 + j * 32 + lane; x[j] = i < n ? src[i] : 0; }
#pragma unroll
                for (int j = 0; j < 16; j++) v += x[j];
            }
            v = __reduce_add_sync(0xffffffffu, v);
            if (lane == 0) { if (slot < 75) s_i[slot - 50] = v; else s_c[slot - 75] = v; }
        }
    }
    if (threadIdx.x < IG_N_OPS) s_corr[threadIdx.x] = 0.0;
    __syncthreads();
    TLP(5);
    const int n_sub = s_c[0];
    const int t = n_sub % 64;
    const RowMut* tab = table + (size_t)k * IG_N_OPS * ns;
    const int* tlen = table_len + (size_t)k * IG_N_OPS * ns;
    // ---- last-block quirk: uniq slots u >= t lose the final (n_sub % 64) contacts of the row-sorted slice
    if (compat_last_block && t > 0 && t < n_uniq) {
        // ordered (hence deterministic) collection of the last t selected contacts of the row-sorted slice:
        // rows from the last one backwards, the whole block scans a row's contacts with a block-wide
        // exclusive scan of the selection flags, keeping the row's last `take` selected contacts in order
        // 1. the tail rows, found in parallel: windows of blockDim rows from the end of the affected-row list,
        //    block-wide scan of their selected-contact counts (thread order = descending row)
        const int* rc_k = row_cnt + (size_t)k * ns;
        if (threadIdx.x == 0) { tr_n = 0; t_need = 0; }
        __syncthreads();
        for (int hi = ci_k.n_rows; hi > 0; hi -= (int)blockDim.x) {
            const int carry = t_need;   // selected contacts in the rows behind this window
            if (carry >= t) break;
            const int ri = hi - 1 - (int)threadIdx.x;
            const int c = ri >= 0 ? rc_k[ri] : 0;
            int x = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            if (lane == 31) t_wsum[w] = x;
            __syncthreads();
            int before = 0, total = 0;
            for (int ww = 0; ww < nwarp; ww++) { const int v = t_wsum[ww]; if (ww < w) before += v; total += v; }
            const int excl = carry + before + x - c;   // tail contacts in later rows
            if (c > 0 && excl < t) {
                const int take = min(c, t - excl);
                const int slot = atomicAdd(&tr_n, 1);  // < 64 rows: each holds at least one tail contact
                tr_ri[slot] = ri; tr_skip[slot] = c - take; tr_off[slot] = t - (excl + take);
            }
            __syncthreads();
            if (threadIdx.x == 0) t_need = carry + total;
            __syncthreads();
        }
        // 2. one warp per tail row: its last `take` selected contacts, in column order, to their place in the tail
        for (int j = w; j < tr_n; j += nwarp) {
            const int ri = tr_ri[j], skip = tr_skip[j], off = tr_off[j];
            const int r = rows[(size_t)k * ns + ri];
            const CoordRec ci = coord[r];
            const long long b0 = row_ptr[r], e0 = row_ptr[r + 1];
            int running = 0;
            for (long long q0 = b0; q0 < e0; q0 += 32) {
                const long long q = q0 + lane;
                int2 c = make_int2(0, 0);
                bool sel = false;
                if (q < e0) {
                    c = cv[q];
                    const CoordRec cj = coord[c.x];
                    sel = (cj.id_c == ci_k.id_a || cj.id_c == ci_k.id_b) && contact_selected(ci, cj, c.y, ci_k);
                }
                const unsigned bal = __ballot_sync(0xffffffffu, sel);
                const int idx = running + __popc(bal & ((1u << lane) - 1));
                if (sel && idx >= skip) { const int slot = off + (idx - skip); t_cv[slot] = c; t_ri[slot] = ri; }
                running += __popc(bal);
            }
        }
        if (threadIdx.x == 0) t_cnt = t;
        __syncthreads();
        const int n_items = t_cnt * (n_uniq - t);
        for (int idx = threadIdx.x; idx < n_items; idx += blockDim.x) {
            const int e = idx % t_cnt, u = t + idx / t_cnt;
            const int2 c = t_cv[e];
            const RowMut a = tab[(size_t)u * ns + t_ri[e]];
            const int rj = rowidx[(size_t)k * ns + c.x] & ((1 << IG_CLS_SHIFT) - 1);
            const RowMut bm = tab[(size_t)u * ns + rj];
            CoordRec cim, cjm;
            cim.dist = a.dist; cim.id_c = a.id_c; cim.pos = a.pos; cim.s_tot = a.s_tot;
            cjm.dist = bm.dist; cjm.id_c = bm.id_c; cjm.pos = bm.pos; cjm.s_tot = bm.s_tot;
            const double ob = (double)c.y;
            t_val[u][e] = contact_term(cim, cjm, tlen[(size_t)u * ns + rj], ob, ob_const(ob), p, l10v, mbar, exz_tab);
        }
        __syncthreads();
        if (threadIdx.x >= t && threadIdx.x < n_uniq) {
            double ssum = 0.0;
            for (int e = 0; e < t_cnt; e++) ssum += t_val[threadIdx.x][e];
            s_corr[threadIdx.x] = ssum;
        }
        __syncthreads();
    }
    TLP(6);
    // ---- scores
    if (threadIdx.x < IG_N_OPS) sc->scores[k * IG_N_OPS + threadIdx.x] = 0.0;
    __syncthreads();
    if (threadIdx.x < n_uniq) {
        const int u = threadIdx.x;
        const double log_e = (double)LOG10E_F;
        const int m = d.uniq[u];
        // Z[m] over ALL sub-fragments = Z_cur(all) - Z_cur(affected rows) + Z_m(affected rows)
        const double z = sc->z_cur - s_z[24] + s_z[u];
        const int n_intra = sc->nintra_cur - s_i[24] + s_i[u];  // int32 wrap-consistent
        const double val_inter = -1.0 * log_e * (n_pix - __int2double_rn(n_intra)) * p.v_inter;
        const double lz = z * log_e + val_inter;
        const double lnz = s_nz[u] - ((u >= t && compat_last_block && t > 0) ? s_corr[u] : 0.0);
        sc->scores[k * IG_N_OPS + m] = lnz + lz + sc->lnz_full - s_nz[24];
        sc->lnz_new[k * IG_N_OPS + m] = sc->lnz_full - s_nz[24] + s_nz[u];  // without the last-block quirk
        sc->z_new[k * IG_N_OPS + m] = z;
        sc->nintra_new[k * IG_N_OPS + m] = n_intra;
    }
    if (threadIdx.x == 0) {
        sc->lsub_cur[k] = s_nz[24];
        sc->ci[k].n_sub = n_sub;
        n_uniq_out[k] = n_uniq;
        n_sub_out[k] = n_sub;
        atomicAdd(&sc->st_contacts, (unsigned long long)s_c[1]);
        atomicAdd(&sc->st_rows, (unsigned long long)ci_k.n_rows);
        atomicAdd(&sc->st_frags, (unsigned long long)(d.A.l_cont + (ci_k.same ? 0 : d.B.l_cont)));
        atomicAdd(&sc->st_selected, (unsigned long long)n_sub);
        atomicAdd(&sc->st_proposals, (unsigned long long)n_uniq);
    }
    TLP(7);
    if (!do_select) return;
    // move selection by the LAST candidate block to finish (saves a dependent launch)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) t_cnt = (atomicAdd(&sc->ticket_fin, 1u) == (unsigned)sc->n_cands - 1) ? 1 : 0;
    __syncthreads();
    if (t_cnt && threadIdx.x < 32) {
        __threadfence();
        select_step(sc, desc_g);
    }
}

// K10: move selection (CL:1435-1446): scores==0 -> -inf; first index of the maximum.
__global__ void k_select(DevScalars* sc) {
    __shared__ double sm[IG_MAX_CANDS * IG_N_OPS];
    const int n = sc->n_cands * IG_N_OPS;
    for (int i = threadIdx.x; i < n; i += blockDim.x) sm[i] = sc->scores[i];
    __syncthreads();
    if (threadIdx.x != 0) return;
    int best = -1;
    double bv = 0.0;
    for (int i = 0; i < n; i++) {
        const double v = sm[i];
        if (v == 0.0) continue;
        if (best < 0 || v > bv) { best = i; bv = v; }
    }
    if (best < 0) best = 0;  // np.argmax of an all-zero filtered vector
    sc->win_cand = best / IG_N_OPS;
    sc->win_op = best % IG_N_OPS;
    sc->likelihood = sm[best];
    sc->n_heads = 0; sc->sum_l_cont = 0; sc->dist_half = 0;  // accumulators of k_post
    sc->q4_hits = 0;                                          // counted by k_apply for THIS move
}
// step path: selection + the bookkeeping of k_post_scalars in one launch (k_apply reads the label base
// from the descriptor, not from sc->max_label, so bumping it here cannot race)
__device__ void select_step(DevScalars* sc, const IgDescriptor* __restrict__ desc_g) {
    const int n = sc->n_cands * IG_N_OPS;
    const int lane = threadIdx.x & 31;  // executed by one full warp
    int best = -1;
    const double T = sc->temperature;
    if (T > 0.0) {
        best = temper_select(sc, n, T);   // a draw among the scored proposals (ig_k_temper.cuh)
    } else {
        // first index of the maximum among the scored (non-zero) proposals (CL:1435-1446)
        double bv = 0.0;
        for (int i = lane; i < n; i += 32) {
            const double v = __ldcg(&sc->scores[i]);
            if (v == 0.0) continue;
            if (best < 0 || v > bv) { best = i; bv = v; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int ob = __shfl_down_sync(0xffffffffu, best, o);
            const double ov = __shfl_down_sync(0xffffffffu, bv, o);
            if (ob >= 0 && (best < 0 || ov > bv || (ov == bv && ob < best))) { best = ob; bv = ov; }
        }
        best = __shfl_sync(0xffffffffu, best, 0);
        if (best < 0) best = 0;
    }
    const int kc = best / IG_N_OPS, op = best % IG_N_OPS;
    const unsigned hit = __ballot_sync(0xffffffffu, lane < desc_g[kc].n_uniq && desc_g[kc].uniq[lane] == op);
    if (lane < 12 && op >= 12) sc->valid[lane] = desc_g[kc].valid[lane];
    if (lane != 0) return;
    sc->win_cand = kc; sc->win_op = op; sc->likelihood = __ldcg(&sc->scores[best]);
    sc->live_likelihood = sc->likelihood;
    sc->n_heads = 0; sc->sum_l_cont = 0; sc->dist_half = 0; sc->q4_hits = 0;
    sc->max_label += 2;
    sc->prev_k = kc; sc->prev_u = hit ? (__ffs(hit) - 1) : 0;
    sc->prev_windowed = (sc->ci[kc].same && sc->ci[kc].is_circ == 0) ? 1 : 0;
    sc->prev_id_a = sc->ci[kc].id_a; sc->prev_n_rows = sc->ci[kc].n_rows;
    sc->lnz_next = __ldcg(&sc->lnz_new[best]); sc->z_next = __ldcg(&sc->z_new[best]); sc->nintra_next = __ldcg(&sc->nintra_new[best]);
    sc->ticket_out = 0;
}
__global__ void k_select_step(DevScalars* sc, const IgDescriptor* __restrict__ desc_g) { select_step(sc, desc_g); }

// Same-linear-contig moves are scored on a WINDOWED slice (slice_sp_mat, KA:565-586): contacts of the
// contig outside the windows keep their distance mathematically, but the reference's next full
// recomputation (CL:1409) sees their float32 coordinates re-rounded.  To keep lnz_full identical to
// that recomputation without rescanning every contact, add exactly those contacts' term changes.
__global__ void __launch_bounds__(IG_THREADS)
k_lnz_outside(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const CoordRec* __restrict__ coord,
              const int* __restrict__ clen, DevScalars* sc, const int* __restrict__ rows, const int* __restrict__ rowidx, int ns,
              const RowMut* __restrict__ table, const int* __restrict__ table_len, float mbar, const float* __restrict__ exz_tab,
              double* __restrict__ part) {
    TL(8);
    if (!sc->prev_windowed) return;
    __shared__ double sm[32];
    __shared__ int is_last;
    const int k = sc->prev_k, u = sc->prev_u;
    const Params p = sc->p;
    const double l10v = sc->log10_vinter;
    const CandInfo ci_k = sc->ci[k];
    const int lane = threadIdx.x & 31;
    const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    const int* my_rows = rows + (size_t)k * ns;
    const int* my_idx = rowidx + (size_t)k * ns;
    const RowMut* tab = table + ((size_t)k * IG_N_OPS + u) * ns;
    const int* tlen = table_len + ((size_t)k * IG_N_OPS + u) * ns;
    double acc = 0.0;
    for (int ri = wg; ri < ci_k.n_rows; ri += nw) {
        const int r = my_rows[ri];
        const CoordRec ci = coord[r];
        const RowMut a = tab[ri];
        for (long long q = row_ptr[r] + lane; q < row_ptr[r + 1]; q += 32) {
            const int2 c = __ldg(&cv[q]);
            const CoordRec cj = coord[c.x];
            if (cj.id_c != ci_k.id_a) continue;               // other contigs: inter-contig term, unchanged
            if (contact_selected(ci, cj, c.y, ci_k)) continue;  // already inside lnz_new
            const int rj = my_idx[c.x] & ((1 << IG_CLS_SHIFT) - 1);
            const RowMut bm = tab[rj];
            CoordRec cim, cjm;
            cim.dist = a.dist; cim.id_c = a.id_c; cim.pos = a.pos; cim.s_tot = a.s_tot;
            cjm.dist = bm.dist; cjm.id_c = bm.id_c; cjm.pos = bm.pos; cjm.s_tot = bm.s_tot;
            const double ob = (double)c.y, obc = ob_const(ob);
            // the full-likelihood kernel takes the circular length from the ROW (KA:4428)
            const double t_old = contact_term(ci, cj, clen[r], ob, obc, p, l10v, mbar, exz_tab);
            const double t_new = contact_term(cim, cjm, tlen[ri], ob, obc, p, l10v, mbar, exz_tab);
            acc += t_new - t_old;
        }
    }
    const double tot = block_sum(acc, sm);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = tot;
        __threadfence();
        is_last = (atomicAdd(&sc->ticket_out, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double v = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) v += ((volatile double*)part)[i];
    const double all = block_sum(v, sm);
    if (threadIdx.x == 0) sc->lnz_next += all;
}

// start of the next step in incremental mode: the coordinates of the rows touched by the last applied
// move are taken from the mutation table (bit-identical to uni_fill_vect_dist on the new scaffold),
// everything else is unchanged; the scalar likelihood pieces were prepared by the previous step.
__global__ void __launch_bounds__(256)
k_commit_coords(CoordRec* __restrict__ coord, int* __restrict__ clen, DevScalars* sc, const int* __restrict__ rows, int ns,
                const RowMut* __restrict__ table, const int* __restrict__ table_len, const FragRec* __restrict__ live,
                const SubRec* __restrict__ sub, SubX* __restrict__ subx, unsigned char* __restrict__ row_dirty) {
    TL(11);
    const int k = sc->prev_k, u = sc->prev_u, n = sc->prev_n_rows;
    const int* my_rows = rows + (size_t)k * ns;
    const RowMut* tab = table + ((size_t)k * IG_N_OPS + u) * ns;
    const int* tlen = table_len + ((size_t)k * IG_N_OPS + u) * ns;
    for (int ri = blockIdx.x * blockDim.x + threadIdx.x; ri < n; ri += gridDim.x * blockDim.x) {
        const int r = my_rows[ri];
        const RowMut m = tab[ri];
        CoordRec c; c.dist = m.dist; c.id_c = m.id_c; c.pos = m.pos; c.s_tot = m.s_tot;
        coord[r] = c; clen[r] = tlen[ri];
        if (row_dirty) row_dirty[r] = 1;   // cached per-contact records of this row are stale (k_lnz_refresh)
        const SubRec sr = sub[r];
        const Frag f = live[sr.parent].f;   // the scaffold after the applied move
        SubX x; x.start_bp = f.start_bp; x.len_ori = f.len_bp * f.ori; x.watson = sr.watson; x.crick = sr.crick;
        subx[r] = x;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        sc->lnz_full = sc->lnz_next; sc->z_cur = sc->z_next; sc->nintra_cur = sc->nintra_next;
    }
}

// K11: apply the winning move to every fragment (test_copy_struct + copy_struct, CL:2094-2151)
__global__ void __launch_bounds__(256)
k_apply(FragRec* __restrict__ live, int nf, DevScalars* sc, const IgDescriptor* __restrict__ desc_g, int forced_cand, int forced_op) {
    TL(9);
    __shared__ IgDescriptor d;
    const int kc = forced_cand >= 0 ? forced_cand : sc->win_cand;
    const int op = forced_op >= 0 ? forced_op : sc->win_op;
    {
        const int* src = reinterpret_cast<const int*>(desc_g + kc);
        int* dst = reinterpret_cast<int*>(&d);
        for (int i = threadIdx.x; i < (int)(sizeof(IgDescriptor) / 4); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    // every thread reads only its own fragment + the descriptor's pivots (loaded before any write): in place is safe
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nf) {
        const Frag f = live[i].f;
        Frag o;
        if (op >= 8 && op < 12) {  // paste may leave a fragment unwritten (Q4): keep + count
            const int ua = (op - 8) >> 1, ub = (op - 8) & 1;
            Frag t1 = ig_split(f, i, d.A, ua, d.max_id);
            Frag t2 = ig_split(t1, i, d.T1B[ua], ub, d.max_id1[ua]);
            int written;
            o = ig_paste(t2, i, d.T2A[ua][ub], d.a, d.T2B[ua][ub], d.b, &written);
            if (!written) atomicAdd(&sc->q4_hits, 1);
        } else {
            o = ig_eval_op(d, op, f, i);
        }
        live[i].f = o;
    }
}
// bookkeeping that must not race with k_apply's reads of sc->max_label (through the descriptor it does not: the
// descriptor carries max_id) -- label counter and list_valid_insert (CL:2125-2126 re-runs get_bounds for ops >= 12)
__global__ void k_post_scalars(DevScalars* sc, const IgDescriptor* __restrict__ desc_g, int forced_cand, int forced_op) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int kc = forced_cand >= 0 ? forced_cand : sc->win_cand;
    const int op = forced_op >= 0 ? forced_op : sc->win_op;
    if (op >= 12) for (int i = 0; i < 12; i++) sc->valid[i] = desc_g[kc].valid[i];
    sc->max_label += 2;
    if (forced_cand >= 0) { sc->n_heads = 0; sc->sum_l_cont = 0; sc->dist_half = 0; }
}
__global__ void __launch_bounds__(256)
k_post(const FragRec* __restrict__ live, int nf, const int* __restrict__ init_prev, const int* __restrict__ init_next,
       const int* __restrict__ orientable, DevScalars* sc, CycleOut* __restrict__ cyc_out, ig_tempered_step* __restrict__ trec_out) {
    TL(10);
    __shared__ int s_heads;
    __shared__ long long s_len, s_half;
    if (threadIdx.x == 0) { s_heads = 0; s_len = 0; s_half = 0; }
    __syncthreads();
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    int heads = 0; long long len = 0; int half = 0;  // half = decrement of d in units of 1/2
    if (f < nf) {
        const Frag g = live[f].f;
        if (g.pos == 0) { heads = 1; len = g.l_cont; }
        // dist_inter_genome, CL:672-715 (init_ori == +1, blacklist empty)
        const int p0 = init_prev[f], n0 = init_next[f];
        int p1 = g.prev, n1 = g.next;
        int swap = 1;
        if ((p1 == p0 && n1 == n0) || (p1 == n0 && n1 == p0)) half += 2;
        if (orientable[f]) {
            if (1 != g.ori) { int tmp = p1; p1 = n1; n1 = tmp; swap = -1; }
            if (p0 == p1) {
                if (p0 == -1 || !orientable[p1]) half += 2;
                else { half += 1; if (1 == swap * live[p1].f.ori) half += 1; }
            }
            if (n0 == n1) {
                if (n0 == -1 || !orientable[n1]) half += 2;
                else { half += 1; if (1 == swap * live[n1].f.ori) half += 1; }
            }
        } else {
            if (p1 == p0 || p1 == n0) half += 2;
            if (n1 == n0 || n1 == p0) half += 2;
        }
    }
    // warp-level reductions first: one shared atomic per warp instead of one per thread
    const int w_heads = __reduce_add_sync(0xffffffffu, heads);
    const int w_half = __reduce_add_sync(0xffffffffu, half);
    long long w_len = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w_len += __shfl_down_sync(0xffffffffu, w_len, o);
    if ((threadIdx.x & 31) == 0) {
        if (w_heads) { atomicAdd(&s_heads, w_heads); atomicAdd((unsigned long long*)&s_len, (unsigned long long)w_len); }
        if (w_half) atomicAdd((unsigned long long*)&s_half, (unsigned long long)w_half);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_heads) atomicAdd(&sc->n_heads, s_heads);
        if (s_len) atomicAdd((unsigned long long*)&sc->sum_l_cont, (unsigned long long)s_len);
        if (s_half) atomicAdd((unsigned long long*)&sc->dist_half, (unsigned long long)s_half);
        if (cyc_out) {  // cycle mode: the last block to finish publishes this step's record and advances the plan
            __threadfence();
            if (atomicAdd(&sc->ticket_post, 1u) == gridDim.x - 1) {
                __threadfence();
                CycleOut o;
                o.likelihood = sc->likelihood; o.lnz_full = sc->lnz_full;
                o.dist_half = *(volatile long long*)&sc->dist_half; o.sum_l_cont = *(volatile long long*)&sc->sum_l_cont;
                o.n_heads = *(volatile int*)&sc->n_heads; o.win_cand = sc->win_cand; o.win_op = sc->win_op; o.q4_hits = sc->q4_hits;
                o.n_proposals = 0;
                for (int i = 0; i < sc->n_cands; i++) o.n_proposals += sc->res_nuniq[i];
                o.id_f_sampled = sc->cands[sc->win_cand];
                cyc_out[sc->step_idx] = o;
                if (sc->temperature > 0.0) trec_out[sc->step_idx] = sc->trec;   // the tempered draw (ig_k_temper.cuh)
                sc->step_idx += 1;
#ifdef IG_TIMELINE
                g_tl_step += 1;
#endif
            }
        }
    }
}
__global__ void k_explode(FragRec* live, int nf, const int* __restrict__ perm) {  // KA:409-426
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nf) return;
    Frag f = live[i].f;
    f.pos = 0; f.start_bp = 0; f.sub_pos = 0; f.id_c = perm[i]; f.prev = -1; f.next = -1;
    f.l_cont = 1; f.l_cont_bp = f.len_bp; f.sub_l_cont = f.sub_len;
    live[i].f = f;
}
// histogram for the initial p(s) fit (CL:2253-2293) on the INITIAL scaffold; integer-exact sums
__global__ void __launch_bounds__(IG_THREADS)
k_histogram(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const int* __restrict__ sym_diag,
            const FragRec* __restrict__ init, const SubRec* __restrict__ sub, int n_rows, double bin_kb, double max_kb,
            int n_bins, unsigned long long* __restrict__ hist, unsigned long long* __restrict__ rows_used) {
    const int lane = threadIdx.x & 31;
    const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (int r = wg; r < n_rows; r += nw) {
        const SubRec si = sub[r];
        const Frag fi = init[si.parent].f;
        const bool used = bin_kb < (double)fi.l_cont_bp / 1000.0;
        if (!used) continue;
        const double s_i = (double)fi.start_bp / 1000.0 + (double)si.watson;
        if (lane == 0) {
            atomicAdd(rows_used, 1ULL);
            if (sym_diag && sym_diag[r] != 0 && 0.0 < max_kb) atomicAdd(&hist[0], (unsigned long long)sym_diag[r]);
        }
        for (long long q = row_ptr[r] + lane; q < row_ptr[r + 1]; q += 32) {
            const int2 c = cv[q];
            const SubRec sj = sub[c.x];
            const Frag fj = init[sj.parent].f;
            if (fj.id_c != fi.id_c) continue;
            const double s_j = (double)fj.start_bp / 1000.0 + (double)sj.watson;
            const double dd = fabs(s_i - s_j);
            if (!(dd < max_kb)) continue;
            const int b = (int)(dd / bin_kb);
            if (b < 0 || b >= n_bins) continue;
            const int mult = 1 + (c.x < n_rows ? 1 : 0);  // symmetric matrix: row r and row c.x both see it
            atomicAdd(&hist[b], (unsigned long long)((long long)c.y * mult));
        }
    }
}

// N1 (SURVEY 8f): K x K thumbnail of the contact map in the CURRENT scaffold order, binned on the
// device (the reference densifies NS x NS on the host, CL:2598-2599).  Integer counts => exact.
__global__ void __launch_bounds__(IG_THREADS)
k_thumbnail(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const int* __restrict__ sub_rank, int ns, int K,
            unsigned int* __restrict__ img) {
    const int lane = threadIdx.x & 31;
    const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (int r = wg; r < ns; r += nw) {
        const int pi = (int)(((long long)sub_rank[r] * K) / ns);
        for (long long q = row_ptr[r] + lane; q < row_ptr[r + 1]; q += 32) {
            const int2 c = cv[q];
            const int pj = (int)(((long long)sub_rank[c.x] * K) / ns);
            atomicAdd(&img[(size_t)pi * K + pj], (unsigned int)c.y);
            if (pi != pj) atomicAdd(&img[(size_t)pj * K + pi], (unsigned int)c.y);
        }
    }
}
