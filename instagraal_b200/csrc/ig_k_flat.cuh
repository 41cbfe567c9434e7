// instagraal_b200 -- flat scoring path of small levels: k_pick + k_eval_flat.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// FLAT scoring path for small levels (yeast scale: a candidate touches a few hundred rows of ~100 contacts).
// There the row-per-warp kernel above is all latency: one tiny work item per warp, each a chain of dependent
// gathers plus a partly filled evaluation queue, and half of the lanes hold contacts outside the slice.  Instead:
//   k_pick      one warp per 32-contact chunk of an affected row (rows own whole chunks of a per-candidate list,
//               offsets = running sum of the padded row lengths from k_rows_small): slice membership, class-pair
//               mask, current-state term; the contacts that need a look under at least one mutation are written
//               compactly (ballot prefix) at the start of their chunk (+ the count), so the list order is fixed;
//   k_eval_flat work item = (one chunk's packed contacts, group of uniq slots): no selection, no gathers by
//               column, no per-row set-up; loop over the group's mutations exactly like the dense schedule of
//               k_score (same eval_pair / queue code), one accumulator reduction per block.
// Results are the same sums in a different (still fixed) order.
#define IG_PICK_PARTS 4
// blocks [first, first + count) of the k_eval_flat grid that work for a candidate: one block per non-empty
// candidate + the rest in proportion to the number of chunks
// (k >= 0: the range of candidate k; k < 0: the candidate whose range holds block `blk`, -1 in *cand if none)
__device__ __forceinline__ void flat_block_range(const DevScalars* __restrict__ sc, int n_cands, int grid, int k, int blk,
                                                 int* first, int* count, int* tiles, int* cand) {
    int t[IG_MAX_CANDS];
#pragma unroll
    for (int c = 0; c < IG_MAX_CANDS; c++) t[c] = (sc->flat_segtotal[c] + 31) >> 5;   // independent loads, issued together
    int tiles_all = 0, n_nonempty = 0;
#pragma unroll
    for (int c = 0; c < IG_MAX_CANDS; c++) { if (c >= n_cands) t[c] = 0; tiles_all += t[c]; n_nonempty += t[c] > 0; }
    const int spare = grid - n_nonempty;
    int b0 = 0;
    *first = 0; *count = 0; *tiles = 0; *cand = -1;
#pragma unroll
    for (int c = 0; c < IG_MAX_CANDS; c++) {
        if (t[c] == 0) continue;
        const int nb = 1 + (int)(((long long)spare * t[c]) / tiles_all);
        const bool hit = k >= 0 ? (c == k) : (blk >= b0 && blk < b0 + nb);
        if (hit) { *first = b0; *count = nb; *tiles = t[c]; *cand = c; }
        b0 += nb;
    }
}
struct __align__(16) FlatRec {   // 64 B
    int pos, start_bp, len_ori; float watson; float crick; int val; float cur_s; int cur_dp;
    int rjc, flags; double t_cur; int ri; unsigned m; int pad[2];
};                               // flags: 1 same contig now, 2 current term deferred, 4 the row's contig is circular

// one selected contact (row end ci / class cls_r, column col) as the evaluation kernels need it; m = uniq slots to look at
// (class-pair table, already restricted to the scored slots); returns with x.m == 0 when nothing is left to evaluate
__device__ __forceinline__ void make_flat_rec(FlatRec& x, unsigned m, int col, int val, int ri, const CoordRec& ci, int cls_r,
                                              const CoordRec& cj, int rjc, const Params& p, double l10v, double inter_const, float mbar,
                                              const float* __restrict__ exz_tab, const unsigned* __restrict__ g_farok, float far_s,
                                              int far_dp, const SubX* __restrict__ subx, const int* __restrict__ clen) {
    x.rjc = rjc;
    x.pos = cj.pos; x.val = val; x.ri = ri;
    x.cur_s = fabsf(ci.dist - cj.dist);
    x.cur_dp = abs(ci.pos - cj.pos);
    const bool cur_same = ci.id_c == cj.id_c;
    if (m && cur_same && ci.s_tot == 0 && x.cur_s >= far_s && x.cur_dp >= far_dp)
        m &= ~__ldg(&g_farok[cls_r * IG_MAX_CLS + (rjc >> IG_CLS_SHIFT)]);
    if (m) {
        const SubX sx = subx[col];
        x.start_bp = sx.start_bp; x.len_ori = sx.len_ori; x.watson = sx.watson; x.crick = sx.crick;
        const double ob = (double)val;
        x.flags = (cur_same ? 1 : 0) | (ci.s_tot != 0 ? 4 : 0);
        x.t_cur = 0.0;
        if (!cur_same) x.t_cur = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + inter_const;
        else if (ci.s_tot != 0) x.t_cur = contact_term(ci, cj, clen[col], ob, 0.0, p, l10v, mbar, exz_tab);
        else if (!((x.cur_s > 0.0f) && (x.cur_s < p.d_max))) x.t_cur = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + (double)exz_tab[x.cur_dp] * LOG10E_F;
        else x.flags |= 2;
        x.pad[0] = 0; x.pad[1] = 0;
    }
    x.m = m;
}

__global__ void __launch_bounds__(IG_THREADS, IG_SCORE_CTAS_PER_SM)
k_pick(const int2* __restrict__ cv, const CoordRec* __restrict__ coord, const int* __restrict__ clen, DevScalars* sc,
       const IgDescriptor* __restrict__ desc_g, const int* __restrict__ rowidx, int ns, int* __restrict__ row_cnt,
       int* __restrict__ flat_cnt, size_t chunk_stride, int* __restrict__ part_c, FlatRec* __restrict__ flat, size_t flat_stride,
       float mbar, const float* __restrict__ exz_tab, const IgClassTab* __restrict__ clstab, const SubX* __restrict__ subx,
       const RowInfo* __restrict__ rinfo) {
    TL(15);
    TLP_DECL();
    const int k = blockIdx.y;
    if (k >= sc->n_cands) return;
    __shared__ int s_sel, s_read;
    const CandInfo ci_k = sc->ci[k];
    const int n_items = ci_k.n_rows * IG_PICK_PARTS;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wg = blockIdx.x * IG_WARPS_PER_BLOCK + w, nw = gridDim.x * IG_WARPS_PER_BLOCK;
    if (threadIdx.x == 0) { s_sel = 0; s_read = 0; }
    __syncthreads();
    if ((int)blockIdx.x * IG_WARPS_PER_BLOCK < n_items) {
        const Params p = sc->p;
        const double l10v = sc->log10_vinter;
        const double inter_const = (double)p.v_inter * LOG10E_F;
        const unsigned allmask = (1u << desc_g[k].n_uniq) - 1u;
        const unsigned* g_mask = clstab[k].mask;
        const unsigned* g_farok = clstab[k].farok;
        const float far_s = clstab[k].far_s;
        const int far_dp = clstab[k].far_dp;
        const int* my_idx = rowidx + (size_t)k * ns;
        FlatRec* my_flat = flat + (size_t)k * flat_stride;
        int* my_cnt = flat_cnt + (size_t)k * chunk_stride;
        TLP(8);   // prologue
        int sel_w = 0, read_w = 0;
        for (int it = wg; it < n_items; it += nw) {
            const int ri = it / IG_PICK_PARTS, part = it - ri * IG_PICK_PARTS;
            const RowInfo info = rinfo[(size_t)k * ns + ri];
            const CoordRec ci = info.ci;
            const unsigned* mrow = g_mask + info.cls * IG_MAX_CLS;
            const long long b = info.b, e = info.b + info.n;
            int row_sel = 0;
            for (long long q0 = b + 32 * part; q0 < e; q0 += 32 * IG_PICK_PARTS) {
                const long long q = q0 + lane;
                FlatRec x;
                x.m = 0;
                if (q < e) {
                    const int2 c = __ldg(&cv[q]);
                    const CoordRec cj = coord[c.x];
                    if ((cj.id_c == ci_k.id_a || cj.id_c == ci_k.id_b) && contact_selected(ci, cj, c.y, ci_k)) {
                        row_sel++;
                        const int rjc = my_idx[c.x];
                        make_flat_rec(x, __ldg(&mrow[rjc >> IG_CLS_SHIFT]) & allmask, c.x, c.y, ri, ci, info.cls, cj, rjc, p, l10v,
                                      inter_const, mbar, exz_tab, g_farok, far_s, far_dp, subx, clen);
                    }
                }
                const unsigned bal = __ballot_sync(0xffffffffu, x.m != 0);
                const long long slot0 = info.seg + (q0 - b);   // this chunk's 32 list slots
                if (x.m) my_flat[slot0 + __popc(bal & ((1u << lane) - 1))] = x;
                if (lane == 0) my_cnt[slot0 >> 5] = __popc(bal);
            }
            row_sel = __reduce_add_sync(0xffffffffu, row_sel);
            if (lane == 0 && row_sel) atomicAdd(&row_cnt[(size_t)k * ns + ri], row_sel);   // zeroed by k_rows_small
            sel_w += row_sel;
            if (part == 0) read_w += info.n;
        }
        TLP(9);   // chunk loop
        if (lane == 0 && (sel_w | read_w)) { atomicAdd(&s_sel, sel_w); atomicAdd(&s_read, read_w); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        part_c[PART_IDX(k, 2, 0, gridDim.x, blockIdx.x)] = s_sel;
        part_c[PART_IDX(k, 2, 1, gridDim.x, blockIdx.x)] = s_read;
    }
}

#define IG_FLAT_ITEMS 2   // smaller slot groups until every warp of a candidate's blocks has this many items
// LIST = false: the flat list of small levels (rows own whole 32-contact chunks, per-chunk counts, fixed order, double sums);
// LIST = true : the pick list of the streaming path (k_stream appends in arbitrary order; sc->flat_segtotal[k] = number of
//               records; fixed-point sums, see acc_add).
template <bool LIST>
__global__ void __launch_bounds__(IG_THREADS, IG_SCORE_CTAS_PER_SM)
k_eval_flat(const DevScalars* __restrict__ sc, const IgDescriptor* __restrict__ desc_g, int ns, const int* __restrict__ flat_cnt,
            size_t chunk_stride, const FlatRec* __restrict__ flat, size_t flat_stride, const RowMut* __restrict__ table,
            const int* __restrict__ table_len, float mbar, const float* __restrict__ exz_tab, double* __restrict__ part_nz,
            const IgClassTab* __restrict__ clstab) {
    TL(6);
    TLP_DECL();
    extern __shared__ double acc_s[];                 // [IG_N_OPS][IG_THREADS]
    __shared__ double red[IG_WARPS_PER_BLOCK][IG_N_OPS];
    __shared__ QEnt queue[IG_WARPS_PER_BLOCK][IG_QCAP];
    // The blocks of ONE grid are dealt to the candidates in proportion to their number of chunks (a candidate in
    // two long contigs has many times the contacts of one in two short ones: equal shares would wait for the
    // largest); inside a candidate the items = (chunk, group of gs uniq slots) are strided over its warps.
    const int n_cands = sc->n_cands;
    int k = -1, b_first = 0, n_blocks_k = 0, tiles_k = 0;
    flat_block_range(sc, n_cands, (int)gridDim.x, -1, (int)blockIdx.x, &b_first, &n_blocks_k, &tiles_k, &k);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = lane; i < IG_N_OPS; i += 32) red[w][i] = 0.0;   // (all-zero bits: also the fixed-point zero)
    __syncwarp();
    if (LIST && k >= 0 && !sc->use_stream[k]) k = -1;   // (cannot happen: candidates scored by k_score leave no picks)
    if (k >= 0) {
    const int n_recs = LIST ? sc->flat_segtotal[k] : 0;
    const int nw = n_blocks_k * IG_WARPS_PER_BLOCK;
    int gs = IG_N_OPS;
    while (gs > 3 && tiles_k * (IG_N_OPS / gs) < IG_FLAT_ITEMS * nw) gs >>= 1;
    const int ng = IG_N_OPS / gs;
    const int n_items = tiles_k * ng;
    const int wg = ((int)blockIdx.x - b_first) * IG_WARPS_PER_BLOCK + w;
    for (int u = 0; u < IG_N_OPS; u++) acc_s[u * IG_THREADS + threadIdx.x] = 0.0;
    const Params p = sc->p;
    const double l10v = sc->log10_vinter;
    const double inter_const = (double)p.v_inter * LOG10E_F;
    double* my_acc = acc_s + threadIdx.x;
    QEnt* myq = queue[w];
    int qn = 0;
    unsigned touched = 0;
    const int n_uniq = desc_g[k].n_uniq;
    const int* cnt = flat_cnt + (size_t)k * chunk_stride;
    const FlatRec* my_flat = flat + (size_t)k * flat_stride;
    const RowMut* tab = table + (size_t)k * IG_N_OPS * ns;
    const int* tlen = table_len + (size_t)k * IG_N_OPS * ns;
    const IgMotion* g_mot = clstab[k].mot;
    TLP(12);  // prologue
    for (int it = wg; it < n_items; it += nw) {
        const int tile = it / ng, grp = it - tile * ng;
        const int u0 = grp * gs;
        if (u0 >= n_uniq) continue;
        const unsigned gmask = ((1u << gs) - 1u) << u0;
        unsigned m = 0;
        Ctc x;
        x.pos = 0; x.start_bp = 0; x.len_ori = 0; x.watson = 0.f; x.crick = 0.f; x.val = 0; x.cur_s = 0.f; x.cur_dp = 0;
        x.rjc = 0; x.t_cur = 0.0; x.flags = 0;
        int ri = 0;
        float row_s_tot = 0.f;
        if (lane < (LIST ? min(32, n_recs - (tile << 5)) : __ldg(&cnt[tile]))) {
            const FlatRec r = my_flat[((size_t)tile << 5) + lane];
            x.pos = r.pos; x.start_bp = r.start_bp; x.len_ori = r.len_ori; x.watson = r.watson; x.crick = r.crick; x.val = r.val;
            x.cur_s = r.cur_s; x.cur_dp = r.cur_dp; x.rjc = r.rjc; x.t_cur = r.t_cur; x.flags = r.flags;
            ri = r.ri;
            m = r.m & gmask;
            row_s_tot = (r.flags & 4) ? 1.0f : 0.0f;   // eval_pair only asks whether the row's contig is circular
        }
        const unsigned um = __reduce_or_sync(0xffffffffu, m);
        if (!um) continue;
        unsigned chg = 0;
        RowMut a_nxt = tab[(size_t)(__ffs(um) - 1) * ns + ri];   // row-end entry, fetched one mutation ahead
#pragma unroll 1
        for (unsigned uw = um; uw; uw &= uw - 1) {
            const int u = __ffs(uw) - 1;
            const RowMut a = a_nxt;
            const unsigned rest = uw & (uw - 1);
            if (rest) a_nxt = tab[(size_t)(__ffs(rest) - 1) * ns + ri];
            float s_m = 0.f; int dp_m = 0; bool push = false;
            if ((m >> u) & 1u) {
                double add;
                if (eval_pair(x, u, a, g_mot, row_s_tot, p, l10v, inter_const, mbar, exz_tab, tab, tlen, ns, s_m, dp_m, push, add)) {
                    chg |= 1u << u;
                    acc_add<LIST>(&my_acc[u * IG_THREADS], add);
                }
            }
            queue_push<LIST>(push, s_m, dp_m, 1u << u, x.val, myq, qn, my_acc, p, l10v, exz_tab);
        }
        queue_push<LIST>((x.flags & 2) && chg, x.cur_s, x.cur_dp, chg | IG_QSUB, x.val, myq, qn, my_acc, p, l10v, exz_tab);
        touched |= __reduce_or_sync(0xffffffffu, chg);
    }
    TLP(13);  // items
    if (qn > 0) { eval_queue<LIST>(myq, qn, my_acc, p, l10v, exz_tab); }
    __syncwarp();
    for (unsigned tw = touched; tw; tw &= tw - 1) {
        const int us = __ffs(tw) - 1;
        if (LIST) {
            long long v = *reinterpret_cast<long long*>(&my_acc[us * IG_THREADS]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) *reinterpret_cast<long long*>(&red[w][us]) = v;
        } else {
            const double v = warp_sum(my_acc[us * IG_THREADS]);
            if (lane == 0) red[w][us] = v;
        }
    }
    TLP(14);  // final flush + reductions
    }
    __syncthreads();
    if (k >= 0 && threadIdx.x < 25) {   // k_finalize reads candidate k's partials from its own block range only
        if (LIST) {   // int64 fixed-point partials (bit pattern stored in the double array; k_finalize adds them as integers)
            long long v = 0;
            if (threadIdx.x < IG_N_OPS) for (int ww = 0; ww < IG_WARPS_PER_BLOCK; ww++) v += *reinterpret_cast<long long*>(&red[ww][threadIdx.x]);
            *reinterpret_cast<long long*>(&part_nz[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)]) = v;
        } else {
            double v = 0.0;
            if (threadIdx.x < IG_N_OPS) for (int ww = 0; ww < IG_WARPS_PER_BLOCK; ww++) v += red[ww][threadIdx.x];
            part_nz[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// STREAMING scoring path of large levels (ig_config.rigid_pruning != 0): one pass over the affected rows' contacts that
// touches 8 bytes per contact and NOTHING else for the contacts that cannot change:
//   * (col, val) pairs with 128-bit loads, two contacts per lane (streamed: evict-first);
//   * is the column in one of the <= 2 affected contigs?  one bit per sub-fragment, the candidate's bitmap staged in
//     SHARED memory (NS / 8 bytes; written by k_rows_write) -- half of a 1 Gb level's contacts are trans/noise contacts
//     and stop here;
//   * the others read 2 bytes of cls16[col] = rigid-motion class + position relative to the slice windows: slice
//     membership (window_selected) and the class-pair bit table (shared memory) say whether ANY mutation can change the
//     contact's term.  With rigid pruning only contacts that cross a breakpoint (or join two contigs) do: a few per cent;
//   * those PICKS get their record built (coordinate gathers, current term) and are appended to the candidate's list
//     (warp-aggregated atomic); k_eval_flat<true> evaluates the list with order-independent fixed-point sums.
// Per row the number of selected contacts goes to row_cnt (last-block quirk of k_finalize), per block the counters to
// part_c.  Candidates that involve a circular contig (every pair may change) are left to k_score.
__global__ void __launch_bounds__(IG_THREADS, 4)
k_stream(const int2* __restrict__ cv, const CoordRec* __restrict__ coord, const int* __restrict__ clen, DevScalars* sc,
         const IgDescriptor* __restrict__ desc_g, const int* __restrict__ rowidx, int ns, int* __restrict__ row_cnt,
         const unsigned* __restrict__ bitmap, int bitmap_words, const unsigned short* __restrict__ cls16,
         int* __restrict__ part_c, FlatRec* __restrict__ list, size_t list_cap, float mbar, const float* __restrict__ exz_tab,
         const IgClassTab* __restrict__ clstab, const SubX* __restrict__ subx, const RowInfo* __restrict__ rinfo) {
    TL(15);
    const int k = blockIdx.y;
    if (k >= sc->n_cands) return;
    if (!sc->use_stream[k]) return;   // k_score writes this candidate's counters
    extern __shared__ unsigned s_bits[];               // [bitmap_words]
    __shared__ unsigned s_mask[IG_MAX_CLS * IG_MAX_CLS];
    __shared__ int s_sel, s_read;
    const CandInfo ci_k = sc->ci[k];
    const int n_rows = ci_k.n_rows;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wg = blockIdx.x * IG_WARPS_PER_BLOCK + w, nw = gridDim.x * IG_WARPS_PER_BLOCK;
    if (threadIdx.x == 0) { s_sel = 0; s_read = 0; }
    // a candidate with few rows (mid-assembly contigs) cuts each row into `parts` interleaved sets of 64-contact trips, one
    // warp each, so that its critical path is one trip and not a whole row
    const int parts = n_rows * 8 <= nw ? 8 : (n_rows * 4 <= nw ? 4 : (n_rows * 2 <= nw ? 2 : 1));
    const int n_items = n_rows * parts;
    if ((int)blockIdx.x * IG_WARPS_PER_BLOCK < n_items) {
        const unsigned* gb = bitmap + (size_t)k * bitmap_words;
        for (int i = threadIdx.x; i < bitmap_words; i += blockDim.x) s_bits[i] = gb[i];
        const unsigned allmask = (1u << desc_g[k].n_uniq) - 1u;
        for (int i = threadIdx.x; i < IG_MAX_CLS * IG_MAX_CLS; i += blockDim.x) s_mask[i] = clstab[k].mask[i] & allmask;
    }
    __syncthreads();
    if ((int)blockIdx.x * IG_WARPS_PER_BLOCK < n_items) {
        const Params p = sc->p;
        const double l10v = sc->log10_vinter;
        const double inter_const = (double)p.v_inter * LOG10E_F;
        const unsigned* g_farok = clstab[k].farok;
        const float far_s = clstab[k].far_s;
        const int far_dp = clstab[k].far_dp;
        const int* my_idx = rowidx + (size_t)k * ns;
        const unsigned short* my_cls = cls16 + (size_t)k * ns;
        FlatRec* my_list = list + (size_t)k * list_cap;
        int sel_w = 0, read_w = 0;
        // software pipeline: the NEXT item's row record and the NEXT trip's contacts are in flight while this trip is classified
        RowInfo info_nxt;
        if (wg < n_items) info_nxt = rinfo[(size_t)k * ns + wg / parts];
        for (int it = wg; it < n_items; it += nw) {
            const int ri = it / parts, part = it - ri * parts;
            const RowInfo info = info_nxt;
            if (it + nw < n_items) info_nxt = rinfo[(size_t)k * ns + (it + nw) / parts];
            const CoordRec ci = info.ci;
            const unsigned* mrow = s_mask + info.cls * IG_MAX_CLS;
            const unsigned fr = window_flags(ci.pos, ci_k);
            const long long b = info.b, e = info.b + info.n;
            int row_sel = 0;
            const long long k_first = (b & ~1LL) + 64 * part, k_step = 64 * parts;
            int4 c2_nxt = make_int4(0, 0, 0, 0);
            if (k_first + 2 * lane < e) c2_nxt = __ldcs(reinterpret_cast<const int4*>(cv + k_first + 2 * lane));
            for (long long k0 = k_first; k0 < e; k0 += k_step) {
                const long long kk = k0 + 2 * lane;
                const int4 c2 = c2_nxt;
                c2_nxt = make_int4(0, 0, 0, 0);
                if (kk + k_step < e) c2_nxt = __ldcs(reinterpret_cast<const int4*>(cv + kk + k_step));
                unsigned m0 = 0, m1 = 0;
                if (kk >= b && kk < e && c2.y > 0 && ((s_bits[c2.x >> 5] >> (c2.x & 31)) & 1u)) {
                    const unsigned cb = my_cls[c2.x];
                    if (window_selected(fr, cb >> 8)) { row_sel++; m0 = mrow[cb & 31u]; }
                }
                if (kk + 1 < e && c2.w > 0 && ((s_bits[c2.z >> 5] >> (c2.z & 31)) & 1u)) {
                    const unsigned cb = my_cls[c2.z];
                    if (window_selected(fr, cb >> 8)) { row_sel++; m1 = mrow[cb & 31u]; }
                }
                // picks (rare): build the record, append it to the candidate's list
#pragma unroll
                for (int half = 0; half < 2; half++) {
                    const unsigned m = half ? m1 : m0;
                    if (!__any_sync(0xffffffffu, m != 0)) continue;
                    FlatRec x;
                    x.m = 0;
                    if (m) {
                        const int col = half ? c2.z : c2.x;
                        make_flat_rec(x, m, col, half ? c2.w : c2.y, ri, ci, info.cls, coord[col], my_idx[col], p, l10v, inter_const,
                                      mbar, exz_tab, g_farok, far_s, far_dp, subx, clen);
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, x.m != 0);
                    if (!bal) continue;
                    int base = 0;
                    if (lane == 0) base = atomicAdd(&sc->flat_segtotal[k], __popc(bal));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (x.m) {
                        const size_t slot = (size_t)base + __popc(bal & ((1u << lane) - 1));
                        if (slot < list_cap) my_list[slot] = x;
                        else sc->list_overflow = 1;
                    }
                }
            }
            row_sel = __reduce_add_sync(0xffffffffu, row_sel);
            if (lane == 0) {   // (zeroed by k_rows_write)
                if (parts == 1) row_cnt[(size_t)k * ns + ri] = row_sel;
                else if (row_sel) atomicAdd(&row_cnt[(size_t)k * ns + ri], row_sel);
            }
            sel_w += row_sel;
            if (part == 0) read_w += info.n;
        }
        if (lane == 0 && (sel_w | read_w)) { atomicAdd(&s_sel, sel_w); atomicAdd(&s_read, read_w); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        part_c[PART_IDX(k, 2, 0, gridDim.x, blockIdx.x)] = s_sel;
        part_c[PART_IDX(k, 2, 1, gridDim.x, blockIdx.x)] = s_read;
    }
}

__device__ void select_step(DevScalars* sc, const IgDescriptor* __restrict__ desc_g);
