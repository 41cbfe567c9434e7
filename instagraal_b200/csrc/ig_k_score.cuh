// instagraal_b200 -- scoring: slice rule, row-end table + zero terms, evaluation queue, the row-per-warp scoring kernel.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// slice_sp_mat membership of one contact (KA:557-606, incl. the precedence quirk Q11 and dat>0)
__device__ __forceinline__ bool contact_selected(const CoordRec& ci, const CoordRec& cj, int val, const CandInfo& c) {
    bool sel;
    if ((cj.id_c == ci.id_c) && c.same && (c.is_circ == 0)) {
        const int x = min(ci.pos, cj.pos), y = max(ci.pos, cj.pos);
        sel = ((x <= c.down_a) && (y >= c.up_a)) || ((y >= c.up_b) && (x <= c.down_b));
    } else {
        sel = ((!c.same) && (cj.id_c == c.id_a)) || (cj.id_c == c.id_b);
    }
    return sel && (val > 0);
}

struct RowMut { float dist; int id_c; int pos; float s_tot; };  // one sub-fragment under one mutation

// transposed partial layout: part[(k * n_slots + slot) * n_blocks + block]
#define PART_IDX(k, nslots, slot, nblocks, blk) ((((size_t)(k) * (nslots) + (slot)) * (nblocks)) + (blk))

// K8a: mutated coordinates of every affected sub-fragment under every scored mutation, evaluated
//      ONCE per (row, mutation) (replaces fill_vect_dist x24, KA:3699-3760) + the zero terms
//      (eval_all_likelihood_on_zero_1st, KA:3919-4002) restricted to the affected contigs.
//      Block (25 warps) per tile of 32 affected rows (lane = row), warp w = uniq slot w, warp 24 = the current state.
#define IG_PRE_THREADS (25 * 32)
__global__ void __launch_bounds__(IG_PRE_THREADS)
k_precompute(const CoordRec* __restrict__ coord, const int* __restrict__ clen, const FragRec* __restrict__ live,
             const SubRec* __restrict__ sub, const DevScalars* __restrict__ sc, const IgDescriptor* __restrict__ desc_g,
             const int* __restrict__ rows, int ns, RowMut* __restrict__ table, int* __restrict__ table_len, float mbar,
             double* __restrict__ part_z,  // [cand][25][gridDim.x]
             int* __restrict__ part_i)     // [cand][25][gridDim.x]
{
    TL(5);
    const int k = blockIdx.y;
    const int n_rows = sc->ci[k].n_rows;
    if (k >= sc->n_cands) return;
    if ((int)blockIdx.x * 32 >= n_rows) {   // no tile for this block
        if (threadIdx.x < 25) {
            part_z[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = 0.0;
            part_i[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = 0;
        }
        return;
    }
    __shared__ IgDescriptor d;
    __shared__ double red[25];   // warp w owns uniq slot w (warp 24: the current state)
    __shared__ int redi[25];
    {
        const int* src = reinterpret_cast<const int*>(desc_g + k);
        int* dst = reinterpret_cast<int*>(&d);
        for (int i = threadIdx.x; i < (int)(sizeof(IgDescriptor) / 4); i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x < 25) { red[threadIdx.x] = 0.0; redi[threadIdx.x] = 0; }
    __syncthreads();
    const Params p = sc->p;
    const int n_uniq = d.n_uniq;
    const int lane = threadIdx.x & 31, slot = threadIdx.x >> 5;
    const int* my_rows = rows + (size_t)k * ns;
    // a block takes tiles of 32 rows (lane = row); warp w evaluates uniq slot w for the tile, so the op is
    // warp-uniform (no divergence between the 24 move functions) and the table writes are coalesced
    if (slot < n_uniq || slot == 24) {
        for (int tile = blockIdx.x; tile * 32 < n_rows; tile += gridDim.x) {
            const int ri = tile * 32 + lane;
            double z = 0.0;
            int ia = 0;
            if (ri < n_rows) {
                const int r = my_rows[ri];
                if (slot < 24) {
                    const SubRec si = sub[r];
                    const Frag fi = live[si.parent].f;
                    const Frag fm = ig_eval_op(d, d.uniq[slot], fi, si.parent);
                    int len;
                    const CoordRec c = coords_of(fm, si, &len);
                    RowMut m; m.dist = c.dist; m.id_c = c.id_c; m.pos = c.pos; m.s_tot = c.s_tot;
                    const size_t ti = ((size_t)k * IG_N_OPS + slot) * ns + ri;
                    table[ti] = m; table_len[ti] = len;
                    if (c.pos == 0) ia = intra_pairs(len);
                    z = zero_term(c.pos, len, c.s_tot, p, mbar);
                } else {
                    const CoordRec ci = coord[r];
                    const int len = clen[r];
                    if (ci.pos == 0) ia = intra_pairs(len);
                    z = zero_term(ci.pos, len, ci.s_tot, p, mbar);
                }
            }
            z = warp_sum(z);
            ia = __reduce_add_sync(0xffffffffu, ia);
            if (lane == 0) { red[slot] += z; redi[slot] += ia; }   // tiles are visited in a fixed order
        }
    }
    __syncthreads();
    if (threadIdx.x < 25) {
        part_z[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = red[threadIdx.x];
        part_i[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = redi[threadIdx.x];
    }
}

// K8b: THE scoring kernel (replaces slice_sp_mat + host sort + prepare_sparse_call +
//      extract_sub_likelihood + eval_sub_likelihood).  grid = (G, n_cands).  Work item = (affected
//      CSR row, group of GS uniq slots); a warp takes one item at a time, its lanes stride the row's
//      contacts with coalesced 8-byte (col,val) loads.  The group size adapts to the amount of work
//      (GS = 24 when there are more rows than warps, down to 1 when a candidate has only a handful
//      of rows) so small assemblies still fill the 148 SMs.  Mutated coordinates of both endpoints
//      come from the table written by k_precompute (row side: warp-uniform broadcast loads; column
//      side: rowidx gather, contiguous across neighbouring contacts).
// The mutation loop is deliberately NOT unrolled and the expensive math is instantiated once: an
// unrolled 24-way body (x4 group sizes) measured 35 warps stalled on instruction fetch per issue
// (ncu "no_instruction", profiles/r1_ncu_k_score_G.txt) -- the kernel has to fit the I-cache.
// Per-thread per-slot accumulators live in shared memory ([slot][thread], conflict-free).
//
// Divergence: for most (contact, mutation) pairs the term is cheap -- bit-identical to the current
// state's term, or the constant inter-contig / out-of-range floor -- and only a few lanes of a warp
// need powf + f64 log10 (ncu: 11 of 32 lanes active on average).  Those evaluations are therefore
// QUEUED per warp in shared memory and executed 32 at a time with all lanes busy; the result is
// added to the executing lane's accumulator (only the sum over lanes matters; the order is fixed,
// hence deterministic).
struct __align__(16) QEnt { float s; int dp; unsigned mask; int val; };  // 16 B; mask bit 31: subtract
#define IG_QCAP 64
#define IG_QSUB 0x80000000u

// term of a linear-contig contact at 0 < s < d_max WITHOUT the part that depends on the observed count only
// (it cancels in t_mut - t_cur)
// Accumulation flavours.  FIXED = false: per-thread double sums, reduced in a fixed order (deterministic because the work
// of a thread is fixed).  FIXED = true (streaming path of large levels, whose pick list is appended in arbitrary order):
// every term is rounded to a 2^-32 fixed-point int64 first, so the total is EXACT integer arithmetic and independent of
// the order -- run-to-run deterministic without fixing who evaluates what (rounding error < 1.2e-10 per term).
#define IG_FIX_SCALE 4294967296.0
template <bool FIXED>
__device__ __forceinline__ void acc_add(double* __restrict__ slot, double t) {
    if (FIXED) *reinterpret_cast<long long*>(slot) += __double2ll_rn(t * IG_FIX_SCALE);
    else *slot += t;
}
template <bool FIXED>
__device__ __noinline__ void eval_queue(const QEnt* __restrict__ q, int n, double* __restrict__ my_acc, const Params& p,
                                        double l10v, const float* __restrict__ exz_tab) {
    const int lane = threadIdx.x & 31;
    if (lane < n) {
        const QEnt e = q[lane];
        const float exf = fmaxf((p.d == 2.0f) ? (p.c1 * powf_pos(e.s, p.slope)) * p.fact
                                              : (p.c1 * powf_pos(e.s, p.slope) * expf((p.d - 2) / (powf_pos(e.s * p.lm / p.kuhn, 2.0f) + p.d))) * p.fact,
                                p.v_inter);  // rippe_contacts for 0 < s < d_max (KA:153-163)
        double t = pxl_term(exf, (double)e.val, 0.0, l10v, p.v_inter) + (double)exz_tab[e.dp] * LOG10E_F;
        if (e.mask & IG_QSUB) t = -t;
        for (unsigned m = e.mask & 0xffffffu; m; m &= m - 1) acc_add<FIXED>(&my_acc[(__ffs(m) - 1) * IG_THREADS], t);
    }
}
// (evaluating two entries per lane in batches of 64 -- two interleaved powf/log10 chains -- was tried: no gain on
//  small levels, 12 % slower on the 1 Gb workload through register pressure)

// one selected contact as the slot loop needs it (column end + current state)
struct Ctc { int pos, start_bp, len_ori; float watson, crick; int val; float cur_s; int cur_dp; int rjc; double t_cur; int flags; };
                                                                                 // flags: 1 same contig now, 2 current term deferred

// term of contact x under uniq slot u: returns false when it is bit-identical to the current state; otherwise
// `add` = t_u - t_cur for the cheap cases, or push = true (s_m, dp_m to be evaluated through the queue; add = -t_cur)
__device__ __forceinline__ bool eval_pair(const Ctc& x, int u, const RowMut a, const IgMotion* __restrict__ g_mot, float row_s_tot,
                                          const Params& p, double l10v, double inter_const, float mbar, const float* __restrict__ exz_tab,
                                          const RowMut* __restrict__ tab, const int* __restrict__ tlen, int ns,
                                          float& s_m, int& dp_m, bool& push, double& add) {
    const int4 mo4 = __ldg(reinterpret_cast<const int4*>(g_mot + (x.rjc >> IG_CLS_SHIFT) * IG_N_OPS + u));  // dbp, dsp, id_c, flip
    const bool m_same = a.id_c == mo4.z;
    const bool cur_same = x.flags & 1;
    const double ob = (double)x.val;
    double t = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + inter_const;  // different contigs: both expectations are v_inter
    if (m_same) {
        if (a.s_tot != 0) {  // circular contig (rare): mutated column end from the table, evaluated in place
            const int rj = x.rjc & ((1 << IG_CLS_SHIFT) - 1);
            const RowMut bm = tab[(size_t)u * ns + rj];
            CoordRec cim, cjm;
            cim.dist = a.dist; cim.id_c = a.id_c; cim.pos = a.pos; cim.s_tot = a.s_tot;
            cjm.dist = bm.dist; cjm.id_c = bm.id_c; cjm.pos = bm.pos; cjm.s_tot = bm.s_tot;
            t = contact_term(cim, cjm, tlen[(size_t)u * ns + rj], ob, 0.0, p, l10v, mbar, exz_tab);
        } else {
            // the column end under this mutation: start_bp and sub-position follow the class motion
            const int len_j = abs(x.len_ori);
            const bool fw = (x.len_ori > 0) != (mo4.w != 0);
            const int sb = mo4.w ? mo4.x - x.start_bp - len_j : x.start_bp + mo4.x;
            const float dj = __int2float_rn(sb) / 1000.0f + (fw ? x.watson : x.crick);  // KA:3751
            const int pj = mo4.w ? mo4.y - 1 - x.pos : x.pos + mo4.y;
            s_m = fabsf(a.dist - dj);
            dp_m = abs(a.pos - pj);
            if (cur_same && row_s_tot == 0 && s_m == x.cur_s && dp_m == x.cur_dp) return false;  // bit-identical inputs
            if (!((s_m > 0.0f) && (s_m < p.d_max)))
                t = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + (double)exz_tab[dp_m] * LOG10E_F;  // floor v_inter
            else { push = true; t = 0.0; }  // needs powf + log10: queue it
        }
    } else if (!cur_same) return false;  // two contigs before and after
    add = t - x.t_cur;  // t_cur = 0 while deferred
    return true;
}

// warp-collective append to the warp's queue of expensive evaluations; a full batch of 32 is evaluated at once
template <bool FIXED = false>
__device__ __forceinline__ void queue_push(bool push, float s, int dp, unsigned mask, int val, QEnt* __restrict__ myq, int& qn,
                                           double* __restrict__ my_acc, const Params& p, double l10v, const float* __restrict__ exz_tab) {
    const unsigned pm = __ballot_sync(0xffffffffu, push);
    if (!pm) return;
    const int lane = threadIdx.x & 31;
    if (push) {
        QEnt en; en.s = s; en.dp = dp; en.mask = mask; en.val = val;
        myq[qn + __popc(pm & ((1u << lane) - 1))] = en;
    }
    qn += __popc(pm);
    __syncwarp();
    if (qn >= 32) {
        eval_queue<FIXED>(myq, 32, my_acc, p, l10v, exz_tab);
        __syncwarp();
        if (lane < qn - 32) { const QEnt mv = myq[32 + lane]; myq[lane] = mv; }
        qn -= 32;
        __syncwarp();
    }
}

// The per-slot sums are DIFFERENCES to the current state: D[u] = sum over the selected contacts whose term
// changes under mutation u of (t_u - t_cur); contacts that do not change contribute nothing and are not
// evaluated at all (score[u] = Lnz_full(cur) + Lz[u] + D[u] is algebraically KA:4029-4046; the part of a term
// that depends on the observed count only cancels and is left out).
//   * Which (contact, mutation) pairs need a look at all is read from the candidate's class-pair bit table.
//   * The mutated coordinate of the COLUMN end is recomputed on the fly from its current start_bp / offsets and
//     the rigid motion of its class under the mutation (same float32 operations as fill_vect_dist, KA:3751, so
//     bit-identical to the reference's 24 coordinate copies) -- no dependent global load inside the slot loop;
//     the ROW end is warp-uniform and staged from the k_precompute table into shared memory once per item.
//   * A pair whose (same-contig flag, s, sub-fragment separation) is bit-identical to the current state is
//     skipped; the rest is either a cheap constant (other contig / outside (0, d_max)) or goes to the queue.
#define IG_GS_DIV 4       // split a row into slot groups while rows * groups < warps / IG_GS_DIV
#define IG_SPARSE_DIV 4   // deal (contact, mutation) pairs to the lanes when fewer than 32 / IG_SPARSE_DIV lanes are busy
__global__ void __launch_bounds__(IG_THREADS, IG_SCORE_CTAS_PER_SM)
k_score(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const CoordRec* __restrict__ coord,
        const int* __restrict__ clen, const DevScalars* __restrict__ sc, const IgDescriptor* __restrict__ desc_g,
        const int* __restrict__ rows, const int* __restrict__ rowidx, int ns, int* __restrict__ row_cnt,
        const RowMut* __restrict__ table, const int* __restrict__ table_len, float mbar, const float* __restrict__ exz_tab,
        double* __restrict__ part_nz,   // [cand][25][gridDim.x]  (24 uniq slots; slot 24 unused = 0)
        int* __restrict__ part_c,       // [cand][2][gridDim.x]   (contacts selected, contacts read)
        const IgClassTab* __restrict__ clstab, const SubX* __restrict__ subx, const RowInfo* __restrict__ rinfo,
        int2 split)                     // (slots per item, parts per row) forced by tests; (0, 0): chosen from the work
{
    TL(6);
    TLB();
    TLP_DECL();
    const int k = blockIdx.y;
    if (k >= sc->n_cands) return;
    if (sc->use_stream[k]) return;                    // scored by k_stream + k_eval_flat<true>
    extern __shared__ double acc_s[];                 // [IG_N_OPS][IG_THREADS]
    __shared__ double red[IG_WARPS_PER_BLOCK][25];
    __shared__ int redi[IG_WARPS_PER_BLOCK][2];
    __shared__ QEnt queue[IG_WARPS_PER_BLOCK][IG_QCAP];
    __shared__ RowMut s_row[IG_WARPS_PER_BLOCK][IG_N_OPS];
    __shared__ unsigned s_chg[IG_WARPS_PER_BLOCK][32];
    __shared__ int s_off[IG_WARPS_PER_BLOCK][32];
    const CandInfo ci_k = sc->ci[k];
    const int n_uniq = desc_g[k].n_uniq;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wg = blockIdx.x * IG_WARPS_PER_BLOCK + w, nw = gridDim.x * IG_WARPS_PER_BLOCK;
    // Work distribution: one warp per (affected row, group of gs uniq slots, part of the row); gs = 24 and one
    // part when there are more rows than warps, fewer slots per item and rows cut into `parts` interleaved
    // chunk sets when a candidate has few rows (yeast-scale assemblies), so that the grid stays occupied and
    // the longest row does not set the kernel's critical path.
    int gs = IG_N_OPS, parts = 1;
    const int want = nw / IG_GS_DIV;
    if (ci_k.n_rows < want) gs = (ci_k.n_rows * 4 >= want) ? 6 : ((ci_k.n_rows * 8 >= want) ? 3 : 1);
    if (ci_k.n_rows * (IG_N_OPS / gs) * 2 <= nw) parts = 2;
    if (ci_k.n_rows * (IG_N_OPS / gs) * 4 <= nw) parts = 4;
    if (split.x) { gs = split.x; parts = split.y; }
    const int ng = IG_N_OPS / gs;
    const int n_items = ci_k.n_rows * ng * parts;
    if ((int)blockIdx.x * IG_WARPS_PER_BLOCK >= n_items) {  // nothing for this block
        if (threadIdx.x < 25) part_nz[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = 0.0;
        if (threadIdx.x < 2) part_c[PART_IDX(k, 2, threadIdx.x, gridDim.x, blockIdx.x)] = 0;
        return;
    }
    const Params p = sc->p;
    const double l10v = sc->log10_vinter;
    const unsigned* g_mask = clstab[k].mask;    // small per-candidate tables: read through L1
    const unsigned* g_farok = clstab[k].farok;
    const IgMotion* g_mot = clstab[k].mot;
    const unsigned* g_rep = clstab[k].repmask;
    const unsigned* g_mem = clstab[k].members;
    const float far_s = clstab[k].far_s;
    const int far_dp = clstab[k].far_dp;
    // whole-row items (all 24 slots in one item): slots whose two classes undergo the same motions are evaluated once, through
    // their representative, and the result is credited to every member of the group (bit-identical terms)
    const bool dedup = gs == IG_N_OPS;
    if (lane < 25) red[w][lane] = 0.0;
    if (lane < 2) redi[w][lane] = 0;
    for (int u = 0; u < IG_N_OPS; u++) acc_s[u * IG_THREADS + threadIdx.x] = 0.0;  // kept zero between items (see the item epilogue)
    __syncwarp();
    const int* my_idx = rowidx + (size_t)k * ns;
    int* my_cnt = row_cnt + (size_t)k * ns;
    const RowMut* tab = table + (size_t)k * IG_N_OPS * ns;
    const int* tlen = table_len + (size_t)k * IG_N_OPS * ns;
    double* my_acc = acc_s + threadIdx.x;
    QEnt* myq = queue[w];
    RowMut* myrow = s_row[w];
    unsigned* mychg = s_chg[w];
    int* myoff = s_off[w];
    // (double)p.v_inter * LOG10E_F below: the constant term of a contact whose endpoints lie in different contigs
    // (KA:4348-4352) minus the ob part, written out at each use -- held in a variable it costs k_score spill slots
    TLP(0);   // block prologue
    for (int it = wg; it < n_items; it += nw) {
        TLB_ITEM();
        const int rg = it / parts, part = it - rg * parts;
        const int ri = rg / ng, g = rg - ri * ng;
        const int q_off = 32 * part, q_step = 32 * parts;
        const int u0 = g * gs;
        if (u0 >= n_uniq && g != 0) continue;
        const int u1 = min(u0 + gs, n_uniq);
        const unsigned gmask = (u1 > u0) ? (((1u << (u1 - u0)) - 1u) << u0) : 0u;
        const RowInfo info = rinfo[(size_t)k * ns + ri];
        const CoordRec ci = info.ci;
        const int cls_r = info.cls;
        const unsigned* mrow = g_mask + cls_r * IG_MAX_CLS;
        const long long b = info.b, e = info.b + info.n;
        __syncwarp();
        if (u0 + lane < u1) myrow[lane] = tab[(size_t)(u0 + lane) * ns + ri];
        __syncwarp();
        TLP(1);   // item set-up (row record, row-end table entries)
        int row_sel = 0;
        int qn = 0;  // warp-uniform queue fill
        unsigned touched = 0;  // slots (relative to u0) that received a term in this item
        // the (col, val) pair and the column's coordinates are fetched one chunk ahead
        // (only when whole rows are processed: short row parts gain nothing from it)
        const bool ahead = parts == 1;
        int2 c_nxt = make_int2(0, 0);
        CoordRec cj_nxt = ci;
        if (ahead && b + q_off + lane < e) { c_nxt = __ldg(&cv[b + q_off + lane]); cj_nxt = coord[c_nxt.x]; }
        for (long long q0 = b + q_off; q0 < e; q0 += q_step) {
            const long long q = q0 + lane;
            int2 c = c_nxt;
            CoordRec cj = cj_nxt;
            if (!ahead && q < e) { c = __ldg(&cv[q]); cj = coord[c.x]; }
            if (ahead && q + q_step < e) c_nxt = __ldg(&cv[q + q_step]);
            unsigned m = 0;
            Ctc x;
            x.pos = 0; x.start_bp = 0; x.len_ori = 0; x.watson = 0.f; x.crick = 0.f; x.val = 0; x.cur_s = 0.f; x.cur_dp = 0;
            x.rjc = 0; x.t_cur = 0.0; x.flags = 0;
            if (q < e) {
                if ((cj.id_c == ci_k.id_a || cj.id_c == ci_k.id_b) && contact_selected(ci, cj, c.y, ci_k)) {
                    row_sel++;
                    x.rjc = my_idx[c.x];
                    x.pos = cj.pos; x.val = c.y;
                    x.cur_s = fabsf(ci.dist - cj.dist);
                    x.cur_dp = abs(ci.pos - cj.pos);
                    const bool cur_same = ci.id_c == cj.id_c;
                    m = __ldg(&mrow[x.rjc >> IG_CLS_SHIFT]) & gmask;
                    // far beyond d_max before and after: every non-reflecting mutation leaves the floor term
                    if (m && cur_same && ci.s_tot == 0 && x.cur_s >= far_s && x.cur_dp >= far_dp)
                        m &= ~__ldg(&g_farok[cls_r * IG_MAX_CLS + (x.rjc >> IG_CLS_SHIFT)]);
                    if (m) {  // current-state term of the lanes that have something to evaluate
                        const SubX sx = subx[c.x];
                        x.start_bp = sx.start_bp; x.len_ori = sx.len_ori; x.watson = sx.watson; x.crick = sx.crick;
                        const double ob = (double)c.y;
                        if (!cur_same) x.t_cur = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + (double)p.v_inter * LOG10E_F;
                        else if (ci.s_tot != 0) x.t_cur = contact_term(ci, cj, clen[c.x], ob, 0.0, p, l10v, mbar, exz_tab);  // circular (rare)
                        else if (!((x.cur_s > 0.0f) && (x.cur_s < p.d_max))) x.t_cur = pxl_term(p.v_inter, ob, 0.0, l10v, p.v_inter) + (double)exz_tab[x.cur_dp] * LOG10E_F;
                        else x.flags |= 2;  // powf + log10: goes through the queue once, with the mask of changed slots
                        x.flags |= cur_same ? 1 : 0;
                    }
                }
            }
            if (ahead && q + q_step < e) cj_nxt = coord[c_nxt.x];
            // mr = the slots to EVALUATE (group representatives when dedup; u0 == 0 then), m = the slots to credit
            const int t_pair = cls_r * IG_MAX_CLS + (x.rjc >> IG_CLS_SHIFT);
            const unsigned mr = (dedup && m) ? (m & __ldg(&g_rep[t_pair])) : m;
            const unsigned um = __reduce_or_sync(0xffffffffu, mr);
            if (!um) continue;
            unsigned chg = 0;
            // number of (contact, mutation) pairs of this chunk
            const int n_pairs = __reduce_add_sync(0xffffffffu, __popc(mr));
            if (n_pairs * IG_SPARSE_DIV > __popc(um) * 32) {
                // DENSE: most lanes take part in most mutations -> loop over the mutations, lane = contact
#pragma unroll 1
                for (unsigned uw = um; uw; uw &= uw - 1) {
                    const int u = __ffs(uw) - 1;
                    float s_m = 0.f; int dp_m = 0; bool push = false;
                    unsigned mem = 1u << (u - u0);
                    if ((mr >> u) & 1u) {
                        double add;
                        if (eval_pair(x, u, myrow[u - u0], g_mot, ci.s_tot, p, l10v, (double)p.v_inter * LOG10E_F, mbar, exz_tab, tab, tlen, ns, s_m, dp_m, push, add)) {
                            if (dedup) mem = __ldg(&g_mem[t_pair * IG_N_OPS + u]) & m;
                            chg |= mem;
                            for (unsigned mm = mem; mm; mm &= mm - 1) my_acc[(__ffs(mm) - 1) * IG_THREADS] += add;
                        }
                    }
                    queue_push(push, s_m, dp_m, mem, x.val, myq, qn, my_acc, p, l10v, exz_tab);
                }
            } else {
                // SPARSE (long contigs: only the contacts that cross a breakpoint change): the pairs are dealt
                // densely to the lanes; the executing lane fetches the contact from its owner by shuffles
                int pre = __popc(mr);   // inclusive prefix over the lanes
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += y; }
                __syncwarp();
                mychg[lane] = 0; myoff[lane] = pre - __popc(mr);
                __syncwarp();
#pragma unroll 1
                for (int base = 0; base < n_pairs; base += 32) {
                    const int pi = base + lane;
                    const bool valid = pi < n_pairs;
                    int src = 0;
                    if (valid) {  // last lane whose exclusive offset is <= pi
#pragma unroll
                        for (int stp = 16; stp > 0; stp >>= 1) if (src + stp < 32 && myoff[src + stp] <= pi) src += stp;
                    }
                    const unsigned msrc = __shfl_sync(0xffffffffu, mr, src);
                    const unsigned mfull = __shfl_sync(0xffffffffu, m, src);
                    Ctc y;
                    y.pos = __shfl_sync(0xffffffffu, x.pos, src); y.start_bp = __shfl_sync(0xffffffffu, x.start_bp, src);
                    y.len_ori = __shfl_sync(0xffffffffu, x.len_ori, src); y.watson = __shfl_sync(0xffffffffu, x.watson, src);
                    y.crick = __shfl_sync(0xffffffffu, x.crick, src); y.val = __shfl_sync(0xffffffffu, x.val, src);
                    y.cur_s = __shfl_sync(0xffffffffu, x.cur_s, src); y.cur_dp = __shfl_sync(0xffffffffu, x.cur_dp, src);
                    y.rjc = __shfl_sync(0xffffffffu, x.rjc, src); y.t_cur = __shfl_sync(0xffffffffu, x.t_cur, src);
                    y.flags = __shfl_sync(0xffffffffu, x.flags, src);
                    float s_m = 0.f; int dp_m = 0; bool push = false;
                    int u = u0;
                    unsigned mem = 0;
                    if (valid) {
                        u = __fns(msrc, 0, pi - myoff[src] + 1);
                        mem = 1u << (u - u0);
                        double add;
                        if (eval_pair(y, u, myrow[u - u0], g_mot, ci.s_tot, p, l10v, (double)p.v_inter * LOG10E_F, mbar, exz_tab, tab, tlen, ns, s_m, dp_m, push, add)) {
                            if (dedup) mem = __ldg(&g_mem[(cls_r * IG_MAX_CLS + (y.rjc >> IG_CLS_SHIFT)) * IG_N_OPS + u]) & mfull;
                            atomicOr(&mychg[src], mem);
                            for (unsigned mm = mem; mm; mm &= mm - 1) my_acc[(__ffs(mm) - 1) * IG_THREADS] += add;
                        }
                    }
                    queue_push(push, s_m, dp_m, mem, y.val, myq, qn, my_acc, p, l10v, exz_tab);
                }
                __syncwarp();
                chg = mychg[lane];
            }
            // the deferred current-state terms, subtracted from every slot that changed
            queue_push((x.flags & 2) && chg, x.cur_s, x.cur_dp, chg | IG_QSUB, x.val, myq, qn, my_acc, p, l10v, exz_tab);
            touched |= __reduce_or_sync(0xffffffffu, chg);
        }
        TLP(2);   // contact loop
        if (qn > 0) { eval_queue<false>(myq, qn, my_acc, p, l10v, exz_tab); }
        __syncwarp();
        // fixed-order accumulation into this warp's slot sums (work items are visited in a fixed order); only
        // the slots that received a term are reduced, and their accumulators are put back to zero
        for (unsigned tw = touched; tw; tw &= tw - 1) {
            const int us = __ffs(tw) - 1;
            const double v = warp_sum(my_acc[us * IG_THREADS]);
            my_acc[us * IG_THREADS] = 0.0;
            if (lane == 0) red[w][u0 + us] += v;
        }
        if (g == 0) {
            row_sel = __reduce_add_sync(0xffffffffu, row_sel);
            if (lane == 0) {
                redi[w][0] += row_sel;
                if (parts > 1) { if (row_sel) atomicAdd(&my_cnt[ri], row_sel); if (part == 0) redi[w][1] += (int)(e - b); }
                else { my_cnt[ri] = row_sel; redi[w][1] += (int)(e - b); }
            }
        }
    }
    TLP(3);   // last queue flush + slot reductions of the items
    __syncthreads();
    TLP(4);   // waiting for the slowest warp of the block
    if (threadIdx.x < 25) {
        double v = 0.0;
        for (int ww = 0; ww < IG_WARPS_PER_BLOCK; ww++) v += red[ww][threadIdx.x];
        part_nz[PART_IDX(k, 25, threadIdx.x, gridDim.x, blockIdx.x)] = v;
    }
    if (threadIdx.x < 2) {
        int iv = 0;
        for (int ww = 0; ww < IG_WARPS_PER_BLOCK; ww++) iv += redi[ww][threadIdx.x];
        part_c[PART_IDX(k, 2, threadIdx.x, gridDim.x, blockIdx.x)] = iv;
    }
}
#define IG_SCORE_SMEM (IG_N_OPS * IG_THREADS * sizeof(double))
