// instagraal_b200 -- per-candidate setup: descriptor, cut fragments, rigid-motion class tables, ordered affected-row list.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// K2: per-candidate setup.  Thread 0 walks the candidates IN ORDER because extract_uniq_mutations
//     of candidate k reads the list_valid_insert left by get_bounds of candidate k-1 (quirk Q3).
__global__ void k_cand_setup(const FragRec* __restrict__ live, DevScalars* sc, IgDescriptor* desc, int n_bounds,
                             int first_flip_eject, const int* __restrict__ plan, int stream_mode) {
    TL(0);
    if (plan) {  // cycle mode: this step's {n_cands, fragment, candidates} come from the cycle plan (a step of <= IG_MAX_CANDS)
        const int* src = plan + (size_t)sc->step_idx * sc->plan_stride;
        if (threadIdx.x < 2 + IG_MAX_CANDS) (&sc->n_cands)[threadIdx.x] = src[threadIdx.x];
        __syncthreads();
    }
    // one lane per candidate: pivots and get_bounds in parallel; only the uniq lists chain through the
    // previous candidate's validity list (quirk Q3), which goes through shared memory
    __shared__ int sv[IG_MAX_CANDS + 1][12];
    const int k = threadIdx.x;
    const int n = sc->n_cands;
    const int a = sc->a;
    const Frag A = live[a].f;
    if (k < 12) sv[0][k] = sc->valid[k];
    Frag B = A;
    int b = a;
    if (k < n) {
        b = sc->cands[k];
        B = live[b].f;
        IgDescriptor& d = desc[k];
        d.a = a; d.b = b; d.max_id = sc->max_label;
        d.A = A; d.B = B;
        ig_get_bounds_positions(A, B, d.valid, d.cut_pos_up, d.cut_pos_down);
        for (int i = 0; i < 12; i++) sv[k + 1][i] = d.valid[i];
        for (int i = 0; i < IG_N_CUT; i++) { d.f_up[i] = -1; d.f_down[i] = -1; }
        // slice windows, KA:526-551 (sub-fragment units of the live scaffold)
        CandInfo& c = sc->ci[k];
        int pfa = A.sub_pos * (A.ori == 1) + (A.sub_pos - A.sub_len) * (A.ori == -1); if (pfa < 0) pfa = 0;
        int pfb = B.sub_pos * (B.ori == 1) + (B.sub_pos - B.sub_len) * (B.ori == -1); if (pfb < 0) pfb = 0;
        c.id_a = A.id_c; c.id_b = B.id_c; c.same = A.id_c == B.id_c; c.is_circ = A.circ;
        c.up_a = max(0, pfa - n_bounds - A.sub_len); c.down_a = min(A.sub_l_cont - 1, pfa + n_bounds + A.sub_len);
        c.up_b = max(0, pfb - B.sub_len); c.down_b = min(B.sub_l_cont - 1, pfb + B.sub_len);
        c.n_rows = 0; c.n_sub = 0; c.row_hi = -1;
        sc->ticket_cuts[k] = 0; sc->ticket_rows[k] = 0;
        // streaming scoring path: not for circular contigs (every class pair may change there: k_score's generic route),
        // and only for candidates of at most stream_mode affected rows (their picks must fit the list)
        const int rows_k = A.sub_l_cont + (A.id_c == B.id_c ? 0 : B.sub_l_cont);
        sc->use_stream[k] = (stream_mode && A.circ == 0 && B.circ == 0 && rows_k <= stream_mode) ? 1 : 0;
        if (stream_mode) sc->flat_segtotal[k] = 0;   // pick-list fill
    }
    if (stream_mode && k >= n && k < IG_MAX_CANDS) { sc->use_stream[k] = 0; sc->flat_segtotal[k] = 0; }
    __syncthreads();
    if (k < n) {
        IgDescriptor& d = desc[k];
        d.n_uniq = ig_uniq_mutations(A, B, sv[k], (k == 0) ? first_flip_eject : 0, d.uniq);
    }
    if (k < 12) sc->valid[k] = sv[n][k];  // state after the last candidate's get_bounds (CL:1854-1870)
    if (k == 0) { sc->ticket_fin = 0; sc->ticket_post = 0; }
}
// K3: cut fragments of get_bounds (KA:2255-2269), all candidates at once; the LAST block to finish a
//     candidate then evaluates every pivot of its descriptor (one thread).
__global__ void __launch_bounds__(256)
k_find_cuts(const FragRec* __restrict__ live, int nf, DevScalars* sc, IgDescriptor* desc, IgClassTab* __restrict__ clstab) {
    TL(1);
    // ONE pass over the scaffold for all candidates of the step (they share the visited fragment A, hence A's contig): a
    // fragment record is read once and tested against every candidate's cut positions
    const int n = sc->n_cands;
    __shared__ int is_last;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nf) {
        const Frag f = live[i].f;
        if (f.id_c == desc[0].A.id_c) {
            for (int k = 0; k < n; k++) {
                IgDescriptor& d = desc[k];
#pragma unroll
                for (int c = 0; c < IG_N_CUT; c++) {
                    if (f.pos == d.cut_pos_down[c]) d.f_down[c] = i;
                    if (f.pos == d.cut_pos_up[c]) d.f_up[c] = i;
                }
            }
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(&sc->ticket_cuts[0], 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    // the last block: warp k evaluates every pivot of candidate k's descriptor
    __threadfence();
    const int k = threadIdx.x >> 5;
    if (k < n) ig_build_descriptor_part(desc[k], [&](int j) { return live[j].f; }, threadIdx.x & 31);
    __syncthreads();
    // breakpoints of the rigid-motion classes (ig_moves.cuh): k_rows_write classifies the rows with them
    if (k < n && (threadIdx.x & 31) == 0) {
        const IgDescriptor& d = desc[k];
        IgClassTab& ct = clstab[k];
        int bpf[IG_MAX_BP + 2], bps[IG_MAX_BP], bpbs[2];
        ig_class_breakpoints(d, bpf, bps, bpf + IG_MAX_BP, bpbs);
        for (int j = 0; j < IG_MAX_BP; j++) ct.bp_sub[j] = bps[j];
        ct.bp_sub_b[0] = bpbs[0]; ct.bp_sub_b[1] = bpbs[1];
        ct.distinct_b = d.A.id_c != d.B.id_c; ct.id_b = d.B.id_c;
    }
}

// K4: rigid-motion classes of each candidate (ig_moves.cuh): one motion per (class, uniq slot) from a class
//     representative, then the class-pair bit table read by k_score.  One block per candidate, on the side
//     stream (only k_score needs the result).
__global__ void __launch_bounds__(IG_N_OPS * 32)
k_classes(const DevScalars* __restrict__ sc, const IgDescriptor* __restrict__ desc, IgClassTab* __restrict__ clstab, int rigid, float mbar) {
    TL(2);
    const int k = blockIdx.x;
    if (k >= sc->n_cands) return;
    __shared__ IgDescriptor d;
    __shared__ int s_bpf[IG_MAX_BP + 2], s_have[IG_MAX_CLS];
    __shared__ IgSig s_sig[IG_MAX_CLS][IG_N_OPS];
    {
        const int* src = reinterpret_cast<const int*>(desc + k);
        int* dst = reinterpret_cast<int*>(&d);
        for (int i = threadIdx.x; i < (int)(sizeof(IgDescriptor) / 4); i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x < IG_MAX_CLS) s_have[threadIdx.x] = 0;
    __syncthreads();
    IgClassTab& ct = clstab[k];
    if (threadIdx.x == 0) {
        int bps[IG_MAX_BP], bpbs[2];
        ig_class_breakpoints(d, s_bpf, bps, s_bpf + IG_MAX_BP, bpbs);
    }
    __syncthreads();
    const int n_uniq = d.n_uniq;
    {   // one uniq slot per warp pass (lanes = class representatives): no divergence between ops
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        int on_b = 0;
        const int pos = lane < IG_MAX_CLS ? ig_class_rep_pos(d, s_bpf, s_bpf + IG_MAX_BP, lane, &on_b) : -1;
        const int cls = pos < 0 ? -1 : (on_b ? IG_CLS_B0 + ig_class_count(s_bpf + IG_MAX_BP, 2, pos) : ig_class_count(s_bpf, IG_MAX_BP, pos));
        if (w == 0 && cls >= 0) s_have[cls] = 1;
        for (int u = w; u < n_uniq; u += (int)(blockDim.x >> 5)) {
            if (cls < 0) continue;
            const IgSig g = ig_class_signature(d, on_b, pos, d.uniq[u]);   // representatives of one class agree
            s_sig[cls][u] = g;
            IgMotion mo; mo.dbp = g.dbp; mo.dsp = g.dsp; mo.id_c = g.id_c; mo.flip = g.flip;
            ct.mot[cls * IG_N_OPS + u] = mo;
        }
    }
    __syncthreads();
    const int circ_a = d.A.circ, circ_b = d.B.circ;
    for (int t = threadIdx.x; t < IG_MAX_CLS * IG_MAX_CLS; t += blockDim.x) {
        const int c1 = t / IG_MAX_CLS, c2 = t - c1 * IG_MAX_CLS;
        unsigned m = 0xffffffu;
        if (s_have[c1] && s_have[c2]) {
            m = 0;
            const int cur_same = (c1 >= IG_CLS_B0) == (c2 >= IG_CLS_B0);
            const int cur_circ = c1 >= IG_CLS_B0 ? circ_b : circ_a;
            for (int u = 0; u < n_uniq; u++)
                if (ig_class_pair_changed(s_sig[c1][u], s_sig[c2][u], cur_same, cur_circ, rigid)) m |= 1u << u;
        }
        ct.mask[t] = m;
        unsigned fo = 0;
        if (s_have[c1] && s_have[c2])
            for (int u = 0; u < n_uniq; u++)
                if (ig_class_pair_far_ok(s_sig[c1][u], s_sig[c2][u])) fo |= 1u << u;
        ct.farok[t] = fo;
        // groups of slots with identical motions of both classes (ig_class_pair_same_motion): lowest slot = representative.
        // Only the row-per-warp kernel reads them: skipped for candidates that take the streaming path (this kernel sits
        // beside the row list on the step's critical path at mid-assembly; the grouping is a few thousand instructions).
        if (sc->use_stream[k]) continue;
        unsigned rep = 0, mem[IG_N_OPS];
#pragma unroll
        for (int u = 0; u < IG_N_OPS; u++) mem[u] = 0;
        if (s_have[c1] && s_have[c2] && !circ_a && !circ_b) {
            for (int u = 0; u < n_uniq; u++) {
                if (!((m >> u) & 1u)) continue;
                int r = -1;
                for (unsigned rr = rep; rr && r < 0; rr &= rr - 1) {
                    const int v = __ffs(rr) - 1;
                    if (ig_class_pair_same_motion(s_sig[c1][v], s_sig[c2][v], s_sig[c1][u], s_sig[c2][u])) r = v;
                }
                if (r < 0) { rep |= 1u << u; mem[u] = 1u << u; } else mem[r] |= 1u << u;
            }
        } else {
            rep = m;
            for (int u = 0; u < IG_N_OPS; u++) mem[u] = 1u << u;
        }
        ct.repmask[t] = rep;
        for (int u = 0; u < IG_N_OPS; u++) ct.members[t * IG_N_OPS + u] = mem[u];
    }
    // margin: twice the largest shift of any class under any non-reflecting mutation
    if (threadIdx.x < 32) {
        int mb = 0, ms = 0;
        for (int c = threadIdx.x; c < IG_MAX_CLS; c += 32)
            if (s_have[c])
                for (int u = 0; u < n_uniq; u++)
                    if (!s_sig[c][u].flip) { mb = max(mb, abs(s_sig[c][u].dbp)); ms = max(ms, abs(s_sig[c][u].dsp)); }
        mb = __reduce_max_sync(0xffffffffu, mb);
        ms = __reduce_max_sync(0xffffffffu, ms);
        if (threadIdx.x == 0) {
            const float d_max = sc->p.d_max;
            ct.far_s = d_max + 2.0f * (__int2float_ru(mb) / 1000.0f) + 1.0f;
            ct.far_dp = (int)ceilf(d_max / mbar) + 2 * ms + 2;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K5-7: ORDERED list of the CSR rows (sub-fragments) that belong to the <=2 affected contigs.
__device__ __forceinline__ bool row_affected(const CoordRec& c, const CandInfo& ci) { return c.id_c == ci.id_a || c.id_c == ci.id_b; }
// Position of a sub-fragment relative to the two slice windows of a same-linear-contig candidate (slice_sp_mat,
// KA:565-586): bit 0 = left of window A (pos < up_a), 1 = right of it (pos > down_a), 2 / 3 = the same for window B.
// A contact (i, j) is selected when, for one of the windows, the two ends are neither both left nor both right of it:
//     min(pos) <= down && max(pos) >= up   <=>   (flags_i & flags_j & 3) == 0   (resp. & 12)
__device__ __forceinline__ unsigned window_flags(int pos, const CandInfo& c) {
    if (!(c.same && c.is_circ == 0)) return 0u;
    return (pos < c.up_a ? 1u : 0u) | (pos > c.down_a ? 2u : 0u) | (pos < c.up_b ? 4u : 0u) | (pos > c.down_b ? 8u : 0u);
}
__device__ __forceinline__ bool window_selected(unsigned fi, unsigned fj) {
    const unsigned both = fi & fj;
    return ((both & 3u) == 0u) || ((both & 12u) == 0u);
}
// (large levels) ONE pass over the coordinates for all candidates of the step: a chunk of 1024 rows is read once and tested
// against every candidate's <= 2 affected contigs
__global__ void __launch_bounds__(IG_ROW_CHUNK)
k_rows_count(const CoordRec* __restrict__ coord, int ns, DevScalars* sc, int* __restrict__ chunk_cnt, int n_chunks) {
    TL(3);
    const int n = sc->n_cands;
    __shared__ int is_last, carry;
    __shared__ int wsum[32];
    __shared__ int s_ida[IG_MAX_CANDS], s_idb[IG_MAX_CANDS];
    if (threadIdx.x < n) { s_ida[threadIdx.x] = sc->ci[threadIdx.x].id_a; s_idb[threadIdx.x] = sc->ci[threadIdx.x].id_b; }
    __syncthreads();
    const int r = blockIdx.x * IG_ROW_CHUNK + threadIdx.x;
    const int idc = r < ns ? coord[r].id_c : -1;
    for (int k = 0; k < n; k++) {
        const bool f = r < ns && (idc == s_ida[k] || idc == s_idb[k]);
        const int cnt = __syncthreads_count(f);
        if (threadIdx.x == 0) chunk_cnt[k * n_chunks + blockIdx.x] = cnt;
    }
    if (threadIdx.x == 0) {
        __threadfence();
        is_last = (atomicAdd(&sc->ticket_rows[0], 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    // the last block to finish turns every candidate's chunk counts into exclusive offsets
    __threadfence();
    for (int k = 0; k < n; k++) {
        if (threadIdx.x == 0) carry = 0;
        __syncthreads();
        volatile int* c = chunk_cnt + k * n_chunks;
        for (int base = 0; base < n_chunks; base += blockDim.x) {
            const int i = base + threadIdx.x;
            const int v = i < n_chunks ? c[i] : 0;
            int x = v;
            const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
            if (lane == 31) wsum[w] = x;
            __syncthreads();
            if (w == 0) {
                int s2 = lane < (blockDim.x >> 5) ? wsum[lane] : 0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s2, o); if (lane >= o) s2 += y; }
                wsum[lane] = s2;
            }
            __syncthreads();
            const int excl = carry + (w ? wsum[w - 1] : 0) + x - v;
            if (i < n_chunks) c[i] = excl;
            __syncthreads();
            if (threadIdx.x == blockDim.x - 1) carry = excl + v;
            __syncthreads();
        }
        if (threadIdx.x == 0) sc->ci[k].n_rows = carry;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(IG_ROW_CHUNK)
k_rows_write(const CoordRec* __restrict__ coord, int ns, const DevScalars* __restrict__ sc, const int* __restrict__ chunk_off,
             int n_chunks, int* __restrict__ rows, int* __restrict__ rowidx, int* __restrict__ row_cnt, int rows_stride,
             const IgClassTab* __restrict__ clstab, const long long* __restrict__ row_ptr, RowInfo* __restrict__ rinfo,
             unsigned* __restrict__ bitmap, int bitmap_words, unsigned short* __restrict__ cls16) {
    TL(4);
    const int n = sc->n_cands;
    __shared__ int wsum[IG_MAX_CANDS][32];
    __shared__ int s_bp[IG_MAX_CANDS][IG_MAX_BP + 4];
    __shared__ int s_ida[IG_MAX_CANDS], s_idb[IG_MAX_CANDS];
    for (int t = threadIdx.x; t < n * (IG_MAX_BP + 4); t += blockDim.x) {
        const int k = t / (IG_MAX_BP + 4), j = t - k * (IG_MAX_BP + 4);
        s_bp[k][j] = reinterpret_cast<const int*>(clstab + k)[j];  // bp_sub, bp_sub_b, distinct_b, id_b
    }
    if (threadIdx.x < n) { s_ida[threadIdx.x] = sc->ci[threadIdx.x].id_a; s_idb[threadIdx.x] = sc->ci[threadIdx.x].id_b; }
    __syncthreads();
    const int r = blockIdx.x * IG_ROW_CHUNK + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    CoordRec cr;
    cr.id_c = -1; cr.pos = 0; cr.dist = 0.f; cr.s_tot = 0.f;
    if (r < ns) cr = coord[r];
    unsigned fmask = 0;   // candidates this row belongs to
    for (int k = 0; k < n; k++) {
        const bool f = r < ns && (cr.id_c == s_ida[k] || cr.id_c == s_idb[k]);
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (f) fmask |= 1u << k;
        if (lane == 0) {
            wsum[k][w] = __popc(b);
            // streaming scoring path: membership bitmap of the affected contigs (one bit per sub-fragment, staged in shared
            // memory by k_stream)
            if (bitmap && r < ns) bitmap[(size_t)k * bitmap_words + (r >> 5)] = b;
        }
    }
    __syncthreads();
    if (w < n) {   // warp k: inclusive scan of candidate k's per-warp counts
        int s = wsum[w][lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        wsum[w][lane] = s;
    }
    __syncthreads();
    for (int k = 0; k < n; k++) {
        const bool f = (fmask >> k) & 1u;
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (!f) continue;
        const int off = chunk_off[k * n_chunks + blockIdx.x] + (w ? wsum[k][w - 1] : 0) + __popc(b & ((1u << lane) - 1));
        rows[(size_t)k * rows_stride + off] = r;
        const int cls = ig_class_of(s_bp[k], s_bp[k] + IG_MAX_BP, s_bp[k][IG_MAX_BP + 2], s_bp[k][IG_MAX_BP + 3], cr.id_c, cr.pos);
        rowidx[(size_t)k * rows_stride + r] = off | (cls << IG_CLS_SHIFT);
        if (cls16) cls16[(size_t)k * rows_stride + r] = (unsigned short)(cls | (window_flags(cr.pos, sc->ci[k]) << 8));
        const long long rb = row_ptr[r];
        RowInfo ri; ri.r = r; ri.cls = cls; ri.n = (int)(row_ptr[r + 1] - rb); ri.pad = 0; ri.b = rb; ri.seg = 0; ri.ci = cr;
        rinfo[(size_t)k * rows_stride + off] = ri;
        row_cnt[(size_t)k * rows_stride + off] = 0;  // k_score (rows cut into parts) and k_stream accumulate into it
    }
}

// K5-7 for small levels (a handful of row chunks): count + scan + write in ONE launch, one block per candidate
// walking the chunks with a running offset (saves a dependent launch of the step's chain).
__global__ void __launch_bounds__(IG_ROW_CHUNK)
k_rows_small(const CoordRec* __restrict__ coord, int ns, DevScalars* sc, int n_chunks, int* __restrict__ rows,
             int* __restrict__ rowidx, int* __restrict__ row_cnt, int rows_stride, const IgClassTab* __restrict__ clstab,
             const long long* __restrict__ row_ptr, RowInfo* __restrict__ rinfo) {
    TL(3);
    const int k = blockIdx.x;
    if (k >= sc->n_cands) return;
    __shared__ int wsum[32], wlen[32];
    __shared__ int s_bp[IG_MAX_BP + 4];
    if (threadIdx.x < IG_MAX_BP + 4) s_bp[threadIdx.x] = reinterpret_cast<const int*>(clstab + k)[threadIdx.x];
    const CandInfo ci_k = sc->ci[k];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int base = 0, seg_base = 0;   // rows so far / stored contacts of those rows (segment offsets of the flat list)
    for (int ch = 0; ch < n_chunks; ch++) {
        const int r = ch * IG_ROW_CHUNK + threadIdx.x;
        CoordRec cr;
        if (r < ns) cr = coord[r];
        const bool f = r < ns && row_affected(cr, ci_k);
        const unsigned b = __ballot_sync(0xffffffffu, f);
        long long rb = 0;
        int rn = 0;
        if (f) { rb = row_ptr[r]; rn = (int)(row_ptr[r + 1] - rb); }
        const int rn_pad = (rn + 31) & ~31;   // rows own whole 32-contact chunks of the flat list
        int lx = rn_pad;   // inclusive warp scan of the padded row lengths
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, lx, o); if (lane >= o) lx += y; }
        __syncthreads();   // wsum / wlen of the previous chunk fully consumed
        if (lane == 0) wsum[w] = __popc(b);
        if (lane == 31) wlen[w] = lx;
        __syncthreads();
        if (w == 0) {
            int s = wsum[lane], l = wlen[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, s, o), z = __shfl_up_sync(0xffffffffu, l, o);
                if (lane >= o) { s += y; l += z; }
            }
            wsum[lane] = s; wlen[lane] = l;
        }
        __syncthreads();
        if (f) {
            const int off = base + (w ? wsum[w - 1] : 0) + __popc(b & ((1u << lane) - 1));
            rows[(size_t)k * rows_stride + off] = r;
            const int cls = ig_class_of(s_bp, s_bp + IG_MAX_BP, s_bp[IG_MAX_BP + 2], s_bp[IG_MAX_BP + 3], cr.id_c, cr.pos);
            rowidx[(size_t)k * rows_stride + r] = off | (cls << IG_CLS_SHIFT);
            RowInfo ri; ri.r = r; ri.cls = cls; ri.n = rn; ri.pad = 0; ri.b = rb; ri.ci = cr;
            ri.seg = (long long)(seg_base + (w ? wlen[w - 1] : 0) + lx - rn_pad);
            rinfo[(size_t)k * rows_stride + off] = ri;
            row_cnt[(size_t)k * rows_stride + off] = 0;
        }
        base += wsum[31]; seg_base += wlen[31];
    }
    if (threadIdx.x == 0) { sc->ci[k].n_rows = base; sc->flat_segtotal[k] = seg_base; }
}
