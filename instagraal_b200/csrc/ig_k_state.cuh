// instagraal_b200 -- state of the current scaffold: coordinates, full likelihood over every contact, tables.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// K0: coordinates of the current scaffold (uni_fill_vect_dist, KA:3763-3822) + its zero term and
//     intra pixel count (eval_likelihood_on_zero with the CORRECT float mean, i.e. without Q1).
__global__ void __launch_bounds__(IG_THREADS)
k_coords(const FragRec* __restrict__ live, const SubRec* __restrict__ sub, CoordRec* __restrict__ coord,
         int* __restrict__ clen, int ns, const DevScalars* __restrict__ sc, float mbar, int use_test,
         double* __restrict__ part_z, int* __restrict__ part_n, int write_coords, SubX* __restrict__ subx,
         unsigned char* __restrict__ row_dirty, const int* __restrict__ pred = nullptr) {
    if (pred && !*pred) return;   // step kind 3: only after an accepted nuisance proposal
    TL(13);
    __shared__ double sm[32];
    __shared__ int sn;
    const Params p = use_test ? sc->p_test : sc->p;
    if (threadIdx.x == 0) sn = 0;
    __syncthreads();
    double z = 0.0;
    int nloc = 0;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < ns; r += gridDim.x * blockDim.x) {
        CoordRec c; int len;
        if (write_coords) {
            SubRec s = sub[r];
            Frag f = live[s.parent].f;
            c = coords_of(f, s, &len);
            coord[r] = c; clen[r] = len;
            SubX x; x.start_bp = f.start_bp; x.len_ori = f.len_bp * f.ori; x.watson = s.watson; x.crick = s.crick;
            subx[r] = x;
            if (row_dirty) row_dirty[r] = 1;   // cached per-contact records of this row are stale (k_lnz_refresh)
        } else { c = coord[r]; len = clen[r]; }
        if (c.pos == 0) nloc += intra_pairs(len);
        z += zero_term(c.pos, len, c.s_tot, p, mbar);
    }
    if (nloc) atomicAdd(&sn, nloc);
    double tot = block_sum(z, sm);
    __syncthreads();
    if (threadIdx.x == 0) { part_z[blockIdx.x] = tot; part_n[blockIdx.x] = sn; }
}

// K1: full likelihood over every stored contact (evaluate_likelihood_sparse, KA:4374-4488).
//     A pure stream over the CSR: 8 bytes per contact + one 16-byte coordinate gather (L1/L2-resident table).
//     Warp per row; every lane takes TWO contacts per trip with one 128-bit load (rows start on any contact: the
//     trip starts at the even index below it, the out-of-row half is masked).  Per contact the term is
//         ob * log10(ex) - ex - obc(ob) + exz * log10(e)                      (KA:251-270, 4322-4353)
//     * obc(ob) (log10 ob!, two f64 log10 + sqrt for ob >= 15) depends on the observed count only: its sum over the
//       level is computed ONCE per handle (k_obc_sum) and subtracted from the first block's partial;
//     * contacts whose expectation is the floor v_inter (other contig, s outside (0, d_max)) need no transcendental:
//       their ob, count and exz are summed as integers / plain adds;
//     * the others (powf + log10) are QUEUED per warp in shared memory and evaluated 32 at a time with every lane
//       busy (near-diagonal and trans contacts alternate inside a row: evaluating in place leaves half of the lanes
//       idle through ~80 instructions); powf_pos is bit-identical to the reference's powf, log10_f32 < 4e-16.
//     Rows of circular contigs and v_inter <= 0 take the generic per-contact routine (contact_term).
struct __align__(8) LnzQ { float s; int val; };
#define IG_LNZ_QCAP 96
__device__ __forceinline__ double lnz_eval(const LnzQ e, const Params& p, double l10v) {
    const float pw = powf_pos(e.s, p.slope);
    float exf;
    if (p.d == 2.0f) exf = __fmul_rn(__fmul_rn(p.c1, pw), p.fact);
    else exf = (p.c1 * pw * expf((p.d - 2) / (powf(e.s * p.lm / p.kuhn, 2.0f) + p.d))) * p.fact;
    exf = fmaxf(exf, p.v_inter);
    const double lg = (exf == p.v_inter) ? l10v : log10_f32(exf);
    return (double)e.val * lg - (double)exf;
}
__global__ void __launch_bounds__(IG_THREADS)
k_full_lnz(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const CoordRec* __restrict__ coord,
           const int* __restrict__ clen, int ns, const DevScalars* __restrict__ sc, float mbar, int use_test,
           const float* __restrict__ exz_tab, double* __restrict__ part) {
    TL(14);
    __shared__ double sm[32];
    __shared__ LnzQ queue[IG_WARPS_PER_BLOCK][IG_LNZ_QCAP];
    const Params p = use_test ? sc->p_test : sc->p;
    const double l10v = use_test ? sc->log10_vinter_test : sc->log10_vinter;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const bool generic = !(p.v_inter > 0.0f);
    LnzQ* myq = queue[w];
    int qn = 0;                      // warp-uniform
    double acc = 0.0, acc_exz = 0.0; // queued terms / expected contacts of the zero term (floats summed in double)
    long long sob = 0;               // observed counts of the floor contacts
    int nfl = 0;                     // number of floor contacts
    for (int r = wg; r < ns; r += nw) {
        const long long b = row_ptr[r], e = row_ptr[r + 1];
        if (b == e) continue;
        const CoordRec ci = coord[r];
        if (generic || ci.s_tot != 0) {   // circular contig (rare) / degenerate floor: the generic routine, obc hoisted all the same
            const int len_i = clen[r];
            for (long long k = b + lane; k < e; k += 32) {
                const int2 c = __ldg(&cv[k]);
                const CoordRec cj = coord[c.x];
                const double ob = (double)c.y;
                // KA:4428: the circular zero term uses the ROW's contig length
                double t;
                if (generic) {   // with v_inter <= 0 a term may vanish entirely (ex == 0, KA:257): keep its own obc
                    const double obc = ob_const(ob);
                    t = contact_term(ci, cj, len_i, ob, obc, p, l10v, mbar, exz_tab) + obc;
                } else t = contact_term(ci, cj, len_i, ob, 0.0, p, l10v, mbar, exz_tab);
                acc += t;
            }
            continue;
        }
        for (long long k0 = (b & ~1LL); k0 < e; k0 += 64) {
            const long long k = k0 + 2 * lane;
            int4 c2 = make_int4(0, 0, 0, 0);
            if (k < e) c2 = __ldcs(reinterpret_cast<const int4*>(cv + k));   // streamed once: do not keep it in L1
            const bool v0 = (k >= b) && (k < e), v1 = (k + 1 < e);
            CoordRec cj0 = ci, cj1 = ci;
            if (v0) cj0 = coord[c2.x];
            if (v1) cj1 = coord[c2.z];
            bool push0 = false, push1 = false;
            float s0 = 0.f, s1 = 0.f;
            if (v0) {
                float exz = p.v_inter;
                if (cj0.id_c == ci.id_c) {
                    s0 = fabsf(ci.dist - cj0.dist);
                    exz = exz_tab[abs(ci.pos - cj0.pos)];
                    push0 = (s0 > 0.0f) && (s0 < p.d_max);
                }
                acc_exz += (double)exz;
                if (!push0) { sob += c2.y; nfl++; }
            }
            if (v1) {
                float exz = p.v_inter;
                if (cj1.id_c == ci.id_c) {
                    s1 = fabsf(ci.dist - cj1.dist);
                    exz = exz_tab[abs(ci.pos - cj1.pos)];
                    push1 = (s1 > 0.0f) && (s1 < p.d_max);
                }
                acc_exz += (double)exz;
                if (!push1) { sob += c2.w; nfl++; }
            }
            // warp-collective append (first contacts of all lanes, then second ones) + evaluation of full batches
            const unsigned m0 = __ballot_sync(0xffffffffu, push0), m1 = __ballot_sync(0xffffffffu, push1);
            if (push0) { LnzQ q; q.s = s0; q.val = c2.y; myq[qn + __popc(m0 & ((1u << lane) - 1))] = q; }
            qn += __popc(m0);
            if (push1) { LnzQ q; q.s = s1; q.val = c2.w; myq[qn + __popc(m1 & ((1u << lane) - 1))] = q; }
            qn += __popc(m1);
            __syncwarp();
            while (qn >= 32) {
                qn -= 32;
                acc += lnz_eval(myq[qn + lane], p, l10v);
            }
            __syncwarp();
        }
    }
    if (lane < qn) acc += lnz_eval(myq[lane], p, l10v);
    // floor contacts: ob * log10(v_inter) - v_inter each (KA:259-262 with ex == v_inter).  The generic routine has no floor
    // sums (sob == nfl == acc_exz == 0), and with v_inter <= 0 log10(v_inter) is -inf or NaN: 0 * -inf would make it NaN
    if (!generic) acc += l10v * (double)sob - (double)p.v_inter * (double)nfl + acc_exz * (double)LOG10E_F;
    double tot = block_sum(acc, sm);
    if (threadIdx.x == 0) part[blockIdx.x] = tot - (blockIdx.x == 0 ? sc->obc_total : 0.0);
}
// sum over every stored contact of the part of its term that depends on the observed count only (KA:259,262)
__global__ void __launch_bounds__(IG_THREADS)
k_obc_sum(const int2* __restrict__ cv, long long nnz, double* __restrict__ part) {
    __shared__ double sm[32];
    double acc = 0.0;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (long long)gridDim.x * blockDim.x) {
        const double ob = (double)max(cv[k].y, 0);
        acc += ob_const(ob);
    }
    const double tot = block_sum(acc, sm);
    if (threadIdx.x == 0) part[blockIdx.x] = tot;
}

// ------------------------------------------------------------------------------------------------
// K1': the same sum as k_full_lnz from CACHED per-contact records -- the nuisance step's likelihood
//      (step_nuisance_parameters -> eval_likelihood_4_nuisance, CL:2961-3051 / 1296-1344) runs after EVERY step_sampler
//      from cycle 5 on (IG:242-252): the parameters change with every call, the scaffold's coordinates only for the rows
//      of the <= 2 contigs the last move touched.  What a contact's term needs from the scaffold is
//          same contig?   s = |dist_i - dist_j| (float32, KA:4322)   dp = |pos_i - pos_j|
//      so these are kept per contact in an 8-byte record {s (negative: other contig), dp | val << dp_bits} that is
//      rebuilt for the rows whose coordinates were rewritten (row_dirty, set by k_coords / k_commit_coords: every row of
//      an affected contig; a contact from an untouched row into a touched contig joined other contigs before and after).
//        k_lnz_refresh  rows flagged dirty: the gather path of k_full_lnz, writing records; rows of circular contigs are
//                       evaluated here on every call with the generic routine (their records say "skip");
//        k_lnz_stream   a flat pass over the records: 8 bytes per contact, no row structure, no gathers but the
//                       L1-resident expected-contact table; floor contacts are counted, the others queued per warp and
//                       evaluated 32 at a time (powf_pos + log10_f32) exactly like k_full_lnz.
//      Same terms, same double accumulation, different (fixed) summation order.
// Record encoding (dp_bits low bits = index into the expected-contact table, the observed count above them):
//   same contig      {s >= 0,  dp}        table[dp]     = expected contacts at separation dp (k_exz_table)
//   other contig     {-1.0f,   ns + 1}    table[ns + 1] = v_inter
//   skip             {-1.0f,   ns + 2}    table[ns + 2] = 0      (rows of circular contigs; the odd padding record)
// so the flat pass needs no case distinction: a record is QUEUED when 0 < s < d_max and is a floor contact otherwise, and
// every record adds table[idx] to the zero term.  Floor contacts are not even counted per record:
//   sum_floor (ob log10 v - v) = log10 v * (V_all - V_queued) - v * (N_all - N_queued)
// with V_all = the level's total observed count (constant) and N_all = the number of records streamed; the skip records
// are in N_all (and, for circular rows, in V_all) and k_lnz_refresh, which evaluates those rows anyway, takes their
// spurious floor terms out again.
__global__ void __launch_bounds__(IG_THREADS)
k_lnz_refresh(const long long* __restrict__ row_ptr, const int2* __restrict__ cv, const CoordRec* __restrict__ coord,
              const int* __restrict__ clen, int ns, const DevScalars* __restrict__ sc, float mbar, int use_test,
              const float* __restrict__ exz_tab, int2* __restrict__ rec, unsigned char* __restrict__ row_dirty, int dp_bits,
              double* __restrict__ part, const int* __restrict__ pred = nullptr) {
    if (pred && !*pred) return;
    TL(14);
    __shared__ double sm[32];
    const Params p = use_test ? sc->p_test : sc->p;
    const double l10v = use_test ? sc->log10_vinter_test : sc->log10_vinter;
    const int lane = threadIdx.x & 31;
    const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    double acc = 0.0;
    // warp w owns the rows r = w (mod nw): the rows of one contig are neighbours in r, so a move's dirty rows land on as many
    // different warps as there are; each warp looks at 32 of its rows at a time (flags read in parallel)
    for (int j0 = 0; wg + (long long)j0 * nw < ns; j0 += 32) {
        const long long r_ll = wg + (long long)(j0 + lane) * nw;
        const int r_l = r_ll < ns ? (int)r_ll : -1;
        bool need = false;
        if (r_l >= 0) {
            const bool circ = coord[r_l].s_tot != 0;
            need = (row_ptr[r_l] != row_ptr[r_l + 1]) && (circ || row_dirty[r_l] != 0);
            if (!need && row_dirty[r_l]) row_dirty[r_l] = 0;   // empty row
        }
        for (unsigned todo = __ballot_sync(0xffffffffu, need); todo; todo &= todo - 1) {
            const int r = wg + (j0 + __ffs(todo) - 1) * nw;
            const long long b = row_ptr[r], e = row_ptr[r + 1];
            const CoordRec ci = coord[r];
            const bool circ = ci.s_tot != 0;
            const bool dirty = row_dirty[r] != 0;
            const int len_i = clen[r];
            for (long long k = b + lane; k < e; k += 32) {
                const int2 c = __ldg(&cv[k]);
                const CoordRec cj = coord[c.x];
                int2 out;
                out.x = __float_as_int(-1.0f);
                if (circ) {   // KA:4428: the circular zero term uses the ROW's contig length; obc is hoisted (sc->obc_total)
                    acc += contact_term(ci, cj, len_i, (double)c.y, 0.0, p, l10v, mbar, exz_tab)
                           - (l10v * (double)c.y - (double)p.v_inter);   // what the flat pass adds for a skip record
                    out.y = (ns + 2) | (c.y << dp_bits);
                } else if (cj.id_c == ci.id_c) {
                    out.x = __float_as_int(fabsf(ci.dist - cj.dist));
                    out.y = abs(ci.pos - cj.pos) | (c.y << dp_bits);
                } else out.y = (ns + 1) | (c.y << dp_bits);
                if (dirty) rec[k] = out;
            }
            __syncwarp();
            if (dirty && lane == 0) row_dirty[r] = 0;
        }
    }
    const double tot = block_sum(acc, sm);
    if (threadIdx.x == 0) part[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(IG_THREADS, 4)
k_lnz_stream(const int4* __restrict__ rec2, long long n_pairs, int n_pad, double val_total, const DevScalars* __restrict__ sc,
             int use_test, const float* __restrict__ exz_tab, int dp_bits, double* __restrict__ part,
             const int* __restrict__ pred = nullptr) {
    if (pred && !*pred) return;
    TL(14);
    __shared__ double sm[32];
    __shared__ LnzQ queue[IG_WARPS_PER_BLOCK][IG_LNZ_QCAP];
    const Params p = use_test ? sc->p_test : sc->p;
    const double l10v = use_test ? sc->log10_vinter_test : sc->log10_vinter;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long wg = (long long)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const long long nw = (long long)((gridDim.x * blockDim.x) >> 5);
    const unsigned dpmask = (1u << dp_bits) - 1u;
    const unsigned lt = (1u << lane) - 1u;
    LnzQ* myq = queue[w];
    int qn = 0, n_queued = 0;         // warp-uniform
    double acc = 0.0, acc_exz = 0.0;  // queued terms / expected contacts of the zero term
    int v_queued = 0;                 // observed counts of the queued contacts
    auto eval = [&](const LnzQ e) {
        v_queued += e.val;
        acc += lnz_eval(e, p, l10v);
    };
    auto append = [&](bool p0, int s0, unsigned y0, bool p1, int s1, unsigned y1) {
        const unsigned m0 = __ballot_sync(0xffffffffu, p0), m1 = __ballot_sync(0xffffffffu, p1);
        const int c0 = __popc(m0), c1 = __popc(m1);
        if (p0) { LnzQ q; q.s = __int_as_float(s0); q.val = (int)(y0 >> dp_bits); myq[qn + __popc(m0 & lt)] = q; }
        if (p1) { LnzQ q; q.s = __int_as_float(s1); q.val = (int)(y1 >> dp_bits); myq[qn + c0 + __popc(m1 & lt)] = q; }
        qn += c0 + c1; n_queued += c0 + c1;
        __syncwarp();
        while (qn >= 32) {
            qn -= 32;
            eval(myq[qn + lane]);
        }
        __syncwarp();
    };
    // n_pairs is a multiple of 64: whole trips only; the next trip's records are in flight while this one is evaluated
    const int4 skip2 = make_int4(__float_as_int(-1.0f), 0, __float_as_int(-1.0f), 0);
    long long base = wg * 64;
    int4 ra = skip2, rb = skip2;
    if (base < n_pairs) { ra = __ldcs(rec2 + base + lane); rb = __ldcs(rec2 + base + 32 + lane); }   // streamed once per call: evict first
    for (; base < n_pairs; base += nw * 64) {
        const long long nxt = base + nw * 64;
        int4 na = skip2, nb = skip2;
        if (nxt < n_pairs) { na = __ldcs(rec2 + nxt + lane); nb = __ldcs(rec2 + nxt + 32 + lane); }
        const float e0 = __ldg(&exz_tab[(unsigned)ra.y & dpmask]), e1 = __ldg(&exz_tab[(unsigned)ra.w & dpmask]);
        const float e2 = __ldg(&exz_tab[(unsigned)rb.y & dpmask]), e3 = __ldg(&exz_tab[(unsigned)rb.w & dpmask]);
        const float s0 = __int_as_float(ra.x), s1 = __int_as_float(ra.z), s2 = __int_as_float(rb.x), s3 = __int_as_float(rb.z);
        append((s0 > 0.0f) && (s0 < p.d_max), ra.x, (unsigned)ra.y, (s1 > 0.0f) && (s1 < p.d_max), ra.z, (unsigned)ra.w);
        append((s2 > 0.0f) && (s2 < p.d_max), rb.x, (unsigned)rb.y, (s3 > 0.0f) && (s3 < p.d_max), rb.z, (unsigned)rb.w);
        acc_exz += ((double)e0 + (double)e1) + ((double)e2 + (double)e3);
        ra = na; rb = nb;
    }
    if (lane < qn) eval(myq[lane]);
    // the queued contacts are not floor contacts: take them out of the closed-form floor sum (block 0 adds its constants)
    acc += acc_exz * (double)LOG10E_F - l10v * (double)v_queued;
    if (lane == 0) acc += (double)p.v_inter * (double)n_queued;
    double tot = block_sum(acc, sm);
    if (threadIdx.x == 0) {
        if (blockIdx.x == 0)
            tot += l10v * val_total - (double)p.v_inter * (2.0 * (double)n_pairs - (double)n_pad) - sc->obc_total;
        part[blockIdx.x] = tot;
    }
}

// generic deterministic final reduction of `n` doubles (and optionally ints) by one block
// pred (all four kernels above too): when given, the kernel returns at once while *pred == 0
__global__ void k_reduce(const double* __restrict__ part, int n, double* out, const int* __restrict__ ipart, int* iout,
                         const int* __restrict__ pred = nullptr) {
    if (pred && !*pred) return;
    __shared__ double sm[32];
    __shared__ int smi;
    if (threadIdx.x == 0) smi = 0;
    __syncthreads();
    double v = 0.0;
    int iv = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { v += part[i]; if (ipart) iv += ipart[i]; }
    if (ipart && iv) atomicAdd(&smi, iv);
    double tot = block_sum(v, sm);
    __syncthreads();
    if (threadIdx.x == 0) { *out = tot; if (iout) *iout = smi; }
}

// exz table: expected contacts at integer sub-fragment separation (linear contigs), KA:4330-4335
__global__ void k_exz_table(float* __restrict__ tab, int n, const DevScalars* __restrict__ sc, float mbar, int use_test) {
    const Params p = use_test ? sc->p_test : sc->p;
    if (blockIdx.x == 0 && threadIdx.x == 0) { tab[n] = p.v_inter; tab[n + 1] = 0.0f; }   // slots of the likelihood records (k_lnz_stream)
    for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < n; d += gridDim.x * blockDim.x) {
        float s_z = __int2float_rn(d) * mbar;
        tab[d] = (s_z < p.d_max) ? rippe_contacts(s_z, p) : p.v_inter;
    }
}
__global__ void k_set_params_dev(DevScalars* sc, const float* __restrict__ p8, int test) {   // parameters from device memory (graph replay)
    Params p;
    p.kuhn = p8[0]; p.lm = p8[1]; p.c1 = p8[2]; p.slope = p8[3]; p.d = p8[4]; p.d_max = p8[5]; p.fact = p8[6]; p.v_inter = p8[7];
    if (test) { sc->p_test = p; sc->log10_vinter_test = log10((double)p.v_inter); }
    else { sc->p = p; sc->log10_vinter = log10((double)p.v_inter); }
}
__global__ void k_set_params(DevScalars* sc, Params p, int test) {
    if (test) { sc->p_test = p; sc->log10_vinter_test = log10((double)p.v_inter); }
    else { sc->p = p; sc->log10_vinter = log10((double)p.v_inter); }
}
