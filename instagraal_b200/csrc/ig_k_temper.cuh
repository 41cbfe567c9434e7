// instagraal_b200 -- production RNG mode: move selection at a chain temperature T > 0 (DESIGN.md 4e).
// Part of ig_kernels.cu (included there after ig_k_rng.cuh; not a stand-alone translation unit).
#pragma once

// At T > 0 a step draws its move among the scored proposals (non-zero, non-NaN score: the set the argmax ranges over) with
// probability w_i / sum(w), w_i = exp((s_i - m) / T), m = the maximum score: the convention of the nuisance step's
// exp((l_nuis - l_t) / T), so a chain at T targets exp(L / T) in both of its move types.  Arithmetic that a restatement
// repeats exactly: the weights lane-parallel (double exp, IEEE subtraction and division), their sum by lane 0 in ascending
// index; the pick is the first index whose running sum exceeds u * S, the last scored index if rounding leaves none,
// index 0 when nothing was scored (as the argmax).  A wide step draws in two stages (ig_k_wide.cuh): the batch b from
// W_b = S_b exp((m_b - M) / T) with u_batch, then the proposal inside it with u, which gives P(b) P(i | b) = w_i / sum(w).
// Draws: philox_uniform(t, cycle, IG_TEMPER_U | IG_TEMPER_U_BATCH, 0, seed), a counter domain neither k_draw_plan
// (draw < 2^31) nor the nuisance step (0x80000000, 0x80000001) uses.
#define IG_TEMPER_U 0x80000002u
#define IG_TEMPER_U_BATCH 0x80000003u

__device__ __forceinline__ bool temper_scored(double v) { return v != 0.0 && !isnan(v); }

// the draw (t, cycle, domain) of the plan step in flight (select_step, k_wide_pick: before k_post advances step_idx)
__device__ __forceinline__ double temper_uniform(const DevScalars* sc, unsigned domain) {
    return philox_uniform((unsigned)sc->step_idx, sc->nuis_cycle, domain, 0u, make_uint2(sc->nuis_key_lo, sc->nuis_key_hi));
}

// one full warp: w[i] = exp((s_i - m) / T) for the scored proposals among scores[0, n), 0 elsewhere.  Returns S (lane 0's
// sum in ascending index) on every lane; *m_out = m (-inf when nothing is scored), *cnt = scored proposals, *last = the
// last scored index (-1: none)
__device__ double temper_weights(const double* scores, int n, double T, double* w, double* m_out, int* cnt, int* last) {
    const int lane = threadIdx.x & 31;
    double m = -INFINITY;
    int c = 0, li = -1;
    for (int i = lane; i < n; i += 32) {
        const double v = __ldcg(&scores[i]);
        if (!temper_scored(v)) continue;
        m = fmax(m, v); c++; li = i;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    c = __reduce_add_sync(0xffffffffu, c);
    li = __reduce_max_sync(0xffffffffu, (unsigned)(li + 1)) - 1;
    for (int i = lane; i < n; i += 32) {
        const double v = __ldcg(&scores[i]);
        w[i] = temper_scored(v) ? exp(__ddiv_rn(__dsub_rn(v, m), T)) : 0.0;
    }
    __syncwarp();
    double S = 0.0;
    if (lane == 0) for (int i = 0; i < n; i++) S = __dadd_rn(S, w[i]);
    *m_out = m; *cnt = c; *last = li;
    return __shfl_sync(0xffffffffu, S, 0);
}

// the first index whose running sum (ascending, as S was formed) exceeds target; `last` when rounding leaves none
__device__ __forceinline__ int temper_pick(const double* w, int n, double target, int last) {
    double cum = 0.0;
    for (int i = 0; i < n; i++) {
        cum = __dadd_rn(cum, w[i]);
        if (cum > target) return i;
    }
    return last;
}

// select_step at T > 0 (one full warp; kept out of line so that the argmax path of k_finalize keeps its registers): the
// drawn flattened index of sc->scores, the same on every lane.  Lane 0 leaves the step's record in sc->trec (k_post
// publishes it; k_wide_finish completes a wide step's).
__device__ __noinline__ int temper_select(DevScalars* sc, int n, double T) {
    __shared__ double s_w[IG_MAX_CANDS * IG_N_OPS];
    double m;
    int cnt, last;
    const double S = temper_weights(sc->scores, n, T, s_w, &m, &cnt, &last);
    int best = 0;
    if ((threadIdx.x & 31) == 0) {
        const double u = temper_uniform(sc, IG_TEMPER_U);
        if (cnt > 0) best = temper_pick(s_w, n, __dmul_rn(u, S), last);
        ig_tempered_step& r = sc->trec;
        r.s_max = m; r.log_w = log(S); r.u = u; r.u_batch = 0.0;
        r.n_scored = cnt; r.batch = 0; r.index = best; r.pad = 0;
    }
    return __shfl_sync(0xffffffffu, best, 0);
}

__global__ void k_set_temperature(DevScalars* sc, double temperature) { sc->temperature = temperature; }
