// instagraal_b200 -- steps of more than IG_MAX_CANDS candidates (up to IG_MAX_NEIGHBOURS): batches of IG_MAX_CANDS.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once
//
// A wide step runs the step's head (refresh or incremental commit) once, then one score-only pass of the usual chain
// (k_cand_setup ... k_finalize without selection) per batch of IG_MAX_CANDS candidates, in candidate order, and then
// scores the winning batch once more with the selecting tail (select_step, k_lnz_outside, k_apply, k_post).  The kernels
// below only move data between the step's scalar record and the wide record: they stage a batch's candidates where
// k_cand_setup reads them, keep every pass's scores and the running maximum, and fix up what the re-scored batch cannot
// know (its index in the whole list, the flip/eject proposal of a batch other than the first, the validity list).
// Everything around the launch sequence (enqueue_wide_step in ig_kernels.cu) is the narrow step's: host step, cycle plan
// (read here at the stride sc->plan_stride), graph cache and step record.
#define IG_MAX_BATCHES ((IG_MAX_NEIGHBOURS + IG_MAX_CANDS - 1) / IG_MAX_CANDS)
struct WideStep {
    int in[2 + IG_MAX_NEIGHBOURS];             // ig_step_wide: n_cands, fragment, sorted candidates
    double scores[IG_MAX_NEIGHBOURS * IG_N_OPS];
    int n_uniq[IG_MAX_NEIGHBOURS], n_sub[IG_MAX_NEIGHBOURS];
    int valid0[IG_MAX_BATCHES][12];             // list_valid_insert each batch started from (quirk Q3)
    int valid_end[12];                          // ... and the one the last batch left
    int n, a;                                   // candidates of the step, visited fragment
    int best_b, n_prop;                         // first batch that reached the maximum (-1: none scored), proposals scored
    double best_v;
    int win_cand, pad;                          // index of the applied move's candidate in the whole list
    // T > 0 (ig_k_temper.cuh): per batch the maximum score m_b, S_b = sum exp((s_i - m_b) / T) and the scored proposals;
    // the step's maximum M, log(sum_b W_b), the batch draw and the scored proposals of the whole step
    double t_m[IG_MAX_BATCHES], t_S[IG_MAX_BATCHES];
    int t_cnt[IG_MAX_BATCHES];
    double t_M, t_logW, t_ub;
    int t_nsc, t_pad;
};

// before batch b: its candidates (8b .. 8b + n_b - 1 of the step's list) into sc, where k_cand_setup reads them, and the
// validity list the batch starts from.  plan = the cycle plan (entry sc->step_idx, stride sc->plan_stride) or nullptr (w->in).
// A batch past the step's candidates (a device-drawn plan with fewer neighbours than asked for) gets n_b = 0: every
// kernel of the pass then does nothing.
__global__ void k_wide_stage(DevScalars* sc, WideStep* w, const int* __restrict__ plan, int b) {
    const int* src = plan ? plan + (size_t)sc->step_idx * sc->plan_stride : w->in;
    const int n = src[0], i = threadIdx.x;
    const int nb = max(0, min(IG_MAX_CANDS, n - b * IG_MAX_CANDS));
    if (i < IG_MAX_CANDS) sc->cands[i] = i < nb ? src[2 + b * IG_MAX_CANDS + i] : 0;
    if (i < 12) w->valid0[b][i] = sc->valid[i];
    if (i == 0) {
        sc->n_cands = nb; sc->a = src[1];
        if (b == 0) { w->n = n; w->a = src[1]; w->best_b = -1; w->best_v = 0.0; w->n_prop = 0; }
    }
}

// after the score-only pass of batch b: its scores and counters into the wide record, the running maximum (first index of
// the maximum over the non-zero scores, CL:1435-1446: a later batch wins only with a strictly larger score)
__global__ void k_wide_stash(const DevScalars* __restrict__ sc, WideStep* w, int b) {
    const int nb = sc->n_cands;
    const double T = sc->temperature;
    if (T > 0.0 && threadIdx.x < 32) {   // the batch's part of the tempered draw
        __shared__ double s_w[IG_MAX_CANDS * IG_N_OPS];
        double m;
        int cnt, last;
        const double S = temper_weights(sc->scores, nb * IG_N_OPS, T, s_w, &m, &cnt, &last);
        if (threadIdx.x == 0) { w->t_m[b] = m; w->t_S[b] = S; w->t_cnt[b] = cnt; }
    }
    for (int i = threadIdx.x; i < nb * IG_N_OPS; i += blockDim.x) w->scores[b * IG_MAX_CANDS * IG_N_OPS + i] = sc->scores[i];
    if (threadIdx.x < nb) {
        w->n_uniq[b * IG_MAX_CANDS + threadIdx.x] = sc->res_nuniq[threadIdx.x];
        w->n_sub[b * IG_MAX_CANDS + threadIdx.x] = sc->res_nsub[threadIdx.x];
    }
    if (threadIdx.x < 12) w->valid_end[threadIdx.x] = sc->valid[threadIdx.x];
    if (threadIdx.x != 0) return;
    int np = 0;
    for (int k = 0; k < nb; k++) np += sc->res_nuniq[k];
    w->n_prop += np;
    int best = -1;
    double bv = 0.0;
    for (int i = 0; i < nb * IG_N_OPS; i++) {
        const double v = sc->scores[i];
        if (v == 0.0) continue;
        if (best < 0 || v > bv) { best = i; bv = v; }
    }
    if (best >= 0 && (w->best_b < 0 || bv > w->best_v)) { w->best_b = b; w->best_v = bv; }
}

// T > 0: the batch drawn with u_batch from W_b = S_b exp((m_b - M) / T), in batch order (ig_k_temper.cuh); the last batch
// with a scored proposal if rounding leaves none, batch 0 when nothing was scored
__device__ __noinline__ int wide_temper_batch(const DevScalars* sc, WideStep* w, double T) {
    const int n_b = (w->n + IG_MAX_CANDS - 1) / IG_MAX_CANDS;
    double M = -INFINITY;
    int nsc = 0, last = -1;
    for (int b = 0; b < n_b; b++) if (w->t_cnt[b] > 0) { M = fmax(M, w->t_m[b]); nsc += w->t_cnt[b]; last = b; }
    auto W = [&](int b) { return w->t_cnt[b] > 0 ? __dmul_rn(w->t_S[b], exp(__ddiv_rn(__dsub_rn(w->t_m[b], M), T))) : 0.0; };
    double sum = 0.0;
    for (int b = 0; b < n_b; b++) sum = __dadd_rn(sum, W(b));
    const double ub = temper_uniform(sc, IG_TEMPER_U_BATCH);
    const double target = __dmul_rn(ub, sum);
    int pick = last < 0 ? 0 : last;
    double cum = 0.0;
    for (int b = 0; b < n_b && last >= 0; b++) {
        cum = __dadd_rn(cum, W(b));
        if (cum > target) { pick = b; break; }
    }
    w->t_M = M; w->t_logW = log(sum); w->t_ub = ub; w->t_nsc = nsc;
    return pick;
}

// before the re-score: the winning batch (batch 0 when nothing was scored, as np.argmax of an all -inf vector; at T > 0 the
// drawn batch) staged like k_wide_stage, from the validity list it started from
__global__ void k_wide_pick(DevScalars* sc, WideStep* w, const int* __restrict__ plan) {
    const int* src = plan ? plan + (size_t)sc->step_idx * sc->plan_stride : w->in;
    __shared__ int s_b;
    const double T = sc->temperature;
    if (threadIdx.x == 0) s_b = T > 0.0 ? wide_temper_batch(sc, w, T) : max(w->best_b, 0);
    __syncthreads();
    const int b = s_b;
    const int nb = max(0, min(IG_MAX_CANDS, w->n - b * IG_MAX_CANDS));
    const int i = threadIdx.x;
    if (i < IG_MAX_CANDS) sc->cands[i] = i < nb ? src[2 + b * IG_MAX_CANDS + i] : 0;
    if (i < 12) sc->valid[i] = w->valid0[b][i];
    __syncthreads();
    if (i == 0) { sc->n_cands = nb; sc->a = w->a; w->best_b = b; }
}

// after k_cand_setup of the re-score (launched with first_flip_eject = 1): the flip / eject proposals belong to the step's
// first candidate only, so a winning batch other than the first loses them again (ig_uniq_mutations as k_cand_setup calls it)
__global__ void k_wide_flip(const DevScalars* __restrict__ sc, IgDescriptor* desc, const WideStep* __restrict__ w) {
    if (threadIdx.x != 0 || w->best_b == 0 || sc->n_cands == 0) return;
    IgDescriptor& d = desc[0];
    d.n_uniq = ig_uniq_mutations(d.A, d.B, w->valid0[w->best_b], 0, d.uniq);
}

// after the tail: the candidate index in the whole list, the step's proposal count (score-only passes), and the validity
// list the reference leaves -- the last batch's, unless the applied op re-ran get_bounds (op >= 12, select_step).  The
// fragment k_post recorded is already right: sc->cands holds the re-scored winning batch.
__global__ void k_wide_finish(DevScalars* sc, WideStep* w, CycleOut* __restrict__ cyc_out, ig_tempered_step* __restrict__ trec_out) {
    const int i = threadIdx.x;
    if (i < 12 && sc->win_op < 12) sc->valid[i] = w->valid_end[i];
    if (i != 0) return;
    w->win_cand = w->best_b * IG_MAX_CANDS + sc->win_cand;
    if (cyc_out) {   // the record k_post just published (it advanced step_idx)
        CycleOut& o = cyc_out[sc->step_idx - 1];
        o.win_cand = w->win_cand; o.n_proposals = w->n_prop;
        if (sc->temperature > 0.0) {   // the record k_post published holds the draw inside the batch: the whole step's
            ig_tempered_step& r = trec_out[sc->step_idx - 1];
            r.s_max = w->t_M; r.log_w = w->t_logW; r.u_batch = w->t_ub; r.n_scored = w->t_nsc;
            r.batch = w->best_b; r.index = w->best_b * IG_MAX_CANDS * IG_N_OPS + r.index;
        }
    }
}
