/* instagraal_b200 -- C ABI of the B200-native scaffolding-MCMC hot path.
 *
 * Drop-in boundary for the reference's `sampler` class (src/instagraal/cuda_lib_gl_single.py,
 * "CL"): every entry point below replaces the pycuda launch sequence of one reference method.
 * Plain C: borrowed, C-contiguous host buffers in, caller-allocated buffers out; nothing returned
 * by pointer outlives the call.  One handle = one chain on one GPU, single host thread, all calls
 * blocking (except ig_run_cycle_device_async).  Every function returns 0 on success or a negative code (message: ig_last_error).
 * There is no CPU path: ig_create fails when no CUDA device is usable.
 */
#ifndef INSTAGRAAL_B200_H
#define INSTAGRAAL_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IG_N_FIELDS 13 /* pos, sub_pos, id_c, start_bp, len_bp, sub_len, circ, prev, next, l_cont,
                          sub_l_cont, l_cont_bp, ori  (struct frag, kernel_sparse_adapt.cu:40-58, minus
                          the inert id/rep/activ/id_d which the facade synthesises) */
#define IG_MAX_CANDS 8        /* candidates of one scoring pass (ig_step_result, ig_run_cycle plans) */
#define IG_MAX_NEIGHBOURS 64  /* candidates of one step: steps of more than IG_MAX_CANDS are scored in passes of
                                 IG_MAX_CANDS (ig_step_wide, ig_run_cycle_wide, ig_run_cycle_device) */
#define IG_N_OPS 24

typedef struct ig_handle ig_handle;

typedef struct ig_config {
    int32_t device;            /* CUDA ordinal (reference: --device, cli/main.py:74-80) */
    int32_t n_frags;           /* NF  = n_new_frags        (CL:170-171) */
    int32_t n_sub_frags;       /* NS  = init_n_sub_frags   (CL:140)     */
    int64_t nnz;               /* strict-upper non-zeros of the level L-1 matrix (CL:615) */
    int32_t max_bounds_insert; /* CL:417-420 */
    float mean_sub_len_kb;     /* float32(mean_len_bp_frags / 1000), CL:231,1120 */
    double n_pix;              /* n_pixl_sub_mat, CL:366 (caller reproduces the int32 wrap, quirk Q8) */
    int32_t compat_last_block; /* 1: reproduce the last-64-contact-block quirk of eval_sub_likelihood
                                  (kernel_sparse_adapt.cu:4362); 0: sum every contact */
    int32_t rigid_pruning;     /* 0 (default): every (contact, mutation) whose coordinates are not bit-identical to
                                  the current state is re-evaluated, reproducing the reference's float32
                                  re-rounding of shifted coordinates (fill_vect_dist, kernel_sparse_adapt.cu:3751);
                                  1: contacts whose two ends undergo the same rigid motion are skipped (their
                                  term cannot change mathematically) -- faster on long contigs, scores differ
                                  from the reference by that rounding noise */
} ig_config;

typedef struct ig_level_data {
    const int32_t* frags13;    /* [13][NF] initial live scaffold, field order of IG_N_FIELDS */
    const int32_t* sub_parent; /* [NS] parent fragment of each sub-fragment   (sub_frags_2_frags.x) */
    const float* sub_watson;   /* [NS] kb from fragment start                  (.y)  SS:703-717 */
    const float* sub_crick;    /* [NS] kb from fragment end                    (.z) */
    const int32_t* sub_j;      /* [NS] index within parent                     (.w) */
    const int64_t* row_ptr;    /* [NS+1] CSR of triu(M + M^T, k=1), canonical row-major (CL:592-609) */
    const int32_t* col;        /* [nnz] */
    const int32_t* val;        /* [nnz] */
    const int32_t* init_prev;  /* [NF] CL:269 */
    const int32_t* init_next;  /* [NF] CL:270 */
    const int32_t* orientable; /* [NF] CL:271-275 */
} ig_level_data;

typedef struct ig_step_result {
    double scores[IG_MAX_CANDS * IG_N_OPS]; /* all_scores, CL:1414-1431 (0.0 = not evaluated) */
    double likelihood;       /* o = all_scores[argmax], CL:1454 */
    double lnz_full;         /* gpu_curr_likelihood_nz, CL:1285 */
    double dist;             /* dist_inter_genome, CL:665-716 */
    int64_t sum_l_cont;      /* sum of contig lengths over contigs (mean_length_contigs numerator) */
    int32_t n_contigs;       /* CL:2736 */
    int32_t op_sampled;      /* CL:1446 */
    int32_t id_f_sampled;    /* CL:1445 */
    int32_t cand_index;      /* index of id_f_sampled in the candidate list */
    int32_t n_uniq[IG_MAX_CANDS];  /* proposals scored per candidate (gpu_n_uniq) */
    int32_t n_sub[IG_MAX_CANDS];   /* contacts selected by slice_sp_mat per candidate (n_sub_vals) */
    int32_t q4_hits;         /* fragments that hit the reference's "nothing written" paste case (Q4) */
    int32_t reserved;
} ig_step_result;

typedef struct ig_cycle_step {   /* compact per-step record of ig_run_cycle (what IG.full_em collects, IG:221-241) */
    double likelihood;       /* o */
    double lnz_full;
    double dist;
    int64_t sum_l_cont;
    int32_t n_contigs, op_sampled, id_f_sampled, cand_index;
    int32_t n_proposals;     /* proposals scored in this step (sum of n_uniq) */
    int32_t q4_hits;
} ig_cycle_step;

typedef struct ig_nuisance_step {   /* one nuisance step of a production-mode cycle (ig_set_device_nuisance), 80 B */
    double likelihood_nuis;    /* eval_likelihood_4_nuisance under p_test (CL:1296-1344) */
    double likelihood_t_after; /* likelihood_t after the step: likelihood_nuis if accepted, else the step's o */
    double u;                  /* acceptance draw */
    double draw;               /* the normal draw added to the moved parameter (NaN: none, d_nuc <= 0) */
    float p_test[8];           /* the proposed parameter set: kuhn, lm, c1, slope, d, d_max, fact, v_inter */
    int32_t id_modif;          /* 0 fact, 1 slope, 2 d_max, 3 d_nuc (= v_inter) */
    int32_t accepted;          /* exp(likelihood_nuis - o) >= u, and valid */
    int32_t valid;             /* 0: non-finite value, fact <= 0, slope >= 0, no d_max root, d_max <= 0 or v_inter <= 0 */
    int32_t pad;
} ig_nuisance_step;

typedef struct ig_tempered_step {   /* the move draw of one step at a chain temperature T > 0 (ig_set_temperature), 48 B */
    double s_max;              /* M, the step's maximum score */
    double log_w;              /* log(sum_i exp((s_i - M) / T)) over the scored proposals (log sum_b W_b of a wide step) */
    double u;                  /* draw inside the (winning) batch: philox_uniform(t, cycle, 0x80000002, 0, seed) */
    double u_batch;            /* batch draw of a wide step: philox_uniform(t, cycle, 0x80000003, 0, seed); 0 in a narrow step */
    int32_t n_scored;          /* scored proposals of the step (non-zero, non-NaN score) */
    int32_t batch;             /* drawn batch of IG_MAX_CANDS candidates (0 in a narrow step) */
    int32_t index;             /* drawn flattened index over the whole step: candidate * IG_N_OPS + op */
    int32_t pad;
} ig_tempered_step;

/* sampler.__init__ device part (CL:92-319: sparse_data_2_gpu, setup_all_gpu_struct, loadProgram) */
int ig_create(const ig_config* cfg, const ig_level_data* data, ig_handle** out);
/* sampler.free_gpu (CL:3167-3177) */
void ig_destroy(ig_handle* h);
const char* ig_last_error(ig_handle* h);
/* _check_gpu probe (cli/endtoend.py:51-83): number of usable CUDA devices, name of device 0 */
int ig_device_count(void);

/* memcpy_htod(gpu_param_simu, ...) (CL:2343-2349, 3033): kuhn, lm, c1, slope, d, d_max, fact, v_inter */
int ig_set_params(ig_handle* h, const float p[8]);
/* GPUStruct.copy_from_gpu / copy_to_gpu (gpustruct.py:94-186).  get: contig ids are relabelled the
 * way modify_gl_cuda_buffer would have left them (0..NC-1, longest contig = NC-1, CL:2715-2806). */
int ig_get_state(ig_handle* h, int32_t* out13xNF);
int ig_set_state(ig_handle* h, const int32_t* in13xNF);
/* gpu_list_valid_insert (CL:421): carried from one get_bounds to the next extract_uniq_mutations (Q3) */
int ig_get_valid_insert(ig_handle* h, int32_t out12[12]);
int ig_set_valid_insert(ig_handle* h, const int32_t in12[12]);
/* bomb_the_genome (CL:1925-1948) with the host-drawn permutation */
int ig_bomb(ig_handle* h, const int32_t* perm);

/* step_sampler (CL:1401-1465) after the host drew + sorted the candidates (CL:1403-1404) */
int ig_step(ig_handle* h, int32_t id_frag, const int32_t* cands, int32_t n_cands, ig_step_result* out);
/* n_steps consecutive step_sampler calls (the inner loop of full_em, IG:217-241) enqueued without any host
 * synchronisation in between; cands8 = [n_steps][IG_MAX_CANDS] sorted candidates, n_cands = [n_steps]. */
int ig_run_cycle(ig_handle* h, int32_t n_steps, const int32_t* frags, const int32_t* cands8, const int32_t* n_cands,
                 ig_cycle_step* out);
/* Steps of up to IG_MAX_NEIGHBOURS candidates (the reference takes any --neighborhood).  The candidates are scored in
 * passes of IG_MAX_CANDS; the move is the first index of the maximum over all of them (CL:1435-1446), as in ig_step.
 * ig_step_wide: scores = [24 * n_cands] all_scores, n_uniq / n_sub = [n_cands]; the scalar fields of `out` are filled,
 * cand_index is the index into the whole candidate list, and out->scores / n_uniq / n_sub hold the first IG_MAX_CANDS
 * candidates' values.  n_cands <= IG_MAX_CANDS is ig_step.
 * ig_run_cycle_wide: ig_run_cycle with cands = [n_steps][width] (width >= every n_cands[t], <= IG_MAX_NEIGHBOURS);
 * ig_run_cycle is this call with width = IG_MAX_CANDS.
 * ig_get_cycle_plan_wide: the plan of the last cycle as [n_steps][2 + width] (n_cands, fragment, candidates); fails when
 * a step had more than width candidates. */
int ig_step_wide(ig_handle* h, int32_t id_frag, const int32_t* cands, int32_t n_cands, ig_step_result* out, double* scores,
                 int32_t* n_uniq, int32_t* n_sub);
int ig_run_cycle_wide(ig_handle* h, int32_t n_steps, const int32_t* frags, const int32_t* cands, int32_t width,
                      const int32_t* n_cands, ig_cycle_step* out);
int ig_get_cycle_plan_wide(ig_handle* h, int32_t n_steps, int32_t width, int32_t* out /* [n_steps][2 + width] */);
/* Production RNG mode (SURVEY 8b "RNG contract"): the neighbour draws of return_neighbours (CL:3103-3141) on the
 * device.  ig_set_neighbour_weights uploads setup_distri_frags (CL:3053-3101) as a CSR: for fragment f the
 * candidates idx[ptr[f]..ptr[f+1]) (f itself excluded), the running sum cdf of their probabilities pk and the
 * number of non-zero pk.  ig_run_cycle_device = ig_run_cycle with every step's candidates drawn by one kernel
 * (Philox4x32-10, key = seed, counter = (step, cycle, draw, attempt); successive draws without replacement,
 * sorted, A dropped): no per-step host work at all.  ig_get_cycle_plan returns what was drawn. */
int ig_set_neighbour_weights(ig_handle* h, const int64_t* ptr, const int32_t* idx, const double* cdf, const int32_t* n_nonzero);
int ig_run_cycle_device(ig_handle* h, int32_t n_steps, const int32_t* frags, int32_t n_neighbours, uint64_t seed,
                        uint32_t cycle, ig_cycle_step* out);   /* n_neighbours <= IG_MAX_NEIGHBOURS */
int ig_get_cycle_plan(ig_handle* h, int32_t n_steps, int32_t* out /* [n_steps][2 + IG_MAX_CANDS] */);
/* The nuisance-parameter step of the production RNG mode (step_nuisance_parameters, CL:2961-3051; full_em runs it after
 * every step_sampler from cycle 5 on, IG:242-252).  While on, ig_run_cycle_device, ig_run_cycles_device_multi and
 * ig_run_cycle_device_async / ig_cycle_wait run one nuisance step on the device after every step, without host work:
 *   draws     Philox4x32-10 with the chain's seed as key, A = (t, cycle, 0x80000000, 0), B = (t, cycle, 0x80000001, 0):
 *             id_modif = A.x >> 30, acceptance u = 53-bit uniform of (A.y, A.z), draw = sigma * Box-Muller normal of (B)
 *   proposal  the float32 arithmetic of the reference's proposal; d_max = the root of rippe(x) = d_nuc in double,
 *             rounded to float32 (DESIGN.md D3) instead of scipy's fsolve
 *   invalid   (non-finite, fact <= 0, slope >= 0, no root, d_max <= 0, v_inter <= 0): rejected, nothing changes
 *   decision  exp(L_nuis - o) >= u with L_nuis = eval_likelihood_4_nuisance under the proposal on the coordinates of
 *             the step's start (quirk Q5); on acceptance the live parameters become the proposal and the next step
 *             recomputes its likelihood sums (decided on the device).
 * Needs the per-contact likelihood records (not with IG_LNZ_CACHE=0), parameters set with v_inter > 0, and no pending
 * asynchronous cycle.  ig_run_cycle (parity mode, host-drawn neighbours) refuses to run while it is on.  Off (the default):
 * every call behaves as without it.  ig_get_nuisance_records returns the per-step records of the last cycle. */
int ig_set_device_nuisance(ig_handle* h, int32_t on);
int ig_get_nuisance_records(ig_handle* h, int32_t n_steps, ig_nuisance_step* out);
/* Chain temperature T >= 0 of the production RNG mode (DESIGN.md 4e).  T = 0 (the default) is the reference's argmax.  At
 * T > 0 every step of ig_run_cycle_device, ig_run_cycles_device_multi and ig_run_cycle_device_async draws its move among the
 * scored proposals with probability exp((s_i - M) / T) / sum, M = the step's maximum score (Philox4x32-10 with the chain's
 * seed as key, counters (t, cycle, 0x80000002, 0) and, for the batch of a step of more than IG_MAX_CANDS candidates,
 * (t, cycle, 0x80000003, 0)), and the nuisance step accepts when exp((L_nuis - o) / T) >= u.  The host-RNG entry points
 * (ig_step, ig_step_wide, ig_run_cycle, ig_run_cycle_wide) refuse to run at T > 0.  ig_set_temperature refuses NaN, +-inf,
 * negative values and a pending asynchronous cycle; it is stream-ordered (the step graphs read T at replay).
 * ig_get_tempered_records returns the per-step draws of the last cycle (written only at T > 0). */
int ig_set_temperature(ig_handle* h, double temperature);
int ig_get_tempered_records(ig_handle* h, int32_t n_steps, ig_tempered_step* out);
/* eval = score every mutation of one (A,B) pair without applying: extract_uniq_mutations +
 * perform_mutations + slice_sparse_mat + extract_current_sub_likelihood + eval_all_sub_likelihood
 * (CL:1417-1431).  Refreshes the coordinates / full likelihood like the head of step_sampler. */
int ig_eval_scores(ig_handle* h, int32_t id_frag, int32_t id_cand, int32_t flip_eject, double out24[24],
                   int32_t* n_uniq, int32_t* n_sub);
/* apply = test_copy_struct + modify_gl_cuda_buffer (CL:2094-2151, 1453) */
int ig_apply(ig_handle* h, int32_t id_frag, int32_t id_cand, int32_t op, ig_step_result* out);
/* eval_likelihood_4_nuisance (CL:1296-1344) when use_stale_coords=1 (coordinates of the last
 * fill_dist_single, quirk Q5); eval_likelihood on fresh coordinates when 0.
 * out3 = { nz likelihood, raw zeros sum Z (before *log_e), (double) n_vals_intra }. */
int ig_full_likelihood(ig_handle* h, const float p[8], int32_t use_stale_coords, double out3[3]);
/* estimate_parameters_rippe, histogram part (CL:2247-2297): per-bin sum over the first n_rows rows
 * of the SYMMETRIC level L-1 matrix of intra-contig contacts at distance < max_kb, on the initial
 * scaffold; hist[n_bins] int64 sums, rows_used = rows whose contig is longer than bin_kb. */
int ig_distance_histogram(ig_handle* h, double bin_kb, double max_kb, int32_t n_rows, int32_t n_bins,
                          int64_t* hist, int64_t* rows_used);

/* display_current_matrix (CL:2555-2606) without densifying NS x NS on the host: K x K binned contact counts
 * in the displayed order given by sub_rank[NS] (SURVEY 8f, N1) */
int ig_contact_thumbnail(ig_handle* h, const int32_t* sub_rank, int32_t K, uint32_t* out);

/* Diagnostics (builds with -DIG_TIMELINE only; -1 otherwise): per step of the last cycle run, per kernel, the earliest
 * block start and latest block end in %globaltimer ns: out[n_steps][16][2]. */
int ig_timeline_reset(ig_handle* h);
int ig_timeline_get(ig_handle* h, int32_t n_steps, uint64_t* out);
/* per block of the LAST k_score launch: start ns, end ns, SM id, work items: out[n_blocks][4] */
int ig_timeline_blocks(ig_handle* h, int32_t n_blocks, uint64_t* out);
/* k_score phase profile: SM cycles of warp 0 of every block, summed per phase (prologue, item set-up, contact loop,
 * final flush + reductions, wait at the block barrier) since the last reset */
int ig_timeline_phases(ig_handle* h, uint64_t* out8, int32_t reset);

/* diagonal of (M + M^T) at level L-1 (self contacts): only the p(s) histogram sees it (CL:2257-2288) */
int ig_set_sym_diag(ig_handle* h, const int32_t* diag);

/* measurement hooks (no reference counterpart): per-kernel CUDA-event timing on the handle's stream
 * and the scoring kernel's algorithmic traffic counters; see bench.py */
int ig_set_profiling(ig_handle* h, int32_t on);
int ig_get_stats(ig_handle* h, double out10[10], int32_t reset);
/* profiling mode only: accumulated ms between consecutive main-stream launches of a step */
int ig_get_kernel_times(ig_handle* h, double out11[11], int32_t reset);
/* refresh_every = N: recompute coordinates + full likelihood over every contact at least every N steps
 * (1 = every step, the reference's own schedule CL:1407-1409; 0 = only after the state was changed from
 * outside); in between they are maintained incrementally (identical up to f64 summation order).
 * use_graph: replay each step as one CUDA graph. */
int ig_set_options(ig_handle* h, int32_t refresh_every, int32_t use_graph);
/* chains that share one GPU (ig_clone): this chain's scoring grids take 1/share of the SMs so the chains' kernels overlap
 * (no counterpart in the reference, which runs one chain per process and GPU); 1 = the whole machine (default) */
int ig_set_gpu_share(ig_handle* h, int32_t share);
/* device milliseconds spent inside the full-likelihood kernel by ig_full_likelihood calls (the nuisance step's
 * eval_likelihood_4_nuisance, CL:1296-1344) and the number of such calls: out2 = { ms, calls } */
int ig_get_nuisance_stats(ig_handle* h, double out2[2], int32_t reset);
/* number of full refreshes among the steps covered by the last ig_get_stats call */
int ig_get_full_refresh_count(ig_handle* h, int64_t* out);

/* self-test of the device math the kernels use in place of libdevice's powf / double log10 (same results: powf_pos is a
 * transcription of powf's main path, bit-identical for x > 0; log10_f32 agrees to < 4e-16): n samples of x log-uniform in
 * [x_lo, x_hi], exponent y; out2 = { inputs where powf_pos != powf bit-wise, max |log10_f32 - log10| }. */
int ig_selftest_math(ig_handle* h, int32_t n, float x_lo, float x_hi, float y, double out2[2]);

/* ---- replica chains (SURVEY 8e: a chain is sequential, so the 8-GPU box runs independent chains, one or more per GPU).
 * The reference has no counterpart: it is single-process, single-GPU (instagraal.py:55 pycuda.autoinit).
 *
 * ig_clone: a further chain on the same level and device.  Own scaffold / scratch / streams; the contacts, sub-fragment
 * table, initial scaffold and neighbour weights are shared with `parent` (freed with the last chain that uses them). */
int ig_clone(ig_handle* parent, ig_handle** out);
/* ig_run_cycle_device for n_chains chains of one device at once: steps enqueued round-robin on the chains' streams, one wait
 * at the end, so the chains run side by side.  frags = [n_chains][n_steps], seeds = [n_chains], out = [n_chains][n_steps]. */
int ig_run_cycles_device_multi(ig_handle** chains, int32_t n_chains, int32_t n_steps, const int32_t* frags, int32_t n_neighbours,
                               const uint64_t* seeds, uint32_t cycle, ig_cycle_step* out);
/* the same, one chain, without waiting: ig_cycle_wait collects the records of the n_steps enqueued steps */
int ig_run_cycle_device_async(ig_handle* h, int32_t n_steps, const int32_t* frags, int32_t n_neighbours, uint64_t seed, uint32_t cycle);
int ig_cycle_wait(ig_handle* h, int32_t n_steps, ig_cycle_step* out);
/* NCCL all-gather of every chain's likelihood + live scaffold, inside the library (libnccl.so.2 is dlopen'ed on first use).
 * ig_nccl_unique_id: rank 0 creates the id, the launcher distributes it (file, environment, MPI, ...).
 * ig_nccl_init: one communicator per process / GPU, owned by `lead`; n_ranks == 1 needs no id and no NCCL.
 * ig_allgather_best: lik / n_contigs = [n_ranks * n_local] (rank-major); best = index of the highest likelihood (lowest index
 * on ties; the same on every rank); ms = device time of pack + all-gather (CUDA events).
 * ig_get_gathered_state: scaffold [13][NF] of chain `index` as of the last all-gather.
 * ig_adopt_gathered: every local chain whose global index differs from `index` restarts from chain `index` of the last
 * all-gather, on the device: scaffold, live parameters, validity list (quirk Q3) and contig-label counter; its next step is a
 * full refresh and it keeps its own seed.  Chain `index`, if local, is not touched.  Asynchronous: enqueued on the lead's
 * stream, each adopting chain's stream waits for it.  p8_out / valid_out / likelihood_out (each may be NULL) receive the
 * adopted chain's parameters, validity list and likelihood. */
int ig_nccl_unique_id(char id_out[128]);
int ig_nccl_init(ig_handle* lead, int32_t rank, int32_t n_ranks, int32_t n_local_chains, const char id[128]);
int ig_allgather_best(ig_handle* lead, ig_handle** local_chains, int32_t n_local, double* lik, int32_t* n_contigs, int32_t* best,
                      float* ms);
int ig_get_gathered_state(ig_handle* lead, int32_t index, int32_t* out13xNF);
/* the live log-likelihood (likelihood_t: the last applied move's score, or L_nuis after an accepted nuisance proposal) of every
 * chain in the last all-gather, out = [n_ranks * n_local] rank-major */
int ig_get_gathered_live_likelihood(ig_handle* lead, double* out);
int ig_adopt_gathered(ig_handle* lead, ig_handle** local_chains, int32_t n_local, int32_t index, float p8_out[8], int32_t valid_out[12],
                      double* likelihood_out);
int ig_nccl_finalize(ig_handle* lead);
/* ---- pyramid build (SURVEY 8f N2; pyramid_sparse.py:331-397 fill_sparse_pyramid_level, :686-722 the contact part of
 * subsample_data_set): bin n contacts (fa, fb 0-based, count nc) of one level.  old2new (may be NULL = identity) maps an
 * old 0-based fragment id to its new 0-based id; each pair is ordered (smaller id first), equal pairs are summed.
 * first_appearance_order = 0: output sorted by (a, b) -- the text file of the next level;
 * first_appearance_order = 1: rows ascending, inside a row in order of first appearance in the input -- the HDF5 layout.
 * out_* must hold n entries; *n_out = number of distinct pairs.  Handle-free; `device` = CUDA ordinal. */
int ig_bin_contacts(int32_t device, int64_t n, const int32_t* fa, const int32_t* fb, const int32_t* nc, const int32_t* old2new,
                    int32_t n_old, int32_t first_appearance_order, int32_t* out_a, int32_t* out_b, int64_t* out_n, int64_t* n_out);
/* device address of the live scaffold records (64 B per fragment) -- diagnostics */
int ig_device_state_ptr(ig_handle* h, void** dev_ptr, int64_t* n_bytes);

#ifdef __cplusplus
}
#endif
#endif
