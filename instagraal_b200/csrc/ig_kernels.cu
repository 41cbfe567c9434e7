// instagraal_b200 -- hand-written CUDA (sm_100a) for the scaffolding-MCMC hot path + its C ABI.
//
// One ig_step() = one reference step_sampler() (cuda_lib_gl_single.py:1401-1465, "CL") with the
// ~700 host<->device crossings collapsed into 11-12 stream-ordered launches (one CUDA-graph replay) and
// ONE blocking D2H of a 6 KB result record; ig_run_cycle / ig_run_cycle_device enqueue a whole sweep.
// Steps of up to 64 candidates take the same host step (ig_step_wide), cycle plan, graph cache and plan step; only the
// launch sequence differs beyond IG_MAX_CANDS (enqueue_step / enqueue_wide_step, ig_k_wide.cuh).
// Design (DESIGN.md has the long form):
//   * contacts: CSR by row sub-fragment of the strict upper triangle, (col,val) interleaved int2;
//     a candidate touches only the rows of the <=2 affected contigs (ordered row list built on
//     device), never the whole COO, and never through the host.
//   * the 24 candidate scaffolds are never materialised.  Every op moves the fragments between two
//     breakpoints rigidly (ig_moves.cuh): k_classes evaluates each op once per class; the row end of a
//     contact comes from a per-(row, mutation) table (k_precompute), the column end is recomputed on
//     the fly from its class motion with the reference's float32 operations.
//   * scores are sums of DIFFERENCES to the current state over the contacts whose term changes;
//     class-pair bit tables say which (contact, mutation) pairs need a look at all.
//   * three scoring paths, one per handle (choose_scoring): flat (k_pick + k_eval_flat, small levels), stream
//     (k_stream + k_eval_flat, large levels) and rows (k_score, a warp per affected row, the largest levels).
//   * all sums in double, fixed (deterministic) reduction order: lane -> warp shuffle -> block ->
//     partial array -> single-block tree.  No floating-point atomics anywhere.
//   * expected contacts in float32 exactly as the reference kernel writes them (same libdevice
//     powf/expf/log10 calls, same association), so per-contact terms are bit-identical to the
//     reference's eval_sub_likelihood (kernel_sparse_adapt.cu:4236-4370, "KA").
// Tensor cores are deliberately unused: sparse gather + transcendental math, no contraction.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/instagraal_b200.h"
#include "ig_moves.cuh"

#define IG_WARPS_PER_BLOCK 8
#define IG_SCORE_CTAS_PER_SM (24 / IG_WARPS_PER_BLOCK)
#define IG_THREADS (IG_WARPS_PER_BLOCK * 32)
#define IG_ROW_CHUNK 1024
#define IG_FLAT_MAX_NNZ 1500000   // levels up to 1.5 M stored contacts take the flat scoring path (list: 64 B x nnz x 8)
#define IG_ROWS_SMALL_CHUNKS 16  // levels of up to 16 Ki sub-fragments build the affected-row list in one launch
#define IG_STREAM_SMEM_MAX (200 * 1024)   // largest membership bitmap (NS / 8 bytes) k_stream stages in shared memory
#define IG_LANE_CUR 24  // lane that owns the current-state zero term in the score kernel

struct Params { float kuhn, lm, c1, slope, d, d_max, fact, v_inter; };  // KA:91-100
struct SubRec { int parent; float watson; float crick; int j; };          // 16 B
struct CoordRec { float dist; int id_c; int pos; float s_tot; };          // 16 B (uni_fill_vect_dist)
struct __align__(16) SubX { int start_bp; int len_ori; float watson; float crick; };  // 16 B: what a rigid motion needs to
                                                                          // recompute a sub-fragment's coordinate (len_ori = len_bp * ori)

struct __align__(16) RowInfo { int r; int cls; int n; int pad; long long b; long long seg; CoordRec ci; };  // 48 B: all
                                   // k_score needs to start on an affected row, in one round trip
struct CandInfo {  // per-candidate slice description (slice_sp_mat prologue, KA:526-551)
    int id_a, id_b, same, is_circ;
    int up_a, down_a, up_b, down_b;
    int n_rows, n_sub, row_hi, pad;
};

struct DevScalars {
    Params p;          // live parameters
    Params p_test;     // nuisance test parameters
    double log10_vinter, log10_vinter_test;
    int max_label;
    int valid[12];     // gpu_list_valid_insert
    int n_cands, a;
    int cands[IG_MAX_CANDS];
    CandInfo ci[IG_MAX_CANDS];
    double lnz_full, z_cur, lsub_cur[IG_MAX_CANDS];
    int nintra_cur;
    int win_cand, win_op;
    int q4_hits;
    int n_heads; long long sum_l_cont; long long dist_half;
    double scores[IG_MAX_CANDS * IG_N_OPS];
    double z_new[IG_MAX_CANDS * IG_N_OPS];    // zero-term sum Z of the whole scaffold under each scored move
    int nintra_new[IG_MAX_CANDS * IG_N_OPS];  // intra pixel count under each scored move
    double lnz_new[IG_MAX_CANDS * IG_N_OPS];  // full non-zero likelihood of the scaffold under each scored move
    double likelihood;
    // incremental maintenance of (coordinates, lnz_full, z_cur, nintra_cur) across steps
    double lnz_next, z_next; int nintra_next;
    int prev_k, prev_u, prev_windowed, prev_id_a, prev_n_rows;
    unsigned int ticket_out, ticket_post;
    int step_idx, plan_stride;   // entry of the cycle plan the next step reads; ints per entry (2 + W), set by whoever writes the plan
    double full_out[3];
    int full_nintra, pad_;
    double obc_total;   // sum over every stored contact of the observed-count-only part of its term (k_obc_sum)
    unsigned int ticket_cuts[IG_MAX_CANDS], ticket_rows[IG_MAX_CANDS], ticket_fin;  // last-block-done counters
    // measurement: algorithmic traffic of the scoring kernel, accumulated over steps
    unsigned long long st_contacts, st_rows, st_frags, st_selected, st_proposals;
    // flat scoring path (small levels): per candidate, list slots owned by the affected rows (padded row lengths)
    int flat_segtotal[IG_MAX_CANDS];
    // per-candidate counters of the step (written by k_finalize): they travel with this record in ONE copy
    int res_nuniq[IG_MAX_CANDS], res_nsub[IG_MAX_CANDS];
    // streaming scoring path of large levels: which candidates take it, overflow of a pick list
    int use_stream[IG_MAX_CANDS];
    int list_overflow, pad2_;
    // production-mode nuisance step (ig_k_nuis.cuh): the key and cycle of the cycle being run, the proposal in flight, and
    // the flag that tells the next step (kind 3) that its likelihood sums are stale (the proposal was accepted)
    unsigned nuis_key_lo, nuis_key_hi, nuis_cycle;
    int nuis_id, nuis_valid, nuis_stale;
    double nuis_u, nuis_draw;
    // chain temperature (ig_set_temperature, read at replay; 0 = the argmax), the chain's live log-likelihood (the applied
    // move's score, or L_nuis after an accepted nuisance proposal: the facade's likelihood_t) and the tempered draw of the
    // step in flight (ig_k_temper.cuh)
    double temperature, live_likelihood;
    ig_tempered_step trec;
};

struct CycleOut {  // compact per-step record of a cycle (k_post; k_wide_finish fixes up a wide step's)
    double likelihood, lnz_full;
    long long dist_half, sum_l_cont;
    int n_heads, win_cand, win_op, q4_hits;
    int n_proposals, id_f_sampled;   // proposals scored by the step, fragment of the applied move's candidate
};

#include "ig_k_common.cuh"   // optional device-side timeline, the reference's device math (textual twins), reduction helpers
#include "ig_k_state.cuh"   // state of the current scaffold: coordinates, full likelihood over every contact, tables
#include "ig_k_setup.cuh"   // per-candidate setup: descriptor, cut fragments, rigid-motion class tables, ordered affected-row list
#include "ig_k_score.cuh"   // scoring: slice rule, row-end table + zero terms, evaluation queue, the row-per-warp scoring kernel
#include "ig_k_flat.cuh"   // flat scoring path of small levels: k_pick + k_eval_flat
#include "ig_k_rng.cuh"   // production RNG mode: Philox4x32-10 neighbour draws of a whole cycle
#include "ig_k_temper.cuh"   // production RNG mode: move selection at a chain temperature T > 0
#include "ig_k_finish.cuh"   // finalisation, move selection, incremental maintenance, apply, contig bookkeeping, histogram, thumbnail
#include "ig_k_nuis.cuh"   // production RNG mode: the nuisance-parameter step after every step of a cycle
#include "ig_k_wide.cuh"   // steps of more than IG_MAX_CANDS candidates: batch staging, running maximum, fix-ups
static_assert(sizeof(ig_nuisance_step) == 80, "ig_nuisance_step is 80 bytes (NUIS_DTYPE in _lib.py)");
static_assert(sizeof(ig_tempered_step) == 48, "ig_tempered_step is 48 bytes (TEMPERED_DTYPE in _lib.py)");

// ================================================================================================
// host side
// the level's read-only arrays: shared by every chain cloned from one handle (ig_clone), freed with the last of them
struct LevelBlock {
    int refs;
    int max_val;   // largest observed count of the level (decides whether the packed likelihood records can hold it)
    double val_total;   // sum of the observed counts of every stored contact
    long long max_row_len;   // longest CSR row (sizes the pick list of the streaming scoring path)
    int* sym_diag;
    long long* nb_ptr; int* nb_idx; double* nb_cdf; int* nb_nnz;
};
// How a step scores its candidates (choose_scoring):
//   PATH_FLAT    k_rows_small -> k_pick -> k_eval_flat<false>
//   PATH_STREAM  k_rows_count / k_rows_write -> k_stream -> k_eval_flat<true>, beside k_score for the candidates k_cand_setup
//                leaves to it (circular contigs; reference-faithful mode: candidates whose picks might not fit the list)
//   PATH_ROWS    k_rows_count / k_rows_write -> k_score (a warp per affected row) for every candidate
enum ScoringPath { PATH_FLAT, PATH_STREAM, PATH_ROWS };
struct ig_replica_state;
struct ig_handle {
    ig_config cfg;
    LevelBlock* lvl;
    ig_replica_state* rep;   // NCCL communicator + gather buffers (ig_nccl_init), owned by the process's lead handle
    int nf, ns;
    long long nnz;
    cudaStream_t stream, side, pf;
    cudaEvent_t ev_coords, ev_lnz, ev_fork, ev_sel, ev_out, ev_cuts, ev_cls, ev_pre, ev_ksc;
    ScoringPath path;   // chosen once per handle (choose_scoring)
    int2 split;         // k_score's (slots per item, parts per row) forced by IG_FORCE_SPLIT; (0, 0): chosen from the work
    int grid_flat; int* flat_cnt; FlatRec* flat_list; size_t flat_stride, chunk_stride;
    unsigned* bitmap; int bitmap_words; unsigned short* cls16; FlatRec* pick_list; size_t pick_cap; int stream_smem;
    int stream_rows_max;   // candidates with at most this many affected rows take the streaming path (exact mode: bounded by the pick list)
    FragRec *live, *init_live;
    SubRec* sub;
    CoordRec* coord;
    int* clen;
    long long* row_ptr;
    int2* cv;
    int *init_prev, *init_next, *orientable;
    DevScalars* sc;
    IgDescriptor* desc;
    float *exz, *exz_test;
    int n_chunks, *chunk_cnt, *rows, *row_cnt;
    int grid_score, grid_score_full;   // scoring grid in use / the whole machine (ig_set_gpu_share)
    double *part_nz, *part_z; int *part_i, *part_c;
    int grid_pre;
    RowMut* table; int *table_len, *rowidx;
    IgClassTab* clstab; int rigid; SubX* subx; RowInfo* rinfo;
    int* cyc_frags;
    double *part_full; int n_part_full;
    // cached per-contact records of the full likelihood (k_lnz_refresh / k_lnz_stream): 8 B x nnz per chain
    cudaGraphExec_t graph_nuis = nullptr; bool nuis_graph_failed = false; float *h_p8 = nullptr, *d_p8 = nullptr;   // nuisance evaluation as one graph
    int2* lnz_rec; unsigned char* row_dirty; int dp_bits; bool lnz_cache; int grid_lnz; long long lnz_pairs; int lnz_pad;
    double *part_zc; int* part_nc; int n_part_zc;
    int *d_nuniq, *d_nsub, *d_perm;
    unsigned long long* d_hist;
    DevScalars* h_sc;  // pinned mirror
    int* h_small;      // pinned scratch (cands, nuniq, nsub)
    bool params_set, coords_fresh, coords_ever; int init_max_label;
    long long label_hi = 0;          // upper bound of the contig labels in use (2 new ones per applied move), see labels_guard
    bool incr_valid; int refresh_every; long long steps_since_full;
    bool vinter_pos;  // live v_inter > 0 (the per-contact records assume it)
    bool lnz_stale;   // the parameters changed since lnz_full / z_cur were computed (the scaffold bookkeeping is intact)
    double* part_out;
    long long last_n_full;
    // one graph per [step kind + 4 * cycle][shape]: shape = candidates in the grid (1 .. IG_MAX_CANDS) of a narrow step,
    // IG_MAX_CANDS + number of batches of a wide step (get_graph)
    cudaGraphExec_t graph[8][IG_MAX_CANDS + IG_MAX_BATCHES + 1];
    // production-mode nuisance step (ig_set_device_nuisance): one graph per handle replayed after every plan step, the
    // per-step records (cyc_cap of them), and whether a nuisance step was enqueued since the plan began
    bool nuis_on = false, nuis_enqueued = false, nuis_graph_dev_failed = false;
    cudaGraphExec_t graph_nuis_dev = nullptr;
    ig_nuisance_step* nuis_rec = nullptr;
    // chain temperature (ig_set_temperature; the device reads its copy in sc) and the per-step records of the tempered draws
    double temperature = 0.0;
    ig_tempered_step* temp_rec = nullptr;
    // the cycle plan [cyc_cap][2 + W] (n_cands, fragment, candidates), W <= cyc_width; plan_width = W of the last cycle
    int* cyc_plan; CycleOut* cyc_out; int cyc_cap, cyc_width, plan_width; bool graph_failed, capturing, use_graph; long long n_full;
    int pending_steps;   // steps enqueued by an asynchronous cycle call and not collected yet
    // steps of more than IG_MAX_CANDS candidates (ig_k_wide.cuh): the wide record + its pinned mirror
    WideStep *wide = nullptr, *h_wide = nullptr;
    // measurement (CUDA events on the launching stream)
    cudaEvent_t ev[6];
    cudaEvent_t evk[16]; double ms_k[16];  // per-kernel event timing of the main stream (profiling mode)
    double ms_step, ms_score, ms_full, ms_nuis; long long n_nuis;
    long long n_launches, n_steps;
    int profile;
    std::string err;
};

static thread_local std::string g_err;
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf[512];                                                                         \
            snprintf(buf, sizeof buf, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            if (h) h->err = buf; else g_err = buf;                                                 \
            return -2;                                                                             \
        }                                                                                          \
    } while (0)
// Host-to-device copy from pageable memory that is COMPLETE when it returns: a plain cudaMemcpy may return once the data
// is staged, and the kernels run on non-blocking streams that are not ordered against the legacy stream it uses.
static inline cudaError_t h2d_sync(void* dst, const void* src, size_t bytes) {
    cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(cudaStreamLegacy);
}

extern "C" const char* ig_last_error(ig_handle* h) { return h ? h->err.c_str() : g_err.c_str(); }
extern "C" int ig_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

template <class T> static int dev_alloc(ig_handle* h, T** p, size_t n) {
    CK(cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)));
    return 0;
}

static int upload_state(ig_handle* h, const int32_t* in13, FragRec* dst) {
    const int nf = h->nf;
    std::vector<FragRec> tmp(nf);
    for (int i = 0; i < nf; i++) {
        int* v = reinterpret_cast<int*>(&tmp[i].f);
        for (int k = 0; k < IG_N_FIELDS; k++) v[k] = in13[(size_t)k * nf + i];
        tmp[i].pad[0] = tmp[i].pad[1] = tmp[i].pad[2] = 0;
    }
    CK(cudaMemcpyAsync(dst, tmp.data(), sizeof(FragRec) * nf, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// The handle's scoring path and what it sizes, decided once per handle: PATH_FLAT up to 16 Ki sub-fragments and 1.5 M
// contacts, otherwise PATH_STREAM while the membership bitmap fits k_stream's shared memory, otherwise PATH_ROWS; the pick
// list of the streaming path; whether the per-contact likelihood records fit the level.  Tests override the choice:
// IG_SCORING_PATH=flat|stream|rows, IG_FORCE_SPLIT=gs,parts (k_score's work split: gs uniq slots per item, rows cut into
// `parts`; it selects no path, so it acts wherever k_score runs: every candidate of the rows path, the candidates the stream
// path leaves to it, none of the flat path), IG_LNZ_CACHE=0|1.  An override that is malformed or that the level cannot
// honour fails ig_create.
static int choose_scoring(ig_handle* h) {
    const bool flat_ok = h->n_chunks <= IG_ROWS_SMALL_CHUNKS, stream_ok = h->stream_smem <= IG_STREAM_SMEM_MAX;
    h->path = (flat_ok && h->nnz <= IG_FLAT_MAX_NNZ) ? PATH_FLAT : stream_ok ? PATH_STREAM : PATH_ROWS;
    if (const char* e = getenv("IG_SCORING_PATH")) {
        if (!strcmp(e, "flat") && flat_ok) h->path = PATH_FLAT;
        else if (!strcmp(e, "stream") && stream_ok) h->path = PATH_STREAM;
        else if (!strcmp(e, "rows")) h->path = PATH_ROWS;
        else {
            h->err = std::string("ig_create: IG_SCORING_PATH=") + e + " is not one of flat, stream, rows that this level can take "
                     "(flat: up to 16 Ki sub-fragments; stream: up to 1.6 M sub-fragments)";
            return -1;
        }
    }
    h->split = make_int2(0, 0);
    if (const char* e = getenv("IG_FORCE_SPLIT")) {
        int gs = 0, parts = 0, len = 0;
        if (sscanf(e, "%d,%d%n", &gs, &parts, &len) != 2 || e[len] || gs <= 0 || IG_N_OPS % gs || parts < 1 || parts > 32) {
            h->err = std::string("ig_create: IG_FORCE_SPLIT=") + e + " is not gs,parts (gs divides 24, 1 <= parts <= 32)";
            return -1;
        }
        h->split = make_int2(gs, parts);
    }
    h->pick_cap = 0; h->stream_rows_max = 0;
    if (h->path == PATH_STREAM) {
        h->pick_cap = std::min<size_t>((size_t)h->nnz + 64, (size_t)2 << 20);   // 64-byte records: 128 MB per candidate slot at most
        // rigid pruning: every linear candidate (a few per cent of its contacts are picked).  Reference-faithful mode: almost
        // every selected contact is a pick, so only candidates whose contacts are sure to fit the pick list take it (the
        // mid-assembly regime: two contigs of a few hundred sub-fragments, where the row-per-warp kernel is all latency)
        h->stream_rows_max = h->rigid ? INT32_MAX : (int)std::min<long long>(INT32_MAX, (long long)h->pick_cap / std::max<long long>(h->lvl->max_row_len, 1));
    }
    // packed likelihood records: table index (sub-fragment separation, or one of two special slots) in the low bits, the
    // observed count above them
    h->dp_bits = 1;
    while ((1 << h->dp_bits) < h->ns + 3) h->dp_bits++;
    h->lnz_cache = h->nnz > 0 && h->dp_bits <= 24 && (long long)h->lvl->max_val < (1LL << (32 - h->dp_bits));
    if (const char* e = getenv("IG_LNZ_CACHE")) {
        if (!strcmp(e, "0")) h->lnz_cache = false;
        else if (strcmp(e, "1") || !h->lnz_cache) {
            h->err = std::string("ig_create: IG_LNZ_CACHE=") + e + " is not 0, or 1 on a level whose counts and size fit the records";
            return -1;
        }
    }
    return 0;
}

// parent != nullptr: a further chain on the same level (ig_clone): the level's read-only arrays are borrowed, not uploaded
static int create_impl(const ig_config* cfg, const ig_level_data* data, ig_handle* parent, ig_handle** out) {
    ig_handle* h = nullptr;
    if (!cfg || (!data && !parent) || !out) { g_err = "ig_create: null argument"; return -1; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        g_err = "ig_create: no CUDA device available (this library has no CPU path)";
        return -3;
    }
    if (cfg->device < 0 || cfg->device >= ndev) { g_err = "ig_create: bad device ordinal"; return -1; }
    if (cfg->n_frags <= 0 || cfg->n_sub_frags <= 0 || cfg->nnz < 0) { g_err = "ig_create: bad sizes"; return -1; }
    if (cfg->n_sub_frags >= (1 << IG_CLS_SHIFT)) { g_err = "ig_create: more than 2^24 sub-fragments"; return -1; }
    h = new ig_handle();
    h->cfg = *cfg; h->nf = cfg->n_frags; h->ns = cfg->n_sub_frags; h->nnz = cfg->nnz;
    h->rigid = cfg->rigid_pruning ? 1 : 0;
    h->params_set = false; h->coords_fresh = false; h->coords_ever = false;
    h->incr_valid = false; h->lnz_stale = false; h->refresh_every = 4096; h->steps_since_full = 0;
    memset(h->graph, 0, sizeof h->graph); h->cyc_plan = nullptr; h->cyc_out = nullptr; h->cyc_frags = nullptr;
    h->cyc_cap = 0; h->cyc_width = 0; h->plan_width = IG_MAX_CANDS;
    h->graph_failed = false; h->capturing = false; h->use_graph = true; h->n_full = 0; h->pending_steps = 0; h->rep = nullptr;
    cudaError_t e0 = cudaSetDevice(cfg->device);
    if (e0 != cudaSuccess) { g_err = std::string("cudaSetDevice: ") + cudaGetErrorString(e0); delete h; return -2; }
#define CKC(x) do { int r_ = (x); if (r_) { g_err = h->err; ig_destroy(h); return r_; } } while (0)
    auto body = [&]() -> int {
        CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&h->pf, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_cuts, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_cls, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_pre, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_ksc, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_coords, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_lnz, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_sel, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming));
        for (int i = 0; i < 6; i++) CK(cudaEventCreate(&h->ev[i]));
        for (int i = 0; i < 16; i++) { CK(cudaEventCreate(&h->evk[i])); h->ms_k[i] = 0.0; }
        h->ms_step = h->ms_score = h->ms_full = 0.0; h->ms_nuis = 0.0; h->n_nuis = 0; h->n_launches = 0; h->n_steps = 0; h->profile = 0;
        const int nf = h->nf, ns = h->ns;
        if (dev_alloc(h, &h->live, nf) || dev_alloc(h, &h->coord, ns) || dev_alloc(h, &h->clen, ns)) return -2;
        if (parent) {
            h->lvl = parent->lvl; h->lvl->refs++;
            h->init_live = parent->init_live; h->sub = parent->sub; h->row_ptr = parent->row_ptr; h->cv = parent->cv;
            h->init_prev = parent->init_prev; h->init_next = parent->init_next; h->orientable = parent->orientable;
        } else {
            h->lvl = new LevelBlock();
            memset(h->lvl, 0, sizeof(LevelBlock)); h->lvl->refs = 1;
            long long mr = 0, tot = 0;
            int mv = 0;
            for (int r = 0; r < ns; r++) mr = std::max(mr, (long long)(data->row_ptr[r + 1] - data->row_ptr[r]));
            for (long long i = 0; i < h->nnz; i++) { mv = std::max(mv, data->val[i]); tot += data->val[i]; }
            h->lvl->max_row_len = mr; h->lvl->max_val = mv; h->lvl->val_total = (double)tot;
            if (dev_alloc(h, &h->init_live, nf) || dev_alloc(h, &h->sub, ns)) return -2;
            if (dev_alloc(h, &h->row_ptr, (size_t)ns + 1) || dev_alloc(h, &h->cv, (size_t)h->nnz + 2)) return -2;
            if (dev_alloc(h, &h->init_prev, nf) || dev_alloc(h, &h->init_next, nf) || dev_alloc(h, &h->orientable, nf)) return -2;
        }
        if (dev_alloc(h, &h->sc, 1) || dev_alloc(h, &h->desc, IG_MAX_CANDS)) return -2;
        if (dev_alloc(h, &h->exz, (size_t)ns + 3) || dev_alloc(h, &h->exz_test, (size_t)ns + 3)) return -2;   // + the two slots of k_lnz_stream
        h->n_chunks = (ns + IG_ROW_CHUNK - 1) / IG_ROW_CHUNK;
        if (dev_alloc(h, &h->chunk_cnt, (size_t)IG_MAX_CANDS * h->n_chunks)) return -2;
        h->bitmap_words = (ns + 31) / 32;
        h->stream_smem = h->bitmap_words * (int)sizeof(unsigned);
        if (int rc = choose_scoring(h)) return rc;
        h->flat_cnt = nullptr; h->flat_list = nullptr; h->flat_stride = (size_t)h->nnz + 32 * (size_t)ns + 32;   // rows own whole 32-contact chunks
        h->chunk_stride = h->flat_stride / 32 + 1;
        if (h->path == PATH_FLAT) {
            if (dev_alloc(h, &h->flat_cnt, (size_t)IG_MAX_CANDS * h->chunk_stride) ||
                dev_alloc(h, &h->flat_list, (size_t)IG_MAX_CANDS * h->flat_stride)) return -2;
        }
        if (dev_alloc(h, &h->rows, (size_t)IG_MAX_CANDS * ns) || dev_alloc(h, &h->row_cnt, (size_t)IG_MAX_CANDS * ns)) return -2;
        h->bitmap = nullptr; h->cls16 = nullptr; h->pick_list = nullptr;
        if (h->path == PATH_STREAM) {   // (the two-pass row list also writes the bitmap and the class words)
            if (dev_alloc(h, &h->bitmap, (size_t)IG_MAX_CANDS * h->bitmap_words) || dev_alloc(h, &h->cls16, (size_t)IG_MAX_CANDS * ns) ||
                dev_alloc(h, &h->pick_list, (size_t)IG_MAX_CANDS * h->pick_cap)) return -2;
            CK(cudaFuncSetAttribute(k_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, h->stream_smem));
        }
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, cfg->device));
        const int sms = prop.multiProcessorCount;
        h->grid_score = sms * IG_SCORE_CTAS_PER_SM;  // 24 resident warps per SM (80 registers per thread; 6 KB of accumulators per warp)
        h->grid_score_full = h->grid_score;
        CK(cudaFuncSetAttribute(k_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IG_SCORE_SMEM));
        CK(cudaFuncSetAttribute(k_eval_flat<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IG_SCORE_SMEM));
        CK(cudaFuncSetAttribute(k_eval_flat<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IG_SCORE_SMEM));
        h->grid_flat = (sms * IG_SCORE_CTAS_PER_SM) / 5;   // k_pick grid per candidate: a step's (usually 5) candidates fill the GPU once
        h->grid_pre = std::min(sms * 2, (ns + 31) / 32);   // 2 resident CTAs of 25 warps per SM; one tile of 32 rows per block at most
        if (dev_alloc(h, &h->part_nz, (size_t)IG_MAX_CANDS * h->grid_score * 25)) return -2;
        if (dev_alloc(h, &h->part_c, (size_t)IG_MAX_CANDS * h->grid_score * 2)) return -2;
        if (dev_alloc(h, &h->part_z, (size_t)IG_MAX_CANDS * h->grid_pre * 25)) return -2;
        if (dev_alloc(h, &h->part_i, (size_t)IG_MAX_CANDS * h->grid_pre * 25)) return -2;
        if (dev_alloc(h, &h->table, (size_t)IG_MAX_CANDS * IG_N_OPS * ns)) return -2;
        if (dev_alloc(h, &h->table_len, (size_t)IG_MAX_CANDS * IG_N_OPS * ns)) return -2;
        if (dev_alloc(h, &h->rowidx, (size_t)IG_MAX_CANDS * ns)) return -2;
        if (dev_alloc(h, &h->clstab, (size_t)IG_MAX_CANDS) || dev_alloc(h, &h->subx, (size_t)ns) || dev_alloc(h, &h->rinfo, (size_t)IG_MAX_CANDS * ns)) return -2;
        h->n_part_full = sms * 8;
        if (dev_alloc(h, &h->part_full, 2 * (size_t)h->n_part_full)) return -2;
        h->lnz_rec = nullptr; h->row_dirty = nullptr; h->grid_lnz = sms * 4;
        if (dev_alloc(h, &h->part_out, h->n_part_full)) return -2;
        h->n_part_zc = sms * 2;
        if (dev_alloc(h, &h->part_zc, h->n_part_zc) || dev_alloc(h, &h->part_nc, h->n_part_zc)) return -2;
        if (dev_alloc(h, &h->d_perm, nf)) return -2;
        h->d_nuniq = h->sc->res_nuniq; h->d_nsub = h->sc->res_nsub;   // device addresses inside the result record
        if (dev_alloc(h, &h->d_hist, 1 << 16)) return -2;
        CK(cudaMallocHost((void**)&h->h_sc, sizeof(DevScalars)));
        CK(cudaMallocHost((void**)&h->h_small, 64 * sizeof(int)));
        CK(cudaMallocHost((void**)&h->h_p8, sizeof(Params)));
        if (dev_alloc(h, &h->d_p8, 8) || dev_alloc(h, &h->wide, 1)) return -2;
        CK(cudaMallocHost((void**)&h->h_wide, sizeof(WideStep)));
        CK(cudaMemsetAsync(h->sc, 0, sizeof(DevScalars), h->stream));
        // uploads
        if (parent) {
            CK(cudaMemcpyAsync(h->live, h->init_live, sizeof(FragRec) * nf, cudaMemcpyDeviceToDevice, h->stream));
        } else {
            if (upload_state(h, data->frags13, h->live)) return -2;
            CK(cudaMemcpy(h->init_live, h->live, sizeof(FragRec) * nf, cudaMemcpyDeviceToDevice));
            {
                std::vector<SubRec> s(ns);
                for (int i = 0; i < ns; i++) {
                    s[i].parent = data->sub_parent[i]; s[i].watson = data->sub_watson[i];
                    s[i].crick = data->sub_crick[i]; s[i].j = data->sub_j[i];
                    if (s[i].parent < 0 || s[i].parent >= nf) { h->err = "ig_create: sub_parent out of range"; return -1; }
                }
                CK(h2d_sync(h->sub, s.data(), sizeof(SubRec) * ns));
            }
            if (data->row_ptr[0] != 0 || data->row_ptr[ns] != h->nnz) { h->err = "ig_create: row_ptr inconsistent with nnz"; return -1; }
            CK(h2d_sync(h->row_ptr, data->row_ptr, sizeof(long long) * ((size_t)ns + 1)));
            {
                const size_t chunk = 1 << 24;
                std::vector<int2> buf(std::min<size_t>(chunk, (size_t)h->nnz));
                for (size_t off = 0; off < (size_t)h->nnz; off += chunk) {
                    const size_t n = std::min(chunk, (size_t)h->nnz - off);
                    for (size_t i = 0; i < n; i++) { buf[i].x = data->col[off + i]; buf[i].y = data->val[off + i]; }
                    CK(h2d_sync(h->cv + off, buf.data(), n * sizeof(int2)));
                }
            }
            CK(cudaMemset(h->cv + h->nnz, 0, 2 * sizeof(int2)));   // k_full_lnz reads contacts in aligned pairs
            CK(h2d_sync(h->init_prev, data->init_prev, sizeof(int) * nf));
            CK(h2d_sync(h->init_next, data->init_next, sizeof(int) * nf));
            CK(h2d_sync(h->orientable, data->orientable, sizeof(int) * nf));
        }
        {   // packed likelihood records (choose_scoring), streamed in whole trips of 64 record pairs
            h->lnz_pairs = ((h->nnz + 1) / 2 + 63) / 64 * 64;
            h->lnz_pad = (int)(2 * h->lnz_pairs - h->nnz);
            if (h->lnz_cache) {
                if (dev_alloc(h, &h->lnz_rec, (size_t)(2 * h->lnz_pairs)) || dev_alloc(h, &h->row_dirty, (size_t)ns)) return -2;
                std::vector<int2> pad(h->lnz_pad);
                for (auto& q : pad) { const float m1 = -1.0f; memcpy(&q.x, &m1, 4); q.y = ns + 2; }   // "skip" records
                if (h->lnz_pad) CK(h2d_sync(h->lnz_rec + h->nnz, pad.data(), sizeof(int2) * pad.size()));
                CK(cudaMemsetAsync(h->row_dirty, 1, (size_t)ns, h->stream));   // every row's records are built on first use
            }
        }
        // factorial table on the device (same libdevice calls as the reference's factorial())
        double* d16;
        CK(cudaMalloc((void**)&d16, 16 * sizeof(double)));
        k_init_tables<<<1, 32, 0, h->stream>>>(d16);
        double h16[16];
        CK(cudaMemcpyAsync(h16, d16, sizeof h16, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpyToSymbol(c_log10_fact, h16, sizeof h16));
        CK(cudaFree(d16));
        {   // log10_f32: bucket centres of the float mantissa
            double2 tab[128];
            for (int i = 0; i < 128; i++) { const double c = 1.0 + (i + 0.5) / 128.0; tab[i].x = 1.0 / c; tab[i].y = log10(c); }
            CK(cudaMemcpyToSymbol(g_log10tab, tab, sizeof tab));
        }
        // observed-count-only part of the likelihood terms, summed once (it depends on neither scaffold nor parameters)
        if (parent) {
            CK(cudaMemcpyAsync(&h->sc->obc_total, &parent->sc->obc_total, sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
        } else {
            k_obc_sum<<<h->n_part_full, IG_THREADS, 0, h->stream>>>(h->cv, h->nnz, h->part_full);
            k_reduce<<<1, 256, 0, h->stream>>>(h->part_full, h->n_part_full, &h->sc->obc_total, nullptr, nullptr);
        }
        CK(cudaStreamSynchronize(h->stream));
        // label counter: labels in the initial scaffold are arbitrary; start above their maximum
        int maxlab = 0;
        if (parent) maxlab = parent->init_max_label;
        else for (int i = 0; i < nf; i++) maxlab = std::max(maxlab, data->frags13[(size_t)2 * nf + i]);
        h->init_max_label = maxlab; h->label_hi = maxlab;
        CK(h2d_sync(&h->sc->max_label, &maxlab, sizeof(int)));
        return 0;
    };
    int rc = body();
    if (rc) { g_err = h->err; ig_destroy(h); return rc; }
    *out = h;
    return 0;
}

extern "C" int ig_create(const ig_config* cfg, const ig_level_data* data, ig_handle** out) {
    if (!data) { g_err = "ig_create: null argument"; return -1; }
    return create_impl(cfg, data, nullptr, out);
}
// A further chain on the SAME level and device (replicas with different seeds, several per GPU): own scaffold, scratch,
// streams and graphs; the contacts, sub-fragment table and initial scaffold (the bulk of the memory: 8 B per contact)
// are shared with `parent` and freed when the last chain using them is destroyed.  The clone starts from the level's
// initial scaffold with no parameters set.
extern "C" int ig_clone(ig_handle* parent, ig_handle** out) {
    if (!parent || !out) { g_err = "ig_clone: null argument"; return -1; }
    return create_impl(&parent->cfg, nullptr, parent, out);
}

// the step graphs of slots first_slot .. 7 (4 and up: cycle graphs) and the device nuisance graph, which bake in the
// cycle buffers and the scoring grids
static void destroy_graphs(ig_handle* h, int first_slot) {
    for (int i = first_slot; i < 8; i++)
        for (cudaGraphExec_t& g : h->graph[i]) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    if (h->graph_nuis_dev) { cudaGraphExecDestroy(h->graph_nuis_dev); h->graph_nuis_dev = nullptr; }
}

static void replica_free(ig_handle* h);
extern "C" void ig_destroy(ig_handle* h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    replica_free(h);
    if (h->lvl && --h->lvl->refs > 0) {   // other chains still use the level's arrays
        h->init_live = nullptr; h->sub = nullptr; h->row_ptr = nullptr; h->cv = nullptr;
        h->init_prev = nullptr; h->init_next = nullptr; h->orientable = nullptr;
    } else if (h->lvl) {
        for (void* q : {(void*)h->lvl->sym_diag, (void*)h->lvl->nb_ptr, (void*)h->lvl->nb_idx, (void*)h->lvl->nb_cdf, (void*)h->lvl->nb_nnz}) if (q) cudaFree(q);
        delete h->lvl;
    }
    h->lvl = nullptr;
    void* ptrs[] = {h->lnz_rec, h->row_dirty, h->bitmap, h->cls16, h->pick_list, h->flat_cnt, h->flat_list, h->clstab, h->subx, h->rinfo, h->cyc_frags, h->live, h->part_out, h->part_c, h->table, h->table_len, h->rowidx, h->init_live, h->sub, h->coord, h->clen, h->row_ptr, h->cv,
                    h->init_prev, h->init_next, h->orientable, h->sc, h->desc, h->exz, h->exz_test, h->chunk_cnt,
                    h->rows, h->row_cnt, h->part_nz, h->part_z, h->part_i, h->part_full, h->part_zc, h->part_nc,
                    h->d_perm, h->d_hist};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (h->h_sc) cudaFreeHost(h->h_sc);
    if (h->h_small) cudaFreeHost(h->h_small);
    if (h->h_p8) cudaFreeHost(h->h_p8);
    if (h->d_p8) cudaFree(h->d_p8);
    if (h->graph_nuis) cudaGraphExecDestroy(h->graph_nuis);
    if (h->nuis_rec) cudaFree(h->nuis_rec);
    if (h->temp_rec) cudaFree(h->temp_rec);
    if (h->wide) cudaFree(h->wide);
    if (h->h_wide) cudaFreeHost(h->h_wide);
    for (int i = 0; i < 6; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    for (int i = 0; i < 16; i++) if (h->evk[i]) cudaEventDestroy(h->evk[i]);
    destroy_graphs(h, 0);
    if (h->cyc_plan) cudaFree(h->cyc_plan);
    if (h->cyc_out) cudaFree(h->cyc_out);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->pf) cudaStreamDestroy(h->pf);
    if (h->ev_cuts) cudaEventDestroy(h->ev_cuts);
    if (h->ev_cls) cudaEventDestroy(h->ev_cls);
    if (h->ev_pre) cudaEventDestroy(h->ev_pre);
    if (h->ev_ksc) cudaEventDestroy(h->ev_ksc);
    if (h->ev_coords) cudaEventDestroy(h->ev_coords);
    if (h->ev_lnz) cudaEventDestroy(h->ev_lnz);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_sel) cudaEventDestroy(h->ev_sel);
    if (h->ev_out) cudaEventDestroy(h->ev_out);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

static int use(ig_handle* h) {
    if (!h) { g_err = "null handle"; return -1; }
    CK(cudaSetDevice(h->cfg.device));
    return 0;
}
static int launch_ok(ig_handle* h, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { h->err = std::string(what) + ": " + cudaGetErrorString(e); return -2; }
    return 0;
}

extern "C" int ig_set_params(ig_handle* h, const float p8[8]) {
    if (use(h)) return -1;
    Params p; memcpy(&p, p8, sizeof p);
    k_set_params<<<1, 1, 0, h->stream>>>(h->sc, p, 0);
    k_exz_table<<<std::min(1024, (h->ns + 256) / 256), 256, 0, h->stream>>>(h->exz, h->ns + 1, h->sc, h->cfg.mean_sub_len_kb, 0);
    if (launch_ok(h, "set_params")) return -2;
    CK(cudaStreamSynchronize(h->stream));
    h->params_set = true;
    h->vinter_pos = p.v_inter > 0.0f;
    h->lnz_stale = true;  // lnz_full / z_cur depend on the parameters: the next step recomputes them (step_kind)
    return 0;
}

// renumber like modify_gl_cuda_buffer (CL:2715-2806): contigs listed in ascending index of their
// head fragment (sequential select_uniq_id_c), stable sort by length descending, id = NC-1-rank.
static void canonical_labels(int nf, int32_t* st13) {
    int32_t* pos = st13; int32_t* id_c = st13 + (size_t)2 * nf; int32_t* l_cont = st13 + (size_t)9 * nf;
    std::vector<int> heads;
    for (int i = 0; i < nf; i++) if (pos[i] == 0) heads.push_back(i);
    std::vector<int> order(heads.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return l_cont[heads[x]] > l_cont[heads[y]]; });
    std::vector<std::pair<int, int>> lut;  // (old label, rank)
    lut.reserve(heads.size());
    for (size_t r = 0; r < order.size(); r++) lut.push_back({id_c[heads[order[r]]], (int)r});
    std::stable_sort(lut.begin(), lut.end(), [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first < b.first; });
    const int nc = (int)heads.size();
    for (int i = 0; i < nf; i++) {
        auto it = std::upper_bound(lut.begin(), lut.end(), std::make_pair(id_c[i], INT32_MAX));
        if (it != lut.begin() && (it - 1)->first == id_c[i]) id_c[i] = (nc - 1) - (it - 1)->second;
    }
}

extern "C" int ig_get_state(ig_handle* h, int32_t* out13) {
    if (use(h)) return -1;
    const int nf = h->nf;
    std::vector<FragRec> tmp(nf);
    CK(cudaMemcpyAsync(tmp.data(), h->live, sizeof(FragRec) * nf, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < nf; i++) {
        const int* v = reinterpret_cast<const int*>(&tmp[i].f);
        for (int k = 0; k < IG_N_FIELDS; k++) out13[(size_t)k * nf + i] = v[k];
    }
    canonical_labels(nf, out13);
    return 0;
}
extern "C" int ig_set_state(ig_handle* h, const int32_t* in13) {
    if (use(h)) return -1;
    if (upload_state(h, in13, h->live)) return -2;
    int maxlab = 0;
    for (int i = 0; i < h->nf; i++) maxlab = std::max(maxlab, in13[(size_t)2 * h->nf + i]);
    CK(h2d_sync(&h->sc->max_label, &maxlab, sizeof(int)));
    h->label_hi = maxlab;
    h->coords_fresh = false;
    h->incr_valid = false;
    return 0;
}
// (the handle's stream is drained first: ig_adopt_gathered writes the list asynchronously, and these copies run on the
// legacy stream, which is not ordered with the handle's non-blocking one)
extern "C" int ig_get_valid_insert(ig_handle* h, int32_t out12[12]) {
    if (use(h)) return -1;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out12, h->sc->valid, 12 * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" int ig_set_valid_insert(ig_handle* h, const int32_t in12[12]) {
    if (use(h)) return -1;
    CK(cudaStreamSynchronize(h->stream));
    CK(h2d_sync(h->sc->valid, in12, 12 * sizeof(int)));
    return 0;
}
extern "C" int ig_bomb(ig_handle* h, const int32_t* perm) {
    if (use(h)) return -1;
    CK(cudaMemcpyAsync(h->d_perm, perm, sizeof(int) * h->nf, cudaMemcpyHostToDevice, h->stream));
    k_explode<<<(h->nf + 255) / 256, 256, 0, h->stream>>>(h->live, h->nf, h->d_perm);
    if (launch_ok(h, "explode")) return -2;
    int maxlab = h->nf;  // perm values are 0..NF-1
    h->label_hi = maxlab;
    CK(cudaMemcpyAsync(&h->sc->max_label, &maxlab, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->coords_fresh = false;
    h->incr_valid = false;
    return 0;
}

// Contig labels are only ever compared for equality, so every applied move simply takes two fresh ones (max_label += 2).
// Long before the int32 counter could wrap (~5e8 steps) the labels are re-based to 0..NC-1 through the canonical
// relabelling of ig_get_state (what the reference does after every step, CL:2715-2806); the next step then refreshes fully.
static int labels_guard(ig_handle* h) {
    h->label_hi += 2;
    if (h->label_hi < (1LL << 30)) return 0;
    std::vector<int32_t> st((size_t)IG_N_FIELDS * h->nf);
    if (int rc = ig_get_state(h, st.data())) return rc;
    return ig_set_state(h, st.data());
}

// rows + precompute + scoring kernels of one pass (after k_cand_setup / k_find_cuts were enqueued, k_classes on h->pf)
#define IG_MARK(i) do { if (h->profile && !h->capturing) cudaEventRecord(h->evk[i], h->stream); } while (0)
static void enqueue_scoring(ig_handle* h, int n) {
    const float mbar = h->cfg.mean_sub_len_kb;
    const FragRec* live = h->live;
    if (h->path == PATH_FLAT) {
        IG_MARK(3);
        k_rows_small<<<n, IG_ROW_CHUNK, 0, h->stream>>>(h->coord, h->ns, h->sc, h->n_chunks, h->rows, h->rowidx, h->row_cnt, h->ns,
                                                        h->clstab, h->row_ptr, h->rinfo);
    } else {
        k_rows_count<<<h->n_chunks, IG_ROW_CHUNK, 0, h->stream>>>(h->coord, h->ns, h->sc, h->chunk_cnt, h->n_chunks);
        IG_MARK(3);
        k_rows_write<<<h->n_chunks, IG_ROW_CHUNK, 0, h->stream>>>(h->coord, h->ns, h->sc, h->chunk_cnt, h->n_chunks, h->rows,
                                                                           h->rowidx, h->row_cnt, h->ns, h->clstab, h->row_ptr, h->rinfo,
                                                                           h->bitmap, h->bitmap_words, h->cls16);
    }
    IG_MARK(4);
    k_precompute<<<dim3(h->grid_pre, n), IG_PRE_THREADS, 0, h->stream>>>(h->coord, h->clen, live, h->sub, h->sc, h->desc, h->rows, h->ns,
                                                                    h->table, h->table_len, mbar, h->part_z, h->part_i);
    if (h->profile && !h->capturing) cudaEventRecord(h->ev[4], h->stream);
    cudaStreamWaitEvent(h->stream, h->ev_cls, 0);
    IG_MARK(5);
    if (h->path == PATH_FLAT) {
        k_pick<<<dim3(h->grid_flat, n), IG_THREADS, 0, h->stream>>>(h->cv, h->coord, h->clen, h->sc, h->desc, h->rowidx, h->ns, h->row_cnt,
                                                                    h->flat_cnt, h->chunk_stride, h->part_c, h->flat_list, h->flat_stride, mbar, h->exz,
                                                                    h->clstab, h->subx, h->rinfo);
        k_eval_flat<false><<<h->grid_score, IG_THREADS, IG_SCORE_SMEM, h->stream>>>(h->sc, h->desc, h->ns, h->flat_cnt, h->chunk_stride, h->flat_list,
                                                                            h->flat_stride, h->table, h->table_len, mbar, h->exz, h->part_nz, h->clstab);
    } else {
        // (streaming mode: k_score only works for the candidates k_stream leaves to it -- circular contigs, and in the
        //  reference-faithful mode the candidates whose picks would not fit the list.  It runs BESIDE the streaming pair on
        //  the third stream -- different candidates, different partials -- and joins before k_finalize.)
        cudaStream_t ks = h->stream;
        if (h->path == PATH_STREAM) {
            ks = h->pf;   // (k_classes ran on it: already ordered)
            cudaEventRecord(h->ev_pre, h->stream);
            cudaStreamWaitEvent(ks, h->ev_pre, 0);
            k_stream<<<dim3(h->grid_score, n), IG_THREADS, h->stream_smem, h->stream>>>(h->cv, h->coord, h->clen, h->sc, h->desc, h->rowidx, h->ns, h->row_cnt,
                                                                             h->bitmap, h->bitmap_words, h->cls16, h->part_c, h->pick_list, h->pick_cap,
                                                                             mbar, h->exz, h->clstab, h->subx, h->rinfo);
            k_eval_flat<true><<<h->grid_score, IG_THREADS, IG_SCORE_SMEM, h->stream>>>(h->sc, h->desc, h->ns, nullptr, 0, h->pick_list, h->pick_cap,
                                                                               h->table, h->table_len, mbar, h->exz, h->part_nz, h->clstab);
        }
        k_score<<<dim3(h->grid_score, n), IG_THREADS, IG_SCORE_SMEM, ks>>>(h->row_ptr, h->cv, h->coord, h->clen, h->sc, h->desc, h->rows,
                                                                          h->rowidx, h->ns, h->row_cnt, h->table, h->table_len, mbar, h->exz,
                                                                          h->part_nz, h->part_c, h->clstab, h->subx, h->rinfo, h->split);
        if (ks != h->stream) {
            cudaEventRecord(h->ev_ksc, ks);
            cudaStreamWaitEvent(h->stream, h->ev_ksc, 0);
        }
    }
    if (h->profile && !h->capturing) cudaEventRecord(h->ev[5], h->stream);
}

static int apply_and_post(ig_handle* h, int forced_cand, int forced_op) {
    const int nf = h->nf;
    h->label_hi += 2;
    k_apply<<<(nf + 255) / 256, 256, 0, h->stream>>>(h->live, nf, h->sc, h->desc, forced_cand, forced_op);
    k_post_scalars<<<1, 1, 0, h->stream>>>(h->sc, h->desc, forced_cand, forced_op);
    k_post<<<(nf + 255) / 256, 256, 0, h->stream>>>(h->live, nf, h->init_prev, h->init_next, h->orientable, h->sc, nullptr, nullptr);
    h->coords_fresh = false;
    h->n_launches += 3;
    return launch_ok(h, "apply");
}

// the result of the last step or scoring pass of n candidates from the scalar record (and the wide record beyond
// IG_MAX_CANDS): `out` holds the first IG_MAX_CANDS candidates' values (applied: and the move), scores / n_uniq / n_sub
// (where given) all n.  copy: download the scalar record first (a step enqueues that copy itself)
static int fetch_result(ig_handle* h, int n, const int32_t* cands, ig_step_result* out, bool applied, bool copy = true,
                        double* scores = nullptr, int32_t* n_uniq = nullptr, int32_t* n_sub = nullptr) {
    if (copy) {
        CK(cudaMemcpyAsync(h->h_sc, h->sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    const DevScalars& s = *h->h_sc;
    if (s.list_overflow) { h->err = "pick list of the streaming scoring path overflowed"; return -4; }
    const bool wide = n > IG_MAX_CANDS;
    const double* sv = wide ? h->h_wide->scores : s.scores;
    const int* nu = wide ? h->h_wide->n_uniq : s.res_nuniq;
    const int* nsub = wide ? h->h_wide->n_sub : s.res_nsub;
    const int m = std::min(n, IG_MAX_CANDS);
    memset(out, 0, sizeof *out);
    for (int i = 0; i < m * IG_N_OPS; i++) out->scores[i] = sv[i];
    for (int i = 0; i < m; i++) { out->n_uniq[i] = nu[i]; out->n_sub[i] = nsub[i]; }
    if (scores) for (int i = 0; i < n * IG_N_OPS; i++) scores[i] = sv[i];
    for (int i = 0; i < n; i++) { if (n_uniq) n_uniq[i] = nu[i]; if (n_sub) n_sub[i] = nsub[i]; }
    out->lnz_full = s.lnz_full;
    out->q4_hits = s.q4_hits;
    if (applied) {
        const int win = wide ? h->h_wide->win_cand : s.win_cand;
        out->likelihood = s.likelihood;
        out->cand_index = win; out->op_sampled = s.win_op;
        out->id_f_sampled = cands[win];
        out->n_contigs = s.n_heads; out->sum_l_cont = s.sum_l_cont;
        out->dist = (3.0 * h->nf - 0.5 * (double)s.dist_half) / (3.0 * h->nf);
    }
    return 0;
}

// Everything one step enqueues (no host synchronisation): used directly and under graph capture.
//   full = 1: fill_dist_single + eval_likelihood over every contact (CL:1407-1409), on the side stream,
//             overlapped with the candidate setup on the main stream;
//   full = 0: incremental refresh from the previous step's mutation table (same values up to f64
//             summation order), O(rows of the last move).
// head of a step: the side streams fork from the main stream, then the refresh or incremental commit of `full` runs on the
// side stream (ev_coords / ev_lnz mark its coordinates and its likelihood sums)
static void enqueue_head(ig_handle* h, int full) {
    const float mbar = h->cfg.mean_sub_len_kb;
    cudaEventRecord(h->ev_fork, h->stream);
    cudaStreamWaitEvent(h->side, h->ev_fork, 0);
    cudaStreamWaitEvent(h->pf, h->ev_fork, 0);
    if (full == 2 || full == 3) {
        // parameters changed, scaffold bookkeeping intact (an accepted nuisance proposal): coordinates as in the incremental
        // step (k_commit_coords flags the rows of the previous move), zero terms and the full non-zero likelihood recomputed
        // under the new parameters -- the latter from the cached per-contact records (k_lnz_refresh + k_lnz_stream).
        // Kind 3 (production-mode nuisance step): the same launches, but the recomputation only runs when the previous
        // step's nuisance proposal was accepted (sc->nuis_stale); otherwise it is the incremental step, kind 0
        const int* pred = full == 3 ? &h->sc->nuis_stale : nullptr;
        k_commit_coords<<<std::min(h->n_part_zc, (h->ns + 255) / 256), 256, 0, h->side>>>(h->coord, h->clen, h->sc, h->rows, h->ns,
                                                                                         h->table, h->table_len, h->live, h->sub, h->subx, h->row_dirty);
        k_coords<<<h->n_part_zc, IG_THREADS, 0, h->side>>>(h->live, h->sub, h->coord, h->clen, h->ns, h->sc, mbar, 0, h->part_zc,
                                                          h->part_nc, 0, h->subx, nullptr, pred);
        k_reduce<<<1, 256, 0, h->side>>>(h->part_zc, h->n_part_zc, &h->sc->z_cur, h->part_nc, &h->sc->nintra_cur, pred);
        cudaEventRecord(h->ev_coords, h->side);
        if (h->profile && !h->capturing) cudaEventRecord(h->ev[2], h->side);
        k_lnz_refresh<<<h->grid_lnz, IG_THREADS, 0, h->side>>>(h->row_ptr, h->cv, h->coord, h->clen, h->ns, h->sc, mbar, 0, h->exz,
                                                               h->lnz_rec, h->row_dirty, h->dp_bits, h->part_full + h->grid_lnz, pred);
        k_lnz_stream<<<h->grid_lnz, IG_THREADS, 0, h->side>>>(reinterpret_cast<const int4*>(h->lnz_rec), h->lnz_pairs, h->lnz_pad,
                                                              h->lvl->val_total, h->sc, 0, h->exz, h->dp_bits, h->part_full, pred);
        if (h->profile && !h->capturing) cudaEventRecord(h->ev[3], h->side);
        k_reduce<<<1, 256, 0, h->side>>>(h->part_full, 2 * h->grid_lnz, &h->sc->lnz_full, nullptr, nullptr, pred);
        cudaEventRecord(h->ev_lnz, h->side);
    } else if (full) {
        k_coords<<<h->n_part_zc, IG_THREADS, 0, h->side>>>(h->live, h->sub, h->coord, h->clen, h->ns, h->sc, mbar, 0, h->part_zc,
                                                          h->part_nc, 1, h->subx, h->row_dirty);
        k_reduce<<<1, 256, 0, h->side>>>(h->part_zc, h->n_part_zc, &h->sc->z_cur, h->part_nc, &h->sc->nintra_cur);
        cudaEventRecord(h->ev_coords, h->side);
        if (h->profile && !h->capturing) cudaEventRecord(h->ev[2], h->side);
        k_full_lnz<<<h->n_part_full, IG_THREADS, 0, h->side>>>(h->row_ptr, h->cv, h->coord, h->clen, h->ns, h->sc, mbar, 0, h->exz,
                                                              h->part_full);
        if (h->profile && !h->capturing) cudaEventRecord(h->ev[3], h->side);
        k_reduce<<<1, 256, 0, h->side>>>(h->part_full, h->n_part_full, &h->sc->lnz_full, nullptr, nullptr);
        cudaEventRecord(h->ev_lnz, h->side);
    } else {
        k_commit_coords<<<std::min(h->n_part_zc, (h->ns + 255) / 256), 256, 0, h->side>>>(h->coord, h->clen, h->sc, h->rows, h->ns,
                                                                                         h->table, h->table_len, h->live, h->sub, h->subx, h->row_dirty);
        cudaEventRecord(h->ev_coords, h->side);
        cudaEventRecord(h->ev_lnz, h->side);
    }
}
// one scoring pass over the candidates in sc (or, plan != nullptr, in the cycle plan's entry sc->step_idx): setup, row list,
// precompute, scoring, k_finalize (do_select: with the move selection); wide_rescore: the re-score of a wide step's winning
// batch (k_wide_flip)
static void enqueue_pass(ig_handle* h, int n, int first_flip_eject, const int* plan, int do_select, bool wide_rescore = false) {
    const float mbar = h->cfg.mean_sub_len_kb;
    const FragRec* live = h->live;
    IG_MARK(0);
    k_cand_setup<<<1, 32, 0, h->stream>>>(live, h->sc, h->desc, h->cfg.max_bounds_insert, first_flip_eject, plan, h->path == PATH_STREAM ? h->stream_rows_max : 0);
    if (wide_rescore) k_wide_flip<<<1, 32, 0, h->stream>>>(h->sc, h->desc, h->wide);
    IG_MARK(1);
    k_find_cuts<<<(h->nf + 255) / 256, 256, 0, h->stream>>>(live, h->nf, h->sc, h->desc, h->clstab);
    cudaEventRecord(h->ev_cuts, h->stream);
    cudaStreamWaitEvent(h->pf, h->ev_cuts, 0);
    k_classes<<<n, IG_N_OPS * 32, 0, h->pf>>>(h->sc, h->desc, h->clstab, h->rigid, h->cfg.mean_sub_len_kb);   // beside the row list; k_score needs it
    cudaEventRecord(h->ev_cls, h->pf);
    cudaStreamWaitEvent(h->stream, h->ev_coords, 0);
    IG_MARK(2);
    enqueue_scoring(h, n);
    const bool flat = h->path == PATH_FLAT;
    cudaStreamWaitEvent(h->stream, h->ev_lnz, 0);
    IG_MARK(6);
    k_finalize<<<n, 1024, 0, h->stream>>>(h->row_ptr, h->cv, h->coord, h->sc, h->desc, h->rows, h->rowidx, h->ns, h->row_cnt, h->table,
                                         h->table_len, mbar, h->exz, h->part_nz, h->part_c, h->grid_score, h->part_z, h->part_i, h->grid_pre,
                                         h->cfg.n_pix, h->cfg.compat_last_block, h->d_nuniq, h->d_nsub, do_select,
                                         flat ? h->grid_flat : h->grid_score, flat ? 1 : 0);
    IG_MARK(7);
}
// the move selected by the last pass: incremental maintenance beside it, apply, contig bookkeeping (+ the cycle record)
static void enqueue_tail(ig_handle* h, int cycle) {
    const float mbar = h->cfg.mean_sub_len_kb;
    IG_MARK(8);
    // independent of apply/post: runs beside them on the side stream, joined before the result copy
    cudaEventRecord(h->ev_sel, h->stream);
    cudaStreamWaitEvent(h->side, h->ev_sel, 0);
    // (not with rigid pruning: there the contacts outside the slice windows keep their terms, as they do mathematically)
    if (!h->rigid)
        k_lnz_outside<<<h->grid_score, IG_THREADS, 0, h->side>>>(h->row_ptr, h->cv, h->coord, h->clen, h->sc, h->rows, h->rowidx, h->ns,
                                                                 h->table, h->table_len, mbar, h->exz, h->part_out);
    cudaEventRecord(h->ev_out, h->side);
    IG_MARK(9);
    k_apply<<<(h->nf + 255) / 256, 256, 0, h->stream>>>(h->live, h->nf, h->sc, h->desc, -1, -1);
    IG_MARK(10);
    k_post<<<(h->nf + 255) / 256, 256, 0, h->stream>>>(h->live, h->nf, h->init_prev, h->init_next, h->orientable, h->sc,
                                                       cycle ? h->cyc_out : nullptr, cycle ? h->temp_rec : nullptr);
    IG_MARK(11);
    cudaStreamWaitEvent(h->stream, h->ev_out, 0);
}
// Everything one step enqueues (no host synchronisation): used directly and under graph capture.  The candidates come from
// the cycle plan (cycle: the step also writes its record) or from the pinned staging of the host step (h_small, h_wide->in).
// A step of up to IG_MAX_CANDS candidates: one selecting pass over its grid_n candidate slots.
static void enqueue_step(ig_handle* h, int full, int grid_n, int cycle) {
    if (!cycle) cudaMemcpyAsync(&h->sc->n_cands, h->h_small, (2 + IG_MAX_CANDS) * sizeof(int), cudaMemcpyHostToDevice, h->stream);
    enqueue_head(h, full);
    enqueue_pass(h, grid_n, 1, cycle ? h->cyc_plan : nullptr, 1);
    enqueue_tail(h, cycle);
    if (!cycle) cudaMemcpyAsync(h->h_sc, h->sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, h->stream);
}
// A step of n_batches * IG_MAX_CANDS candidate slots (ig_k_wide.cuh): the head once, one score-only pass per batch, the
// winning batch scored again with the selecting tail.  Every pass is launched for a full batch (the grid of IG_MAX_CANDS
// candidates, whatever the batch holds), so the re-score repeats its batch's pass launch for launch and its scores, hence
// its selection, are bit-identical to that pass's.
static void enqueue_wide_step(ig_handle* h, int full, int n_batches, int cycle) {
    const int* plan = cycle ? h->cyc_plan : nullptr;
    if (!cycle) cudaMemcpyAsync(h->wide->in, h->h_wide->in, sizeof(h->wide->in), cudaMemcpyHostToDevice, h->stream);
    enqueue_head(h, full);
    for (int b = 0; b < n_batches; b++) {
        k_wide_stage<<<1, 32, 0, h->stream>>>(h->sc, h->wide, plan, b);
        enqueue_pass(h, IG_MAX_CANDS, b == 0 ? 1 : 0, nullptr, 0);
        k_wide_stash<<<1, 256, 0, h->stream>>>(h->sc, h->wide, b);
    }
    k_wide_pick<<<1, 32, 0, h->stream>>>(h->sc, h->wide, plan);
    enqueue_pass(h, IG_MAX_CANDS, 1, nullptr, 1, true);
    enqueue_tail(h, cycle);
    k_wide_finish<<<1, 32, 0, h->stream>>>(h->sc, h->wide, cycle ? h->cyc_out : nullptr, cycle ? h->temp_rec : nullptr);
    if (!cycle) {
        cudaMemcpyAsync(h->h_sc, h->sc, sizeof(DevScalars), cudaMemcpyDeviceToHost, h->stream);
        cudaMemcpyAsync(h->h_wide, h->wide, sizeof(WideStep), cudaMemcpyDeviceToHost, h->stream);
    }
}
static int n_batches_of(int n) { return (n + IG_MAX_CANDS - 1) / IG_MAX_CANDS; }
// the launches of a step of grid_n candidate slots
static int enqueue_any_step(ig_handle* h, int full, int grid_n, int cycle) {
    if (grid_n > IG_MAX_CANDS) enqueue_wide_step(h, full, n_batches_of(grid_n), cycle);
    else enqueue_step(h, full, grid_n, cycle);
    return launch_ok(h, "enqueue_step");
}

// 0: incremental step; 1: coordinates and likelihood sums from scratch (scaffold replaced from outside, periodic refresh);
// 2: likelihood sums only (parameters changed; needs the per-contact records and v_inter > 0, which the records assume);
// 3: kind 2 decided on the device (a step after a production-mode nuisance step: see enqueue_plan_step)
static int step_kind(const ig_handle* h) {
    if (!h->incr_valid || (h->refresh_every > 0 && h->steps_since_full >= h->refresh_every)) return 1;
    if (h->lnz_stale) return (h->lnz_cache && h->vinter_pos) ? 2 : 1;
    return 0;
}
// kernel launches of enqueue_head (per kind) and of one enqueue_pass: k_cand_setup, k_find_cuts, k_classes, the row list
// (flat: one launch, else two), k_precompute, the scoring kernels (flat: k_pick + k_eval_flat; stream: k_stream +
// k_eval_flat + k_score; rows: k_score) and k_finalize
static int head_launches(int kind) { return kind >= 2 ? 6 : kind ? 4 : 1; }
static int pass_launches(const ig_handle* h) { return h->path == PATH_STREAM ? 10 : 8; }
// ... of a step of grid_n candidate slots: head, pass, tail (k_lnz_outside unless rigid, k_apply, k_post); a wide step adds
// one pass with k_wide_stage and k_wide_stash per batch, and k_wide_pick, k_wide_flip, k_wide_finish
static int step_launches(const ig_handle* h, int kind, int grid_n) {
    const int wide = grid_n > IG_MAX_CANDS ? n_batches_of(grid_n) * (pass_launches(h) + 2) + 3 : 0;
    return head_launches(kind) + pass_launches(h) + (h->rigid ? 2 : 3) + wide;
}

// capture what `enqueue` launches on the handle's stream into `exec`; a failed capture leaves it null and sets `failed`
// (the caller then launches directly)
template <class F>
static void capture(ig_handle* h, cudaGraphExec_t& exec, bool& failed, F enqueue) {
    cudaGraph_t g = nullptr;
    h->capturing = true;
    cudaError_t e = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal);
    if (e == cudaSuccess) {
        enqueue();
        e = cudaStreamEndCapture(h->stream, &g);
    }
    h->capturing = false;
    if (e == cudaSuccess && g) e = cudaGraphInstantiate(&exec, g, 0);
    if (g) cudaGraphDestroy(g);
    if (e != cudaSuccess || !exec) { exec = nullptr; failed = true; cudaGetLastError(); }
}
// the graph of a step of grid_n candidate slots (captured on first use; nullptr once a capture failed)
static cudaGraphExec_t get_graph(ig_handle* h, int full, int grid_n, int cycle) {
    cudaGraphExec_t& ge = h->graph[full + 4 * cycle][grid_n <= IG_MAX_CANDS ? grid_n : IG_MAX_CANDS + n_batches_of(grid_n)];
    if (!ge && !h->graph_failed) capture(h, ge, h->graph_failed, [&] { enqueue_any_step(h, full, grid_n, cycle); });
    return ge;
}
// one step on the handle's stream: the graph ge (get_graph), or its launches when there is none
static int launch_step(ig_handle* h, cudaGraphExec_t ge, int full, int grid_n, int cycle) {
    if (ge) { CK(cudaGraphLaunch(ge, h->stream)); }
    else if (enqueue_any_step(h, full, grid_n, cycle)) return -2;
    h->n_launches += step_launches(h, full, grid_n);
    return 0;
}
// the handle's bookkeeping after a step of kind `kind` (host step or plan step; kind 3 counts as incremental)
static void after_step(ig_handle* h, int kind) {
    const bool refresh = kind == 1 || kind == 2;
    h->steps_since_full = refresh ? 1 : h->steps_since_full + 1;
    h->n_full += refresh ? 1 : 0;
    h->incr_valid = true; h->lnz_stale = false;
    h->coords_fresh = false; h->coords_ever = true;
}

extern "C" int ig_step(ig_handle* h, int32_t id_frag, const int32_t* cands, int32_t n_cands, ig_step_result* out) {
    if (use(h)) return -1;
    if (n_cands <= 0 || n_cands > IG_MAX_CANDS) { h->err = "n_cands out of range"; return -1; }
    return ig_step_wide(h, id_frag, cands, n_cands, out, nullptr, nullptr, nullptr);
}

// step_sampler: enqueue_step up to IG_MAX_CANDS candidates, enqueue_wide_step beyond
extern "C" int ig_step_wide(ig_handle* h, int32_t id_frag, const int32_t* cands, int32_t n_cands, ig_step_result* out, double* scores,
                            int32_t* n_uniq, int32_t* n_sub) {
    if (use(h)) return -1;
    if (!out || !cands) { h->err = "ig_step_wide: null argument"; return -1; }
    if (n_cands <= 0 || n_cands > IG_MAX_NEIGHBOURS) { h->err = "ig_step_wide: n_cands out of range (1 .. IG_MAX_NEIGHBOURS = 64)"; return -1; }
    if (!h->params_set) { h->err = "ig_step: parameters not set (ig_set_params)"; return -1; }
    if (h->temperature > 0.0) { h->err = "ig_step: the chain temperature is > 0 (tempered selection needs the seeded production mode, "
                                         "ig_run_cycle_device); set it back with ig_set_temperature(h, 0)"; return -1; }
    if (id_frag < 0 || id_frag >= h->nf) { h->err = "id_frag out of range"; return -1; }
    for (int i = 0; i < n_cands; i++) if (cands[i] < 0 || cands[i] >= h->nf) { h->err = "candidate out of range"; return -1; }
    for (int i = 0; i < n_cands; i++) if (cands[i] == id_frag) { h->err = "candidate equals the visited fragment (reference quirk Q4; see DESIGN.md D1)"; return -1; }
    if (int rc = labels_guard(h)) return rc;
    const bool wide = n_cands > IG_MAX_CANDS;
    int* in = wide ? h->h_wide->in : h->h_small;
    in[0] = n_cands; in[1] = id_frag;
    for (int i = 0; i < (wide ? IG_MAX_NEIGHBOURS : IG_MAX_CANDS); i++) in[2 + i] = i < n_cands ? cands[i] : 0;
    const int full = step_kind(h);
    cudaGraphExec_t ge = (h->use_graph && !h->profile) ? get_graph(h, full, n_cands, 0) : nullptr;   // (profiling: per-kernel marks)
    cudaEventRecord(h->ev[0], h->stream);
    if (int rc = launch_step(h, ge, full, n_cands, 0)) return rc;
    cudaEventRecord(h->ev[1], h->stream);
    CK(cudaStreamSynchronize(h->stream));
    after_step(h, full);
    if (int rc = fetch_result(h, n_cands, cands, out, true, false, scores, n_uniq, n_sub)) return rc;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->ms_step += ms;
    if (h->profile) {
        if (full && cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]) == cudaSuccess) h->ms_full += ms;
        if (cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) h->ms_score += ms;
        for (int i = 0; i < 11; i++)
            if (cudaEventElapsedTime(&ms, h->evk[i], h->evk[i + 1]) == cudaSuccess) h->ms_k[i] += ms;
    }
    h->n_steps++;
    return 0;
}

// A whole MCMC cycle (or any run of steps) enqueued without a single host synchronisation in between:
// the host uploads the plan {fragment, sorted candidates} of every step (drawn with the reference's own
// RNG calls, which do not depend on the chain state), every step is one CUDA-graph replay that reads its
// plan entry and writes a compact record on the device, and the host synchronises once at the end.
// Semantically identical to n_steps calls of ig_step (IG.full_em inner loop, instagraal.py:217-241).

// The buffers of a cycle of n_steps steps whose plan entries hold `width` candidate slots: the plan [n_steps][2 + width],
// the step records, the visiting order, the nuisance and tempered records.  They only grow; the cycle graphs bake them in.
static int cycle_buffers(ig_handle* h, int n_steps, int width) {
    if (n_steps > h->cyc_cap || width > h->cyc_width) {
        const int cap = std::max(n_steps, h->cyc_cap), w = std::max(width, h->cyc_width);
        for (void* q : {(void*)h->cyc_plan, (void*)h->cyc_out, (void*)h->cyc_frags, (void*)h->nuis_rec, (void*)h->temp_rec}) if (q) cudaFree(q);
        h->cyc_plan = nullptr; h->cyc_out = nullptr; h->cyc_frags = nullptr; h->nuis_rec = nullptr; h->temp_rec = nullptr;
        h->cyc_cap = 0; h->cyc_width = 0;
        destroy_graphs(h, 4);
        if (dev_alloc(h, &h->cyc_plan, (size_t)cap * (2 + w)) || dev_alloc(h, &h->cyc_out, (size_t)cap) ||
            dev_alloc(h, &h->cyc_frags, (size_t)cap) || dev_alloc(h, &h->nuis_rec, (size_t)cap) || dev_alloc(h, &h->temp_rec, (size_t)cap)) return -2;
        h->cyc_cap = cap; h->cyc_width = w;
    }
    h->plan_width = width;
    return 0;
}

// the nuisance step of the production mode (ig_k_nuis.cuh) after the step just enqueued: propose, evaluate the proposal
// with exactly the launches of ig_full_likelihood(p_test, use_stale_coords = 1), decide, promote, record
static void enqueue_nuisance(ig_handle* h) {
    const float mbar = h->cfg.mean_sub_len_kb;
    k_nuis_propose<<<1, 1, 0, h->stream>>>(h->sc);
    k_exz_table<<<std::min(1024, (h->ns + 256) / 256), 256, 0, h->stream>>>(h->exz_test, h->ns + 1, h->sc, mbar, 1);
    k_coords<<<h->n_part_zc, IG_THREADS, 0, h->stream>>>(h->live, h->sub, h->coord, h->clen, h->ns, h->sc, mbar, 1,
                                                        h->part_zc, h->part_nc, 0, h->subx, h->row_dirty);
    k_reduce<<<1, 256, 0, h->stream>>>(h->part_zc, h->n_part_zc, &h->sc->full_out[1], h->part_nc, &h->sc->full_nintra);
    k_lnz_refresh<<<h->grid_lnz, IG_THREADS, 0, h->stream>>>(h->row_ptr, h->cv, h->coord, h->clen, h->ns, h->sc, mbar, 1, h->exz_test,
                                                             h->lnz_rec, h->row_dirty, h->dp_bits, h->part_full + h->grid_lnz);
    k_lnz_stream<<<h->grid_lnz, IG_THREADS, 0, h->stream>>>(reinterpret_cast<const int4*>(h->lnz_rec), h->lnz_pairs, h->lnz_pad,
                                                            h->lvl->val_total, h->sc, 1, h->exz_test, h->dp_bits, h->part_full);
    k_reduce<<<1, 256, 0, h->stream>>>(h->part_full, 2 * h->grid_lnz, &h->sc->full_out[0], nullptr, nullptr);
    k_nuis_accept<<<1, 1, 0, h->stream>>>(h->sc, h->nuis_rec, h->cfg.n_pix);
    k_nuis_copy_exz<<<std::min(1024, (h->ns + 258) / 256), 256, 0, h->stream>>>(h->exz, h->exz_test, h->ns + 3, h->sc);
}
#define IG_LAUNCHES_NUIS 9
static int launch_nuisance(ig_handle* h) {
    if (h->use_graph && !h->graph_nuis_dev && !h->nuis_graph_dev_failed)
        capture(h, h->graph_nuis_dev, h->nuis_graph_dev_failed, [&] { enqueue_nuisance(h); });
    if (h->use_graph && h->graph_nuis_dev) { CK(cudaGraphLaunch(h->graph_nuis_dev, h->stream)); }
    else enqueue_nuisance(h);
    h->n_launches += IG_LAUNCHES_NUIS;
    return launch_ok(h, "nuisance step");
}
// the plan's next step (entry sc->step_idx) on the handle's stream, its grid built for grid_n candidate slots (a wide step
// beyond IG_MAX_CANDS), then the production-mode nuisance step when it is on
static int enqueue_plan_step(ig_handle* h, int grid_n) {
    if (int rc = labels_guard(h)) return rc;
    int full = step_kind(h);
    // after a nuisance step of this plan the host cannot know whether the parameters changed: kind 3 decides on the device
    if (full == 0 && h->nuis_on && h->nuis_enqueued) full = 3;
    if (int rc = launch_step(h, h->use_graph ? get_graph(h, full, grid_n, 1) : nullptr, full, grid_n, 1)) return rc;
    after_step(h, full);
    if (h->nuis_on) {
        if (int rc = launch_nuisance(h)) return rc;
        h->nuis_enqueued = true;
    }
    return 0;
}
static int begin_plan(ig_handle* h) {
    CK(cudaMemsetAsync(&h->sc->step_idx, 0, sizeof(int), h->stream));
    cudaEventRecord(h->ev[0], h->stream);
    return 0;
}
// wait for the n_steps enqueued steps and convert their device records
static int collect_plan(ig_handle* h, int n_steps, ig_cycle_step* out) {
    cudaEventRecord(h->ev[1], h->stream);
    std::vector<CycleOut> res(n_steps);
    int overflow = 0;
    CK(cudaMemcpyAsync(res.data(), h->cyc_out, sizeof(CycleOut) * n_steps, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&overflow, &h->sc->list_overflow, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->pending_steps = 0;
    if (h->nuis_on && h->nuis_enqueued) {
        // the last step's nuisance decision: an accepted proposal leaves the sums stale for the next step (ig_step or the
        // first step of the next cycle, both decided on the host: kind 2)
        int stale = 0; Params p;
        CK(cudaMemcpyAsync(&stale, &h->sc->nuis_stale, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(&p, &h->sc->p, sizeof(Params), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemsetAsync(&h->sc->nuis_stale, 0, sizeof(int), h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (stale) h->lnz_stale = true;
        h->vinter_pos = p.v_inter > 0.0f;   // (always: a proposal with v_inter <= 0 is never accepted)
    }
    h->nuis_enqueued = false;
    if (overflow) { h->err = "pick list of the streaming scoring path overflowed"; return -4; }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->ms_step += ms;
    h->n_steps += n_steps;
    for (int t = 0; t < n_steps; t++) {
        const CycleOut& r = res[t];
        ig_cycle_step& o = out[t];
        o.likelihood = r.likelihood; o.lnz_full = r.lnz_full;
        o.dist = (3.0 * h->nf - 0.5 * (double)r.dist_half) / (3.0 * h->nf);
        o.sum_l_cont = r.sum_l_cont; o.n_contigs = r.n_heads; o.op_sampled = r.win_op; o.cand_index = r.win_cand;
        o.id_f_sampled = r.id_f_sampled;
        o.q4_hits = r.q4_hits; o.n_proposals = r.n_proposals;
    }
    return 0;
}
template <class GridN>
static int run_plan(ig_handle* h, int n_steps, GridN grid_n, ig_cycle_step* out) {
    if (begin_plan(h)) return -2;
    for (int t = 0; t < n_steps; t++) if (int rc = enqueue_plan_step(h, grid_n(t))) return rc;
    return collect_plan(h, n_steps, out);
}

extern "C" int ig_run_cycle(ig_handle* h, int32_t n_steps, const int32_t* frags, const int32_t* cands8, const int32_t* n_cands,
                            ig_cycle_step* out) {
    return ig_run_cycle_wide(h, n_steps, frags, cands8, IG_MAX_CANDS, n_cands, out);
}
// cands = [n_steps][width].  The plan holds every step at the stride 2 + W, W = max(IG_MAX_CANDS, longest list): a step of
// more than IG_MAX_CANDS candidates runs as a wide step, the others as narrow steps of their own size
extern "C" int ig_run_cycle_wide(ig_handle* h, int32_t n_steps, const int32_t* frags, const int32_t* cands, int32_t width,
                                 const int32_t* n_cands, ig_cycle_step* out) {
    if (use(h)) return -1;
    if (!h->params_set) { h->err = "ig_run_cycle: parameters not set"; return -1; }
    if (h->nuis_on) { h->err = "ig_run_cycle: the device nuisance step is on (it needs the seeded production mode, ig_run_cycle_device); "
                                "turn it off with ig_set_device_nuisance(h, 0)"; return -1; }
    if (h->temperature > 0.0) { h->err = "ig_run_cycle: the chain temperature is > 0 (tempered selection needs the seeded production mode, "
                                         "ig_run_cycle_device); set it back with ig_set_temperature(h, 0)"; return -1; }
    if (width <= 0 || width > IG_MAX_NEIGHBOURS) { h->err = "ig_run_cycle: width out of range (1 .. IG_MAX_NEIGHBOURS = 64)"; return -1; }
    if (n_steps <= 0) return 0;
    int n_max = 0;
    for (int t = 0; t < n_steps; t++) {
        const int n = n_cands[t];
        if (n > width) { h->err = "ig_run_cycle: a step has more candidates than the width of the candidate array"; return -1; }
        if (n <= 0 || frags[t] < 0 || frags[t] >= h->nf) { h->err = "ig_run_cycle: bad plan entry"; return -1; }
        for (int i = 0; i < n; i++) {
            const int c = cands[(size_t)t * width + i];
            if (c < 0 || c >= h->nf || c == frags[t]) { h->err = "ig_run_cycle: candidate out of range or equal to the visited fragment"; return -1; }
        }
        n_max = std::max(n_max, n);
    }
    const int w = std::max(IG_MAX_CANDS, n_max), stride = 2 + w;
    std::vector<int> plan((size_t)n_steps * stride, 0);
    for (int t = 0; t < n_steps; t++) {
        int* p = &plan[(size_t)t * stride];
        p[0] = n_cands[t]; p[1] = frags[t];
        for (int i = 0; i < n_cands[t]; i++) p[2 + i] = cands[(size_t)t * width + i];
    }
    if (cycle_buffers(h, n_steps, w)) return -2;
    CK(cudaMemcpyAsync(h->cyc_plan, plan.data(), plan.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(&h->sc->plan_stride, &stride, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    return run_plan(h, n_steps, [&](int t) { return n_cands[t]; }, out);
}

// setup_distri_frags (CL:3053-3101) on the device: per fragment the candidate fragments (self excluded), the
// running sum of their probabilities pk, and the number of non-zero pk (CL:3113).
extern "C" int ig_set_neighbour_weights(ig_handle* h, const int64_t* ptr, const int32_t* idx, const double* cdf, const int32_t* n_nonzero) {
    if (use(h)) return -1;
    if (!ptr || !n_nonzero) { h->err = "ig_set_neighbour_weights: null argument"; return -1; }
    const size_t n = (size_t)ptr[h->nf];
    LevelBlock* L = h->lvl;
    CK(cudaDeviceSynchronize());   // chains sharing the level may still be drawing from the old arrays
    for (void* q : {(void*)L->nb_ptr, (void*)L->nb_idx, (void*)L->nb_cdf, (void*)L->nb_nnz}) if (q) cudaFree(q);
    L->nb_ptr = nullptr; L->nb_idx = nullptr; L->nb_cdf = nullptr; L->nb_nnz = nullptr;
    if (dev_alloc(h, &L->nb_ptr, (size_t)h->nf + 1) || dev_alloc(h, &L->nb_idx, n + 1) || dev_alloc(h, &L->nb_cdf, n + 1) ||
        dev_alloc(h, &L->nb_nnz, (size_t)h->nf)) return -2;
    CK(h2d_sync(L->nb_ptr, ptr, sizeof(long long) * ((size_t)h->nf + 1)));
    if (n) {
        CK(h2d_sync(L->nb_idx, idx, sizeof(int) * n));
        CK(h2d_sync(L->nb_cdf, cdf, sizeof(double) * n));
    }
    CK(h2d_sync(L->nb_nnz, n_nonzero, sizeof(int) * (size_t)h->nf));
    return 0;
}

// One sweep of step_sampler over `frags` with the neighbour draws made ON THE DEVICE (Philox4x32-10 keyed by
// (seed, cycle, step, draw)): the host uploads the visiting order, one kernel draws every step's candidates,
// then the steps replay without host synchronisation.  Needs ig_set_neighbour_weights.
static int prepare_device_plan(ig_handle* h, int32_t n_steps, const int32_t* frags, int32_t n_neighbours, uint64_t seed, uint32_t cycle) {
    if (!h->params_set) { h->err = "ig_run_cycle_device: parameters not set"; return -1; }
    if (!h->lvl->nb_ptr) { h->err = "ig_run_cycle_device: neighbour weights not set (ig_set_neighbour_weights)"; return -1; }
    if (n_neighbours <= 0 || n_neighbours > IG_MAX_NEIGHBOURS) { h->err = "ig_run_cycle_device: n_neighbours out of range (1 .. IG_MAX_NEIGHBOURS = 64)"; return -1; }
    if (h->nf < 2) { h->err = "ig_run_cycle_device: needs at least two fragments"; return -1; }
    if (h->pending_steps) { h->err = "ig_run_cycle_device: an asynchronous cycle is still pending (ig_cycle_wait)"; return -1; }
    for (int t = 0; t < n_steps; t++) if (frags[t] < 0 || frags[t] >= h->nf) { h->err = "ig_run_cycle_device: fragment out of range"; return -1; }
    if (h->nuis_on && !(h->lnz_cache && h->vinter_pos)) {
        h->err = "ig_run_cycle_device: the device nuisance step needs the per-contact likelihood records and v_inter > 0"; return -1;
    }
    const int w = std::max(IG_MAX_CANDS, (int)n_neighbours);   // every step's grid: n_neighbours slots (enqueue_plan_step)
    if (cycle_buffers(h, n_steps, w)) return -2;
    CK(cudaMemcpyAsync(h->cyc_frags, frags, sizeof(int) * (size_t)n_steps, cudaMemcpyHostToDevice, h->stream));
    if (h->nuis_on || h->temperature > 0.0) {   // the key and cycle of the nuisance and tempered-selection draws
        k_nuis_begin<<<1, 1, 0, h->stream>>>(h->sc, (unsigned)(seed & 0xffffffffu), (unsigned)(seed >> 32), cycle);
        h->n_launches += 1;
    }
    auto* draw = w == IG_MAX_CANDS ? k_draw_plan<IG_MAX_CANDS> : k_draw_plan<IG_MAX_NEIGHBOURS>;
    draw<<<(n_steps + 127) / 128, 128, 0, h->stream>>>(h->cyc_plan, w, h->sc, h->cyc_frags, n_steps, n_neighbours, h->nf, h->lvl->nb_ptr,
                                                       h->lvl->nb_idx, h->lvl->nb_cdf, h->lvl->nb_nnz, (unsigned)(seed & 0xffffffffu),
                                                       (unsigned)(seed >> 32), cycle);
    if (launch_ok(h, "draw_plan")) return -2;
    h->n_launches += 1;
    return 0;
}
extern "C" int ig_run_cycle_device(ig_handle* h, int32_t n_steps, const int32_t* frags, int32_t n_neighbours, uint64_t seed,
                                   uint32_t cycle, ig_cycle_step* out) {
    if (use(h)) return -1;
    if (n_steps <= 0) return 0;
    if (int rc = prepare_device_plan(h, n_steps, frags, n_neighbours, seed, cycle)) return rc;
    return run_plan(h, n_steps, [&](int) { return (int)n_neighbours; }, out);
}

// Several chains of ONE device advanced together (replica chains, ig_clone): the same as one ig_run_cycle_device call per
// chain, but the steps are enqueued round-robin on the chains' own streams before anything is waited for, so the GPU runs
// them side by side -- a yeast-scale chain keeps a B200 under 25 % busy, eight of them fill it.  frags = [n_chains][n_steps]
// (each chain's visiting order), seeds = [n_chains], out = [n_chains][n_steps].  Every chain's trajectory is bit-identical
// to what ig_run_cycle_device gives it alone (tests/test_gpu_parity.py).
extern "C" int ig_run_cycles_device_multi(ig_handle** hs, int32_t n_chains, int32_t n_steps, const int32_t* frags, int32_t n_neighbours,
                                          const uint64_t* seeds, uint32_t cycle, ig_cycle_step* out) {
    if (!hs || n_chains <= 0) { g_err = "ig_run_cycles_device_multi: no chains"; return -1; }
    if (n_steps <= 0) return 0;
    for (int c = 0; c < n_chains; c++) {
        ig_handle* h = hs[c];
        if (use(h)) return -1;
        if (int rc = prepare_device_plan(h, n_steps, frags + (size_t)c * n_steps, n_neighbours, seeds[c], cycle)) { g_err = h->err; return rc; }
        if (begin_plan(h)) return -2;
    }
    // (several steps per graph launch were tried: the launching host thread is not the bottleneck, no gain)
    for (int t = 0; t < n_steps; t++)
        for (int c = 0; c < n_chains; c++)
            if (int rc = enqueue_plan_step(hs[c], n_neighbours)) { g_err = hs[c]->err; return rc; }
    int rc_all = 0;
    for (int c = 0; c < n_chains; c++)
        if (int rc = collect_plan(hs[c], n_steps, out + (size_t)c * n_steps)) { g_err = hs[c]->err; rc_all = rc; }
    return rc_all;
}
// Asynchronous form for callers that drive the chains themselves: enqueue now, collect later.
extern "C" int ig_run_cycle_device_async(ig_handle* h, int32_t n_steps, const int32_t* frags, int32_t n_neighbours, uint64_t seed, uint32_t cycle) {
    if (use(h)) return -1;
    if (n_steps <= 0) return 0;
    if (int rc = prepare_device_plan(h, n_steps, frags, n_neighbours, seed, cycle)) return rc;
    if (begin_plan(h)) return -2;
    for (int t = 0; t < n_steps; t++) if (int rc = enqueue_plan_step(h, n_neighbours)) return rc;
    h->pending_steps = n_steps;
    return 0;
}
extern "C" int ig_cycle_wait(ig_handle* h, int32_t n_steps, ig_cycle_step* out) {
    if (use(h)) return -1;
    if (n_steps != h->pending_steps) { h->err = "ig_cycle_wait: n_steps does not match the pending cycle"; return -1; }
    if (n_steps <= 0) return 0;
    return collect_plan(h, n_steps, out);
}

// download the plan of the last cycle ([n_steps][2 + IG_MAX_CANDS]: n_cands, fragment, candidates) -- tests / logging
extern "C" int ig_get_cycle_plan(ig_handle* h, int32_t n_steps, int32_t* out) {
    return ig_get_cycle_plan_wide(h, n_steps, IG_MAX_CANDS, out);
}
// the same as [n_steps][2 + width]
extern "C" int ig_get_cycle_plan_wide(ig_handle* h, int32_t n_steps, int32_t width, int32_t* out) {
    if (use(h)) return -1;
    if (n_steps > h->cyc_cap) { h->err = "ig_get_cycle_plan: no such plan"; return -1; }
    if (width <= 0 || width > IG_MAX_NEIGHBOURS) { h->err = "ig_get_cycle_plan: width out of range (1 .. IG_MAX_NEIGHBOURS = 64)"; return -1; }
    if (n_steps <= 0) return 0;
    const int src_w = h->plan_width;
    std::vector<int> src((size_t)n_steps * (2 + src_w));
    CK(cudaMemcpy(src.data(), h->cyc_plan, src.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (int t = 0; t < n_steps; t++) {
        const int* p = &src[(size_t)t * (2 + src_w)];
        int* q = out + (size_t)t * (2 + width);
        if (p[0] > width) { h->err = "ig_get_cycle_plan: a step of the last cycle has more candidates than width"; return -1; }
        q[0] = p[0]; q[1] = p[1];
        for (int i = 0; i < width; i++) q[2 + i] = i < p[0] ? p[2 + i] : 0;
    }
    return 0;
}

extern "C" int ig_set_device_nuisance(ig_handle* h, int32_t on) {
    if (use(h)) return -1;
    if (h->pending_steps) { h->err = "ig_set_device_nuisance: an asynchronous cycle is still pending (ig_cycle_wait)"; return -1; }
    if (on) {
        if (!h->lnz_cache) {
            h->err = "ig_set_device_nuisance: this handle has no per-contact likelihood records (IG_LNZ_CACHE=0, or a level whose "
                     "counts / size do not fit them); the device nuisance step evaluates its proposals from them";
            return -1;
        }
        if (!h->params_set) { h->err = "ig_set_device_nuisance: parameters not set (ig_set_params)"; return -1; }
        if (!h->vinter_pos) { h->err = "ig_set_device_nuisance: the live v_inter must be > 0"; return -1; }
    }
    h->nuis_on = on != 0;
    return 0;
}
// the chain temperature of the tempered selection (ig_k_temper.cuh), written stream-ordered into the scalar record: the
// captured step graphs read it at replay, so they stay valid and no launch is added to a step
extern "C" int ig_set_temperature(ig_handle* h, double temperature) {
    if (use(h)) return -1;
    if (!(temperature >= 0.0) || !std::isfinite(temperature)) { h->err = "ig_set_temperature: the temperature must be finite and >= 0"; return -1; }
    if (h->pending_steps) { h->err = "ig_set_temperature: an asynchronous cycle is still pending (ig_cycle_wait)"; return -1; }
    k_set_temperature<<<1, 1, 0, h->stream>>>(h->sc, temperature);
    if (launch_ok(h, "set_temperature")) return -2;
    h->temperature = temperature;
    return 0;
}
extern "C" int ig_get_tempered_records(ig_handle* h, int32_t n_steps, ig_tempered_step* out) {
    if (use(h)) return -1;
    if (n_steps == 0) return 0;
    if (n_steps < 0 || n_steps > h->cyc_cap || !h->temp_rec) { h->err = "ig_get_tempered_records: no such records"; return -1; }
    CK(cudaMemcpyAsync(out, h->temp_rec, sizeof(ig_tempered_step) * (size_t)n_steps, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
extern "C" int ig_get_nuisance_records(ig_handle* h, int32_t n_steps, ig_nuisance_step* out) {
    if (use(h)) return -1;
    if (n_steps == 0) return 0;
    if (n_steps < 0 || n_steps > h->cyc_cap || !h->nuis_rec) { h->err = "ig_get_nuisance_records: no such records"; return -1; }
    CK(cudaMemcpyAsync(out, h->nuis_rec, sizeof(ig_nuisance_step) * (size_t)n_steps, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// measurement / parity knobs: refresh_every = N -> recompute the coordinates and the full likelihood
// over every contact at least every N steps (1 = every step, exactly the reference's schedule;
// 0 = only when the state was changed from outside); use_graph = replay the step as one CUDA graph.
extern "C" int ig_set_options(ig_handle* h, int32_t refresh_every, int32_t use_graph) {
    if (!h) return -1;
    h->refresh_every = refresh_every;
    h->use_graph = use_graph ? true : false;
    return 0;
}

// Several chains on one GPU (ig_clone): each chain's scoring grids take 1 / share of the machine, so that the kernels of
// different chains run side by side instead of queueing behind each other's full-machine grids (a yeast-scale scoring
// kernel is latency-bound: 8 chains at share 4 deliver 1.2x the aggregate of full grids on T, 1.14x on the 1 Gb level).
// Changes the grouping of the f64 partial sums (not the terms): compare chains run with the SAME share bit for bit.
extern "C" int ig_set_gpu_share(ig_handle* h, int32_t share) {
    if (use(h)) return -1;
    if (share < 1) { h->err = "ig_set_gpu_share: share must be >= 1"; return -1; }
    if (h->pending_steps) { h->err = "ig_set_gpu_share: an asynchronous cycle is still pending"; return -1; }
    CK(cudaStreamSynchronize(h->stream));
    destroy_graphs(h, 0);
    h->grid_score = std::max(8, h->grid_score_full / share);
    h->grid_flat = std::max(1, h->grid_score / 5);
    return 0;
}

// the head of step_sampler (fill_dist_single + eval_likelihood, CL:1407-1409) and a score-only pass of one candidate
extern "C" int ig_eval_scores(ig_handle* h, int32_t id_frag, int32_t id_cand, int32_t flip_eject, double out24[24],
                              int32_t* n_uniq, int32_t* n_sub) {
    if (use(h)) return -1;
    if (!h->params_set) { h->err = "ig_eval_scores: parameters not set"; return -1; }
    h->incr_valid = false;
    if (id_frag < 0 || id_frag >= h->nf) { h->err = "id_frag out of range"; return -1; }
    if (id_cand < 0 || id_cand >= h->nf) { h->err = "candidate out of range"; return -1; }
    int* hs = h->h_small;
    hs[0] = 1; hs[1] = id_frag;
    for (int i = 0; i < IG_MAX_CANDS; i++) hs[2 + i] = i == 0 ? id_cand : 0;
    CK(cudaMemcpyAsync(&h->sc->n_cands, hs, (2 + IG_MAX_CANDS) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    enqueue_head(h, 1);
    enqueue_pass(h, 1, flip_eject, nullptr, 0);
    if (launch_ok(h, "eval_scores")) return -2;
    h->n_launches += head_launches(1) + pass_launches(h);
    h->coords_fresh = true; h->coords_ever = true;
    ig_step_result r;
    if (fetch_result(h, 1, &id_cand, &r, false, true, out24, n_uniq, n_sub)) return -2;
    return 0;
}

extern "C" int ig_apply(ig_handle* h, int32_t id_frag, int32_t id_cand, int32_t op, ig_step_result* out) {
    if (use(h)) return -1;
    if (op < 0 || op >= IG_N_OPS) { h->err = "ig_apply: bad op"; return -1; }
    h->incr_valid = false;
    if (id_frag < 0 || id_frag >= h->nf || id_cand < 0 || id_cand >= h->nf) { h->err = "ig_apply: fragment out of range"; return -1; }
    int* hs = h->h_small;
    hs[0] = 1; hs[1] = id_frag; hs[2] = id_cand;
    CK(cudaMemcpyAsync(&h->sc->n_cands, hs, 3 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    int32_t saved[12];
    CK(cudaMemcpyAsync(saved, h->sc->valid, sizeof saved, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const FragRec* live = h->live;
    k_cand_setup<<<1, 32, 0, h->stream>>>(live, h->sc, h->desc, h->cfg.max_bounds_insert, 0, nullptr, 0);
    k_find_cuts<<<dim3((h->nf + 255) / 256, 1), 256, 0, h->stream>>>(live, h->nf, h->sc, h->desc, h->clstab);
    // test_copy_struct only re-runs get_bounds for op >= 12 (CL:2121-2126): restore the list otherwise
    CK(cudaMemcpyAsync(h->sc->valid, saved, sizeof saved, cudaMemcpyHostToDevice, h->stream));
    if (apply_and_post(h, 0, op)) return -2;
    ig_step_result r;
    if (fetch_result(h, 1, &id_cand, &r, true)) return -2;
    r.op_sampled = op; r.id_f_sampled = id_cand; r.cand_index = 0;
    if (out) *out = r;
    return 0;
}

// everything one nuisance-likelihood evaluation enqueues (test parameters in the pinned h->h_p8): used directly and under
// graph capture.  write_coords = 0: on the coordinates of the last fill (quirk Q5)
static void enqueue_full_likelihood(ig_handle* h, int write_coords, bool records) {
    const float mbar = h->cfg.mean_sub_len_kb;
    cudaMemcpyAsync(h->d_p8, h->h_p8, sizeof(Params), cudaMemcpyHostToDevice, h->stream);
    k_set_params_dev<<<1, 1, 0, h->stream>>>(h->sc, h->d_p8, 1);
    k_exz_table<<<std::min(1024, (h->ns + 256) / 256), 256, 0, h->stream>>>(h->exz_test, h->ns + 1, h->sc, mbar, 1);
    k_coords<<<h->n_part_zc, IG_THREADS, 0, h->stream>>>(h->live, h->sub, h->coord, h->clen, h->ns, h->sc, mbar, 1,
                                                        h->part_zc, h->part_nc, write_coords, h->subx, h->row_dirty);
    k_reduce<<<1, 256, 0, h->stream>>>(h->part_zc, h->n_part_zc, &h->sc->full_out[1], h->part_nc, &h->sc->full_nintra);
    cudaEventRecord(h->ev[2], h->stream);
    if (records) {
        // records of the rows whose coordinates were rewritten since the last call (+ circular contigs), then the flat pass
        k_lnz_refresh<<<h->grid_lnz, IG_THREADS, 0, h->stream>>>(h->row_ptr, h->cv, h->coord, h->clen, h->ns, h->sc, mbar, 1, h->exz_test,
                                                                 h->lnz_rec, h->row_dirty, h->dp_bits, h->part_full + h->grid_lnz);
        k_lnz_stream<<<h->grid_lnz, IG_THREADS, 0, h->stream>>>(reinterpret_cast<const int4*>(h->lnz_rec), h->lnz_pairs, h->lnz_pad,
                                                                h->lvl->val_total, h->sc, 1, h->exz_test, h->dp_bits, h->part_full);
        cudaEventRecord(h->ev[3], h->stream);
        k_reduce<<<1, 256, 0, h->stream>>>(h->part_full, 2 * h->grid_lnz, &h->sc->full_out[0], nullptr, nullptr);
    } else {
        k_full_lnz<<<h->n_part_full, IG_THREADS, 0, h->stream>>>(h->row_ptr, h->cv, h->coord, h->clen, h->ns, h->sc, mbar, 1,
                                                                h->exz_test, h->part_full);
        cudaEventRecord(h->ev[3], h->stream);
        k_reduce<<<1, 256, 0, h->stream>>>(h->part_full, h->n_part_full, &h->sc->full_out[0], nullptr, nullptr);
    }
    // full_out[3] + full_nintra: 32 contiguous bytes of the scalar record
    cudaMemcpyAsync(&h->h_sc->full_out[0], &h->sc->full_out[0], 3 * sizeof(double) + 2 * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
}

extern "C" int ig_full_likelihood(ig_handle* h, const float p8[8], int32_t use_stale_coords, double out3[3]) {
    if (use(h)) return -1;
    Params p; memcpy(&p, p8, sizeof p);
    memcpy(h->h_p8, p8, sizeof(Params));
    const int write = (use_stale_coords && h->coords_ever) ? 0 : 1;
    if (write) { h->coords_ever = true; h->coords_fresh = true; }
    const bool records = h->lnz_cache && p.v_inter > 0.0f;
    // the nuisance step's evaluation (stale coordinates, records) replays as ONE CUDA graph: 8 launches + 2 copies otherwise
    bool graphed = false;
    if (!write && records && h->use_graph && !h->nuis_graph_failed) {
        if (!h->graph_nuis) capture(h, h->graph_nuis, h->nuis_graph_failed, [&] { enqueue_full_likelihood(h, 0, true); });
        if (h->graph_nuis) { CK(cudaGraphLaunch(h->graph_nuis, h->stream)); graphed = true; }
    }
    if (!graphed) enqueue_full_likelihood(h, write, records);
    if (launch_ok(h, "full_likelihood")) return -2;
    h->n_launches += records ? 7 : 6;
    CK(cudaStreamSynchronize(h->stream));
    {   // device time of the likelihood kernels (always measured: two events per call)
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]) == cudaSuccess) { h->ms_nuis += ms; h->n_nuis++; }
        else { cudaGetLastError(); if (graphed) h->nuis_graph_failed = true; }   // (events recorded by graph nodes must stay measurable)
    }
    out3[0] = h->h_sc->full_out[0];
    out3[1] = h->h_sc->full_out[1];
    out3[2] = (double)h->h_sc->full_nintra;
    return 0;
}

extern "C" int ig_distance_histogram(ig_handle* h, double bin_kb, double max_kb, int32_t n_rows, int32_t n_bins,
                                     int64_t* hist, int64_t* rows_used) {
    if (use(h)) return -1;
    if (n_bins <= 0 || n_bins > (1 << 16) - 1) { h->err = "ig_distance_histogram: n_bins out of range"; return -1; }
    if (n_rows > h->ns) n_rows = h->ns;
    CK(cudaMemsetAsync(h->d_hist, 0, sizeof(unsigned long long) * (n_bins + 1), h->stream));
    k_histogram<<<h->n_part_full, IG_THREADS, 0, h->stream>>>(h->row_ptr, h->cv, h->lvl->sym_diag, h->init_live, h->sub, n_rows, bin_kb,
                                                             max_kb, n_bins, h->d_hist, h->d_hist + n_bins);
    if (launch_ok(h, "histogram")) return -2;
    std::vector<unsigned long long> tmp(n_bins + 1);
    CK(cudaMemcpyAsync(tmp.data(), h->d_hist, sizeof(unsigned long long) * (n_bins + 1), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n_bins; i++) hist[i] = (int64_t)tmp[i];
    *rows_used = (int64_t)tmp[n_bins];
    return 0;
}

extern "C" int ig_set_sym_diag(ig_handle* h, const int32_t* diag) {
    if (use(h)) return -1;
    if (!h->lvl->sym_diag) { if (dev_alloc(h, &h->lvl->sym_diag, h->ns)) return -2; }
    CK(cudaMemcpyAsync(h->lvl->sym_diag, diag, sizeof(int) * h->ns, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int ig_device_state_ptr(ig_handle* h, void** dev_ptr, int64_t* n_bytes) {
    if (use(h)) return -1;
    CK(cudaStreamSynchronize(h->stream));
    *dev_ptr = h->live;
    *n_bytes = (int64_t)sizeof(FragRec) * h->nf;
    return 0;
}

// measurement: device time (CUDA events on the handle's stream) and algorithmic traffic counters.
// out[0..2] = ms in ig_step total / in k_score / in k_full_lnz (the latter two only while
// profiling is on); out[3] = kernel launches; out[4] = steps; out[5..9] = contacts read, rows,
// fragments, contacts selected, proposals scored by the scoring kernel.
extern "C" int ig_get_stats(ig_handle* h, double out10[10], int32_t reset) {
    if (use(h)) return -1;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->h_sc, h->sc, sizeof(DevScalars), cudaMemcpyDeviceToHost));
    out10[0] = h->ms_step; out10[1] = h->ms_score; out10[2] = h->ms_full;
    out10[3] = (double)h->n_launches; out10[4] = (double)h->n_steps;
    h->last_n_full = h->n_full;
    out10[5] = (double)h->h_sc->st_contacts; out10[6] = (double)h->h_sc->st_rows; out10[7] = (double)h->h_sc->st_frags;
    out10[8] = (double)h->h_sc->st_selected; out10[9] = (double)h->h_sc->st_proposals;
    if (reset) {
        h->ms_step = h->ms_score = h->ms_full = 0.0; h->n_launches = 0; h->n_steps = 0; h->n_full = 0;
        CK(cudaMemset(&h->sc->st_contacts, 0, 5 * sizeof(unsigned long long)));
    }
    return 0;
}
// device self-test of the two transcribed math routines against the library ones (tests/test_gpu_math.py):
// n samples of x log-uniform in [x_lo, x_hi] with exponent y; out[0] = number of inputs where powf_pos differs from powf
// in any bit, out[1] = max |log10_f32(x) - log10((double)x)|
__global__ void k_selftest_math(int n, float x_lo, float x_hi, float y, unsigned long long* n_bad, double* max_err) {
    const float l0 = log2f(x_lo), l1 = log2f(x_hi);
    unsigned long long bad = 0;
    double worst = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned hsh = (unsigned)i * 2654435761u; hsh ^= hsh >> 15; hsh *= 2246822519u; hsh ^= hsh >> 13;
        const float x = exp2f(l0 + (l1 - l0) * ((float)(hsh >> 8) * (1.0f / 16777216.0f)));
        if (__float_as_uint(powf_pos(x, y)) != __float_as_uint(powf(x, y))) bad++;
        worst = fmax(worst, fabs(log10_f32(x) - log10((double)x)));
    }
    if (bad) atomicAdd(n_bad, bad);
    atomicMax((unsigned long long*)max_err, (unsigned long long)__double_as_longlong(worst));   // non-negative doubles order like integers
}
extern "C" int ig_selftest_math(ig_handle* h, int32_t n, float x_lo, float x_hi, float y, double out2[2]) {
    if (use(h)) return -1;
    unsigned long long* d = nullptr;
    if (dev_alloc(h, &d, 2)) return -2;
    CK(cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), h->stream));
    k_selftest_math<<<296, 256, 0, h->stream>>>(n, x_lo, x_hi, y, d, reinterpret_cast<double*>(d + 1));
    if (launch_ok(h, "selftest_math")) return -2;
    unsigned long long r[2];
    CK(cudaMemcpyAsync(r, d, sizeof r, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    out2[0] = (double)r[0];
    memcpy(&out2[1], &r[1], sizeof(double));
    return 0;
}

extern "C" int ig_set_profiling(ig_handle* h, int32_t on) {
    if (!h) return -1;
    h->profile = on ? 1 : 0;
    return 0;
}

// device ms spent in the full-likelihood kernel by ig_full_likelihood calls (nuisance step) and their number
extern "C" int ig_get_nuisance_stats(ig_handle* h, double out2[2], int32_t reset) {
    if (!h) return -1;
    out2[0] = h->ms_nuis; out2[1] = (double)h->n_nuis;
    if (reset) { h->ms_nuis = 0.0; h->n_nuis = 0; }
    return 0;
}

extern "C" int ig_get_full_refresh_count(ig_handle* h, int64_t* out) {
    if (!h) return -1;
    *out = h->last_n_full;
    return 0;
}

// profiling mode only: accumulated ms between consecutive main-stream launches of a step, in order:
// cand_setup, find_cuts(+wait coords), rows_count, rows_write, precompute, score(+wait lnz), finalize,
// select, lnz_outside, apply, post
extern "C" int ig_get_kernel_times(ig_handle* h, double out11[11], int32_t reset) {
    if (!h) return -1;
    for (int i = 0; i < 11; i++) { out11[i] = h->ms_k[i]; if (reset) h->ms_k[i] = 0.0; }
    return 0;
}

// display_current_matrix (CL:2555-2606) without the NS x NS host densification: sub_rank[s] = position of
// sub-fragment s in the displayed order (computed by the caller from ig_get_state like CL:2563-2585);
// out = K*K uint32 symmetric binned contact counts of the strict upper triangle.
extern "C" int ig_contact_thumbnail(ig_handle* h, const int32_t* sub_rank, int32_t K, uint32_t* out) {
    if (use(h)) return -1;
    if (K <= 0 || K > 8192) { h->err = "ig_contact_thumbnail: K out of range"; return -1; }
    int* d_rank = nullptr; unsigned int* d_img = nullptr;
    if (dev_alloc(h, &d_rank, h->ns) || dev_alloc(h, &d_img, (size_t)K * K)) return -2;
    CK(cudaMemcpyAsync(d_rank, sub_rank, sizeof(int) * h->ns, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(d_img, 0, sizeof(unsigned int) * (size_t)K * K, h->stream));
    k_thumbnail<<<h->n_part_full, IG_THREADS, 0, h->stream>>>(h->row_ptr, h->cv, d_rank, h->ns, K, d_img);
    if (launch_ok(h, "thumbnail")) return -2;
    CK(cudaMemcpyAsync(out, d_img, sizeof(unsigned int) * (size_t)K * K, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(d_rank); cudaFree(d_img);
    return 0;
}

// timeline of the last cycle run (IG_TIMELINE builds only): out[n_steps][IG_TL_KERNELS][2] = earliest block start /
// latest block end of each kernel in %globaltimer ns (~0 / 0 when the kernel did not run in that step)
extern "C" int ig_timeline_reset(ig_handle* h) {
    if (use(h)) return -1;
#ifdef IG_TIMELINE
    std::vector<unsigned long long> init((size_t)IG_TL_STEPS * IG_TL_KERNELS * 2);
    for (size_t i = 0; i < init.size(); i += 2) { init[i] = ~0ull; init[i + 1] = 0ull; }
    CK(cudaMemcpyToSymbol(g_tl, init.data(), init.size() * sizeof(unsigned long long)));
    int zero = 0;
    CK(cudaMemcpyToSymbol(g_tl_step, &zero, sizeof zero));
    return 0;
#else
    h->err = "library built without -DIG_TIMELINE";
    return -1;
#endif
}
extern "C" int ig_timeline_blocks(ig_handle* h, int32_t n_blocks, uint64_t* out) {
    if (use(h)) return -1;
#ifdef IG_TIMELINE
    if (n_blocks > IG_TL_BLOCKS) n_blocks = IG_TL_BLOCKS;
    CK(cudaMemcpyFromSymbol(out, g_tlb, (size_t)n_blocks * 4 * sizeof(unsigned long long)));
    return 0;
#else
    (void)n_blocks; (void)out;
    h->err = "library built without -DIG_TIMELINE";
    return -1;
#endif
}
extern "C" int ig_timeline_phases(ig_handle* h, uint64_t* out8, int32_t reset) {
    if (use(h)) return -1;
#ifdef IG_TIMELINE
    CK(cudaMemcpyFromSymbol(out8, g_tlp, 16 * sizeof(unsigned long long)));
    if (reset) { unsigned long long z[16] = {0}; CK(cudaMemcpyToSymbol(g_tlp, z, sizeof z)); }
    return 0;
#else
    (void)out8; (void)reset;
    h->err = "library built without -DIG_TIMELINE";
    return -1;
#endif
}
extern "C" int ig_timeline_get(ig_handle* h, int32_t n_steps, uint64_t* out) {
    if (use(h)) return -1;
#ifdef IG_TIMELINE
    if (n_steps > IG_TL_STEPS) n_steps = IG_TL_STEPS;
    CK(cudaMemcpyFromSymbol(out, g_tl, (size_t)n_steps * IG_TL_KERNELS * 2 * sizeof(unsigned long long)));
    return 0;
#else
    (void)n_steps; (void)out;
    h->err = "library built without -DIG_TIMELINE";
    return -1;
#endif
}

#include "ig_replicas.cuh"   // replica chains across GPUs: NCCL all-gather inside the library

#include "ig_pyramid.cuh"   // pyramid build: binning of a level's contact list (handle-free entry point)
