// instagraal_b200 -- replica chains across GPUs: NCCL all-gather of every chain's likelihood and live scaffold, inside the
// library (no PyTorch in the product).  Part of ig_kernels.cu (host side; included last).
//
// One process per GPU owns 1..n chains of the same level (ig_create + ig_clone).  Once per cycle (or every few hundred
// steps) ig_allgather_best packs, per local chain, a 128-byte header {likelihood, n_contigs, parameters, validity list,
// label counter} + the live scaffold records (64 B x NF) straight from device memory into one send buffer, all-gathers it
// over NVLink (ncclAllGather on the lead handle's stream; NCCL is dlopen'ed, so the library loads without it), compacts the
// headers on the device and copies only those to the host: every rank then takes the same decision (best chain = highest
// likelihood, lowest global index on ties).  The winner's record stays in the receive buffer of every rank
// (ig_get_gathered_state), and ig_adopt_gathered restarts the local chains from it on the device.
// The reference has no counterpart (single process, single GPU); a chain is inherently sequential, so there is no data-path
// collective: replicas only (SURVEY 8e).
#pragma once
#include <dlfcn.h>

struct IgNcclId { char internal[128]; };
struct IgNccl {
    void* lib;
    int (*GetUniqueId)(IgNcclId*);
    int (*CommInitRank)(void**, int, IgNcclId, int);
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t);
    int (*CommDestroy)(void*);
    const char* (*GetErrorString)(int);
};
static IgNccl g_nccl = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
static int nccl_load(std::string& err) {
    if (g_nccl.lib) return 0;
    const char* names[] = {getenv("IG_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* n : names) if (n && (lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!lib) { err = std::string("cannot dlopen libnccl.so.2: ") + dlerror(); return -1; }
    g_nccl.GetUniqueId = (int (*)(IgNcclId*))dlsym(lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, IgNcclId, int))dlsym(lib, "ncclCommInitRank");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(lib, "ncclAllGather");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy) { err = "libnccl lacks the expected symbols"; return -1; }
    g_nccl.lib = lib;
    return 0;
}

// Everything a chain carries besides its scaffold, so that another chain can take over its whole state (ig_adopt_gathered):
// the live parameters (in the order of k_set_params_dev), the carried validity list (quirk Q3) and the label counter.
struct ReplicaHeader {
    double likelihood; int n_contigs; int n_frags;
    float p8[8];
    int valid[12];
    int max_label, pad0;
    double live_likelihood;   // the chain's likelihood_t: `likelihood` (the last applied move's score) is stale after an
                              // accepted nuisance proposal
    int pad[4];
};
static_assert(sizeof(ReplicaHeader) == 128, "ReplicaHeader is 128 bytes (the scaffold records that follow it stay 64-B aligned)");
struct ig_replica_state {
    void* comm;
    int rank, n_ranks, n_local;
    bool gathered;             // an all-gather completed since ig_nccl_init (recv / h_heads hold its result)
    size_t rec_bytes;          // header + NF scaffold records
    char *send, *recv;         // [n_local] / [n_ranks * n_local] records
    ReplicaHeader* heads;      // compact headers on the device, [n_ranks * n_local]
    ReplicaHeader* h_heads;    // pinned
    cudaEvent_t ev0, ev1, ev_chain;
};

__global__ void k_replica_header(const DevScalars* __restrict__ sc, int nf, ReplicaHeader* out) {
    ReplicaHeader r;
    r.likelihood = sc->likelihood; r.n_contigs = sc->n_heads; r.n_frags = nf;
    const float* p = &sc->p.kuhn;
    for (int i = 0; i < 8; i++) r.p8[i] = p[i];
    for (int i = 0; i < 12; i++) r.valid[i] = sc->valid[i];
    r.max_label = sc->max_label; r.pad0 = 0;
    r.live_likelihood = sc->live_likelihood;
    for (int i = 0; i < 4; i++) r.pad[i] = 0;
    *out = r;
}
// a chain takes over the gathered chain's parameters (as k_set_params_dev sets them), validity list and label counter
__global__ void k_replica_adopt(const ReplicaHeader* __restrict__ src, DevScalars* sc) {
    const ReplicaHeader& r = *src;
    Params p;
    p.kuhn = r.p8[0]; p.lm = r.p8[1]; p.c1 = r.p8[2]; p.slope = r.p8[3]; p.d = r.p8[4]; p.d_max = r.p8[5]; p.fact = r.p8[6]; p.v_inter = r.p8[7];
    sc->p = p; sc->log10_vinter = log10((double)p.v_inter);
    for (int i = 0; i < 12; i++) sc->valid[i] = r.valid[i];
    sc->max_label = r.max_label;
    sc->live_likelihood = r.live_likelihood;
}
__global__ void k_replica_compact(const char* __restrict__ recv, size_t rec_bytes, int n, ReplicaHeader* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = *reinterpret_cast<const ReplicaHeader*>(recv + (size_t)i * rec_bytes);
}

extern "C" int ig_nccl_unique_id(char id_out[128]) {
    std::string err;
    if (nccl_load(err)) { g_err = err; return -5; }
    IgNcclId id;
    const int rc = g_nccl.GetUniqueId(&id);
    if (rc) { g_err = std::string("ncclGetUniqueId: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return -5; }
    memcpy(id_out, id.internal, 128);
    return 0;
}

static void replica_free(ig_handle* h) {
    ig_replica_state* r = h->rep;
    if (!r) return;
    if (r->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(r->comm);
    if (r->send) cudaFree(r->send);
    if (r->recv) cudaFree(r->recv);
    if (r->heads) cudaFree(r->heads);
    if (r->h_heads) cudaFreeHost(r->h_heads);
    if (r->ev0) cudaEventDestroy(r->ev0);
    if (r->ev1) cudaEventDestroy(r->ev1);
    if (r->ev_chain) cudaEventDestroy(r->ev_chain);
    delete r;
    h->rep = nullptr;
}

// One communicator per process / GPU, owned by `lead` (any handle of the process).  n_ranks == 1 needs neither an id
// nor NCCL (the "all-gather" is a device copy): several chains on a single GPU.
extern "C" int ig_nccl_init(ig_handle* h, int32_t rank, int32_t n_ranks, int32_t n_local_chains, const char id[128]) {
    if (use(h)) return -1;
    if (n_ranks <= 0 || rank < 0 || rank >= n_ranks || n_local_chains <= 0) { h->err = "ig_nccl_init: bad rank / size"; return -1; }
    replica_free(h);
    ig_replica_state* r = new ig_replica_state();
    memset(r, 0, sizeof *r);
    h->rep = r;
    r->rank = rank; r->n_ranks = n_ranks; r->n_local = n_local_chains;
    r->rec_bytes = sizeof(ReplicaHeader) + sizeof(FragRec) * (size_t)h->nf;
    CK(cudaMalloc((void**)&r->send, r->rec_bytes * n_local_chains));
    CK(cudaMalloc((void**)&r->recv, r->rec_bytes * n_local_chains * n_ranks));
    CK(cudaMalloc((void**)&r->heads, sizeof(ReplicaHeader) * n_local_chains * n_ranks));
    CK(cudaMallocHost((void**)&r->h_heads, sizeof(ReplicaHeader) * n_local_chains * n_ranks));
    CK(cudaEventCreate(&r->ev0)); CK(cudaEventCreate(&r->ev1));
    CK(cudaEventCreateWithFlags(&r->ev_chain, cudaEventDisableTiming));
    if (n_ranks > 1) {
        if (!id) { h->err = "ig_nccl_init: null id"; return -1; }
        if (nccl_load(h->err)) return -5;
        IgNcclId nid;
        memcpy(nid.internal, id, 128);
        const int rc = g_nccl.CommInitRank(&r->comm, n_ranks, nid, rank);
        if (rc) { h->err = std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return -5; }
    }
    return 0;
}

// All-gather of {likelihood, n_contigs, live scaffold} of the n_local chains of every rank.  lik / n_contigs =
// [n_ranks * n_local] in rank-major order; best = index of the highest likelihood (lowest index on ties), identical on
// every rank; ms = device time of pack + all-gather + header compaction (CUDA events on the lead's stream).
extern "C" int ig_allgather_best(ig_handle* h, ig_handle** local, int32_t n_local, double* lik, int32_t* n_contigs, int32_t* best,
                                 float* ms) {
    if (use(h)) return -1;
    ig_replica_state* r = h->rep;
    if (!r) { h->err = "ig_allgather_best: ig_nccl_init not called"; return -1; }
    if (n_local != r->n_local) { h->err = "ig_allgather_best: number of local chains differs from ig_nccl_init"; return -1; }
    for (int c = 0; c < n_local; c++) if (!local[c] || local[c]->nf != h->nf || local[c]->cfg.device != h->cfg.device) { h->err = "ig_allgather_best: chains must share level and device"; return -1; }
    for (int c = 0; c < n_local; c++) {   // the pack waits for everything the chain has enqueued so far
        if (local[c] == h) continue;
        CK(cudaEventRecord(r->ev_chain, local[c]->stream));
        CK(cudaStreamWaitEvent(h->stream, r->ev_chain, 0));
    }
    CK(cudaEventRecord(r->ev0, h->stream));
    for (int c = 0; c < n_local; c++) {
        char* dst = r->send + r->rec_bytes * c;
        k_replica_header<<<1, 1, 0, h->stream>>>(local[c]->sc, h->nf, reinterpret_cast<ReplicaHeader*>(dst));
        CK(cudaMemcpyAsync(dst + sizeof(ReplicaHeader), local[c]->live, sizeof(FragRec) * (size_t)h->nf, cudaMemcpyDeviceToDevice, h->stream));
    }
    const size_t bytes = r->rec_bytes * n_local;
    if (r->n_ranks > 1) {
        const int rc = g_nccl.AllGather(r->send, r->recv, bytes, /* ncclInt8 */ 0, r->comm, h->stream);
        if (rc) { h->err = std::string("ncclAllGather: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return -5; }
    } else {
        CK(cudaMemcpyAsync(r->recv, r->send, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    const int n_all = r->n_ranks * n_local;
    k_replica_compact<<<(n_all + 63) / 64, 64, 0, h->stream>>>(r->recv, r->rec_bytes, n_all, r->heads);
    CK(cudaEventRecord(r->ev1, h->stream));
    CK(cudaMemcpyAsync(r->h_heads, r->heads, sizeof(ReplicaHeader) * n_all, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (launch_ok(h, "allgather_best")) return -2;
    h->n_launches += 2 * n_local + 1;
    r->gathered = true;
    int b = 0;
    for (int i = 0; i < n_all; i++) {
        if (lik) lik[i] = r->h_heads[i].likelihood;
        if (n_contigs) n_contigs[i] = r->h_heads[i].n_contigs;
        if (r->h_heads[i].likelihood > r->h_heads[b].likelihood) b = i;
    }
    if (best) *best = b;
    if (ms) { *ms = 0.f; cudaEventElapsedTime(ms, r->ev0, r->ev1); }
    return 0;
}

// live log-likelihood (likelihood_t) of every chain in the last all-gather, [n_ranks * n_local] rank-major
extern "C" int ig_get_gathered_live_likelihood(ig_handle* h, double* out) {
    if (use(h)) return -1;
    ig_replica_state* r = h->rep;
    if (!r || !r->gathered) { h->err = "ig_get_gathered_live_likelihood: no all-gather since ig_nccl_init (ig_allgather_best)"; return -1; }
    for (int i = 0; i < r->n_ranks * r->n_local; i++) out[i] = r->h_heads[i].live_likelihood;
    return 0;
}

// scaffold of chain `index` (rank-major, as in ig_allgather_best) from the last all-gather, canonical contig labels
extern "C" int ig_get_gathered_state(ig_handle* h, int32_t index, int32_t* out13) {
    if (use(h)) return -1;
    ig_replica_state* r = h->rep;
    if (!r || index < 0 || index >= r->n_ranks * r->n_local) { h->err = "ig_get_gathered_state: no such chain"; return -1; }
    const int nf = h->nf;
    std::vector<FragRec> tmp(nf);
    CK(cudaMemcpyAsync(tmp.data(), r->recv + r->rec_bytes * index + sizeof(ReplicaHeader), sizeof(FragRec) * nf, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < nf; i++) {
        const int* v = reinterpret_cast<const int*>(&tmp[i].f);
        for (int k = 0; k < IG_N_FIELDS; k++) out13[(size_t)k * nf + i] = v[k];
    }
    canonical_labels(nf, out13);
    return 0;
}

// Every local chain other than `index` restarts from chain `index` of the last all-gather, device to device: its scaffold
// records (raw contig labels: labels are only compared for equality, see labels_guard), parameters, validity list and label
// counter, then its live expected-contact table is rebuilt.  The host flags become those of ig_set_state + ig_set_params, so
// the chain's next step is a full refresh (kind 1).  Always read from recv, never from the source handle: one rank and N
// ranks run the same code, and a local source chain is left untouched.  Everything is enqueued on the lead's stream, which
// the gather used (a later gather is ordered after these copies out of recv); each adopting chain's stream waits for it.
extern "C" int ig_adopt_gathered(ig_handle* h, ig_handle** local, int32_t n_local, int32_t index, float p8_out[8], int32_t valid_out[12],
                                 double* likelihood_out) {
    if (use(h)) return -1;
    ig_replica_state* r = h->rep;
    if (!r) { h->err = "ig_adopt_gathered: ig_nccl_init not called"; return -1; }
    if (!r->gathered) { h->err = "ig_adopt_gathered: no all-gather since ig_nccl_init (ig_allgather_best)"; return -1; }
    if (index < 0 || index >= r->n_ranks * r->n_local) { h->err = "ig_adopt_gathered: no such chain"; return -1; }
    if (n_local != r->n_local) { h->err = "ig_adopt_gathered: number of local chains differs from ig_nccl_init"; return -1; }
    for (int c = 0; c < n_local; c++)
        if (!local[c] || local[c]->nf != h->nf || local[c]->ns != h->ns || local[c]->cfg.device != h->cfg.device) {
            h->err = "ig_adopt_gathered: chains must share level and device"; return -1;
        }
    for (int c = 0; c < n_local; c++)
        if (local[c]->pending_steps) { h->err = "ig_adopt_gathered: an asynchronous cycle is still pending (ig_cycle_wait)"; return -1; }
    const ReplicaHeader& src = r->h_heads[index];
    const char* rec = r->recv + r->rec_bytes * index;
    int n_adopt = 0;
    for (int c = 0; c < n_local; c++) {   // the copies wait for everything the chain has enqueued so far
        if (r->rank * n_local + c == index || local[c] == h) continue;
        CK(cudaEventRecord(r->ev_chain, local[c]->stream));
        CK(cudaStreamWaitEvent(h->stream, r->ev_chain, 0));
    }
    for (int c = 0; c < n_local; c++) {
        if (r->rank * n_local + c == index) continue;
        ig_handle* t = local[c];
        CK(cudaMemcpyAsync(t->live, rec + sizeof(ReplicaHeader), sizeof(FragRec) * (size_t)h->nf, cudaMemcpyDeviceToDevice, h->stream));
        k_replica_adopt<<<1, 1, 0, h->stream>>>(reinterpret_cast<const ReplicaHeader*>(rec), t->sc);
        k_exz_table<<<std::min(1024, (t->ns + 256) / 256), 256, 0, h->stream>>>(t->exz, t->ns + 1, t->sc, t->cfg.mean_sub_len_kb, 0);
        n_adopt++;
    }
    if (launch_ok(h, "adopt_gathered")) return -2;
    h->n_launches += 2 * n_adopt;
    CK(cudaEventRecord(r->ev_chain, h->stream));
    for (int c = 0; c < n_local; c++) {
        if (r->rank * n_local + c == index) continue;
        ig_handle* t = local[c];
        if (t != h) CK(cudaStreamWaitEvent(t->stream, r->ev_chain, 0));
        t->label_hi = src.max_label;
        t->coords_fresh = false; t->incr_valid = false;
        t->lnz_stale = true; t->params_set = true;
        t->vinter_pos = src.p8[7] > 0.0f;
    }
    if (p8_out) memcpy(p8_out, src.p8, sizeof src.p8);
    if (valid_out) memcpy(valid_out, src.valid, sizeof src.valid);
    if (likelihood_out) *likelihood_out = src.likelihood;
    return 0;
}
extern "C" int ig_nccl_finalize(ig_handle* h) {
    if (use(h)) return -1;
    replica_free(h);
    return 0;
}
