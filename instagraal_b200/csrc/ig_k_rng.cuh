// instagraal_b200 -- production RNG mode: Philox4x32-10 neighbour draws of a whole cycle.
// Part of ig_kernels.cu (included there, in this order; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// Production RNG mode (SURVEY 8b): the neighbour draws of a whole cycle on the device.
// Philox4x32-10 keyed by the seed, counter = (step, cycle, draw index, attempt); one thread per step.
// Distribution = return_neighbours (CL:3103-3141): min(delta, #non-zero weights) fragments drawn without
// replacement with probability proportional to the level's contact counts (successive draws, a drawn
// fragment is rejected when drawn again), or `delta` distinct uniform fragments when A has no neighbour;
// then sorted (CL:1404) and A itself dropped (DESIGN.md D1).  The stream differs from NumPy's by design
// (the tests hold a NumPy restatement of this kernel).
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ double philox_uniform(unsigned step, unsigned cycle, unsigned draw, unsigned attempt, uint2 key) {
    const uint4 r = philox4x32_10(make_uint4(step, cycle, draw, attempt), key);
    const unsigned long long bits = ((unsigned long long)r.x << 32) | r.y;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);  // 53 bits -> [0, 1)
}
// MAXC = the most draws a plan entry can hold (IG_MAX_CANDS, or IG_MAX_NEIGHBOURS for wider plans), width = its number of
// candidate slots (plan stride 2 + width, written to sc->plan_stride).  Draw i has the counter (t, cycle, i, attempt) in
// both instantiations, so a wide plan's first IG_MAX_CANDS draws are the narrow plan's.
template <int MAXC>
__global__ void k_draw_plan(int* __restrict__ plan, int width, DevScalars* sc, const int* __restrict__ frags, int n_steps, int delta,
                            int nf, const long long* __restrict__ nb_ptr, const int* __restrict__ nb_idx,
                            const double* __restrict__ nb_cdf, const int* __restrict__ nb_nnz, unsigned seed_lo, unsigned seed_hi,
                            unsigned cycle) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t == 0) sc->plan_stride = 2 + width;
    if (t >= n_steps) return;
    const uint2 key = make_uint2(seed_lo, seed_hi);
    const int a = frags[t];
    const long long b = nb_ptr[a], e = nb_ptr[a + 1];
    const int len = (int)(e - b);
    int got[MAXC];
    int n = 0;
    if (len > 0) {
        const int n_max = min(delta, nb_nnz[a]);
        const double total = nb_cdf[e - 1];
        for (int i = 0; i < n_max; i++) {
            int pick = -1;
            for (unsigned att = 0; att < 256u && pick < 0; att++) {
                const double u = philox_uniform((unsigned)t, cycle, (unsigned)i, att, key) * total;
                int lo = 0, hi = len - 1;  // first j with cdf[j] > u
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (nb_cdf[b + mid] > u) hi = mid; else lo = mid + 1; }
                const int c = nb_idx[b + lo];
                bool dup = false;
                for (int j = 0; j < n; j++) dup |= (got[j] == c);
                if (!dup) pick = c;
            }
            if (pick < 0) {  // a weight so dominant that 256 redraws all hit it: take the first free non-zero entry
                for (int j = 0; j < len && pick < 0; j++) {
                    const double wj = nb_cdf[b + j] - (j ? nb_cdf[b + j - 1] : 0.0);
                    const int c = nb_idx[b + j];
                    bool dup = false;
                    for (int q = 0; q < n; q++) dup |= (got[q] == c);
                    if (wj > 0.0 && !dup) pick = c;
                }
            }
            if (pick >= 0) got[n++] = pick;
        }
    } else {
        const int n_max = min(delta, nf - 1);
        for (int i = 0; i < n_max; i++) {
            int pick = -1;
            for (unsigned att = 0; att < 256u && pick < 0; att++) {
                const int c = min(nf - 1, (int)(philox_uniform((unsigned)t, cycle, (unsigned)i, att, key) * (double)nf));
                bool dup = (c == a);
                for (int j = 0; j < n; j++) dup |= (got[j] == c);
                if (!dup) pick = c;
            }
            if (pick >= 0) got[n++] = pick;
        }
    }
    // sorted, without A itself
    for (int i = 1; i < n; i++) { const int v = got[i]; int j = i - 1; while (j >= 0 && got[j] > v) { got[j + 1] = got[j]; j--; } got[j + 1] = v; }
    int* p = plan + (size_t)t * (2 + width);
    int m = 0;
    for (int i = 0; i < n; i++) if (got[i] != a) p[2 + m++] = got[i];
    for (int i = m; i < width; i++) p[2 + i] = 0;
    p[0] = m; p[1] = a;
}
