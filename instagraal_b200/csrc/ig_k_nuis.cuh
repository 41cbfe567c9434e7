// instagraal_b200 -- production RNG mode: the nuisance-parameter step (step_nuisance_parameters, CL:2961-3051) on the device.
// Part of ig_kernels.cu (included there after ig_k_rng.cuh; not a stand-alone translation unit).
#pragma once

// ------------------------------------------------------------------------------------------------
// After every step of a production-mode cycle (ig_set_device_nuisance), one proposal for the p(s) parameters:
//   k_nuis_propose   one thread: draws, proposal, d_max root, validity -> sc->p_test (+ log10 of its v_inter)
//   (k_exz_table, k_coords without write, k_reduce, k_lnz_refresh, k_lnz_stream, k_reduce under p_test: exactly the
//    sequence of ig_full_likelihood(p_test, use_stale_coords = 1), the reference's eval_likelihood_4_nuisance)
//   k_nuis_accept    one thread: L_nuis composed as eval_likelihood_4_nuisance does (CL:1296-1344), Metropolis decision
//                    against the step's o, promotion of the parameters, the step's record, the "sums are stale" flag
//   k_nuis_copy_exz  the live expected-contact table := the test table, only after an acceptance
// Draws (key = the chain's seed, as for its neighbour draws; counters in a domain k_draw_plan never uses, draw < 2^31):
//   A = philox(t, cycle, 0x80000000, 0), B = philox(t, cycle, 0x80000001, 0)
//   id_modif = A.x >> 30 (choice(4), CL:2976), u = 53-bit uniform of (A.y, A.z) (the acceptance draw),
//   z = sqrt(-2 ln(1 - u1)) cos(2 pi u2) with u1, u2 the 53-bit uniforms of (B.x, B.y), (B.z, B.w); draw = sigma z.
// Proposal: the float32 arithmetic of sampler._nuisance_finish under NumPy's promotion rules (float32 + Python float is a
// float32 add); the d_max that goes with it is the root of rippe(x) = y (deviation D3, DESIGN.md) instead of scipy's
// fsolve on |y - rippe(x)|.  The tests hold a NumPy restatement of all of this.

__device__ __forceinline__ double nuis_u53(unsigned hi, unsigned lo) {   // as philox_uniform builds it
    const unsigned long long bits = ((unsigned long long)hi << 32) | lo;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);
}
// float32 x^y, x^y evaluated in double and rounded once (the correctly rounded powf on every input the proposal meets)
__device__ __forceinline__ float nuis_powf(float x, float y) { return __double2float_rn(pow((double)x, (double)y)); }
// 10 ** (log10(v) - 2) of _nuisance_draws as a float32 chain, each operation rounded once
__device__ __forceinline__ float nuis_sigma(float v) {
    const float l = __double2float_rn(log10((double)v));
    return __double2float_rn(pow(10.0, (double)__fadd_rn(l, -2.0f)));
}
// c1 = float32((0.53 * (lm / kuhn) ** slope) * kuhn ** -3) (CL:2990 and the three others)
__device__ __forceinline__ float nuis_c1(float kuhn, float lm, float slope) {
    return __fmul_rn(__fmul_rn(0.53f, nuis_powf(__fdiv_rn(lm, kuhn), slope)), nuis_powf(kuhn, -3.0f));
}

// d_max of a parameter set: x > 0 with rippe(x) = A 0.53 kuhn^-3 (lm x / kuhn)^slope exp((dd - 2) / ((lm x / kuhn)^2 + dd)) = y,
// in double.  dd == 2 (what the p(s) fit always returns): closed form.  Otherwise safeguarded Newton on
// g(L) = log rippe(e^L) - log y from the closed-form start inside a sign-change bracket (bisection when Newton leaves it),
// to 1e-14 in L (relative in x).  Returns 0 when there is no root (A <= 0, y <= 0, slope >= 0, non-finite inputs, no
// bracket within |L| <= 700).
__host__ __device__ inline int nuis_dmax_root(double kuhn, double lm, double slope, double dd, double A, double y, double* out) {
    *out = NAN;
    if (!(A > 0.0) || !(y > 0.0) || !(slope < 0.0) || !(kuhn > 0.0) || !(lm > 0.0) || !isfinite(A) || !isfinite(y) ||
        !isfinite(slope) || !isfinite(kuhn) || !isfinite(lm) || !isfinite(dd))
        return 0;
    const double c = A * 0.53 * pow(kuhn, -3.0);
    const double x0 = (kuhn / lm) * pow(y / c, 1.0 / slope);
    if (dd == 2.0) {
        if (!(x0 > 0.0) || !isfinite(x0)) return 0;
        *out = x0;
        return 1;
    }
    const double k = lm / kuhn, lk = log(k), lc = log(c), ly = log(y);
    auto g = [&](double L) { const double q2 = k * k * exp(2.0 * L); return lc + slope * (lk + L) + (dd - 2.0) / (q2 + dd) - ly; };
    auto dg = [&](double L) { const double q2 = k * k * exp(2.0 * L); const double den = q2 + dd; return slope - (dd - 2.0) * 2.0 * q2 / (den * den); };
    double L = (x0 > 0.0 && isfinite(x0)) ? log(x0) : 0.0;
    double a = L, b = L, ga = g(L), gb = ga;
    if (ga == 0.0) { *out = exp(L); return isfinite(*out) && *out > 0.0; }
    for (double s = 1.0; !(ga > 0.0 && gb < 0.0) && !(ga < 0.0 && gb > 0.0); s *= 2.0) {   // grow a bracket around L
        if (s > 1400.0) return 0;
        a = fmax(L - s, -700.0); b = fmin(L + s, 700.0);
        ga = g(a); gb = g(b);
        if (!isfinite(ga) || !isfinite(gb)) return 0;
    }
    const bool rising = gb > 0.0;
    for (int it = 0; it < 200; it++) {
        const double gl = g(L);
        if (gl == 0.0) break;
        if ((gl > 0.0) == rising) b = L; else a = L;
        double Ln = L - gl / dg(L);
        if (!(Ln > a && Ln < b)) Ln = 0.5 * (a + b);
        const double step = fabs(Ln - L);
        L = Ln;
        if (step <= 1e-14 * fmax(1.0, fabs(L)) || b - a <= 1e-14 * fmax(1.0, fabs(L))) break;
    }
    *out = exp(L);
    return isfinite(*out) && *out > 0.0;
}

// the seed and cycle of the cycle being enqueued (once per cycle: the nuisance graph and the tempered selection read them
// from the record)
__global__ void k_nuis_begin(DevScalars* sc, unsigned seed_lo, unsigned seed_hi, unsigned cycle) {
    sc->nuis_key_lo = seed_lo; sc->nuis_key_hi = seed_hi; sc->nuis_cycle = cycle;
}

__global__ void k_nuis_propose(DevScalars* sc) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned t = (unsigned)(sc->step_idx - 1), cyc = sc->nuis_cycle;   // k_post has advanced step_idx
    const uint2 key = make_uint2(sc->nuis_key_lo, sc->nuis_key_hi);
    const uint4 A = philox4x32_10(make_uint4(t, cyc, 0x80000000u, 0u), key);
    const uint4 B = philox4x32_10(make_uint4(t, cyc, 0x80000001u, 0u), key);
    const int id = (int)(A.x >> 30);
    const double u = nuis_u53(A.y, A.z);
    const double u1 = nuis_u53(B.x, B.y), u2 = nuis_u53(B.z, B.w);
    const double z = __dmul_rn(sqrt(__dmul_rn(-2.0, log(1.0 - u1))), cos(__dmul_rn(2.0 * M_PI, u2)));
    const Params p = sc->p;
    Params q = p;
    double draw = NAN;   // NaN: no draw (id 3 with d_nuc <= 0: sigma_d_nuc <= 0, draw = None in _nuisance_draws)
    double root = NAN;
    int have_root = 1;
    if (id == 0) {
        draw = __dmul_rn((double)nuis_sigma(p.fact), z);
        q.fact = __fadd_rn(p.fact, __double2float_rn(draw));
        have_root = nuis_dmax_root(q.kuhn, q.lm, q.slope, q.d, q.fact, q.v_inter, &root);
    } else if (id == 1) {
        draw = __dmul_rn(0.005, z);
        q.slope = __fadd_rn(p.slope, __double2float_rn(draw));
        have_root = nuis_dmax_root(q.kuhn, q.lm, q.slope, q.d, q.fact, q.v_inter, &root);
    } else if (id == 2) {
        draw = __dmul_rn(100.0, z);
        q.d_max = __fadd_rn(p.d_max, __double2float_rn(draw));
        // new d_nuc = peval(new_d_max, [kuhn, lm, slope, d, fact]): param[3] = d is the amplitude (quirk Q7), exp term 1
        const float k3 = nuis_powf(p.kuhn, -3.0f);
        const float pw = nuis_powf(__fdiv_rn(__fmul_rn(p.lm, q.d_max), p.kuhn), p.slope);
        q.v_inter = __fmul_rn(p.d, __fmul_rn(__fmul_rn(0.53f, k3), pw));
    } else {
        if (nuis_sigma(p.v_inter) > 0.0f) {
            draw = __dmul_rn((double)nuis_sigma(p.v_inter), z);
            q.v_inter = __fadd_rn(p.v_inter, __double2float_rn(draw));
        }
        have_root = nuis_dmax_root(q.kuhn, q.lm, q.slope, q.d, q.fact, q.v_inter, &root);
    }
    if (id != 2) q.d_max = __double2float_rn(root);   // NaN when there is no root
    q.c1 = nuis_c1(q.kuhn, q.lm, q.slope);
    const float* f = &q.kuhn;
    bool finite = true;
    for (int i = 0; i < 8; i++) finite = finite && isfinite(f[i]);
    const int valid = have_root && finite && q.fact > 0.0f && q.slope < 0.0f && q.d_max > 0.0f && q.v_inter > 0.0f;
    // the likelihood kernels that follow run whatever the validity (the graph is fixed): they only do arithmetic on q
    sc->p_test = q;
    sc->log10_vinter_test = log10((double)q.v_inter);
    sc->nuis_id = id; sc->nuis_valid = valid; sc->nuis_u = u; sc->nuis_draw = draw;
}

__global__ void k_nuis_accept(DevScalars* sc, ig_nuisance_step* __restrict__ rec, double n_pix) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    // eval_likelihood_4_nuisance (CL:1296-1344 as the facade composes it), operation for operation, no contraction
    const double log_e = 0.43429448190325182;
    const Params q = sc->p_test;
    const double intra = __dmul_rn(sc->full_out[1], log_e);
    const double inter = __dmul_rn(__dmul_rn(__dmul_rn(log_e, __dsub_rn(n_pix, (double)sc->full_nintra)), -1.0), (double)q.v_inter);
    const double l_nuis = __dadd_rn(sc->full_out[0], __dadd_rn(intra, inter));
    const double l_t = sc->likelihood;
    const double u = sc->nuis_u;
    const int valid = sc->nuis_valid;
    // temperature() is 1.0 in the reference, the chain temperature T when one is set (DESIGN.md 4e); a NaN ratio is never >= u
    const double T = sc->temperature;
    const int acc = valid && (exp(__dsub_rn(l_nuis, l_t) / (T > 0.0 ? T : 1.0)) >= u);
    if (acc) { sc->p = q; sc->log10_vinter = sc->log10_vinter_test; sc->live_likelihood = l_nuis; }
    sc->nuis_stale = acc;   // the next step's likelihood sums are stale exactly when this proposal was accepted
    ig_nuisance_step r;
    r.likelihood_nuis = l_nuis; r.likelihood_t_after = acc ? l_nuis : l_t; r.u = u; r.draw = sc->nuis_draw;
    const float* f = &q.kuhn;
    for (int i = 0; i < 8; i++) r.p_test[i] = f[i];
    r.id_modif = sc->nuis_id; r.accepted = acc; r.valid = valid; r.pad = 0;
    rec[sc->step_idx - 1] = r;
}

// after an acceptance: the live expected-contact table (+ its two record slots) := the one built for p_test, which holds
// the values k_exz_table computes for the new live parameters
__global__ void k_nuis_copy_exz(float* __restrict__ exz, const float* __restrict__ exz_test, int n, const DevScalars* __restrict__ sc) {
    if (!sc->nuis_stale) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) exz[i] = exz_test[i];
}
