// Device helpers shared by every kernel family: transfer function, stimulus lookup, Philox noise.
// Arithmetic follows the reference's operation order with explicit round-to-nearest intrinsics (no FMA
// contraction) wherever the reference computes elementwise in fp32, so that the only differences to the
// CPU path are the summation order of W.r and the last-ulp behaviour of tanhf/expf.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "odecol_internal.h"

namespace odecol {

#define ODECOL_DEVINL __device__ __forceinline__

// ---- phi and its derivative ---------------------------------------------------------------------------------
// reference src/utils.py:13-28: x_nom = a x - b; z = 80 tanh(-d x_nom / 80); r = x_nom / (1 - exp(z)).
ODECOL_DEVINL float phi(float x) {
    const float x_nom = __fsub_rn(__fmul_rn(48.0f, x), 981.0f);
    float z = __fmul_rn(-0.0089f, x_nom);
    z = __fmul_rn(80.0f, tanhf(__fdiv_rn(z, 80.0f)));
    const float den = __fsub_rn(1.0f, expf(z));
    return __fdiv_rn(x_nom, den);
}

// r = phi(x) and dr/dx in one pass (what autograd assembles from the pieces above).
ODECOL_DEVINL void phi_dphi(float x, float& r, float& dr) {
    const float x_nom = __fsub_rn(__fmul_rn(48.0f, x), 981.0f);
    const float z = __fmul_rn(-0.0089f, x_nom);
    const float th = tanhf(__fdiv_rn(z, 80.0f));
    const float e = expf(__fmul_rn(80.0f, th));
    const float den = __fsub_rn(1.0f, e);
    const float inv = __fdiv_rn(1.0f, den);
    r = __fdiv_rn(x_nom, den);
    // d r / d x_nom = 1/den + x_nom/den^2 * e * dz'/dx_nom,  dz'/dx_nom = (1 - th^2) * (-d)
    const float dzp = (1.0f - th * th) * (-0.0089f);
    dr = 48.0f * (inv + r * inv * e * dzp);
}

// ---------------------------------------------------------------------------------------------------------------
// fast, FP32-accurate elementwise math (the staged families' epilogues; the on-chip family on request); phi within 5e-6 of
// float64 over its whole range (tests/test_gpu_rate_range.py)
// ---------------------------------------------------------------------------------------------------------------
ODECOL_DEVINL float exp_fast(float x) {            // |x| < 87
    const float n = rintf(x * 1.4426950408889634f);
    float f = fmaf(n, -0.693145751953125f, x);
    f = fmaf(n, -1.42860682030941723212e-6f, f);
    float p;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p) : "f"(f * 1.4426950408889634f));
    return p * __int_as_float(((int)n + 127) << 23);
}
// tanh on the argument range of phi's soft clamp, z = 80 tanh(-0.0089 x_nom / 80): Taylor through u^11, < 3e-8 relative for
// |u| <= 0.4 (x_nom within +-3595, i.e. V - A between -54 and +95), the argument CLAMPED beyond.  Out there exp(z) is below
// 1e-13 or above 1e13 either way, so phi = x_nom / (1 - exp(z)) does not see the difference in float32 (|delta r| < 1e-9);
// a branch to an exp-based formula cost every evaluation a divergence point and doubled the code (round-2 SASS: 45 static
// instructions per phi, 16 BSSY / BSYNC pairs per four elements).
ODECOL_DEVINL float tanh_small(float u) {
    u = fminf(fmaxf(u, -0.4f), 0.4f);
    const float s = u * u;
    float p = fmaf(s, -8.8632355299021965e-3f, 2.1869488536155203e-2f);   // -1382/155925, 62/2835
    p = fmaf(s, p, -5.3968253968253968e-2f);                               // -17/315
    p = fmaf(s, p, 1.3333333333333333e-1f);                                // 2/15
    p = fmaf(s, p, -3.3333333333333333e-1f);                               // -1/3
    return fmaf(u * s, p, u);
}
// exp(80 th) for phi's soft-clamped exponent as ONE multiply and ex2.approx (the SFU splits integer and fraction itself):
// the exponent z = 80 th is only known to 2^-24 relative in float32 whichever way it is formed (|z| <= 30.4 -> up to 2e-6
// relative in exp(z), in the reference's own arithmetic as well), and where exp(z) matters to phi -- |z| of order one, the
// cancellation in 1 - exp(z) -- the error is the SFU's 2^-22, with or without a Cody-Waite reduction in front of it.  So the
// reduction (rint, two fmas, int conversion, exponent insertion: 8 of phi's 25 instructions) bought no accuracy.
ODECOL_DEVINL float exp80_fast(float th) {
    float p;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p) : "f"(th * 115.41560327111707f));      // 80 log2(e)
    return p;
}
// 1 / x as the bare SFU instruction (__fdividef / div.approx wrap it in a range check and two conditional rescalings for
// denominators below 2^-126: 1 - exp(z) only gets there AT phi's removable pole, where the reference itself returns NaN)
ODECOL_DEVINL float rcp_fast(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// phi's removable pole at x = 981/48 (x_nom = 0, phi -> 1/0.0089 = 112.36 Hz, phi' -> 24): phi is smooth there, but the
// quotient x_nom / (1 - exp(z)) cancels.  An error eps in exp(z) becomes eps / |v| in phi and about 2 eps / v^2 in phi'
// (v = -z, about 0.43 (x - 981/48)); at the pole itself the quotient is 0 * inf = NaN.  Inside |v| < kPhiPoleBand
// (|x - 981/48| < 0.58) the fast path takes the same function without a quotient of small numbers: phi = G(v) / 0.0089 with
// G = R(u) B(v), R = u / tanh u (u = 0.0089 x_nom / 80 = atanh(v / 80), so R = 1 + v^2 / 19200 + O(v^4 1e-8)) and
// B(v) = v / (1 - exp(-v)) = 1 + v/2 + v^2/12 - v^4/720 + O(v^6 / 30240); phi' = 48 G'(v) (1 - tanh^2 u).  In the band
// the series is off by less than 1e-7 in phi and 6e-7 in phi' (float32 emulation against float64); the quotient, with
// ex2.approx one ulp off, would be off by 2e-7 and 2e-6 at the band's edge.  The choice is a select, not a branch.
// The reference arithmetic (phi, phi_dphi above) keeps the quotient, NaN included.
constexpr float kPhiPoleBand = 0.25f;
constexpr float kG2 = 1.0f / 12.0f + 1.0f / 19200.0f, kG3 = 1.0f / 38400.0f, kG4 = -1.0f / 720.0f + 1.0f / 230400.0f;

ODECOL_DEVINL float phi_fast(float x) {
    const float x_nom = fmaf(48.0f, x, -981.0f);
    const float th = tanh_small(x_nom * (-0.0089f / 80.0f));
    const float v = -80.0f * th;
    const float G = fmaf(v, fmaf(v, fmaf(v, fmaf(v, kG4, kG3), kG2), 0.5f), 1.0f);
    const float r = x_nom * rcp_fast(1.0f - exp80_fast(th));
    return fabsf(v) < kPhiPoleBand ? (1.0f / 0.0089f) * G : r;
}

// phi' = 48 (s1 + s2 (1 - th^2)): s1 = inv and s2 = -0.0089 r inv e from the quotient; in the band, with G = R(u) B(v)
// differentiated factor by factor, s1 = R'(u) B / 80 (R' = 2u/3) and s2 = R B'(v).  (This form, rather than G'(v), is
// the one that keeps the register-resident reverse kernel k_rk4_bwd_small<40, true> within 168 registers without spilling.)
ODECOL_DEVINL void phi_dphi_fast(float x, float& r, float& dr) {
    const float x_nom = fmaf(48.0f, x, -981.0f);
    const float a = x_nom * (-0.0089f / 80.0f);          // -u
    const float th = tanh_small(a);
    const float e = exp80_fast(th);
    const float inv = rcp_fast(1.0f - e);
    const float v = -80.0f * th, w = v * v;
    const float R = fmaf(a * a, 1.0f / 3.0f, 1.0f);
    const float B = fmaf(v, fmaf(v, fmaf(w, -1.0f / 720.0f, 1.0f / 12.0f), 0.5f), 1.0f);   // 1 + v/2 + v^2/12 - v^4/720
    const float dB = fmaf(v, fmaf(w, -1.0f / 180.0f, 1.0f / 6.0f), 0.5f);                 // 1/2 + v/6 - v^3/180
    const bool near = fabsf(v) < kPhiPoleBand;
    const float rq = x_nom * inv;
    r = near ? (1.0f / 0.0089f) * R * B : rq;
    const float s1 = near ? a * B * (-1.0f / 120.0f) : inv;
    const float s2 = near ? R * dB : rq * inv * e * (-0.0089f);
    dr = 48.0f * fmaf(s2, 1.0f - th * th, s1);
}

// ---- stimulus lookup (reference src/utils.py:31-46) ------------------------------------------------------------
// Finds idx in [1, K-1] with searchsorted(right=True) semantics starting from a hint; returns clamped time.
ODECOL_DEVINL float knot_locate(const float* __restrict__ kt, int K, float t, int& idx) {
    const float tc = fminf(fmaxf(t, __ldg(kt)), __ldg(kt + K - 1));
    int i = idx;
    i = i < 1 ? 1 : (i > K - 1 ? K - 1 : i);
    while (i > 1 && __ldg(kt + i - 1) > tc) --i;        // want kt[i-1] <= tc
    while (i < K - 1 && __ldg(kt + i) <= tc) ++i;       // want kt[i] > tc (or i == K-1)
    idx = i;
    return tc;
}

ODECOL_DEVINL float knot_value(const float* __restrict__ kt, const float* __restrict__ ku_trial, int n_in,
                               int idx, float tc, int c) {
    const float x0 = __ldg(kt + idx - 1), x1 = __ldg(kt + idx);
    const float y0 = __ldg(ku_trial + (size_t)(idx - 1) * n_in + c);
    const float y1 = __ldg(ku_trial + (size_t)idx * n_in + c);
    const float slope = __fdiv_rn(__fsub_rn(y1, y0), __fsub_rn(x1, x0));
    return __fadd_rn(y0, __fmul_rn(slope, __fsub_rn(tc, x0)));
}

// One stimulus channel per lane with the interval cached in registers: as long as the query time stays inside the knot
// interval found last (the common case: four stage times per step, a handful of knots per trial) the lookup is two
// compares and the interpolation y0 + slope (tc - x0); the arithmetic and its order are those of knot_value, so the
// result is bit-identical to the uncached path.
struct KnotLane {
    float lo, hi;            // validity of the cached interval: lo <= tc < hi  (+-inf at the ends: held values)
    float x0, y0, slope;
    int idx;
    ODECOL_DEVINL void reset() { lo = 1.0f; hi = 0.0f; idx = 1; x0 = y0 = slope = 0.0f; }   // empty interval: first query locates
    ODECOL_DEVINL float value(const float* __restrict__ kt, const float* __restrict__ ku_trial, int K, int n_in, int ch, float t) {
        const float tc = fminf(fmaxf(t, __ldg(kt)), __ldg(kt + K - 1));
        if (!(lo <= tc && tc < hi)) {
            (void)knot_locate(kt, K, t, idx);
            x0 = __ldg(kt + idx - 1);
            const float x1 = __ldg(kt + idx);
            y0 = __ldg(ku_trial + (size_t)(idx - 1) * n_in + ch);
            const float y1 = __ldg(ku_trial + (size_t)idx * n_in + ch);
            slope = __fdiv_rn(__fsub_rn(y1, y0), __fsub_rn(x1, x0));
            lo = idx == 1 ? -INFINITY : x0;
            hi = idx == K - 1 ? INFINITY : x1;
        }
        return __fadd_rn(y0, __fmul_rn(slope, __fsub_rn(tc, x0)));
    }
};

// ---- elementwise drift given the total synaptic input ------------------------------------------------------------
// total = (ff + bias + rec); reference: coupled_columns.py:225-233.
ODECOL_DEVINL void drift(const Consts& c, float V, float A, float F, float r, float kappa, float total_raw,
                         float& dV, float& dA, float& dF) {
    const float total = __fmul_rn(total_raw, c.tau_s);
    dV = __fdiv_rn(__fadd_rn(-V, __fmul_rn(total, c.R)), c.tau_m);
    dA = __fdiv_rn(__fadd_rn(-A, __fmul_rn(kappa, r)), c.tau_a);
    dF = __fdiv_rn(__fadd_rn(-F, r), c.tau_s);
}

// ---- Philox4x32-10 ---------------------------------------------------------------------------------------------
struct Philox {
    uint32_t k0, k1;
    ODECOL_DEVINL Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
    ODECOL_DEVINL uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            const uint32_t n0 = hi1 ^ c1 ^ a, n2 = hi0 ^ c3 ^ b;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};

// one standard normal from two 32-bit words (Box-Muller, u1 in (0,1])
ODECOL_DEVINL float normal_from_bits(uint32_t a, uint32_t b) {
    const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
    const float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// Virtual Brownian tree: W(t) on [T0, T0 + span] for one trial.  The query time is quantised to
// q / 2^24 of the span (integer path, so every kernel family walks the same nodes), bisection over 24 levels
// with Brownian-bridge midpoints, linear inside the leaf.  Deterministic in (seed, trial, t), hence
// W(a,c) = W(a,b) + W(b,c) under step rejection and results do not depend on sharding or kernel family.
constexpr int kBrownianDepth = 24;
constexpr uint32_t kBrownianRootLevel = 0xFFFFFFFFu;

ODECOL_DEVINL void brownian_path(float T0, float span, float t, uint32_t& q, float& frac) {
    float u = (t - T0) / span;
    u = fminf(fmaxf(u, 0.0f), 1.0f) * 16777216.0f;
    float fl = floorf(u);
    if (fl > 16777215.0f) fl = 16777215.0f;
    q = (uint32_t)fl;
    frac = fminf(u - fl, 1.0f);
}

// normal deviate of tree node (level, index-within-level); level == kBrownianRootLevel is W(T0+span)/sqrt(span)
ODECOL_DEVINL float brownian_node(const Philox& px, uint64_t trial, uint32_t level, uint32_t index) {
    const uint4 bits = px((uint32_t)trial, (uint32_t)(trial >> 32), level, index);
    return normal_from_bits(bits.x, bits.y);
}

// combine: z[l] is the deviate of the node visited at level l, zroot the root deviate
template <typename ZF>
ODECOL_DEVINL float brownian_combine(float span, uint32_t q, float frac, float zroot, ZF z) {
    float wa = 0.0f, wb = sqrtf(span) * zroot;
    float half_sd = 0.5f * sqrtf(span);            // 0.5*sqrt(width), width halves per level
#pragma unroll 1
    for (int level = 0; level < kBrownianDepth; ++level) {
        const float wm = 0.5f * (wa + wb) + half_sd * z(level);
        if ((q >> (kBrownianDepth - 1 - level)) & 1u) wa = wm; else wb = wm;
        half_sd *= 0.70710678118654752f;
    }
    return wa + frac * (wb - wa);
}

// sequential version (one thread per trial)
ODECOL_DEVINL float brownian_tree(const Philox& px, uint64_t trial, float T0, float span, float t) {
    uint32_t q; float frac;
    brownian_path(T0, span, t, q, frac);
    const float zroot = brownian_node(px, trial, kBrownianRootLevel, 0u);
    return brownian_combine(span, q, frac, zroot, [&](int level) {
        const uint32_t index = level == 0 ? 0u : (q >> (kBrownianDepth - level));
        return brownian_node(px, trial, (uint32_t)level, index);
    });
}

// ---- Levy-area-consistent virtual Brownian tree (adaptive srk) -----------------------------------------------------------
// The srk scheme consumes, per step, the increment W and the space-time Levy area U = int (W_r - W_t0) dr; under step
// rejection both must stay consistent on every sub-interval (W(a,c) = W(a,b) + W(b,c), U(a,c) = U(a,b) + U(b,c) +
// (c - b) W(a,b)), which is what torchsde's BrownianInterval guarantees.  Here every dyadic interval of the tree carries
// (W, H) with H = U / h - W / 2 the normalised space-time Levy area (H ~ N(0, h / 12), independent of W); bisecting an
// interval of length h draws Z ~ N(0, h / 16), N ~ N(0, h / 12) (Foster, Lyons & Oberhauser 2020, Theorem 6; verified
// against the conditional law of the four half-interval variables in tests/test_oracle_selfcheck.py):
//     W_left = W/2 + 3/2 H + Z      H_left  = H/4 - Z/2 + N/2
//     W_right = W/2 - 3/2 H - Z     H_right = H/4 - Z/2 - N/2
// A query walks the 24 levels once and returns the CUMULATIVE pair W(t) = W(T0, t), I(t) = int_{T0}^{t} W(T0, r) dr in
// double precision; for a step [a, b]:  W = W(b) - W(a),  U = I(b) - I(a) - (b - a) W(a)  (the difference of the I's
// cancels to ~h^1.5, hence the doubles).  Node deviates are keyed by (seed, trial, level | 0x40000000, index): a stream
// separate from the W-only tree of the Euler-Maruyama solvers.
constexpr uint32_t kLevyLevelTag = 0x40000000u;
constexpr uint32_t kLevyRootLevel = 0x7FFFFFFFu;

ODECOL_DEVINL void levy_node(const Philox& px, uint64_t trial, uint32_t level, uint32_t index, float& z, float& n) {
    const uint4 bits = px((uint32_t)trial, (uint32_t)(trial >> 32), level | kLevyLevelTag, index);
    z = normal_from_bits(bits.x, bits.y);
    n = normal_from_bits(bits.z, bits.w);
}

// zn(level, z, n) yields the two deviates of the node visited at `level` (level == kBrownianDepth: the root's W and H)
template <typename ZN>
ODECOL_DEVINL void levy_combine(float span, uint32_t q, float frac, ZN zn, double& W, double& I) {
    float z, n;
    zn(kBrownianDepth, z, n);
    double h = (double)span;
    double Wab = sqrt(h) * (double)z, Hab = sqrt(h / 12.0) * (double)n;
    double Wa = 0.0, Ia = 0.0;
#pragma unroll 1
    for (int level = 0; level < kBrownianDepth; ++level) {
        zn(level, z, n);
        const double Z = 0.25 * sqrt(h) * (double)z, Nn = sqrt(h / 12.0) * (double)n;
        const double W1 = 0.5 * Wab + 1.5 * Hab + Z, H1 = 0.25 * Hab - 0.5 * Z + 0.5 * Nn;
        const double hh = 0.5 * h;
        if ((q >> (kBrownianDepth - 1 - level)) & 1u) {          // right half: move the left edge to the midpoint
            Ia += hh * Wa + hh * (H1 + 0.5 * W1);
            Wa += W1;
            Wab = 0.5 * Wab - 1.5 * Hab - Z;
            Hab = 0.25 * Hab - 0.5 * Z - 0.5 * Nn;
        } else {
            Wab = W1; Hab = H1;
        }
        h = hh;
    }
    const double fr = (double)frac;                              // linear inside the leaf (span / 2^24 long)
    W = Wa + fr * Wab;
    I = Ia + fr * h * Wa + 0.5 * fr * fr * h * Wab;
}

// sequential version (one thread per query)
ODECOL_DEVINL void levy_tree(const Philox& px, uint64_t trial, float T0, float span, float t, double& W, double& I) {
    uint32_t q; float frac;
    brownian_path(T0, span, t, q, frac);
    levy_combine(span, q, frac, [&](int level, float& z, float& n) {
        if (level == kBrownianDepth) levy_node(px, trial, kLevyRootLevel, 0u, z, n);
        else levy_node(px, trial, (uint32_t)level, level == 0 ? 0u : (q >> (kBrownianDepth - level)), z, n);
    }, W, I);
}

// ---- torchsde srk (Roessler SRI2, SRID2 tableau) pieces shared by the on-chip and the staged kernels ---------------
struct Srid2 {
    static constexpr float quarter = 0.25f, half = 0.5f;
    static constexpr float a0 = (float)(1.0 / 6), a1 = (float)(1.0 / 6), a2 = (float)(2.0 / 3);
};

// (W, U) of step k for one trial: host tables or Philox (U | W ~ N(h W / 2, h^3 / 12)).  The W deviate is the one the
// fixed-step Euler-Maruyama kernel draws for the same (seed, trial, step), so both methods see the same path.
ODECOL_DEVINL void srk_increments(const float* __restrict__ dWs, const float* __restrict__ dUs, const Philox& px,
                                  unsigned long long trial, long long k, int B, int b, float h, float& dw, float& du) {
    if (dWs) {
        dw = __ldg(dWs + (size_t)k * B + b);
        du = __ldg(dUs + (size_t)k * B + b);
    } else {
        const uint4 bits = px((uint32_t)trial, (uint32_t)(trial >> 32), (uint32_t)k, 0x80000000u | (uint32_t)(k >> 32));
        dw = sqrtf(h) * normal_from_bits(bits.x, bits.y);
        du = 0.5f * h * dw + sqrtf(h * h * h * (1.0f / 12.0f)) * normal_from_bits(bits.z, bits.w);
    }
}

// g_weight of the four stages (thread-uniform scalars)
ODECOL_DEVINL void srk_g_weights(float h, float dw, float du, float gw[4]) {
    const float rdt = __fdiv_rn(1.0f, h), sq = __fsqrt_rn(h);
    const float i_kk = __fmul_rn(__fsub_rn(__fmul_rn(dw, dw), h), 0.5f);
    const float i_kkk = __fdiv_rn(__fsub_rn(__fmul_rn(__fmul_rn(dw, dw), dw), __fmul_rn(__fmul_rn(3.0f, h), dw)), 6.0f);
    // beta rows as float32 (torch multiplies a float32 tensor by the Python scalar cast to float32)
    constexpr float b1[4] = {-1.f, (float)(4.0 / 3), (float)(2.0 / 3), 0.f};
    constexpr float b2[4] = {1.f, (float)(-4.0 / 3), (float)(1.0 / 3), 0.f};
    constexpr float b3[4] = {2.f, (float)(-4.0 / 3), (float)(-2.0 / 3), 0.f};
    constexpr float b4[4] = {-2.f, (float)(5.0 / 3), (float)(-2.0 / 3), 1.f};
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        float w = __fadd_rn(__fmul_rn(b1[s], dw), __fdiv_rn(__fmul_rn(b2[s], i_kk), sq));
        w = __fadd_rn(w, __fmul_rn(__fmul_rn(b3[s], du), rdt));
        gw[s] = __fadd_rn(w, __fmul_rn(__fmul_rn(b4[s], i_kkk), rdt));
    }
}

// H0 of stage 3 for one state component: y + (1/4 f0) h + ((1 g) U) / h + (1/4 f1) h + ((1/2 g) U) / h
ODECOL_DEVINL float srk_h2(float y, float f0, float f1, float g, float h, float du, float rdt) {
    float v = __fadd_rn(y, __fmul_rn(__fmul_rn(Srid2::quarter, f0), h));
    v = __fadd_rn(v, __fmul_rn(__fmul_rn(g, du), rdt));
    v = __fadd_rn(v, __fmul_rn(__fmul_rn(Srid2::quarter, f1), h));
    return __fadd_rn(v, __fmul_rn(__fmul_rn(__fmul_rn(Srid2::half, g), du), rdt));
}

// ---- Dormand-Prince 5(4) tableau (Shampine's variant, as torchdiffeq tabulates it) ---------------------------------
struct DP {
    // float32(coefficient), as torchdiffeq casts its float64 tableau to y0.dtype
    static constexpr float a1 = (float)(1.0 / 5), a2 = (float)(3.0 / 10), a3 = (float)(4.0 / 5), a4 = (float)(8.0 / 9);
    static constexpr float b10 = (float)(1.0 / 5);
    static constexpr float b20 = (float)(3.0 / 40), b21 = (float)(9.0 / 40);
    static constexpr float b30 = (float)(44.0 / 45), b31 = (float)(-56.0 / 15), b32 = (float)(32.0 / 9);
    static constexpr float b40 = (float)(19372.0 / 6561), b41 = (float)(-25360.0 / 2187), b42 = (float)(64448.0 / 6561),
                           b43 = (float)(-212.0 / 729);
    static constexpr float b50 = (float)(9017.0 / 3168), b51 = (float)(-355.0 / 33), b52 = (float)(46732.0 / 5247),
                           b53 = (float)(49.0 / 176), b54 = (float)(-5103.0 / 18656);
    static constexpr float b60 = (float)(35.0 / 384), b62 = (float)(500.0 / 1113), b63 = (float)(125.0 / 192),
                           b64 = (float)(-2187.0 / 6784), b65 = (float)(11.0 / 84);
    static constexpr float e0 = (float)(35.0 / 384 - 1951.0 / 21600), e2 = (float)(500.0 / 1113 - 22642.0 / 50085),
                           e3 = (float)(125.0 / 192 - 451.0 / 720), e4 = (float)(-2187.0 / 6784 + 12231.0 / 42400),
                           e5 = (float)(11.0 / 84 - 649.0 / 6300), e6 = (float)(-1.0 / 60);
    static constexpr float m0 = (float)(6025192743.0 / 30085553152.0 / 2), m2 = (float)(51252292925.0 / 65400821598.0 / 2),
                           m3 = (float)(-2691868925.0 / 45128329728.0 / 2), m4 = (float)(187940372067.0 / 1594534317056.0 / 2),
                           m5 = (float)(-1776094331.0 / 19743644256.0 / 2), m6 = (float)(11237099.0 / 235043384.0 / 2);
};

}  // namespace odecol
