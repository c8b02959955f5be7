// Staged (large-N) Euler-Maruyama: the drift's contraction runs on the tensor cores (kernel of stage_tc.cuh with a
// plain right-hand-side epilogue), the stepping logic in small elementwise kernels around it.  At N >= 256 the
// contraction dominates (2 N^2 flops per trial and evaluation against ~60 bytes of bookkeeping), so the extra pass over
// the state costs nothing measurable and keeps the torchsde loop semantics readable:
//
//   fixed step   per step:   f = drift(t_k, y)  [tensor]  ->  y += f h + sigma dW, outputs, next operand   [elementwise]
//   adaptive     per round:  f0 [tensor] -> full step + first half step [elementwise] -> f(mid) [tensor]
//                            -> second half step + per-trial error sums [elementwise] -> per-trial controller
//                            (torchsde update_step_size, accept/reject, Brownian tree queries) -> commit [elementwise]
// Every trial carries its own time and step size; finished trials idle.  Replaces torchsde.sdeint(method='euler') for
// networks beyond the on-chip family (BASELINE.json config 5).
//
// Unlike the other entry points these two synchronise the stream: the fixed-step schedule is replayed on the host from
// a copy of ts, and the adaptive loop polls an "all trials finished" flag every 16 rounds.
#include <vector>
#include "stage_tc.cuh"

namespace odecol {
namespace tc {

// ---- tensor-core right-hand side: f[b] = drift(y[b], W_aug . r_aug[b]) -------------------------------------------------
struct RhsEpi {
    DevProblem p;
    const float* y;        // (B, 3N)
    const float* Rhi; const float* Rlo;   // operand of this evaluation (r = hi + lo); FP16 pairs when wscale != NULL
    float* f;              // (B, 3N)
    int KPa;               // elements per operand row (KP16 in the 16-bit format)
    const float* wscale = nullptr;   // 16-bit operand format: [0] = 1 / (power-of-two scale of the FP16 weight planes); NULL = TF32
    float ws;
    float inv_tm, inv_ta, inv_ts;
    const float* loc;      // (B, N) within-column input W_local (*) r, or NULL (lateral-gain sweeps: DevProblem::lat_gain)
    ODECOL_DEVINL void prepare() { ws = wscale ? __ldg(wscale) : 1.0f; }
    ODECOL_DEVINL void rows(int, int i, int n0, int, int g, int TNq, const float (&tot)[kMaxQ]) const {
        if (i >= p.N) return;
        const __half* Rh16 = reinterpret_cast<const __half*>(Rhi);
        const __half* Rl16 = reinterpret_cast<const __half*>(Rlo);
        const int N = p.N;
        const float kap = __ldg(p.kappa + i);
#pragma unroll 4
        for (int j = 0; j < kMaxQ; ++j) {
            const int b = n0 + g * TNq + j;
            if (j >= TNq || b >= p.B) break;
            const float* yb = y + (size_t)b * 3 * N + i;
            const float r = wscale ? __half2float(Rh16[(size_t)b * KPa + i]) + __half2float(Rl16[(size_t)b * KPa + i]) * 4.8828125e-4f
                                   : Rhi[(size_t)b * KPa + i] + Rlo[(size_t)b * KPa + i];
            // lateral-gain sweep: the contraction holds g_b-scaled lateral input (its stimulus / bias columns were divided
            // by g_b in the operand), the within-column input comes from the operand kernel
            const float tj = tot[j] * ws;
            const float cur = loc ? fmaf(__ldg(p.lat_gain + b), tj, loc[(size_t)b * N + i]) : tj;
            const float total = cur * p.c.tau_s;
            float* fb = f + (size_t)b * 3 * N + i;
            fb[0] = (total * p.c.R - yb[0]) * inv_tm;
            fb[N] = (kap * r - yb[N]) * inv_ta;
            fb[2 * N] = (r - yb[2 * N]) * inv_ts;
        }
    }
    ODECOL_DEVINL void tile_done(int, int, int, int, int) const {}
};

// ---- operand r_aug(t_b, y_b), split hi / lo --------------------------------------------------------------------------------
// Destination of one trial's operand row (and, in lateral-gain sweeps, of its within-column input plane).
struct OperandDst {
    float* hi; float* lo; float* loc;       // loc == NULL unless DevProblem::lat_gain is set
    int KPa;                                // elements per operand row
    unsigned int* ovf;                      // != NULL: 16-bit operand format -- hi / lo are planes of FP16 (x = xh + xl / 2048) with
                                            // KPa halves per row; *ovf is raised when a value does not fit FP16
};

// one operand value in the destination's format: (hi, lo) as the floats the contraction will see
ODECOL_DEVINL void operand_split(const OperandDst& d, float x, float& h, float& l, F16x2& t) {
    if (d.ovf) {
        t = f16_split2(x);
        h = __half2float(__ushort_as_half(t.h));
        l = __half2float(__ushort_as_half(t.l)) * 4.8828125e-4f;
    } else {
        h = tf32_rna(x);
        l = tf32_rna(x - h);
    }
}

// Populations k .. k+3 of trial b from their stage state: r = phi(V - A) -> hi / lo (16-byte stores).  In a lateral-gain sweep
// the within-column input W_local (*) r of the four populations is formed here as well: the eight rates of a column sit in
// the registers of two neighbouring lanes (lane pairs exchange their four by shuffle), so nothing is re-read.  Every lane
// of the warp must call this (in_range = false for lanes past N); `pair8` says whether the shuffle path applies (N % 8 == 0).
ODECOL_DEVINL void operand_block4(const DevProblem& p, const OperandDst& d, int b, int k, bool in_range, const float4& V,
                                  const float4& A, bool pair8) {
    float r[4], h[4], l[4];
    F16x2 t[4];
    bool big = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        r[e] = in_range ? phi_fast((&V.x)[e] - (&A.x)[e]) : 0.f;
        big |= !(fabsf(r[e]) <= kF16Limit);
        operand_split(d, r[e], h[e], l[e], t[e]);
    }
    const size_t ro = (size_t)b * d.KPa;
    if (in_range && d.ovf) {
        if (big) *d.ovf = 1u;
        uint16_t* h16 = reinterpret_cast<uint16_t*>(d.hi) + ro + k;
        uint16_t* l16 = reinterpret_cast<uint16_t*>(d.lo) + ro + k;
        *reinterpret_cast<uint2*>(h16) = make_uint2((uint32_t)t[0].h | ((uint32_t)t[1].h << 16), (uint32_t)t[2].h | ((uint32_t)t[3].h << 16));
        *reinterpret_cast<uint2*>(l16) = make_uint2((uint32_t)t[0].l | ((uint32_t)t[1].l << 16), (uint32_t)t[2].l | ((uint32_t)t[3].l << 16));
    } else if (in_range) {
        st4(d.hi + ro + k, make_float4(h[0], h[1], h[2], h[3]));
        st4(d.lo + ro + k, make_float4(l[0], l[1], l[2], l[3]));
    }
    if (d.loc && pair8) {
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = __shfl_xor_sync(0xffffffffu, h[e] + l[e], 1);      // r as RhsEpi reads it: hi + lo
        if (in_range) {
            const bool upper = (k & 4) != 0;                 // this lane holds populations 4..7 of its column
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            if (p.W_local) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 w0 = ld4(p.W_local + (size_t)(k + e) * 8), w1 = ld4(p.W_local + (size_t)(k + e) * 8 + 4);
                    const float4& wm = upper ? w1 : w0;      // weights onto this lane's own four sources
                    const float4& wo = upper ? w0 : w1;      // ... and onto the partner lane's
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[e] = fmaf((&wm.x)[j], h[j] + l[j], fmaf((&wo.x)[j], o[j], acc[e]));
                }
            }
            st4(d.loc + (size_t)b * p.N + k, make_float4(acc[0], acc[1], acc[2], acc[3]));
        }
    }
}

// stimulus channels at time tq, the constant-one column (both divided by g_b in a lateral-gain sweep, so that
// g_b * (W_aug . r_aug) scales the recurrent input only), and -- when the lane-pair path does not apply -- the
// within-column input from the rates just written.  Called by all threads of the trial's CTA after the population loop.
ODECOL_DEVINL void operand_tail(const DevProblem& p, const OperandDst& d, int b, float tq, bool pair8) {
    const int N = p.N, Kaug = N + p.n_in + 1;
    const float ginv = d.loc ? __fdiv_rn(1.0f, __ldg(p.lat_gain + b)) : 1.0f;
    const size_t ro = (size_t)b * d.KPa;
    int idx = 1;
    const float tcl = knot_locate(p.knot_t, p.K, tq, idx);
    const float* ku = p.knot_u + (size_t)b * p.knot_stride_b;
    for (int k = N + threadIdx.x; k < Kaug; k += blockDim.x) {
        const float v = k < N + p.n_in ? knot_value(p.knot_t, ku, p.n_in, idx, tcl, k - N) * ginv : ginv;
        if (d.ovf) {
            if (!(fabsf(v) <= kF16Limit)) *d.ovf = 1u;
            const F16x2 t = f16_split2(v);
            reinterpret_cast<uint16_t*>(d.hi)[ro + k] = t.h;
            reinterpret_cast<uint16_t*>(d.lo)[ro + k] = t.l;
        } else {
            const float h = tf32_rna(v);
            d.hi[ro + k] = h;
            d.lo[ro + k] = tf32_rna(v - h);
        }
    }
    if (d.loc && !pair8) {
        __syncthreads();
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            const int c0 = i & ~7;
            float acc = 0.f;
            if (p.W_local) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (c0 + j < N) {
                        const float rj = d.ovf ? __half2float(reinterpret_cast<const __half*>(d.hi)[ro + c0 + j]) +
                                                     __half2float(reinterpret_cast<const __half*>(d.lo)[ro + c0 + j]) * 4.8828125e-4f
                                               : d.hi[ro + c0 + j] + d.lo[ro + c0 + j];
                        acc = fmaf(__ldg(p.W_local + (size_t)i * 8 + j), rj, acc);
                    }
            }
            d.loc[(size_t)b * N + i] = acc;
        }
    }
}

ODECOL_DEVINL bool aligned16(const void* q) { return ((uintptr_t)q & 15) == 0; }

// one CTA per trial, per-trial time (NULL -> shared time t_shared); N must be a multiple of 4 (the staged entry points check)
__global__ void k_em_operand(DevProblem p, const float* __restrict__ y, const float* __restrict__ t_trial,
                             float t_shared, float* __restrict__ hi, float* __restrict__ lo, int KPa,
                             const int* __restrict__ active = nullptr, float* __restrict__ loc = nullptr,
                             unsigned int* __restrict__ ovf = nullptr) {
    const int b = blockIdx.x, N = p.N;
    if (active && !active[b]) return;          // adaptive sweeps: a finished trial's drift is never read again
    const OperandDst d{hi, lo, loc, KPa, ovf};
    const float* yb = y + (size_t)b * 3 * N;
    const bool pair8 = (N & 7) == 0 && (!p.W_local || aligned16(p.W_local));
    // four populations per thread and iteration through 16-byte accesses (with one scalar load pair in flight per thread
    // the kernel ran at 3.7 TB/s, latency-bound)
    for (int k0 = 0; k0 < N; k0 += 4 * blockDim.x) {
        const int k = k0 + 4 * threadIdx.x;
        const bool in = k < N;
        float4 V = make_float4(0.f, 0.f, 0.f, 0.f), A = V;
        if (in) { V = ld4(yb + k); A = ld4(yb + N + k); }
        operand_block4(p, d, b, k, in, V, A, pair8);
    }
    operand_tail(p, d, b, t_trial ? t_trial[b] : t_shared, pair8);
}

// ---- fixed step ---------------------------------------------------------------------------------------------------
struct EmStepArgs {
    DevProblem p;
    float* y; const float* f; float* y_prev;      // y updated in place, previous state kept for the interpolation
    const float* dW; unsigned long long seed; long long trial_offset; long long kstep;
    float t0, t1;                                 // this step
    float* y_out; int j_lo, j_hi;                 // outputs emitted after this step: ts[j], j in [j_lo, j_hi)
    const float* ts;
};

__global__ void k_em_step(EmStepArgs a) {
    const int N = a.p.N, B = a.p.B;
    const size_t total = (size_t)B * 3 * N;
    const float h = __fsub_rn(a.t1, a.t0);
    const Philox px(a.seed);
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / (3 * N)), comp = (int)(e % (3 * N));
        float dw;
        if (a.dW) dw = a.dW[(size_t)a.kstep * B + b];
        else {
            const unsigned long long trial = (unsigned long long)(a.trial_offset + b);
            const uint4 bits = px((uint32_t)trial, (uint32_t)(trial >> 32), (uint32_t)a.kstep, 0x80000000u | (uint32_t)(a.kstep >> 32));
            dw = sqrtf(h) * normal_from_bits(bits.x, bits.y);
        }
        const float sg = (a.p.sigma ? __ldg(a.p.sigma + comp) : 0.f) * (a.p.sigma_scale ? __ldg(a.p.sigma_scale + b) : 1.f);
        const float y0 = a.y[e];
        const float y1 = __fadd_rn(__fadd_rn(y0, __fmul_rn(a.f[e], h)), __fmul_rn(sg, dw));
        a.y_prev[e] = y0;
        a.y[e] = y1;
        for (int j = a.j_lo; j < a.j_hi; ++j) {
            const float out_t = __ldg(a.ts + j);
            const float w0 = __fdiv_rn(__fsub_rn(a.t1, out_t), h), w1 = __fdiv_rn(__fsub_rn(out_t, a.t0), h);
            a.y_out[(size_t)j * total + e] = __fadd_rn(__fmul_rn(w0, y0), __fmul_rn(w1, y1));
        }
    }
}

// ---- adaptive: per-trial controller state -------------------------------------------------------------------------------
struct TrialState {
    float* t_cur; float* t_prev; float* t_mid; float* t_next;   // (B)
    double* step; double* prev_ratio; int* has_prev;
    float* w_cur; float* dw_full; float* dw_1; float* dw_2;
    double* err2;
    int* next_out; int* n_acc; int* n_rej; int* status; int* active; int* accept;
    int* n_active;          // single counter
};

__global__ void k_ad_init(DevProblem p, TrialState s, const float* __restrict__ ts, int T, float dt0, unsigned long long seed,
                          long long trial_offset) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    const float t_begin = ts[0], t_end = ts[T - 1];
    s.t_cur[b] = t_begin; s.t_prev[b] = t_begin;
    s.step[b] = (double)dt0; s.prev_ratio[b] = 0.0; s.has_prev[b] = 0;
    s.w_cur[b] = 0.f; s.err2[b] = 0.0;
    s.next_out[b] = 1; s.n_acc[b] = 0; s.n_rej[b] = 0; s.status[b] = ODECOL_ST_OK; s.active[b] = 1; s.accept[b] = 0;
    // first attempt
    const float next_t = fminf(__fadd_rn(t_begin, dt0), t_end);
    const float mid_t = __fmul_rn(0.5f, __fadd_rn(t_begin, next_t));
    s.t_next[b] = next_t; s.t_mid[b] = mid_t;
    const Philox px(seed);
    const unsigned long long trial = (unsigned long long)(trial_offset + b);
    const float span = t_end - t_begin;
    const float wm = brownian_tree(px, trial, t_begin, span, mid_t), wn = brownian_tree(px, trial, t_begin, span, next_t);
    s.dw_full[b] = wn; s.dw_1[b] = wm; s.dw_2[b] = wn - wm;
    if (b == 0) *s.n_active = p.B;
}

// full step and first half step from f0; writes y_full, y_mid AND the operand of the drift evaluation at (t_mid, y_mid).
// One CTA per trial (finished trials cost nothing); a thread handles four populations per iteration -- their V, A and F
// components through 16-byte accesses -- so the rates of y_mid are formed from registers (the separate operand kernel
// re-read y_mid: 8 bytes per population and a launch per round).  Per element the operations of torchsde's Euler step in
// their order.
__global__ void k_ad_half1(DevProblem p, TrialState s, const float* __restrict__ y, const float* __restrict__ f0,
                           float* __restrict__ y_full, float* __restrict__ y_mid, OperandDst d) {
    const int N = p.N, b = blockIdx.x;
    if (!s.active[b]) return;
    const float tc = s.t_cur[b], tm = s.t_mid[b], tn = s.t_next[b];
    const float h = __fsub_rn(tn, tc), h1 = __fsub_rn(tm, tc);
    const float dwf = s.dw_full[b], dw1 = s.dw_1[b];
    const float sc = p.sigma_scale ? __ldg(p.sigma_scale + b) : 1.f;
    const size_t base = (size_t)b * 3 * N;
    const bool sig_vec = p.sigma && aligned16(p.sigma);
    const bool pair8 = (N & 7) == 0 && (!p.W_local || aligned16(p.W_local));
    for (int k0 = 0; k0 < N; k0 += 4 * blockDim.x) {
        const int k = k0 + 4 * threadIdx.x;
        const bool in = k < N;
        float4 ymV = make_float4(0.f, 0.f, 0.f, 0.f), ymA = ymV;
        if (in) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const size_t e0 = base + (size_t)c * N + k;
                const float4 Y = ld4(y + e0), F = ld4(f0 + e0);
                float4 S = make_float4(0.f, 0.f, 0.f, 0.f);
                if (sig_vec) S = ld4(p.sigma + c * N + k);
                else if (p.sigma) S = make_float4(__ldg(p.sigma + c * N + k), __ldg(p.sigma + c * N + k + 1), __ldg(p.sigma + c * N + k + 2),
                                                  __ldg(p.sigma + c * N + k + 3));
                float4 yf, ym;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float sg = (&S.x)[e] * sc, y0 = (&Y.x)[e], f = (&F.x)[e];
                    (&yf.x)[e] = __fadd_rn(__fadd_rn(y0, __fmul_rn(f, h)), __fmul_rn(sg, dwf));
                    (&ym.x)[e] = __fadd_rn(__fadd_rn(y0, __fmul_rn(f, h1)), __fmul_rn(sg, dw1));
                }
                st4(y_full + e0, yf);
                st4(y_mid + e0, ym);
                if (c == 0) ymV = ym;
                if (c == 1) ymA = ym;
            }
        }
        operand_block4(p, d, b, k, in, ymV, ymA, pair8);
    }
    operand_tail(p, d, b, tm, pair8);
}

// second half step from f(mid), error sums per trial
__global__ void k_ad_half2(DevProblem p, TrialState s, const float* __restrict__ y_mid, const float* __restrict__ fm,
                           const float* __restrict__ y_full, float* __restrict__ y_half, float rtol, float atol) {
    const int N = p.N;
    const int b = blockIdx.x;
    if (!s.active[b]) return;
    const float h2 = __fsub_rn(s.t_next[b], s.t_mid[b]);
    const float dw2 = s.dw_2[b];
    double acc = 0.0;
    const float sc = p.sigma_scale ? __ldg(p.sigma_scale + b) : 1.f;
    const size_t base = (size_t)b * 3 * N;
    const bool vec = (N & 3) == 0 && (((uintptr_t)y_mid | (uintptr_t)fm | (uintptr_t)y_full | (uintptr_t)y_half | (uintptr_t)p.sigma) & 15) == 0;
    if (vec) {                                  // four components per thread and iteration, 16-byte accesses
        for (int comp = 4 * threadIdx.x; comp < 3 * N; comp += 4 * blockDim.x) {
            const float4 YM = ld4(y_mid + base + comp), FM = ld4(fm + base + comp), YF = ld4(y_full + base + comp);
            const float4 S = p.sigma ? ld4(p.sigma + comp) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 YH;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float sg = (&S.x)[e] * sc;
                const float yh = __fadd_rn(__fadd_rn((&YM.x)[e], __fmul_rn((&FM.x)[e], h2)), __fmul_rn(sg, dw2));
                (&YH.x)[e] = yh;
                const float yf = (&YF.x)[e];
                const float tol = __fadd_rn(atol, __fmul_rn(rtol, fmaxf(fabsf(yf), fabsf(yh))));
                const float q = __fdiv_rn(__fsub_rn(yf, yh), tol);
                acc += (double)q * q;
            }
            st4(y_half + base + comp, YH);
        }
    } else {
        for (int comp = threadIdx.x; comp < 3 * N; comp += blockDim.x) {
            const size_t e = base + comp;
            const float sg = (p.sigma ? __ldg(p.sigma + comp) : 0.f) * sc;
            const float yh = __fadd_rn(__fadd_rn(y_mid[e], __fmul_rn(fm[e], h2)), __fmul_rn(sg, dw2));
            y_half[e] = yh;
            const float yf = y_full[e];
            const float tol = __fadd_rn(atol, __fmul_rn(rtol, fmaxf(fabsf(yf), fabsf(yh))));
            const float q = __fdiv_rn(__fsub_rn(yf, yh), tol);
            acc += (double)q * q;
        }
    }
    __shared__ double red[32];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
        s.err2[b] = t;
    }
}

// torchsde adaptive_stepping.update_step_size + accept/reject per trial, then the next attempt's times and increments
__global__ void k_ad_control(DevProblem p, TrialState s, const float* __restrict__ ts, int T, float dt_min,
                             unsigned long long seed, long long trial_offset, long long max_attempts) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B || !s.active[b]) return;
    const float t_begin = ts[0], t_end = ts[T - 1];
    const double err = (double)(float)sqrt(s.err2[b] / (3.0 * p.N));
    int acc = 0;
    if (!(err == err)) {
        s.status[b] = ODECOL_ST_NONFINITE; s.active[b] = 0; s.accept[b] = 0; atomicSub(s.n_active, 1);
        return;
    }
    double step = s.step[b];
    {
        const double pfac = err > 1.0 ? 0.0 : 0.13, ifac = err > 1.0 ? 1.0 / 1.5 : 1.0 / 4.5;
        const double ratio = 0.9 / err;
        const double pr = s.has_prev[b] ? s.prev_ratio[b] : ratio;
        double factor = pow(ratio, ifac) * pow(ratio / pr, pfac);
        double facmin = 0.2;
        if (err <= 1.0) { s.prev_ratio[b] = ratio; s.has_prev[b] = 1; facmin = 1.0; }
        factor = fmin(1.4, fmax(facmin, factor));
        step *= factor;
    }
    if (step < (double)dt_min) { step = (double)dt_min; s.has_prev[b] = 0; }
    s.step[b] = step;
    float t_cur = s.t_cur[b];
    if (err <= 1.0 || step <= (double)dt_min) {
        acc = 1;
        s.t_prev[b] = t_cur;
        t_cur = s.t_next[b];
        s.t_cur[b] = t_cur;
        s.w_cur[b] += s.dw_full[b];
        s.n_acc[b] += 1;
    } else {
        s.n_rej[b] += 1;
    }
    s.accept[b] = acc;
    if ((long long)s.n_acc[b] + s.n_rej[b] >= max_attempts) { s.status[b] = ODECOL_ST_MAXSTEPS; s.active[b] = 0; atomicSub(s.n_active, 1); return; }
    // next attempt (also after the final accept: k_ad_commit decides whether the trial is finished)
    const float next_t = fminf(__fadd_rn(t_cur, (float)step), t_end);
    const float mid_t = __fmul_rn(0.5f, __fadd_rn(t_cur, next_t));
    s.t_next[b] = next_t; s.t_mid[b] = mid_t;
    const Philox px(seed);
    const unsigned long long trial = (unsigned long long)(trial_offset + b);
    const float span = t_end - t_begin;
    const float w0 = s.w_cur[b];
    const float wm = brownian_tree(px, trial, t_begin, span, mid_t), wn = brownian_tree(px, trial, t_begin, span, next_t);
    s.dw_full[b] = wn - w0; s.dw_1[b] = wm - w0; s.dw_2[b] = wn - wm;
}

// commit accepted steps: state, outputs reached by the new time, finished trials -- and the operand of the next attempt's
// first drift evaluation, f(t_cur, y), formed from the committed state in registers.  A rejected attempt leaves y, t_cur
// and therefore that operand untouched (the attempt's midpoint evaluation uses the other operand set).
__global__ void k_ad_commit(DevProblem p, TrialState s, const float* __restrict__ ts, int T, float* __restrict__ y,
                            float* __restrict__ y_prev, const float* __restrict__ y_half, float* __restrict__ y_out,
                            OperandDst d) {
    const int N = p.N, b = blockIdx.x;
    if (!s.active[b] || !s.accept[b]) return;
    const float t_prev = s.t_prev[b], t_cur = s.t_cur[b];
    const float spn = __fsub_rn(t_cur, t_prev);
    int j = s.next_out[b];
    const size_t total = (size_t)p.B * 3 * N;
    const bool pair8 = (N & 7) == 0 && (!p.W_local || aligned16(p.W_local));
    for (int k0 = 0; k0 < N; k0 += 4 * blockDim.x) {
        const int k = k0 + 4 * threadIdx.x;
        const bool in = k < N;
        float4 V = make_float4(0.f, 0.f, 0.f, 0.f), A = V;
        if (in) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const size_t e = (size_t)b * 3 * N + (size_t)c * N + k;
                const float4 Y0 = ld4(y + e), Y1 = ld4(y_half + e);
                st4(y_prev + e, Y0);
                st4(y + e, Y1);
                for (int jj = j; jj < T && __ldg(ts + jj) <= t_cur; ++jj) {
                    const float out_t = __ldg(ts + jj);
                    const float w0 = __fdiv_rn(__fsub_rn(t_cur, out_t), spn), w1 = __fdiv_rn(__fsub_rn(out_t, t_prev), spn);
                    float4 O;
#pragma unroll
                    for (int q = 0; q < 4; ++q) (&O.x)[q] = __fadd_rn(__fmul_rn(w0, (&Y0.x)[q]), __fmul_rn(w1, (&Y1.x)[q]));
                    st4(y_out + (size_t)jj * total + e, O);
                }
                if (c == 0) V = Y1;
                if (c == 1) A = Y1;
            }
        }
        operand_block4(p, d, b, k, in, V, A, pair8);
    }
    operand_tail(p, d, b, t_cur, pair8);
    __syncthreads();
    if (threadIdx.x == 0) {
        while (j < T && ts[j] <= t_cur) ++j;
        s.next_out[b] = j;
        if (j >= T) { s.active[b] = 0; atomicSub(s.n_active, 1); }
    }
}

__global__ void k_em_fill_nan(DevProblem p, const int* __restrict__ status, const int* __restrict__ next_out, int T,
                              float* __restrict__ y_out) {
    const int b = blockIdx.x, N = p.N;
    if (status[b] == ODECOL_ST_OK) return;
    const size_t total = (size_t)p.B * 3 * N;
    const float qnan = __int_as_float(0x7fc00000);
    for (int j = next_out[b]; j < T; ++j)
        for (int comp = threadIdx.x; comp < 3 * N; comp += blockDim.x) y_out[(size_t)j * total + (size_t)b * 3 * N + comp] = qnan;
}

// end of an adaptive solve: NaN for the outputs a stopped trial never reached, then the per-trial statistics
template <class State>
static int adaptive_finish(const DevProblem& p, const State& S, int T, float* y_out, int* n_accept, int* n_reject, int* status,
                           cudaStream_t s) {
    k_em_fill_nan<<<p.B, 128, 0, s>>>(p, S.status, S.next_out, T, y_out);
    count_launch();
    const size_t B = p.B;
    if (n_accept && cudaMemcpyAsync(n_accept, S.n_acc, sizeof(int) * B, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (n_reject && cudaMemcpyAsync(n_reject, S.n_rej, sizeof(int) * B, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (status && cudaMemcpyAsync(status, S.status, sizeof(int) * B, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

// grid of the elementwise kernels over n elements
static int ew_grid(size_t n) {
    const size_t g = (n + 255) / 256;
    return (int)(g < 148 * 16 ? g : 148 * 16);
}

// workspace pieces, each 1024-byte aligned
struct Carve {
    size_t o = 0;
    size_t take(size_t bytes) { const size_t r = o; o += (bytes + 1023) / 1024 * 1024; return r; }
};

// per-trial arrays carved one after another from one workspace piece, 16-byte aligned
struct TrialCarve {
    char* at;
    template <class T> void operator()(T*& dst, size_t n) { dst = reinterpret_cast<T*>(at); at += (n * sizeof(T) + 15) / 16 * 16; }
};

// ---- one drift evaluation of the staged solvers on the tensor cores ----------------------------------------------------
// The drift part of a staged workspace: W_aug split into two planes, `sets` operand sets of two planes, and on request
// each set's within-column input plane (lateral-gain sweeps) and the aux slot of the 16-bit format.  The planes are sized
// for TF32 pairs (KPa floats per row); the 16-bit format keeps its rows of KP16 halves in the same buffers
// (2 KP16 <= 4 KPa bytes).  Operand planes have `rows` rows: Bp, or Bp rounded up to 32 for the adjoint, whose dW
// contraction reads them in blocks of 32 trials; the tensor maps cover Bp.  StagedDrift::init zeroes the bytes from the
// first operand plane up to zero_end.
struct DriftLayout {
    int Np, KPa, KP16, TN, Bp, rows, sets;
    bool loc, aux;
    size_t off_W[2], off_R[2][2], off_loc[2], off_aux, zero_end;
};

static DriftLayout drift_layout(Carve& c, const DevProblem& p, int sets, bool loc, bool aux, bool dw_rows) {
    DriftLayout L;
    L.Np = round_up(p.N, BM);
    L.KPa = round_up(p.N + p.n_in + 1, BK);
    L.KP16 = round_up(p.N + p.n_in + 1, BK16);
    L.TN = pick_tile_n(L.Np / BM, p.B);
    L.Bp = round_up(p.B, L.TN);
    L.rows = dw_rows ? round_up(L.Bp, 32) : L.Bp;
    L.sets = sets;
    L.loc = loc && p.lat_gain;
    L.aux = aux;
    for (int i = 0; i < 2; ++i) L.off_W[i] = c.take(4ull * L.Np * L.KPa);
    for (int q = 0; q < sets; ++q)
        for (int i = 0; i < 2; ++i) L.off_R[q][i] = c.take(4ull * L.rows * L.KPa);
    L.zero_end = c.o;
    for (int q = 0; q < sets && L.loc; ++q) L.off_loc[q] = c.take(4ull * p.B * p.N);
    if (aux) L.off_aux = c.take(64);
    return L;
}

// kRetryTf32: a solve in the 16-bit operand format met a value that does not fit FP16 and has to be repeated in TF32
static constexpr int kRetryTf32 = 1 << 20;

// f[b] = drift(t_b, y_b): k_em_operand writes r_aug(t_b, y_b) into an operand set, the tensor-core contraction against the
// split W_aug runs with the RhsEpi epilogue.  In the 16-bit format (f16) W_aug, scaled by a power of two, and the operands
// are FP16 pairs, and an operand value that does not fit FP16 raises the overflow flag in aux[2].
struct StagedDrift {
    DevProblem p;
    cudaStream_t s;
    bool f16;
    int KPr;                                      // elements per operand row in the format in use
    float* W[2];                                  // split W_aug: hi, lo
    float* R[2][2] = {};                          // operand sets: [set][hi, lo]
    float* loc[2] = {};                           // within-column input plane of each set (lateral-gain sweeps), else NULL
    float* aux = nullptr;                         // [0] 1 / weight scale, [1] max|W| bits, [2] overflow flag
    CUtensorMap mW[2], mR[2][2];
    TileShape tsh;

    unsigned int* ovf() const { return f16 ? reinterpret_cast<unsigned int*>(aux + 2) : nullptr; }

    // zero the operand planes (their padding stays zero) and the aux slot, split W_aug in the format, encode the maps
    int init(const DevProblem& p_, char* w, const DriftLayout& L, bool f16_, cudaStream_t s_) {
        p = p_; s = s_; f16 = f16_;
        KPr = f16 ? L.KP16 : L.KPa;
        auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
        for (int i = 0; i < 2; ++i) W[i] = F(L.off_W[i]);
        for (int q = 0; q < L.sets; ++q) {
            for (int i = 0; i < 2; ++i) R[q][i] = F(L.off_R[q][i]);
            loc[q] = L.loc ? F(L.off_loc[q]) : nullptr;
        }
        if (L.aux) aux = F(L.off_aux);
        const int Kaug = p.N + p.n_in + 1;
        if (cudaMemsetAsync(R[0][0], 0, L.zero_end - L.off_R[0][0], s) != cudaSuccess) return ODECOL_E_CUDA;
        if (f16) {
            if (cudaMemsetAsync(aux, 0, 64, s) != cudaSuccess) return ODECOL_E_CUDA;
            k_absmax<<<148, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, reinterpret_cast<unsigned int*>(aux + 1));
            k_split16_w<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, reinterpret_cast<__half*>(W[0]), reinterpret_cast<__half*>(W[1]),
                                            L.Np, L.KP16, reinterpret_cast<unsigned int*>(aux + 1), aux);
            count_launch(2);
        } else {
            k_split_pad<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, W[0], W[1], L.Np, L.KPa);
            count_launch();
        }
        auto map = [&](CUtensorMap* m, const float* base, int rows, int box_rows) {
            return f16 ? make_map16(m, base, rows, L.KP16, L.KP16, box_rows, false) : make_map(m, base, rows, L.KPa, L.KPa, box_rows);
        };
        for (int i = 0; i < 2; ++i)
            if (!map(&mW[i], W[i], L.Np, BM)) return ODECOL_E_CUDA;
        for (int q = 0; q < L.sets; ++q)
            for (int i = 0; i < 2; ++i)
                if (!map(&mR[q][i], R[q][i], L.Bp, L.TN)) return ODECOL_E_CUDA;
        tsh = TileShape{L.Np / BM, L.Bp / L.TN, L.TN, f16 ? L.KP16 / BK16 : L.KPa / BK, 0};
        return ODECOL_OK;
    }
    // r_aug(t, y) into operand set `set`; t_trial != NULL: one time per trial, else t_shared for all
    void operand(int set, const float* y, const float* t_trial, float t_shared) {
        k_em_operand<<<p.B, 128, 0, s>>>(p, y, t_trial, t_shared, R[set][0], R[set][1], KPr, nullptr, loc[set], ovf());
        count_launch();
    }
    // where k_ad_half1 / k_ad_commit write the operand of set `set`
    OperandDst dst(int set) const { return OperandDst{R[set][0], R[set][1], loc[set], KPr, ovf()}; }
    // f = drift(y) from the operand in set `set`
    int contract(int set, const float* y, float* f) const {
        RhsEpi e;
        e.p = p; e.y = y; e.Rhi = R[set][0]; e.Rlo = R[set][1]; e.f = f; e.KPa = KPr; e.loc = loc[set]; e.wscale = f16 ? aux : nullptr;
        e.inv_tm = 1.0f / p.c.tau_m; e.inv_ta = 1.0f / p.c.tau_a; e.inv_ts = 1.0f / p.c.tau_s;
        if (f16) return launch_contract16(mW[0], mW[1], mR[set][0], mR[set][1], tsh, e, s);
        return launch_contract(mW[0], mW[1], mR[set][0], mR[set][1], tsh, e, s);
    }
    int eval(int set, const float* y, const float* t_trial, float t_shared, float* f) {
        operand(set, y, t_trial, t_shared);
        return contract(set, y, f);
    }
    // Synchronises the stream, in the 16-bit format after copying the overflow flag: kRetryTf32 when an operand value did
    // not fit FP16, else ODECOL_OK (or ODECOL_E_CUDA)
    int overflowed() const {
        unsigned int h = 0;
        if (f16 && cudaMemcpyAsync(&h, ovf(), sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
        if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
        return h ? kRetryTf32 : ODECOL_OK;
    }
};

// The forward solves read FP16 pairs in their drift contractions (half the tensor-core instructions and operand bytes of
// the TF32 split: the contraction is 93 % of a round at N = 8192 and runs at 0.89 of the tensor roofline) unless their
// switch is set to 0.  Each switch is read once per process.
enum F16Switch { kEm16, kDp16, kSrk16 };
static bool f16_switch(F16Switch sw) {
    auto on = [](const char* name) { const char* e = getenv(name); return e ? atoi(e) != 0 : true; };
    switch (sw) {
        case kEm16: { static const bool v = on("ODECOL_EM16"); return v; }
        case kDp16: { static const bool v = on("ODECOL_DP16"); return v; }
        default: { static const bool v = on("ODECOL_SRK16"); return v; }
    }
}
// solve(f16) in the 16-bit format when the switch and `allow` say so; kRetryTf32 (an operand value did not fit FP16, read
// at the host's polls) repeats the solve in the TF32 format
template <class Solve>
static int solve_f16_or_tf32(F16Switch sw, bool allow, Solve&& solve) {
    const int rc = solve(f16_switch(sw) && allow);
    return rc == kRetryTf32 ? solve(false) : rc;
}

// torchsde's float32 fixed-step loop (integrate()), replayed on the host from a copy of ts (data independent):
// step(k, t0, t1, j_lo, j_hi) runs step k from t0 to t1, after which the outputs ts[j], j in [j_lo, j_hi), are due.
// n_steps receives the number of steps.
template <class Step>
static int fixed_step_walk(const float* ts_dev, int T, float dt, cudaStream_t s, long long& n_steps, Step&& step) {
    std::vector<float> ts(T);
    if (cudaMemcpyAsync(ts.data(), ts_dev, sizeof(float) * T, cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
    volatile float curr = ts[0];
    const float t_end = ts[T - 1];
    long long k = 0;
    for (int j = 1; j < T;) {
        const float c0 = curr;
        volatile float nx = c0 + dt;
        const float next_t = nx < t_end ? nx : t_end;
        int j_hi = j;
        while (j_hi < T && ts[j_hi] <= next_t) ++j_hi;            // outputs the loop emits once curr_t >= ts[j]
        const int rc = step(k, c0, next_t, j, j_hi);
        if (rc != ODECOL_OK) return rc;
        curr = next_t;
        j = j_hi;
        if (++k > (1LL << 40)) return ODECOL_E_SHAPE;
    }
    n_steps = k;
    return ODECOL_OK;
}

struct EmLayout {
    DriftLayout drift;
    size_t off_f, off_fm, off_yfull, off_ymid, off_yhalf, off_y, off_yprev, off_state, total;
};

static EmLayout em_layout(const DevProblem& p) {
    EmLayout L;
    Carve c;
    // two operand sets: the adaptive sweep keeps the operand of f(t_cur, y) (set 0) across a rejected attempt while the
    // midpoint evaluation f(t_mid, y_mid) uses set 1
    L.drift = drift_layout(c, p, 2, /*loc=*/true, /*aux=*/true, /*dw_rows=*/false);
    const size_t st = 4ull * p.B * 3 * p.N;
    L.off_f = c.take(st); L.off_fm = c.take(st); L.off_yfull = c.take(st); L.off_ymid = c.take(st); L.off_yhalf = c.take(st);
    L.off_y = c.take(st); L.off_yprev = c.take(st);
    L.off_state = c.take(128ull * p.B + 1024);
    L.total = c.o;
    return L;
}

}  // namespace tc

size_t stage_em_fwd_workspace_bytes(const DevProblem& p, int) { return tc::em_layout(p).total; }

static int em_fwd_impl(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                       uint64_t seed, int64_t trial_offset, float dt, int adaptive, float rtol, float atol, float dt_min,
                       int* n_accept, int* n_reject, int* status, float* y_steps, void* ws, size_t ws_bytes, cudaStream_t s,
                       bool f16) {
    using namespace tc;
    const EmLayout L = em_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
    float *f0 = F(L.off_f), *fm = F(L.off_fm), *yfull = F(L.off_yfull), *ymid = F(L.off_ymid), *yhalf = F(L.off_yhalf);
    float *y = F(L.off_y), *yprev = F(L.off_yprev);
    const size_t st = (size_t)p.B * 3 * p.N;

    StagedDrift drift;
    int rc = drift.init(p, w, L.drift, f16, s);
    if (rc != ODECOL_OK) return rc;
    if (cudaMemcpyAsync(y, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaMemcpyAsync(yprev, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaMemcpyAsync(y_out, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (y_steps && cudaMemcpyAsync(y_steps, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;

    if (!adaptive) {
        long long n_steps = 0;
        rc = fixed_step_walk(ts_dev, T, dt, s, n_steps, [&](long long k, float t0, float t1, int j_lo, int j_hi) -> int {
            const int r = drift.eval(0, y, nullptr, t0, f0);
            if (r != ODECOL_OK) return r;
            EmStepArgs a;
            a.p = p; a.y = y; a.f = f0; a.y_prev = yprev; a.dW = dW; a.seed = seed; a.trial_offset = trial_offset; a.kstep = k;
            a.t0 = t0; a.t1 = t1; a.y_out = y_out; a.j_lo = j_lo; a.j_hi = j_hi; a.ts = ts_dev;
            k_em_step<<<ew_grid(st), 256, 0, s>>>(a);
            count_launch();
            if (y_steps && cudaMemcpyAsync(y_steps + (size_t)(k + 1) * st, y, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
                return ODECOL_E_CUDA;
            return ODECOL_OK;
        });
        if (rc != ODECOL_OK) return rc;
        if (f16 && (rc = drift.overflowed()) != ODECOL_OK) return rc;     // did every operand value fit FP16?
        if (n_accept || n_reject || status) {
            std::vector<int> hk(p.B, (int)n_steps), hz(p.B, 0);
            if (n_accept && cudaMemcpyAsync(n_accept, hk.data(), sizeof(int) * p.B, cudaMemcpyHostToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
            if (n_reject && cudaMemcpyAsync(n_reject, hz.data(), sizeof(int) * p.B, cudaMemcpyHostToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
            if (status && cudaMemcpyAsync(status, hz.data(), sizeof(int) * p.B, cudaMemcpyHostToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
            if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;      // host vectors go out of scope
        }
        return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
    }

    // ---- adaptive: per-trial controller state carved from the workspace
    TrialState S;
    const size_t B = p.B;
    TrialCarve g{w + L.off_state};
    g(S.step, B); g(S.prev_ratio, B); g(S.err2, B);
    g(S.t_cur, B); g(S.t_prev, B); g(S.t_mid, B); g(S.t_next, B);
    g(S.w_cur, B); g(S.dw_full, B); g(S.dw_1, B); g(S.dw_2, B);
    g(S.has_prev, B); g(S.next_out, B); g(S.n_acc, B); g(S.n_rej, B); g(S.status, B); g(S.active, B); g(S.accept, B);
    g(S.n_active, 1);

    std::vector<float> tse(2);
    if (cudaMemcpyAsync(&tse[0], ts_dev, sizeof(float), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaMemcpyAsync(&tse[1], ts_dev + T - 1, sizeof(float), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
    const double span = (double)tse[1] - (double)tse[0];
    const long long max_attempts = (long long)(4.0 * span / dt_min) + 4LL * T + 1024;
    const int tb = (p.B + 127) / 128;
    k_ad_init<<<tb, 128, 0, s>>>(p, S, ts_dev, T, dt, seed, trial_offset);
    count_launch();
    drift.operand(0, y, S.t_cur, 0.f);
    int h_active = p.B;
    for (long long round = 0; round < max_attempts && h_active > 0; ++round) {
        // the midpoint evaluation f(t_mid, y_mid) reads operand set 1 (written by k_ad_half1), so that the operand of
        // f(t_cur, y) in set 0 (written by k_ad_commit) survives a rejected attempt
        if ((rc = drift.contract(0, y, f0)) != ODECOL_OK) return rc;
        k_ad_half1<<<p.B, 256, 0, s>>>(p, S, y, f0, yfull, ymid, drift.dst(1));
        if ((rc = drift.contract(1, ymid, fm)) != ODECOL_OK) return rc;
        k_ad_half2<<<p.B, 256, 0, s>>>(p, S, ymid, fm, yfull, yhalf, rtol, atol);
        k_ad_control<<<tb, 128, 0, s>>>(p, S, ts_dev, T, dt_min, seed, trial_offset, max_attempts);
        k_ad_commit<<<p.B, 256, 0, s>>>(p, S, ts_dev, T, y, yprev, yhalf, y_out, drift.dst(0));
        count_launch(4);
        if ((round & 15) == 15) {
            if (cudaMemcpyAsync(&h_active, S.n_active, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
            if ((rc = drift.overflowed()) != ODECOL_OK) return rc;
        }
    }
    if (f16 && (rc = drift.overflowed()) != ODECOL_OK) return rc;         // rounds since the last poll
    return adaptive_finish(p, S, T, y_out, n_accept, n_reject, status, s);
}

int stage_em_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                 uint64_t seed, int64_t trial_offset, float dt, int adaptive, float rtol, float atol, float dt_min,
                 int* n_accept, int* n_reject, int* status, float* y_steps, void* ws, size_t ws_bytes, cudaStream_t s) {
    return tc::solve_f16_or_tf32(tc::kEm16, true, [&](bool f16) {
        return em_fwd_impl(p, ts_dev, T, y0, y_out, dW, seed, trial_offset, dt, adaptive, rtol, atol, dt_min, n_accept, n_reject,
                           status, y_steps, ws, ws_bytes, s, f16);
    });
}


// One drift evaluation of the staged solvers, f[b] = forward(t[b], y[b]), as the sweeps above run it: operand kernel,
// tensor-core contraction, RhsEpi -- always in TF32 operand pairs.  The forward solves run the same unit in FP16 pairs
// unless their switch is 0 (f16_switch below).
int stage_drift(const DevProblem& p, const float* t_trial, const float* y, float* f, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const EmLayout L = em_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    StagedDrift drift;
    const int rc = drift.init(p, static_cast<char*>(ws), L.drift, false, s);
    return rc != ODECOL_OK ? rc : drift.eval(0, y, t_trial, 0.f, f);
}


// ---------------------------------------------------------------------------------------------------------------
// Staged Dormand-Prince 5(4): torchdiffeq's default solver for networks beyond the on-chip family.  Same structure as
// the adaptive Euler-Maruyama above -- every trial carries its own (t, dt), one ROUND = one attempted step of every
// unfinished trial: six stage evaluations (stage state elementwise -> operand -> tensor-core drift), then one kernel
// per trial block that forms the embedded error, takes the accept / reject decision and runs the step-size controller
// exactly like k_dopri5_fwd_small (RMS over the trial's whole state in float64, controller in float64, time in
// float64, state and tableau in float32), emits every output time inside an accepted step through the quartic dense
// output and commits the step.  With a record (training) it leaves every accepted step for the staged reverse sweep,
// stage_dopri5_bwd below.
// ---------------------------------------------------------------------------------------------------------------
namespace tc {

struct DpState {
    double* t; double* dt; double* red;      // (B) current time, step size, reduction scratch
    float* t_stage;                          // (B) time of the stage being evaluated
    int* next_out; int* n_acc; int* n_rej; int* status; int* active;
    int* n_active;
    float* k[7];                             // (B, 3N) stage slopes; k[0] = f(t, y) (FSAL)
    float* y; float* ys;                     // (B, 3N) accepted state, stage state / candidate
};

ODECOL_DEVINL double dp_block_sum(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
    __syncthreads();
    return s;
}

// Hairer's initial step, part 1: d0, d1 -> h0; ys = y + h0 f0; stage time t0 + h0.   One CTA per trial.
__global__ void k_dp_init1(DevProblem p, DpState s, const float* __restrict__ ts, float rtol, float atol) {
    __shared__ double sh[8];
    const int b = blockIdx.x, n3 = 3 * p.N;
    const size_t o = (size_t)b * n3;
    double a0 = 0.0, a1 = 0.0;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) {
        const float y = s.y[o + c], f = s.k[0][o + c];
        const float sc = __fadd_rn(atol, __fmul_rn(fabsf(y), rtol));
        const float q0 = __fdiv_rn(y, sc), q1 = __fdiv_rn(f, sc);
        a0 += (double)q0 * q0; a1 += (double)q1 * q1;
    }
    a0 = dp_block_sum(a0, sh); a1 = dp_block_sum(a1, sh);
    const float d0 = (float)sqrt(a0 / n3), d1 = (float)sqrt(a1 / n3);
    float h0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : __fdiv_rn(__fmul_rn(0.01f, d0), d1);
    h0 = fabsf(h0);
    for (int c = threadIdx.x; c < n3; c += blockDim.x) s.ys[o + c] = __fadd_rn(s.y[o + c], __fmul_rn(h0, s.k[0][o + c]));
    if (threadIdx.x == 0) {
        const double t0 = (double)ts[0];
        s.t[b] = t0;
        s.t_stage[b] = (float)(t0 + (double)h0);
        s.red[2 * b] = (double)h0; s.red[2 * b + 1] = (double)d1;
        s.next_out[b] = 1; s.n_acc[b] = 0; s.n_rej[b] = 0; s.status[b] = ODECOL_ST_OK; s.active[b] = 1;
        if (b == 0) *s.n_active = p.B;
    }
}

// part 2: d2 from f1 = k[1] -> dt
__global__ void k_dp_init2(DevProblem p, DpState s, float rtol, float atol) {
    __shared__ double sh[8];
    const int b = blockIdx.x, n3 = 3 * p.N;
    const size_t o = (size_t)b * n3;
    const float h0 = (float)s.red[2 * b], d1 = (float)s.red[2 * b + 1];
    double a2 = 0.0;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) {
        const float sc = __fadd_rn(atol, __fmul_rn(fabsf(s.y[o + c]), rtol));
        const float q = __fdiv_rn(__fsub_rn(s.k[1][o + c], s.k[0][o + c]), sc);
        a2 += (double)q * q;
    }
    a2 = dp_block_sum(a2, sh);
    if (threadIdx.x == 0) {
        const float d2 = fabsf(__fdiv_rn((float)sqrt(a2 / n3), h0));
        float h1;
        if (d1 <= 1e-15f && d2 <= 1e-15f) h1 = fmaxf(1e-6f, __fmul_rn(h0, 1e-3f));
        else h1 = powf(__fdiv_rn(0.01f, fmaxf(d1, d2)), 0.2f);
        s.dt[b] = (double)fminf(__fmul_rn(100.f, h0), fabsf(h1));
    }
}

// stage state of stage S (1..6) of the current attempt and its evaluation time
template <int S>
__global__ void k_dp_stage(DevProblem p, DpState s) {
    const int n3 = 3 * p.N;
    const size_t total = (size_t)p.B * n3;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / n3);
        if (!s.active[b]) continue;
        const float dtf = (float)s.dt[b];
        float acc;
        if (S == 1) acc = s.k[0][e] * (DP::b10 * dtf);
        if (S == 2) acc = fmaf(s.k[1][e], DP::b21 * dtf, s.k[0][e] * (DP::b20 * dtf));
        if (S == 3) acc = fmaf(s.k[2][e], DP::b32 * dtf, fmaf(s.k[1][e], DP::b31 * dtf, s.k[0][e] * (DP::b30 * dtf)));
        if (S == 4) acc = fmaf(s.k[3][e], DP::b43 * dtf, fmaf(s.k[2][e], DP::b42 * dtf, fmaf(s.k[1][e], DP::b41 * dtf, s.k[0][e] * (DP::b40 * dtf))));
        if (S == 5) acc = fmaf(s.k[4][e], DP::b54 * dtf, fmaf(s.k[3][e], DP::b53 * dtf, fmaf(s.k[2][e], DP::b52 * dtf,
                          fmaf(s.k[1][e], DP::b51 * dtf, s.k[0][e] * (DP::b50 * dtf)))));
        if (S == 6) acc = fmaf(s.k[5][e], DP::b65 * dtf, fmaf(s.k[4][e], DP::b64 * dtf, fmaf(s.k[3][e], DP::b63 * dtf,
                          fmaf(s.k[2][e], DP::b62 * dtf, s.k[0][e] * (DP::b60 * dtf)))));
        s.ys[e] = __fadd_rn(s.y[e], acc);
        if (e == (size_t)b * n3) {
            const double t0 = s.t[b];
            const float t0f = (float)t0;
            const float al = S == 1 ? DP::a1 : S == 2 ? DP::a2 : S == 3 ? DP::a3 : DP::a4;
            s.t_stage[b] = S <= 4 ? __fadd_rn(t0f, __fmul_rn(al, dtf)) : (float)(t0 + s.dt[b]);
        }
    }
}

// error ratio, accept / reject, controller, dense output of every output time inside an accepted step, commit
// rec.y != NULL (training mode): every accepted step leaves its start state, t0 and dt, and every output the index of the
// accepted step it lies in with its dense-output abscissa -- what stage_dopri5_bwd differentiates through
__global__ void k_dp_finish(DevProblem p, DpState s, const float* __restrict__ ts, int T, float rtol, float atol,
                            int max_steps, float* __restrict__ y_out, Dopri5Record rec) {
    __shared__ double sh[8];
    __shared__ int sh_acc, sh_j0, sh_j1, sh_n;
    const int b = blockIdx.x, n3 = 3 * p.N;
    if (!s.active[b]) return;
    const size_t o = (size_t)b * n3;
    const size_t total = (size_t)p.B * n3;
    const double t0 = s.t[b], dt = s.dt[b], t1 = t0 + dt;
    const float dtf = (float)dt;
    double acc = 0.0;
    int bad = 0;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) {
        const size_t e = o + c;
        const float err = fmaf(s.k[6][e], DP::e6 * dtf, fmaf(s.k[5][e], DP::e5 * dtf, fmaf(s.k[4][e], DP::e4 * dtf,
                          fmaf(s.k[3][e], DP::e3 * dtf, fmaf(s.k[2][e], DP::e2 * dtf, s.k[0][e] * (DP::e0 * dtf))))));
        const float y0 = s.y[e], y1 = s.ys[e];
        const float tol = __fadd_rn(atol, __fmul_rn(rtol, fmaxf(fabsf(y0), fabsf(y1))));
        const float q = __fdiv_rn(err, tol);
        acc += (double)q * q;
        bad |= !isfinite(y0);
    }
    acc = dp_block_sum(acc, sh);
    bad = __syncthreads_or(bad);
    const float ratio = (float)sqrt(acc / n3);
    if (threadIdx.x == 0) {
        int st = ODECOL_ST_OK, accept = 0;
        if (bad || !(ratio == ratio)) st = ODECOL_ST_NONFINITE;
        else if (!(t0 + dt > t0)) st = ODECOL_ST_UNDERFLOW;
        else accept = ratio <= 1.0f;
        int j0 = s.next_out[b], j1 = j0;
        sh_n = s.n_acc[b];
        if (st == ODECOL_ST_OK && accept && rec.y && sh_n >= rec.cap) { st = ODECOL_ST_MAXSTEPS; accept = 0; }   // record full
        if (st == ODECOL_ST_OK) {
            if (accept) {
                while (j1 < T && (double)ts[j1] <= t1) ++j1;      // outputs reached by this step: next_t <= st_t1
                s.n_acc[b] += 1;
                if (rec.y) { rec.t0[(size_t)b * rec.cap + sh_n] = t0; rec.dt[(size_t)b * rec.cap + sh_n] = dt; }
            } else {
                s.n_rej[b] += 1;
            }
            const double r64 = (double)ratio;
            double ndt;
            if (r64 == 0.0) ndt = dt * 10.0;
            else { const double df = r64 < 1.0 ? 1.0 : 0.2; ndt = dt * fmin(10.0, fmax(0.9 / pow(r64, 0.2), df)); }
            s.dt[b] = ndt;
            if (accept) { s.t[b] = t1; s.next_out[b] = j1; }
            if (j1 >= T) { s.active[b] = 0; atomicSub(s.n_active, 1); }
            else if (s.n_acc[b] + s.n_rej[b] >= max_steps) { st = ODECOL_ST_MAXSTEPS; }
        }
        if (st != ODECOL_ST_OK) { s.status[b] = st; s.active[b] = 0; atomicSub(s.n_active, 1); accept = 0; }
        sh_acc = accept; sh_j0 = j0; sh_j1 = j1;
    }
    __syncthreads();
    if (!sh_acc) return;
    const int j0 = sh_j0, j1 = sh_j1;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) {
        const size_t e = o + c;
        const float f0 = s.k[0][e], f1 = s.k[6][e], y0c = s.y[e], y1c = s.ys[e];
        if (rec.y) rec.y[((size_t)sh_n * p.B + b) * n3 + c] = y0c;
        if (j1 > j0) {
            const float ymid = __fadd_rn(y0c, fmaf(s.k[6][e], DP::m6 * dtf, fmaf(s.k[5][e], DP::m5 * dtf, fmaf(s.k[4][e], DP::m4 * dtf,
                               fmaf(s.k[3][e], DP::m3 * dtf, fmaf(s.k[2][e], DP::m2 * dtf, s.k[0][e] * (DP::m0 * dtf)))))));
            const float ca = 2.f * dtf * (f1 - f0) - 8.f * (y1c + y0c) + 16.f * ymid;
            const float cb = dtf * (5.f * f0 - 3.f * f1) + 18.f * y0c + 14.f * y1c - 32.f * ymid;
            const float cc = dtf * (f1 - 4.f * f0) - 11.f * y0c - 5.f * y1c + 16.f * ymid;
            const float cd = dtf * f0;
            for (int j = j0; j < j1; ++j) {
                const float x = (float)(((double)ts[j] - t0) / (t1 - t0));
                if (rec.y && c == 0) { rec.out_step[(size_t)b * T + j] = sh_n; rec.out_x[(size_t)b * T + j] = x; }
                float tot = __fadd_rn(y0c, __fmul_rn(x, cd));
                float xp = __fmul_rn(x, x);
                tot = __fadd_rn(tot, __fmul_rn(xp, cc));
                xp = __fmul_rn(xp, x);
                tot = __fadd_rn(tot, __fmul_rn(xp, cb));
                xp = __fmul_rn(xp, x);
                tot = __fadd_rn(tot, __fmul_rn(xp, ca));
                y_out[(size_t)j * total + e] = tot;
            }
        }
        s.y[e] = y1c;
        s.k[0][e] = f1;
    }
}

struct DpLayout {
    DriftLayout drift;
    size_t off_k[7], off_y, off_ys, off_state, total;
};

static DpLayout dp_layout(const DevProblem& p) {
    DpLayout L;
    Carve c;
    L.drift = drift_layout(c, p, 1, /*loc=*/false, /*aux=*/true, /*dw_rows=*/false);
    const size_t st = 4ull * p.B * 3 * p.N;
    for (int i = 0; i < 7; ++i) L.off_k[i] = c.take(st);
    L.off_y = c.take(st); L.off_ys = c.take(st);
    L.off_state = c.take(64ull * p.B + 1024);
    L.total = c.o;
    return L;
}

}  // namespace tc

size_t stage_dopri5_fwd_workspace_bytes(const DevProblem& p, int) { return tc::dp_layout(p).total; }

// f16: the six drift contractions of a round read FP16 pairs, as in em_fwd_impl (kRetryTf32 when a value did not fit).
static int dopri5_fwd_impl(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, float rtol, float atol,
                           int max_steps, int* n_accept, int* n_reject, int* status, const Dopri5Record& rec, void* ws,
                           size_t ws_bytes, cudaStream_t s, bool f16) {
    using namespace tc;
    const DpLayout L = dp_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    const size_t st = (size_t)p.B * 3 * p.N;
    const size_t B = p.B;
    DpState S;
    for (int i = 0; i < 7; ++i) S.k[i] = reinterpret_cast<float*>(w + L.off_k[i]);
    S.y = reinterpret_cast<float*>(w + L.off_y); S.ys = reinterpret_cast<float*>(w + L.off_ys);
    TrialCarve g{w + L.off_state};
    g(S.t, B); g(S.dt, B); g(S.red, 2 * B); g(S.t_stage, B);
    g(S.next_out, B); g(S.n_acc, B); g(S.n_rej, B); g(S.status, B); g(S.active, B);
    g(S.n_active, 1);

    StagedDrift drift;
    int rc = drift.init(p, w, L.drift, f16, s);
    if (rc != ODECOL_OK) return rc;
    if (cudaMemcpyAsync(S.y, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaMemcpyAsync(y_out, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    const int eg = ew_grid(st);
    float t_first = 0.f;
    if (cudaMemcpyAsync(&t_first, ts_dev, sizeof(float), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
    // f(t_stage[b], ys[b]) -> k[stage] for every trial (finished trials compute along harmlessly: rows are independent)
    if ((rc = drift.eval(0, S.y, nullptr, t_first, S.k[0])) != ODECOL_OK) return rc;        // f0 = f(t[0], y0)
    k_dp_init1<<<p.B, 256, 0, s>>>(p, S, ts_dev, rtol, atol);
    if ((rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[1])) != ODECOL_OK) return rc;         // f(t0 + h0, y0 + h0 f0)
    k_dp_init2<<<p.B, 256, 0, s>>>(p, S, rtol, atol);
    count_launch(2);
    int h_active = p.B;
    for (long long round = 0; round < (long long)max_steps && h_active > 0; ++round) {
        k_dp_stage<1><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[1]); if (rc) return rc;
        k_dp_stage<2><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[2]); if (rc) return rc;
        k_dp_stage<3><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[3]); if (rc) return rc;
        k_dp_stage<4><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[4]); if (rc) return rc;
        k_dp_stage<5><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[5]); if (rc) return rc;
        k_dp_stage<6><<<eg, 256, 0, s>>>(p, S); rc = drift.eval(0, S.ys, S.t_stage, 0.f, S.k[6]); if (rc) return rc;
        k_dp_finish<<<p.B, 256, 0, s>>>(p, S, ts_dev, T, rtol, atol, max_steps, y_out, rec);
        count_launch(7);
        if ((round & 15) == 15) {
            if (cudaMemcpyAsync(&h_active, S.n_active, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
            if ((rc = drift.overflowed()) != ODECOL_OK) return rc;
        }
    }
    if (f16 && (rc = drift.overflowed()) != ODECOL_OK) return rc;         // rounds since the last poll
    return adaptive_finish(p, S, T, y_out, n_accept, n_reject, status, s);
}

int stage_dopri5_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, float rtol, float atol,
                     int max_steps, int* n_accept, int* n_reject, int* status, const Dopri5Record& rec, void* ws,
                     size_t ws_bytes, cudaStream_t s) {
    // Forward-only solves take the 16-bit format.  Training (rec.y != NULL) stays on TF32 pairs: on the stiff parity network the
    // discrete adjoint through a stability-limited step sequence is ill-conditioned (on-chip and staged TF32 gradients already
    // differ by 2e-2 there), and the step sequence the FP16 rounding produced amplified it 300-fold (profiles/r2_session4.md).
    return tc::solve_f16_or_tf32(tc::kDp16, rec.y == nullptr, [&](bool f16) {
        return dopri5_fwd_impl(p, ts_dev, T, y0, y_out, rtol, atol, max_steps, n_accept, n_reject, status, rec, ws, ws_bytes, s, f16);
    });
}


// ---------------------------------------------------------------------------------------------------------------
// Staged torchsde srk (Roessler SRI2, fixed step) for networks beyond the on-chip family: three tensor-core drift
// evaluations per step (stages at t0, t0 + h, t0 + h/2; the fourth has weight 0), the stage states, the step and the
// interpolated outputs in elementwise kernels -- the arithmetic of k_srk_fwd_small.  The (W, U) of a step are formed
// once per trial (host tables or Philox) together with the four g_weights.  Forward only.
// ---------------------------------------------------------------------------------------------------------------
namespace tc {

struct SrkNoise { float* dw; float* du; float* gw; };    // (B), (B), (B, 4)

__global__ void k_srk_noise(DevProblem p, SrkNoise nz, const float* __restrict__ dWs, const float* __restrict__ dUs,
                            unsigned long long seed, long long trial_offset, long long kstep, float h) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.B) return;
    const Philox px(seed);
    float dw, du, gw[4];
    srk_increments(dWs, dUs, px, (unsigned long long)(trial_offset + b), kstep, p.B, b, h, dw, du);
    srk_g_weights(h, dw, du, gw);
    nz.dw[b] = dw; nz.du[b] = du;
#pragma unroll
    for (int q = 0; q < 4; ++q) nz.gw[4 * b + q] = gw[q];
}

// which: 1 -> H = y + f0 h;  2 -> H = y + 1/4 (f0 + f1) h + 3/2 sigma U / h  (srk_h2's operation order)
__global__ void k_srk_stage(DevProblem p, SrkNoise nz, int which, const float* __restrict__ y, const float* __restrict__ f0,
                            const float* __restrict__ f1, float h, float* __restrict__ H) {
    const int n3 = 3 * p.N;
    const size_t total = (size_t)p.B * n3;
    const float rdt = __fdiv_rn(1.0f, h);
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        if (which == 1) { H[e] = __fadd_rn(y[e], __fmul_rn(f0[e], h)); continue; }
        const int b = (int)(e / n3), comp = (int)(e % n3);
        const float sg = (p.sigma ? __ldg(p.sigma + comp) : 0.f) * (p.sigma_scale ? __ldg(p.sigma_scale + b) : 1.f);
        H[e] = srk_h2(y[e], f0[e], f1[e], sg, h, nz.du[b], rdt);
    }
}

struct SrkStepArgs {
    DevProblem p; SrkNoise nz;
    float* y; float* y_prev; const float* f0; const float* f1; const float* f2;
    float t0, t1; float* y_out; int j_lo, j_hi; const float* ts;
};

__global__ void k_srk_step(SrkStepArgs a) {
    const int n3 = 3 * a.p.N;
    const size_t total = (size_t)a.p.B * n3;
    const float h = __fsub_rn(a.t1, a.t0);
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / n3), comp = (int)(e % n3);
        const float sg = (a.p.sigma ? __ldg(a.p.sigma + comp) : 0.f) * (a.p.sigma_scale ? __ldg(a.p.sigma_scale + b) : 1.f);
        const float* gw = a.nz.gw + 4 * b;
        const float y0 = a.y[e];
        float v = __fadd_rn(__fadd_rn(y0, __fmul_rn(__fmul_rn(Srid2::a0, a.f0[e]), h)), __fmul_rn(sg, gw[0]));
        v = __fadd_rn(__fadd_rn(v, __fmul_rn(__fmul_rn(Srid2::a1, a.f1[e]), h)), __fmul_rn(sg, gw[1]));
        v = __fadd_rn(__fadd_rn(v, __fmul_rn(__fmul_rn(Srid2::a2, a.f2[e]), h)), __fmul_rn(sg, gw[2]));
        const float y1 = __fadd_rn(v, __fmul_rn(sg, gw[3]));
        a.y_prev[e] = y0;
        a.y[e] = y1;
        for (int j = a.j_lo; j < a.j_hi; ++j) {
            const float out_t = __ldg(a.ts + j);
            const float w0 = __fdiv_rn(__fsub_rn(a.t1, out_t), h), w1 = __fdiv_rn(__fsub_rn(out_t, a.t0), h);
            a.y_out[(size_t)j * total + e] = __fadd_rn(__fmul_rn(w0, y0), __fmul_rn(w1, y1));
        }
    }
}

__global__ void k_status_finite(DevProblem p, const float* __restrict__ y, int* __restrict__ status) {
    const int b = blockIdx.x, n3 = 3 * p.N;
    int bad = 0;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) bad |= !isfinite(y[(size_t)b * n3 + c]);
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) status[b] = bad ? ODECOL_ST_NONFINITE : ODECOL_ST_OK;
}

}  // namespace tc

size_t stage_srk_fwd_workspace_bytes(const DevProblem& p, int) { return tc::em_layout(p).total; }

// f16: the three drift contractions of a step read FP16 pairs, as in em_fwd_impl (kRetryTf32 when a value did not fit: the
// flag is read once, after the last step).
static int srk_fwd_impl(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                        const float* dU, uint64_t seed, int64_t trial_offset, float dt, int* status, float* y_steps, void* ws,
                        size_t ws_bytes, cudaStream_t s, bool f16) {
    using namespace tc;
    const EmLayout L = em_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
    float *f0 = F(L.off_f), *f1 = F(L.off_fm), *f2 = F(L.off_yfull), *H = F(L.off_ymid);
    float *y = F(L.off_y), *yprev = F(L.off_yprev);
    SrkNoise nz;
    nz.dw = F(L.off_state); nz.du = nz.dw + p.B; nz.gw = nz.du + p.B;          // 6 floats per trial of the 128-byte slot
    const size_t st = (size_t)p.B * 3 * p.N;
    StagedDrift drift;
    int rc = drift.init(p, w, L.drift, f16, s);
    if (rc != ODECOL_OK) return rc;
    if (cudaMemcpyAsync(y, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaMemcpyAsync(y_out, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (y_steps && cudaMemcpyAsync(y_steps, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    const int eg = ew_grid(st);
    long long n_steps = 0;
    rc = fixed_step_walk(ts_dev, T, dt, s, n_steps, [&](long long k, float t0, float t1, int j_lo, int j_hi) -> int {
        volatile float hv = t1 - t0;
        const float h = hv;
        volatile float t1v = t0 + h, thv = t0 + 0.5f * h;           // stage times in float32, as the on-chip kernel forms them
        k_srk_noise<<<(p.B + 127) / 128, 128, 0, s>>>(p, nz, dW, dU, (unsigned long long)seed, (long long)trial_offset, k, h);
        int r = drift.eval(0, y, nullptr, t0, f0); if (r) return r;
        k_srk_stage<<<eg, 256, 0, s>>>(p, nz, 1, y, f0, f1, h, H);
        r = drift.eval(0, H, nullptr, t1v, f1); if (r) return r;
        k_srk_stage<<<eg, 256, 0, s>>>(p, nz, 2, y, f0, f1, h, H);
        r = drift.eval(0, H, nullptr, thv, f2); if (r) return r;
        SrkStepArgs a;
        a.p = p; a.nz = nz; a.y = y; a.y_prev = yprev; a.f0 = f0; a.f1 = f1; a.f2 = f2; a.t0 = t0; a.t1 = t1;
        a.y_out = y_out; a.j_lo = j_lo; a.j_hi = j_hi; a.ts = ts_dev;
        k_srk_step<<<eg, 256, 0, s>>>(a);
        count_launch(4);
        if (y_steps && cudaMemcpyAsync(y_steps + (size_t)(k + 1) * st, y, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
            return ODECOL_E_CUDA;
        return ODECOL_OK;
    });
    if (rc != ODECOL_OK) return rc;
    if (f16 && (rc = drift.overflowed()) != ODECOL_OK) return rc;         // did every operand value fit FP16?
    if (status) { k_status_finite<<<p.B, 128, 0, s>>>(p, y, status); count_launch(); }
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

int stage_srk_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                  const float* dU, uint64_t seed, int64_t trial_offset, float dt, int* status, float* y_steps, void* ws,
                  size_t ws_bytes, cudaStream_t s) {
    return tc::solve_f16_or_tf32(tc::kSrk16, true, [&](bool f16) {
        return srk_fwd_impl(p, ts_dev, T, y0, y_out, dW, dU, seed, trial_offset, dt, status, y_steps, ws, ws_bytes, s, f16);
    });
}


// ---------------------------------------------------------------------------------------------------------------
// Staged discrete adjoints of the fixed-step stochastic solvers (Euler-Maruyama, srk) for networks beyond the on-chip
// family.  Building block: the vector-Jacobian product of ONE drift evaluation, b = J(Y, t)^T a, which also accumulates
// grad_W_aug += (gamma a_V)^T r_aug(Y, t):
//   prep        r, phi' of Y;  r_aug and gamma a_V split into hi / lo operands            (elementwise)
//   W^T . (gamma a_V) on the tensor cores, epilogue  b_V = -a_V / tau_m + phi' g,  b_A = -a_A / tau_a - phi' g,
//               b_F = -a_F / tau_s,  g = W^T (gamma a_V) + kappa a_A / tau_a + a_F / tau_s      (same algebra as
//               BwdCtx::stage_bwd of the on-chip family)
//   dW          the MN-major contraction of stage_tc_bwd.cu over the two operand buffers
// The reverse loops around it are those of k_em_bwd_small / k_srk_bwd_small, replayed on the host schedule.
// ---------------------------------------------------------------------------------------------------------------
namespace tc {

struct VjpEpi {
    DevProblem p;
    const float* a;        // (B, 3N) cotangent of the drift
    const float* D;        // (B, N)  phi'(V - A)
    float* b;              // (B, 3N) out
    float inv_tm, inv_ta, inv_ts;
    ODECOL_DEVINL void prepare() {}
    ODECOL_DEVINL void rows(int, int j, int n0, int, int g, int TNq, const float (&tot)[kMaxQ]) const {
        if (j >= p.N) return;
        const int N = p.N;
        const float kap = __ldg(p.kappa + j);
#pragma unroll 4
        for (int q = 0; q < kMaxQ; ++q) {
            const int t = n0 + g * TNq + q;
            if (q >= TNq || t >= p.B) break;
            const float* at = a + (size_t)t * 3 * N + j;
            const float aV = at[0], aA = at[N], aF = at[2 * N];
            const float d = D[(size_t)t * N + j];
            const float gg = tot[q] + kap * aA * inv_ta + aF * inv_ts;
            float* bt = b + (size_t)t * 3 * N + j;
            bt[0] = -aV * inv_tm + d * gg;
            bt[N] = -aA * inv_ta - d * gg;
            bt[2 * N] = -aF * inv_ts;
        }
    }
    ODECOL_DEVINL void tile_done(int, int, int, int, int) const {}
};

// operands of one VJP: r_aug(Y, t) -> (Rhi, Rlo) rows of KPa, gamma a_V -> (AVhi, AVlo) rows of NPk, phi' -> D
// t_trial != NULL: one evaluation time per trial; active != NULL: trials with active[b] == 0 contribute a zero cotangent
// (their rows of the gamma a_V operand are zero, so they add nothing to grad_W_aug)
__global__ void k_vjp_prep(DevProblem p, const float* __restrict__ Y, float tq, const float* __restrict__ a, float gamma,
                           float* __restrict__ Rhi, float* __restrict__ Rlo, int KPa, float* __restrict__ AVhi,
                           float* __restrict__ AVlo, int NPk, float* __restrict__ D,
                           const float* __restrict__ t_trial = nullptr, const int* __restrict__ active = nullptr) {
    const int b = blockIdx.x, N = p.N, Kaug = N + p.n_in + 1;
    const float* yb = Y + (size_t)b * 3 * N;
    int idx = 1;
    if (t_trial) tq = t_trial[b];
    const bool on = !active || active[b] != 0;
    const float tcl = knot_locate(p.knot_t, p.K, tq, idx);
    const float* ku = p.knot_u + (size_t)b * p.knot_stride_b;
    for (int k = threadIdx.x; k < Kaug; k += blockDim.x) {
        float v;
        if (k < N) {
            float dr;
            phi_dphi_fast(yb[k] - yb[N + k], v, dr);
            D[(size_t)b * N + k] = dr;
            const float av = on ? gamma * a[(size_t)b * 3 * N + k] : 0.f;
            const float h = tf32_rna(av);
            AVhi[(size_t)b * NPk + k] = h;
            AVlo[(size_t)b * NPk + k] = tf32_rna(av - h);
        } else if (k < N + p.n_in) v = knot_value(p.knot_t, ku, p.n_in, idx, tcl, k - N);
        else v = 1.0f;
        const float h = tf32_rna(v);
        Rhi[(size_t)b * KPa + k] = h;
        Rlo[(size_t)b * KPa + k] = tf32_rna(v - h);
    }
}

// out = c0 x0 + c1 x1 + c2 x2 + c3 x3 (NULL terms skipped); out may alias any input
__global__ void k_lincomb(size_t n, float* out, float c0, const float* x0, float c1, const float* x1, float c2,
                          const float* x2, float c3, const float* x3) {
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        float v = 0.f;
        if (x0) v += c0 * x0[e];
        if (x1) v += c1 * x1[e];
        if (x2) v += c2 * x2[e];
        if (x3) v += c3 * x3[e];
        out[e] = v;
    }
}

// lam += w1 g_j, pend += w0 g_j for the (selected) output gradient row j
__global__ void k_add_out_grad(DevProblem p, const float* __restrict__ grad_row, const int* __restrict__ sel, int G, float w1,
                               float w0, float* __restrict__ lam, float* __restrict__ pend) {
    const size_t total = (size_t)p.B * G;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / G), g = (int)(e % G);
        const int comp = sel ? sel[g] : g;
        const float v = grad_row[e];
        const size_t at = (size_t)b * 3 * p.N + comp;
        lam[at] += w1 * v;
        if (pend) pend[at] += w0 * v;
    }
}

struct AdjLayout {
    DriftLayout drift;          // TF32; operand planes of Bp32 rows
    int NPk;
    size_t off_AVhi, off_AVlo, off_WThi, off_WTlo, off_D;
    size_t off_lam, off_pend, off_a, off_b[3], off_f[2], off_H[2], off_noise, total;
};

static AdjLayout adj_layout(const DevProblem& p) {
    AdjLayout L;
    Carve c;
    L.drift = drift_layout(c, p, 1, /*loc=*/false, /*aux=*/false, /*dw_rows=*/true);
    const int Np = L.drift.Np, rows = L.drift.rows;
    L.NPk = Np;
    // the gamma a_V operand right behind r_aug: the drift's init zeroes both
    L.off_AVhi = c.take(4ull * rows * L.NPk); L.off_AVlo = c.take(4ull * rows * L.NPk);
    L.drift.zero_end = c.o;
    L.off_WThi = c.take(4ull * Np * L.NPk); L.off_WTlo = c.take(4ull * Np * L.NPk);
    L.off_D = c.take(4ull * p.B * p.N);
    const size_t st = 4ull * p.B * 3 * p.N;
    L.off_lam = c.take(st); L.off_pend = c.take(st); L.off_a = c.take(st);
    for (int i = 0; i < 3; ++i) L.off_b[i] = c.take(st);
    for (int i = 0; i < 2; ++i) L.off_f[i] = c.take(st);
    for (int i = 0; i < 2; ++i) L.off_H[i] = c.take(st);
    L.off_noise = c.take(32ull * p.B + 64);
    L.total = c.o;
    return L;
}

// transpose of the leading n x n block, split, padded (the W^T operand)
static __global__ void k_split_pad_WT(const float* __restrict__ src, int n, int ld, float* __restrict__ hi, float* __restrict__ lo,
                                      int rows_p, int cols_p) {
    const size_t total = (size_t)rows_p * cols_p;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols_p), c = (int)(e % cols_p);
        const float x = (r < n && c < n) ? src[(size_t)c * ld + r] : 0.0f;
        const float h = tf32_rna(x);
        hi[e] = h;
        lo[e] = tf32_rna(x - h);
    }
}

// shared state of a staged reverse sweep
struct AdjCtx {
    DevProblem p; AdjLayout L; cudaStream_t s; char* w;
    StagedDrift drift;                  // f = drift(Y, t); its operand set also holds r_aug(Y, t) for the VJPs
    CUtensorMap mWThi, mWTlo, mAVhi, mAVlo;
    TileShape tsB;
    float gamma;
    float* grad_W;
    float* F(size_t off) const { return reinterpret_cast<float*>(w + off); }

    int init(const DevProblem& p_, void* ws, size_t ws_bytes, float* grad_W_, cudaStream_t s_) {
        p = p_; L = adj_layout(p_); s = s_; w = static_cast<char*>(ws); grad_W = grad_W_;
        if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
        if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
        gamma = p.c.tau_s * p.c.R / p.c.tau_m;
        if (cudaMemsetAsync(w + L.off_lam, 0, L.off_a - L.off_lam, s) != cudaSuccess) return ODECOL_E_CUDA;
        if (cudaMemsetAsync(grad_W, 0, sizeof(float) * (size_t)p.N * p.ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
        const int rc = drift.init(p, w, L.drift, false, s);
        if (rc != ODECOL_OK) return rc;
        const DriftLayout& D = L.drift;
        k_split_pad_WT<<<296, 256, 0, s>>>(p.W_aug, p.N, p.ld_w, F(L.off_WThi), F(L.off_WTlo), D.Np, L.NPk);
        count_launch();
        if (!make_map(&mWThi, F(L.off_WThi), D.Np, L.NPk, L.NPk, BM) || !make_map(&mWTlo, F(L.off_WTlo), D.Np, L.NPk, L.NPk, BM) ||
            !make_map(&mAVhi, F(L.off_AVhi), D.Bp, L.NPk, L.NPk, D.TN) || !make_map(&mAVlo, F(L.off_AVlo), D.Bp, L.NPk, L.NPk, D.TN))
            return ODECOL_E_CUDA;
        tsB = TileShape{D.Np / BM, D.Bp / D.TN, D.TN, L.NPk / BK, 0};
        return ODECOL_OK;
    }
    size_t st() const { return (size_t)p.B * 3 * p.N; }

    // b = J(Y, t)^T a;  grad_W += (gamma a_V)^T r_aug(Y, t).  t_trial != NULL: one time per trial, else t_shared for all;
    // active != NULL: trials with active[b] == 0 are masked (adaptive solvers)
    int vjp(const float* Y, const float* t_trial, float t_shared, const int* active, const float* a, float* b) {
        const DriftLayout& D = L.drift;
        k_vjp_prep<<<p.B, 128, 0, s>>>(p, Y, t_shared, a, gamma, drift.R[0][0], drift.R[0][1], D.KPa, F(L.off_AVhi), F(L.off_AVlo),
                                       L.NPk, F(L.off_D), t_trial, active);
        count_launch();
        VjpEpi e;
        e.p = p; e.a = a; e.D = F(L.off_D); e.b = b;
        e.inv_tm = 1.0f / p.c.tau_m; e.inv_ta = 1.0f / p.c.tau_a; e.inv_ts = 1.0f / p.c.tau_s;
        int rc = launch_contract(mWThi, mWTlo, mAVhi, mAVlo, tsB, e, s);
        if (rc) return rc;
        return tc_dw_accumulate(F(L.off_AVhi), F(L.off_AVlo), drift.R[0][0], drift.R[0][1], D.rows, D.Np, D.KPa, p.N,
                                p.N + p.n_in + 1, p.ld_w, grad_W, s);
    }
    void lincomb(float* out, float c0, const float* x0, float c1 = 0.f, const float* x1 = nullptr, float c2 = 0.f,
                 const float* x2 = nullptr, float c3 = 0.f, const float* x3 = nullptr) {
        k_lincomb<<<ew_grid(st()), 256, 0, s>>>(st(), out, c0, x0, c1, x1, c2, x2, c3, x3);
        count_launch();
    }
};

// the float32 step schedule of torchsde's integrate loop, on the host: step start times, and for every output the solver
// state it ends on with its two interpolation weights (what k_em_schedule computes on the device)
struct HostSchedule {
    std::vector<float> tk, w0, w1;
    std::vector<int> step_of;
    int build(const float* ts_dev, int T, float dt, cudaStream_t s) {
        std::vector<float> ts(T);
        if (cudaMemcpyAsync(ts.data(), ts_dev, sizeof(float) * T, cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
        if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
        const float t_end = ts[T - 1];
        volatile float curr = ts[0], prev = ts[0];
        step_of.assign(T, 0); w0.assign(T, 0.f); w1.assign(T, 1.f);
        tk.assign(1, ts[0]);
        int k = 0;
        for (int j = 1; j < T; ++j) {
            const float out_t = ts[j];
            while (curr < out_t) {
                volatile float nx = curr + dt;
                const float next_t = nx < t_end ? nx : t_end;
                prev = curr; curr = next_t;
                tk.push_back(next_t);
                ++k;
            }
            volatile float spn = curr - prev, a0 = curr - out_t, a1 = out_t - prev;
            step_of[j] = k;
            w0[j] = a0 / spn; w1[j] = a1 / spn;
        }
        return ODECOL_OK;
    }
};

}  // namespace tc

size_t stage_sde_bwd_workspace_bytes(const DevProblem& p, int) { return tc::adj_layout(p).total; }

// which = 0: Euler-Maruyama, 1: srk (needs the increments: host tables or Philox)
int stage_sde_bwd(int which, const DevProblem& p, const float* ts_dev, int T, const float* y_steps, int64_t n_steps,
                  const float* dW, const float* dU, uint64_t seed, int64_t trial_offset, const float* grad_y, const int* sel,
                  int G, float dt, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    AdjCtx cx;
    int rc = cx.init(p, ws, ws_bytes, grad_W, s);
    if (rc) return rc;
    HostSchedule sch;
    rc = sch.build(ts_dev, T, dt, s);
    if (rc) return rc;
    const int nsteps = (int)sch.tk.size() - 1;
    if (nsteps != (int)n_steps) return ODECOL_E_SHAPE;
    const AdjLayout& L = cx.L;
    const size_t st = cx.st();
    float *lam = cx.F(L.off_lam), *pend = cx.F(L.off_pend), *a = cx.F(L.off_a);
    float *b0 = cx.F(L.off_b[0]), *b1 = cx.F(L.off_b[1]), *b2 = cx.F(L.off_b[2]);
    float *f0 = cx.F(L.off_f[0]), *f1 = cx.F(L.off_f[1]), *H1 = cx.F(L.off_H[0]), *H2 = cx.F(L.off_H[1]);
    SrkNoise nz;
    nz.dw = cx.F(L.off_noise); nz.du = nz.dw + p.B; nz.gw = nz.du + p.B;
    const int gg = ew_grid((size_t)p.B * G);
    int j = T - 1;
    for (int k = nsteps - 1; k >= 0; --k) {
        cx.lincomb(lam, 1.f, lam, 1.f, pend);                               // lam += pend
        if (cudaMemsetAsync(pend, 0, sizeof(float) * st, s) != cudaSuccess) return ODECOL_E_CUDA;
        while (j >= 1 && sch.step_of[j] == k + 1) {
            k_add_out_grad<<<gg, 256, 0, s>>>(p, grad_y + (size_t)j * p.B * G, sel, G, sch.w1[j], sch.w0[j], lam, pend);
            count_launch();
            --j;
        }
        const float t0 = sch.tk[k];
        volatile float hv = sch.tk[k + 1] - sch.tk[k];
        const float h = hv;
        const float* yk = y_steps + (size_t)k * st;
        if (which == 0) {
            cx.lincomb(a, h, lam);
            rc = cx.vjp(yk, nullptr, t0, nullptr, a, b0); if (rc) return rc;
            cx.lincomb(lam, 1.f, lam, 1.f, b0);
        } else {
            volatile float t1v = t0 + h, thv = t0 + 0.5f * h;
            k_srk_noise<<<(p.B + 127) / 128, 128, 0, s>>>(p, nz, dW, dU, (unsigned long long)seed, (long long)trial_offset, k, h);
            count_launch();
            rc = cx.drift.eval(0, yk, nullptr, t0, f0); if (rc) return rc;
            k_srk_stage<<<ew_grid(st), 256, 0, s>>>(p, nz, 1, yk, f0, f1, h, H1);
            rc = cx.drift.eval(0, H1, nullptr, t1v, f1); if (rc) return rc;
            k_srk_stage<<<ew_grid(st), 256, 0, s>>>(p, nz, 2, yk, f0, f1, h, H2);
            count_launch(2);
            const float h23 = h * Srid2::a2, h6 = h * Srid2::a0, h4 = h * 0.25f;
            cx.lincomb(a, h23, lam);
            rc = cx.vjp(H2, nullptr, thv, nullptr, a, b2); if (rc) return rc;
            cx.lincomb(a, h6, lam, h4, b2);
            rc = cx.vjp(H1, nullptr, t1v, nullptr, a, b1); if (rc) return rc;
            cx.lincomb(a, h6, lam, h4, b2, h, b1);
            rc = cx.vjp(yk, nullptr, t0, nullptr, a, b0); if (rc) return rc;
            cx.lincomb(lam, 1.f, lam, 1.f, b2, 1.f, b1, 1.f, b0);
        }
    }
    cx.lincomb(lam, 1.f, lam, 1.f, pend);
    if (j >= 0) {                                                           // output 0 is y0 itself
        k_add_out_grad<<<gg, 256, 0, s>>>(p, grad_y, sel, G, 1.f, 0.f, lam, nullptr);
        count_launch();
    }
    if (grad_y0 && cudaMemcpyAsync(grad_y0, lam, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

// ---------------------------------------------------------------------------------------------------------------
// Staged discrete adjoint of dopri5 for networks beyond the on-chip family: the algebra of k_dopri5_bwd_small (reverse
// sweep over the ACCEPTED steps the forward pass recorded; per step the seven stages are recomputed, then the adjoint
// runs through the dense-output quartic, the FSAL row and the tableau) with the drift evaluations and their
// vector-Jacobian products on the tensor cores.  Trials accept different numbers of steps, so the sweep runs in ROUNDS:
// in round r trial b handles its accepted step n_accept[b] - 1 - r (finished trials idle, masked out of every update and
// of grad_W_aug).  What it replaces: loss.backward() through torchdiffeq's unrolled adaptive solver
// (reference scripts/xor_ode.py:114,177, scripts/parity_ode.py:233,250) for the synthetic large networks.
// ---------------------------------------------------------------------------------------------------------------
namespace tc {

struct DpAdj {
    int* nidx; int* act; int* first; int* jptr;      // (B) step index of this round, n >= 0, n == 0, next output to consume
    float* dtf;                                      // (B)
    float* tst[7];                                   // (B) stage times
    float* Ys[7]; float* k[7]; float* kb[7];         // (B, 3N)
    float* yb0; float* yb1; float* lam; float* carry; float* bout;
};

// per trial: which accepted step this round handles, its t0 / dt, its start state
__global__ void k_dpb_begin(DevProblem p, DpAdj d, DpState s, Dopri5Record rec, const int* __restrict__ n_accept, int round) {
    const int b = blockIdx.x, n3 = 3 * p.N;
    const int n = n_accept[b] - 1 - round;
    if (threadIdx.x == 0) {
        d.nidx[b] = n; d.act[b] = n >= 0; d.first[b] = n == 0; s.active[b] = n >= 0;
        if (n >= 0) {
            const double t0 = rec.t0[(size_t)b * rec.cap + n], dt = rec.dt[(size_t)b * rec.cap + n];
            s.t[b] = t0; s.dt[b] = dt;
            d.dtf[b] = (float)dt; d.tst[0][b] = (float)t0;
        }
    }
    if (n < 0) return;
    const float* src = rec.y + ((size_t)n * p.B + b) * n3;
    float* dst = d.Ys[0] + (size_t)b * n3;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) dst[c] = src[c];
}

// adjoint of the dense output for every output inside this step; initial kbar / ybar (k_dopri5_bwd_small, same order)
__global__ void k_dpb_dense(DevProblem p, DpAdj d, Dopri5Record rec, int T, const float* __restrict__ grad_y,
                            const int* __restrict__ inv, int G) {
    const int b = blockIdx.x, n3 = 3 * p.N, B = p.B;
    if (!d.act[b]) return;
    const int n = d.nidx[b];
    const float dtf = d.dtf[b];
    const int j_hi = d.jptr[b];
    int j_lo = j_hi;
    while (j_lo >= 1 && rec.out_step[(size_t)b * T + j_lo] == n) --j_lo;          // outputs (j_lo, j_hi] lie in this step
    const float cmid[7] = {DP::m0, 0.f, DP::m2, DP::m3, DP::m4, DP::m5, DP::m6};
    const size_t o = (size_t)b * n3;
    for (int c = threadIdx.x; c < n3; c += blockDim.x) {
        const int gi = inv[c];
        float ca = 0.f, cb = 0.f, cc = 0.f, cd = 0.f, ce = 0.f;
        if (gi >= 0)
            for (int j = j_hi; j > j_lo; --j) {
                const float x = rec.out_x[(size_t)b * T + j];
                const float x2 = x * x, x3 = x2 * x, x4 = x3 * x;
                const float g = grad_y[((size_t)j * B + b) * G + gi];
                ce += g; cd += x * g; cc += x2 * g; cb += x3 * g; ca += x4 * g;
            }
        const float ymidb = 16.f * ca - 32.f * cb + 16.f * cc;
        d.yb0[o + c] = ce - 8.f * ca + 18.f * cb - 11.f * cc + ymidb;
        d.yb1[o + c] = d.lam[o + c] - 8.f * ca + 14.f * cb - 5.f * cc;
#pragma unroll
        for (int m = 0; m < 7; ++m) {
            float v = dtf * cmid[m] * ymidb;
            if (m == 0) v += dtf * (-2.f * ca + 5.f * cb - 4.f * cc + cd);                    // f0 = k1
            if (m == 6) v += dtf * (2.f * ca - 3.f * cb + cc) + d.carry[o + c];               // f1 = k7 (+ the next step's k1)
            d.kb[m][o + c] = v;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) d.jptr[b] = j_lo;
}

// Ybar_st = [st == 6] ybar1 + J(Y_st)^T kbar_st (in bout), pushed through tableau row st
template <int ST>
__global__ void k_dpb_push(DevProblem p, DpAdj d) {
    const int n3 = 3 * p.N;
    const size_t total = (size_t)p.B * n3;
    const float beta[6][6] = {
        {DP::b10, 0.f, 0.f, 0.f, 0.f, 0.f}, {DP::b20, DP::b21, 0.f, 0.f, 0.f, 0.f}, {DP::b30, DP::b31, DP::b32, 0.f, 0.f, 0.f},
        {DP::b40, DP::b41, DP::b42, DP::b43, 0.f, 0.f}, {DP::b50, DP::b51, DP::b52, DP::b53, DP::b54, 0.f},
        {DP::b60, 0.f, DP::b62, DP::b63, DP::b64, DP::b65}};
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / n3);
        if (!d.act[b]) continue;
        const float dtf = d.dtf[b];
        float Yb = d.bout[e];
        if (ST == 6) Yb += d.yb1[e];
        d.yb0[e] += Yb;
#pragma unroll
        for (int m = 0; m < 6; ++m)
            if (m < ST) d.kb[m][e] += dtf * beta[ST - 1][m] * Yb;
    }
}

// end of the round: hand kbar_1 to the previous step (its k7) or, at a trial's first step, add J(y0)^T kbar_1 (in bout)
__global__ void k_dpb_end(DevProblem p, DpAdj d, int have_first) {
    const int n3 = 3 * p.N;
    const size_t total = (size_t)p.B * n3;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / n3);
        if (!d.act[b]) continue;
        if (d.first[b]) { d.lam[e] = d.yb0[e] + (have_first ? d.bout[e] : 0.f); d.carry[e] = 0.f; }
        else { d.lam[e] = d.yb0[e]; d.carry[e] = d.kb[0][e]; }
    }
}

__global__ void k_dpb_init(DevProblem p, DpAdj d, int T) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.B) d.jptr[b] = T - 1;
}

struct DpAdjLayout { AdjLayout A; size_t off_planes, off_small, off_inv, total; };
static DpAdjLayout dp_adj_layout(const DevProblem& p) {
    DpAdjLayout L;
    L.A = adj_layout(p);
    Carve c{L.A.total};
    const size_t st = 4ull * p.B * 3 * p.N;
    L.off_planes = c.take(26 * st);                                   // Ys, k, kb (7 each), yb0, yb1, lam, carry, bout
    L.off_small = c.take(256ull * p.B + 4096);
    L.off_inv = c.take(4ull * (3 * p.N + 4));
    L.total = c.o;
    return L;
}

}  // namespace tc

size_t stage_dopri5_bwd_workspace_bytes(const DevProblem& p, int) { return tc::dp_adj_layout(p).total; }

int stage_dopri5_bwd(const DevProblem& p, int T, const Dopri5Record& rec, const int* n_accept, const float* grad_y,
                     const int* sel, int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const DpAdjLayout L = dp_adj_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    AdjCtx cx;
    int rc = cx.init(p, ws, ws_bytes, grad_W, s);
    if (rc) return rc;
    char* w = static_cast<char*>(ws);
    const size_t st = cx.st(), B = p.B;
    if (cudaMemsetAsync(w + L.off_planes, 0, L.total - L.off_planes, s) != cudaSuccess) return ODECOL_E_CUDA;
    float* pl = reinterpret_cast<float*>(w + L.off_planes);
    DpAdj d;
    for (int i = 0; i < 7; ++i) { d.Ys[i] = pl + (size_t)i * st; d.k[i] = pl + (size_t)(7 + i) * st; d.kb[i] = pl + (size_t)(14 + i) * st; }
    d.yb0 = pl + 21 * st; d.yb1 = pl + 22 * st; d.lam = pl + 23 * st; d.carry = pl + 24 * st; d.bout = pl + 25 * st;
    TrialCarve g{w + L.off_small};
    g(d.nidx, B); g(d.act, B); g(d.first, B); g(d.jptr, B); g(d.dtf, B);
    for (int i = 0; i < 7; ++i) g(d.tst[i], B);
    DpState S;                                        // the forward stage kernels (k_dp_stage) run on this view
    g(S.t, B); g(S.dt, B);
    S.red = nullptr; S.next_out = S.n_acc = S.n_rej = S.status = nullptr; S.n_active = nullptr;
    S.active = d.act;
    for (int i = 0; i < 7; ++i) S.k[i] = d.k[i];
    S.y = d.Ys[0];
    int* inv = reinterpret_cast<int*>(w + L.off_inv);
    k_tc_build_inv<<<1, 256, 0, s>>>(sel, G, 3 * p.N, inv);
    k_dpb_init<<<(p.B + 127) / 128, 128, 0, s>>>(p, d, T);
    count_launch(2);
    // accepted-step counts decide the number of rounds and where first steps fall (one synchronisation, like the forward pass)
    std::vector<int> nacc(p.B);
    if (cudaMemcpyAsync(nacc.data(), n_accept, sizeof(int) * B, cudaMemcpyDeviceToHost, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess) return ODECOL_E_CUDA;
    int rounds = 0;
    for (int b = 0; b < p.B; ++b) { if (nacc[b] > rec.cap) return ODECOL_E_SHAPE; if (nacc[b] > rounds) rounds = nacc[b]; }
    std::vector<char> has_first(rounds + 1, 0);
    for (int b = 0; b < p.B; ++b) if (nacc[b] >= 1) has_first[nacc[b] - 1] = 1;
    const int eg = ew_grid(st);
    for (int r = 0; r < rounds; ++r) {
        k_dpb_begin<<<p.B, 256, 0, s>>>(p, d, S, rec, n_accept, r);
        count_launch();
        // ---- recompute the seven stages (stage 0 = the recorded start state at t0)
        rc = cx.drift.eval(0, d.Ys[0], d.tst[0], 0.f, d.k[0]); if (rc) return rc;
#define ODECOL_DPB_STAGE(ST)                                                        \
        S.ys = d.Ys[ST]; S.t_stage = d.tst[ST];                                     \
        k_dp_stage<ST><<<eg, 256, 0, s>>>(p, S); count_launch();                    \
        rc = cx.drift.eval(0, d.Ys[ST], d.tst[ST], 0.f, d.k[ST]); if (rc) return rc;
        ODECOL_DPB_STAGE(1) ODECOL_DPB_STAGE(2) ODECOL_DPB_STAGE(3) ODECOL_DPB_STAGE(4) ODECOL_DPB_STAGE(5) ODECOL_DPB_STAGE(6)
#undef ODECOL_DPB_STAGE
        // ---- dense output adjoint, then stages 7 .. 2
        k_dpb_dense<<<p.B, 256, 0, s>>>(p, d, rec, T, grad_y, inv, G);
        count_launch();
#define ODECOL_DPB_BACK(ST)                                                                            \
        rc = cx.vjp(d.Ys[ST], d.tst[ST], 0.f, d.act, d.kb[ST], d.bout); if (rc) return rc;            \
        k_dpb_push<ST><<<eg, 256, 0, s>>>(p, d); count_launch();
        ODECOL_DPB_BACK(6) ODECOL_DPB_BACK(5) ODECOL_DPB_BACK(4) ODECOL_DPB_BACK(3) ODECOL_DPB_BACK(2) ODECOL_DPB_BACK(1)
#undef ODECOL_DPB_BACK
        if (has_first[r]) { rc = cx.vjp(d.Ys[0], d.tst[0], 0.f, d.first, d.kb[0], d.bout); if (rc) return rc; }
        k_dpb_end<<<eg, 256, 0, s>>>(p, d, has_first[r] ? 1 : 0);
        count_launch();
    }
    // output 0 is y0 itself
    k_add_out_grad<<<ew_grid((size_t)p.B * G), 256, 0, s>>>(p, grad_y, sel, G, 1.f, 0.f, d.lam, nullptr);
    count_launch();
    if (grad_y0 && cudaMemcpyAsync(grad_y0, d.lam, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

}  // namespace odecol
