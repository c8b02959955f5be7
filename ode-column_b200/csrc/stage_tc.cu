// Family T drivers: forward RK4 stages on the tensor cores and the diagnostic contraction (kernels in stage_tc.cuh).
#include <cstdlib>
#include "stage_tc.cuh"

namespace odecol {
namespace tc {

// ---------------------------------------------------------------------------------------------------------------
// diagnostic: the contraction core alone, C[n][m] = sum_k A[m][k] B[n][k]
// ---------------------------------------------------------------------------------------------------------------
struct StoreEpi {
    float* C; int M, N, ldc;
    ODECOL_DEVINL void prepare() {}
    ODECOL_DEVINL void rows(int, int i, int n0, int, int g, int TNq, const float (&tot)[kMaxQ]) const {
        if (i >= M) return;
#pragma unroll
        for (int j = 0; j < kMaxQ; ++j) {
            const int b = n0 + g * TNq + j;
            if (j < TNq && b < N) C[(size_t)b * ldc + i] = tot[j];
        }
    }
    ODECOL_DEVINL void tile_done(int, int, int, int, int) const {}
};

struct ContractLayout { int Mp, Np, Kp, TN; size_t off_Ahi, off_Alo, off_Bhi, off_Blo, total; };
static ContractLayout contract_layout(int M, int N, int K) {
    ContractLayout L;
    L.Mp = round_up(M, BM); L.Kp = round_up(K, BK);
    L.TN = pick_tile_n(L.Mp / BM, N);
    L.Np = round_up(N, L.TN);
    size_t o = 0;
    auto take = [&](size_t floats) { const size_t r = o; o += (floats * 4 + 1023) / 1024 * 1024; return r; };
    L.off_Ahi = take((size_t)L.Mp * L.Kp); L.off_Alo = take((size_t)L.Mp * L.Kp);
    L.off_Bhi = take((size_t)L.Np * L.Kp); L.off_Blo = take((size_t)L.Np * L.Kp);
    L.total = o;
    return L;
}


// initial operand (r_aug at t_ptr[0], split hi/lo), constant-one column + zero padding of the second operand buffer,
// and the tile-major copy of y0.  One CTA per (padded) trial.
__global__ void k_tc_init(DevProblem p, TileGeom tg, const float* __restrict__ y, const float* __restrict__ t_ptr,
                          float* __restrict__ hi0, float* __restrict__ lo0, float* __restrict__ hi1, float* __restrict__ lo1,
                          float* __restrict__ V0T, float* __restrict__ A0T, float* __restrict__ F0T, int KPa) {
    const int b = blockIdx.x, N = p.N, Kaug = N + p.n_in + 1;
    const size_t ro = (size_t)b * KPa;
    const int nt = b / tg.TN, g = (b % tg.TN) / tg.TNq, jq = (b % tg.TN) % tg.TNq;
    const int q = jq >> 2, e4 = jq & 3;
    if (b >= p.B) {
        for (int k = threadIdx.x; k < KPa; k += blockDim.x) { hi0[ro + k] = 0.f; lo0[ro + k] = 0.f; hi1[ro + k] = 0.f; lo1[ro + k] = 0.f; }
        for (int i = threadIdx.x; i < tg.Np; i += blockDim.x) {
            const size_t o = tg.off(nt, g, q, i) + e4;
            V0T[o] = 0.f; A0T[o] = 0.f; F0T[o] = 0.f;
        }
        return;
    }
    const float* yb = y + (size_t)b * 3 * N;
    int idx = 1;
    const float tcl = knot_locate(p.knot_t, p.K, __ldg(t_ptr), idx);
    const float* ku = p.knot_u + (size_t)b * p.knot_stride_b;
    for (int k = threadIdx.x; k < KPa; k += blockDim.x) {
        float v = 0.f, one = 0.f;
        if (k < N) v = phi_fast(yb[k] - yb[N + k]);
        else if (k < N + p.n_in) v = knot_value(p.knot_t, ku, p.n_in, idx, tcl, k - N);
        else if (k == Kaug - 1) { v = 1.f; one = 1.f; }
        const float h = tf32_rna(v);
        hi0[ro + k] = h; lo0[ro + k] = tf32_rna(v - h);
        hi1[ro + k] = one; lo1[ro + k] = 0.f;
    }
    for (int i = threadIdx.x; i < tg.Np; i += blockDim.x) {
        const size_t o = tg.off(nt, g, q, i) + e4;
        const bool in = i < N;
        const float V = in ? yb[i] : 0.f, A = in ? yb[N + i] : 0.f, F = in ? yb[2 * N + i] : 0.f;
        V0T[o] = V; A0T[o] = A; F0T[o] = F;
    }
}

struct TcFwdLayout {
    int Np, Bp, KPa, TN, KP16;
    size_t off_Whi, off_Wlo, off_Rhi[2], off_Rlo[2], off_K[3], off_Y[2], off_done, off_inv, total;
    size_t off_W16[2], off_R16[2], off_wscale;      // mixed 16-bit operand format of the persistent forward kernel
};

static TcFwdLayout tc_fwd_layout(const DevProblem& p) {
    TcFwdLayout L;
    L.Np = round_up(p.N, BM);
    L.KPa = round_up(p.N + p.n_in + 1, BK);
    L.TN = pick_tile_n(L.Np / BM, p.B);
    L.Bp = round_up(p.B, L.TN);
    size_t o = 0;
    auto take = [&](size_t floats) { const size_t r = o; o += (floats * 4 + 1023) / 1024 * 1024; return r; };
    L.off_Whi = take((size_t)L.Np * L.KPa); L.off_Wlo = take((size_t)L.Np * L.KPa);
    for (int i = 0; i < 2; ++i) { L.off_Rhi[i] = take((size_t)L.Bp * L.KPa); L.off_Rlo[i] = take((size_t)L.Bp * L.KPa); }
    const size_t plane = (size_t)L.Np * L.Bp;
    for (int i = 0; i < 3; ++i) L.off_K[i] = take(plane);            // V slope of stages 1..3
    for (int i = 0; i < 2; ++i) L.off_Y[i] = take(3 * plane);
    L.off_done = take((size_t)(L.Bp / L.TN) + 64);          // one uint32 per trial tile (floats == 4 bytes)
    L.off_inv = take(3ull * p.N + 4);                       // component -> selection position (checkpoint mode) + F flag
    L.KP16 = round_up(p.N + p.n_in + 1, BK16);
    for (int i = 0; i < 2; ++i) L.off_W16[i] = take(((size_t)L.Np * L.KP16 + 1) / 2);          // FP16: half a float each
    for (int i = 0; i < 2; ++i) L.off_R16[i] = take((size_t)L.Bp * L.KP16);                    // two FP16 planes
    L.off_wscale = take(4);
    L.total = o;
    return L;
}

}  // namespace tc

void tc_launch_init(const DevProblem& p, const tc::TileGeom& tg, const float* y0, const float* t_dev, float* hi0, float* lo0,
                    float* hi1, float* lo1, float* V0T, float* A0T, float* F0T, int KPa, int Bp, cudaStream_t s) {
    tc::k_tc_init<<<Bp, 128, 0, s>>>(p, tg, y0, t_dev, hi0, lo0, hi1, lo1, V0T, A0T, F0T, KPa);
}

int tc_rk4_fwd_persistent(const DevProblem& p, const float* t_dev, int T, const float* y0, float* y_out, int out_every,
                          float* Whi, float* Wlo, float* const Rhi[2], float* const Rlo[2], float* const KT[3],
                          float* const YT[2], unsigned int* done, int Np, int Bp, int KPa, int TN, const tc::CkptView* ck,
                          const tc::Mixed16* mx, cudaStream_t s);

namespace tc {
static Mixed16 mixed16_view(const TcFwdLayout& L, char* w) {
    Mixed16 m;
    for (int i = 0; i < 2; ++i) { m.W16[i] = w + L.off_W16[i]; m.R16[i] = reinterpret_cast<uint16_t*>(w + L.off_R16[i]); }
    m.wscale = reinterpret_cast<float*>(w + L.off_wscale);
    m.KP16 = L.KP16;
    return m;
}
}  // namespace tc

static bool persistent_enabled() {
    const char* v = getenv("ODECOL_PERSISTENT");
    return v ? atoi(v) != 0 : true;
}

size_t tc_rk4_fwd_workspace_bytes(const DevProblem& p, int) { return tc::tc_fwd_layout(p).total; }

int tc_rk4_fwd(const DevProblem& p, const float* t_dev, int T, const float* y0, float* y_out, int out_every, void* ws,
               size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const TcFwdLayout L = tc_fwd_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
    float *Whi = F(L.off_Whi), *Wlo = F(L.off_Wlo);
    float* Rhi[2] = {F(L.off_Rhi[0]), F(L.off_Rhi[1])};
    float* Rlo[2] = {F(L.off_Rlo[0]), F(L.off_Rlo[1])};
    float* KT[3] = {F(L.off_K[0]), F(L.off_K[1]), F(L.off_K[2])};
    float* YT[2] = {F(L.off_Y[0]), F(L.off_Y[1])};
    const int Kaug = p.N + p.n_in + 1;
    const size_t st = (size_t)p.B * 3 * p.N;
    const TileGeom tg{L.Bp / L.TN, L.Np, L.TN, L.TN / 4};
    // long contractions (K > 32 * kChunkMin) go through k_tc_contract, which accumulates in chunks (stage_tc.cuh); the
    // persistent kernel keeps the rotating-accumulator scheme that is accurate up to that length
    if (persistent_enabled() && L.KPa / BK <= kChunkMin) {
        const Mixed16 mx = mixed16_view(L, w);
        return tc_rk4_fwd_persistent(p, t_dev, T, y0, y_out, out_every, Whi, Wlo, Rhi, Rlo, KT, YT,
                                     reinterpret_cast<unsigned int*>(w + L.off_done), L.Np, L.Bp, L.KPa, L.TN, nullptr, &mx, s);
    }

    k_split_pad<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, Whi, Wlo, L.Np, L.KPa);
    k_tc_init<<<L.Bp, 128, 0, s>>>(p, tg, y0, t_dev, Rhi[0], Rlo[0], Rhi[1], Rlo[1], YT[0], YT[0] + tg.plane(),
                                   YT[0] + 2 * tg.plane(), L.KPa);
    count_launch(2);
    if (cudaMemcpyAsync(y_out, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    CUtensorMap mWhi, mWlo, mRhi[2], mRlo[2];
    bool ok = make_map(&mWhi, Whi, L.Np, L.KPa, L.KPa, BM) && make_map(&mWlo, Wlo, L.Np, L.KPa, L.KPa, BM);
    for (int i = 0; i < 2; ++i)
        ok = ok && make_map(&mRhi[i], Rhi[i], L.Bp, L.KPa, L.KPa, L.TN) && make_map(&mRlo[i], Rlo[i], L.Bp, L.KPa, L.KPa, L.TN);
    if (!ok) return ODECOL_E_CUDA;
    const TileShape ts{L.Np / BM, L.Bp / L.TN, L.TN, L.KPa / BK, 0};
    int cur = 0;
    auto launch = [&](auto& e) { return launch_contract(mWhi, mWlo, mRhi[cur], mRlo[cur], ts, e, s); };
    for (int n = 0; n < T - 1; ++n) {
        const int j = n + 1;
        const bool emit = (j % out_every == 0) || (j == T - 1);
        const size_t r = (j % out_every == 0) ? (size_t)(j / out_every) : (size_t)((T - 2) / out_every + 1);
        auto fill = [&](auto& e) {
            e.p = p; e.tg = tg; e.t = t_dev; e.n = n; e.KPa = L.KPa;
            const size_t pl = tg.plane();
            e.V0T = YT[n & 1]; e.A0T = YT[n & 1] + pl; e.F0T = YT[n & 1] + 2 * pl;
            e.V1T = YT[(n + 1) & 1]; e.A1T = YT[(n + 1) & 1] + pl; e.F1T = YT[(n + 1) & 1] + 2 * pl;
            e.traj_row = emit ? y_out + r * st : nullptr; e.ysel_row = nullptr; e.inv = nullptr; e.G = 0;
            e.K1T = KT[0]; e.K2T = KT[1]; e.K3T = KT[2];
            e.Rhi_nxt = Rhi[cur ^ 1]; e.Rlo_nxt = Rlo[cur ^ 1]; e.DRT_nxt = nullptr;
            e.inv_tm = 1.0f / p.c.tau_m; e.inv_ta = 1.0f / p.c.tau_a; e.inv_ts = 1.0f / p.c.tau_s;
            e.t0 = e.t1 = e.dt = 0.f;
        };
        for (int S = 1; S <= 4; ++S) {
            int rc;
            if (S == 1) { FwdEpiT<1> e; fill(e); rc = launch(e); }
            else if (S == 2) { FwdEpiT<2> e; fill(e); rc = launch(e); }
            else if (S == 3) { FwdEpiT<3> e; fill(e); rc = launch(e); }
            else { FwdEpiT<4> e; fill(e); rc = launch(e); }
            if (rc != ODECOL_OK) return rc;
            cur ^= 1;
        }
    }
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}


// ---------------------------------------------------------------------------------------------------------------
// checkpoint mode (training with a component selection): no (T, B, 3N) trajectory; the forward sweep leaves the V/A
// state and the three V slopes of every step (20 bytes per population, trial and step) and the selected components
// ---------------------------------------------------------------------------------------------------------------
size_t tc_rk4_ckpt_bytes(const DevProblem& p, int T) {
    const tc::TcFwdLayout L = tc::tc_fwd_layout(p);
    if (L.KPa / tc::BK > tc::kChunkMin) return 0;      // checkpoint mode lives in the persistent kernel: see tc_rk4_fwd
    const size_t plane = 4ull * L.Np * L.Bp;
    return plane * (2ull * T + 3ull * (T - 1));
}

int tc_rk4_fwd_ckpt(const DevProblem& p, const float* t_dev, int T, const float* y0, const int* sel, int G, float* y_sel,
                    void* ckpt, size_t ckpt_bytes, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const TcFwdLayout L = tc_fwd_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (L.KPa / BK > kChunkMin) return ODECOL_E_UNSUPPORTED;       // see tc_rk4_ckpt_bytes
    if (!ckpt || ckpt_bytes < tc_rk4_ckpt_bytes(p, T)) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
    float* Rhi[2] = {F(L.off_Rhi[0]), F(L.off_Rhi[1])};
    float* Rlo[2] = {F(L.off_Rlo[0]), F(L.off_Rlo[1])};
    float* KT[3] = {F(L.off_K[0]), F(L.off_K[1]), F(L.off_K[2])};
    float* YT[2] = {F(L.off_Y[0]), F(L.off_Y[1])};
    int* inv = reinterpret_cast<int*>(w + L.off_inv);
    const size_t plane = (size_t)L.Np * L.Bp;
    k_tc_build_inv<<<1, 256, 0, s>>>(sel, G, 3 * p.N, inv);
    k_tc_gather_sel<<<296, 256, 0, s>>>(y0, sel, G, p.B, 3 * p.N, y_sel);
    count_launch(2);
    CkptView ck;
    ck.VA = static_cast<float*>(ckpt); ck.K = ck.VA + 2 * plane * (size_t)T; ck.y_sel = y_sel; ck.inv = inv; ck.G = G;
    const Mixed16 mx = mixed16_view(L, w);
    return tc_rk4_fwd_persistent(p, t_dev, T, y0, nullptr, 1, F(L.off_Whi), F(L.off_Wlo), Rhi, Rlo, KT, YT,
                                 reinterpret_cast<unsigned int*>(w + L.off_done), L.Np, L.Bp, L.KPa, L.TN, &ck, &mx, s);
}

size_t tc_contract_workspace_bytes(int M, int N, int K) { return tc::contract_layout(M, N, K).total; }

int tc_contract(const float* A, const float* B, float* C, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const ContractLayout L = contract_layout(M, N, K);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    char* w = static_cast<char*>(ws);
    float* Ahi = reinterpret_cast<float*>(w + L.off_Ahi); float* Alo = reinterpret_cast<float*>(w + L.off_Alo);
    float* Bhi = reinterpret_cast<float*>(w + L.off_Bhi); float* Blo = reinterpret_cast<float*>(w + L.off_Blo);
    k_split_pad<<<296, 256, 0, s>>>(A, M, K, K, Ahi, Alo, L.Mp, L.Kp);
    k_split_pad<<<296, 256, 0, s>>>(B, N, K, K, Bhi, Blo, L.Np, L.Kp);
    count_launch(2);
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    if (!make_map(&ma_hi, Ahi, L.Mp, L.Kp, L.Kp, BM) || !make_map(&ma_lo, Alo, L.Mp, L.Kp, L.Kp, BM) ||
        !make_map(&mb_hi, Bhi, L.Np, L.Kp, L.Kp, L.TN) || !make_map(&mb_lo, Blo, L.Np, L.Kp, L.Kp, L.TN))
        return ODECOL_E_CUDA;
    const TileShape ts{L.Mp / BM, L.Np / L.TN, L.TN, L.Kp / BK, 0};
    StoreEpi epi{C, M, N, M};
    return launch_contract(ma_hi, ma_lo, mb_hi, mb_lo, ts, epi, s);
}

}  // namespace odecol
