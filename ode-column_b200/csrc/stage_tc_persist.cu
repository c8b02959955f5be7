// Family T, persistent variant: ONE cooperative launch runs the whole rk4 time loop (all steps, all four stages).
//
// Each CTA keeps the (population tile, trial tile) pairs it owns for the entire solve.  Stage q+1 of a trial tile needs
// the operand rows written by the stage-q epilogues of ALL population tiles of that trial tile -- a dependency between
// the 4 CTAs of a group only -- so instead of a kernel boundary per stage the TMA producer waits on a per-trial-tile
// counter in global memory (release/acquire + cross-proxy fence).  Consequences:
//   * the epilogue of (stage q, tile A) overlaps the contraction of (stage q, tile B) AND the contraction of
//     (stage q+1, tile A) overlaps the epilogue of (stage q, tile B): in steady state only the epilogues are exposed;
//   * no per-launch prologue (barrier init, TMEM allocation, descriptor fetch) and no drain/fill bubble between stages;
//   * 6,000 launches per forward solve become one.
// All CTAs must be co-resident (they wait on each other), hence cudaLaunchCooperativeKernel with grid <= #SMs.
#include "stage_tc.cuh"

namespace odecol {
namespace tc {

struct PersistArgs {
    DevProblem p;
    TileGeom tg;
    TileShape ts;
    const float* t;
    int T, out_every, KPa;
    float* y_out;              // (rows, B, 3N)
    float* YT[2];              // tile-major state, ping-pong per step
    float* KT[3];
    float* Rhi[2]; float* Rlo[2];
    uint16_t* R16[2]; size_t r16_plane; int KP16; const float* wscale;     // 16-bit operand format (F16 kernel)
    unsigned int* ovf;         // F16 kernel: raised when an operand value does not fit FP16
    const unsigned int* run_if;  // TF32 kernel launched as the fallback of the F16 kernel: return at once unless *run_if != 0
    unsigned int* done;        // [NT] cumulative count of finished (population-tile) epilogues per trial tile
    CkptView ck;               // ck.VA != NULL: checkpoint mode (V/A state and V slopes per step, selected output)
    float inv_tm, inv_ta, inv_ts;
};

template <int S, bool F16>
ODECOL_DEVINL FwdEpiT<S, F16> persist_epi(const PersistArgs& a, int n, int q) {
    FwdEpiT<S, F16> e;
    e.p = a.p; e.tg = a.tg; e.t = a.t; e.n = n; e.KPa = a.KPa;
    const size_t pl = a.tg.plane();
    const int j = n + 1;
    e.F0T = a.YT[n & 1] + 2 * pl; e.F1T = a.YT[j & 1] + 2 * pl;
    if (a.ck.VA) {
        e.V0T = a.ck.VA + 2 * pl * (size_t)n; e.A0T = e.V0T + pl;
        e.V1T = a.ck.VA + 2 * pl * (size_t)j; e.A1T = e.V1T + pl;
        e.K1T = a.ck.K + 3 * pl * (size_t)n; e.K2T = e.K1T + pl; e.K3T = e.K2T + pl;
        e.traj_row = nullptr;
        e.ysel_row = a.ck.y_sel + (size_t)j * a.p.B * a.ck.G; e.inv = a.ck.inv; e.G = a.ck.G;
    } else {
        e.V0T = a.YT[n & 1]; e.A0T = e.V0T + pl; e.V1T = a.YT[j & 1]; e.A1T = e.V1T + pl;
        e.K1T = a.KT[0]; e.K2T = a.KT[1]; e.K3T = a.KT[2];
        const bool emit = (j % a.out_every == 0) || (j == a.T - 1);
        const size_t r = (j % a.out_every == 0) ? (size_t)(j / a.out_every) : (size_t)((a.T - 2) / a.out_every + 1);
        e.traj_row = emit ? a.y_out + r * ((size_t)a.p.B * 3 * a.p.N) : nullptr;
        e.ysel_row = nullptr; e.inv = nullptr; e.G = 0;
    }
    e.Rhi_nxt = a.Rhi[(q + 1) & 1]; e.Rlo_nxt = a.Rlo[(q + 1) & 1];
    e.R16_nxt = a.R16[(q + 1) & 1]; e.r16_plane = a.r16_plane; e.KP16 = a.KP16; e.wscale = a.wscale; e.ovf = a.ovf;
    e.DRT_nxt = nullptr;
    e.inv_tm = a.inv_tm; e.inv_ta = a.inv_ta; e.inv_ts = a.inv_ts;
    return e;
}

template <int S, bool F16>
ODECOL_DEVINL void persist_epilogue(const PersistArgs& a, int n, int q, int m_tile, int row, int n0, int nt, int g, int TNq,
                                    const float (&tot)[kMaxQ], int etid) {
    FwdEpiT<S, F16> e = persist_epi<S, F16>(a, n, q);
    e.prepare();
    e.rows(m_tile, row, n0, nt, g, TNq, tot);
    e.tile_done(m_tile, n0, a.ts.TN, etid, kEpiWarps * 32);
}

// F16: the 16-bit operand format (stage_tc.cuh): two FP16 planes per operand, K blocks of 64 elements (the same 60 KB ring
// stages cover twice the K), three kind::f16 products per K step, the cross accumulator scaled by 2^-11 on the way out.
template <bool F16>
__global__ void __launch_bounds__(kThreads, 1)
k_tc_rk4_fwd_persistent(const __grid_constant__ CUtensorMap mW_hi, const __grid_constant__ CUtensorMap mW_lo,
                        const __grid_constant__ CUtensorMap mR_hi0, const __grid_constant__ CUtensorMap mR_lo0,
                        const __grid_constant__ CUtensorMap mR_hi1, const __grid_constant__ CUtensorMap mR_lo1,
                        PersistArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 2];
    __shared__ uint32_t tmem_base_slot;
    if (!F16 && a.run_if && *a.run_if == 0u) return;      // fallback launch of a 16-bit solve that met no overflow
    const TileShape ts = a.ts;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
    constexpr int RSTAGES = STAGES;
    constexpr int KEL = F16 ? BK16 : BK;              // operand elements per K block (one 128-byte row either way)
    const uint32_t a_bytes = BM * 128, b_bytes = (uint32_t)ts.TN * 128;
    const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]);
    const uint32_t tfull = smem_u32(&bars[2 * STAGES]), tempty = smem_u32(&bars[2 * STAGES + 1]);
    const int tiles = ts.MT * ts.NT;
    const uint32_t acc_stride = (uint32_t)ts.TN;
    uint32_t ncols = 32;
    while (ncols < (kMainAcc + 1) * acc_stride) ncols <<= 1;
    const int n_seq = 4 * (a.T - 1);                  // stage sequence numbers q = 4 n + (s - 1)

    if (threadIdx.x == 0) {
        for (int s = 0; s < RSTAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, kEpiWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;
    if (kEpiRegs && warp < kEpiWarp0) setmaxnreg_dec<32>();

    if (warp == kTmaWarp) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int q = 0; q < n_seq; ++q) {
                const CUtensorMap* mb_hi = (q & 1) ? &mR_hi1 : &mR_hi0;
                const CUtensorMap* mb_lo = (q & 1) ? &mR_lo1 : &mR_lo0;
                for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                    const int nt = tile / ts.MT, m0 = (tile % ts.MT) * BM, n0 = nt * ts.TN;
                    // operand rows of this trial tile are complete once every population tile finished stage q-1
                    const unsigned int need = (unsigned int)ts.MT * (unsigned int)q;
                    uint32_t spins = 0;
                    while (ld_acquire_u32(a.done + nt) < need) {
                        __nanosleep(64);
                        if (++spins > (1u << 26)) __trap();
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");      // generic-proxy writes -> TMA (async proxy) reads
                    for (int kb = 0; kb < ts.KB; ++kb) {
                        mbar_wait(empty0 + 8 * stage, phase ^ 1);
                        const uint32_t base = ring + stage * stage_bytes, fb = full0 + 8 * stage;
                        mbar_expect_tx(fb, stage_bytes);
                        tma_load_2d(base, &mW_hi, fb, kb * KEL, m0);
                        tma_load_2d(base + a_bytes, &mW_lo, fb, kb * KEL, m0);
                        tma_load_2d(base + 2 * a_bytes, mb_hi, fb, kb * KEL, n0);
                        tma_load_2d(base + 2 * a_bytes + b_bytes, mb_lo, fb, kb * KEL, n0);
                        if (++stage == RSTAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0) {
            const uint32_t idesc = F16 ? make_idesc16(ts.TN) : make_idesc(ts.TN);
            const uint32_t d_small = tmem_base + kMainAcc * acc_stride;
            int stage = 0; uint32_t phase = 0, tphase = 0;
            for (int q = 0; q < n_seq; ++q) {
                for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                    mbar_wait(tempty, tphase ^ 1);
                    tc_fence_after();
                    int j = 0;
                    for (int kb = 0; kb < ts.KB; ++kb) {
                        mbar_wait(full0 + 8 * stage, phase);
                        tc_fence_after();
                        const uint32_t base = ring + stage * stage_bytes;
                        const uint64_t a_hi = make_smem_desc(base), a_lo = make_smem_desc(base + a_bytes);
                        const uint64_t b_hi = make_smem_desc(base + 2 * a_bytes), b_lo = make_smem_desc(base + 2 * a_bytes + b_bytes);
#pragma unroll
                        for (int k = 0; k < 4; ++k, ++j) {             // 32 operand bytes per step: K = 8 (TF32) or 16 (F16)
                            const uint64_t adv = (uint64_t)(k * 32 >> 4);
                            const uint32_t d_main = tmem_base + (uint32_t)(j % kMainAcc) * acc_stride;
                            if (F16) {
                                umma_f16(d_small, a_lo + adv, b_hi + adv, idesc, j != 0);
                                umma_f16(d_small, a_hi + adv, b_lo + adv, idesc, 1);
                                umma_f16(d_main, a_hi + adv, b_hi + adv, idesc, j >= kMainAcc);
                            } else {
                                umma_tf32(d_small, a_lo + adv, b_hi + adv, idesc, j != 0);
                                umma_tf32(d_small, a_hi + adv, b_lo + adv, idesc, 1);
                                umma_tf32(d_main, a_hi + adv, b_hi + adv, idesc, j >= kMainAcc);
                            }
                        }
                        umma_commit(empty0 + 8 * stage);
                        if (++stage == RSTAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(tfull);
                    tphase ^= 1;
                }
            }
        }
    } else if (warp >= kEpiWarp0) {
        if (kEpiRegs) setmaxnreg_inc<(kEpiRegs ? kEpiRegs : 96)>();
        const int ew = warp - kEpiWarp0;
        const int quarter = warp & 3;
        const int g = ew >> 2;
        const int etid = ew * 32 + lane;
        const int TNq = ts.TN >> 2;
        uint32_t tphase = 0;
        for (int q = 0; q < n_seq; ++q) {
            const int n = q >> 2, s = (q & 3) + 1;
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                const int m_tile = tile % ts.MT, nt = tile / ts.MT, n0 = nt * ts.TN;
                const int row = m_tile * BM + quarter * 32 + lane;
                float tot[kMaxQ];
                mbar_wait(tfull, tphase);
                tc_fence_after();
                const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(g * TNq);
#pragma unroll
                for (int qq = 0; qq < kMaxQ / 4; ++qq) {
                    if (4 * qq < TNq) {
                        uint32_t u[kMainAcc + 1][4];
#pragma unroll
                        for (int c = 0; c <= kMainAcc; ++c) tmem_ld4_issue(lane_base + c * acc_stride + 4 * qq, u[c]);
                        tmem_ld_wait();
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float sum = __uint_as_float(u[kMainAcc][e]);
                            if (F16) sum *= 4.8828125e-4f;             // the low planes carry 2^11
#pragma unroll
                            for (int c = 0; c < kMainAcc; ++c) sum += __uint_as_float(u[c][e]);
                            tot[4 * qq + e] = sum;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty);
                tphase ^= 1;
                switch (s) {
                    case 1: persist_epilogue<1, F16>(a, n, q, m_tile, row, n0, nt, g, TNq, tot, etid); break;
                    case 2: persist_epilogue<2, F16>(a, n, q, m_tile, row, n0, nt, g, TNq, tot, etid); break;
                    case 3: persist_epilogue<3, F16>(a, n, q, m_tile, row, n0, nt, g, TNq, tot, etid); break;
                    default: persist_epilogue<4, F16>(a, n, q, m_tile, row, n0, nt, g, TNq, tot, etid); break;
                }
                // publish: all epilogue warps' writes of this tile, then one release increment
                __threadfence();
                asm volatile("bar.sync 1, %0;" ::"r"(kEpiWarps * 32) : "memory");
                if (etid == 0) atomicAdd(a.done + nt, 1u);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

}  // namespace tc

// workspace = the per-stage forward layout plus the dependency counters; reuses tc_fwd_layout's buffers.
// mx != NULL: buffers of the mixed 16-bit operand format (stage_tc.cuh) -- used unless ODECOL_FWD16=0.
int tc_rk4_fwd_persistent(const DevProblem& p, const float* t_dev, int T, const float* y0, float* y_out, int out_every,
                          float* Whi, float* Wlo, float* const Rhi[2], float* const Rlo[2], float* const KT[3],
                          float* const YT[2], unsigned int* done, int Np, int Bp, int KPa, int TN, const tc::CkptView* ck,
                          const tc::Mixed16* mx, cudaStream_t s) {
    using namespace tc;
    const int Kaug = p.N + p.n_in + 1;
    const size_t st = (size_t)p.B * 3 * p.N;
    const TileGeom tg{Bp / TN, Np, TN, TN / 4};
    static const bool fwd16_env = [] { const char* e = getenv("ODECOL_FWD16"); return e ? atoi(e) != 0 : true; }();
    const bool f16 = mx && fwd16_env;
    const TileShape tsh{Np / BM, Bp / TN, TN, f16 ? mx->KP16 / BK16 : KPa / BK, 0};
    const int tiles = tsh.MT * tsh.NT;
    int grid = tiles < num_sms() ? tiles : num_sms();
    // every trial tile's population tiles must be owned by co-resident CTAs: guaranteed by the cooperative launch

    k_split_pad<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, Whi, Wlo, Np, KPa);
    extern void tc_launch_init(const DevProblem&, const TileGeom&, const float*, const float*, float*, float*, float*, float*,
                               float*, float*, float*, int, int, cudaStream_t);
    const size_t pl = tg.plane();
    float* V0 = ck ? ck->VA : YT[0];
    tc_launch_init(p, tg, y0, t_dev, Rhi[0], Rlo[0], Rhi[1], Rlo[1], V0, V0 + pl, YT[0] + 2 * pl, KPa, Bp, s);
    count_launch(2);
    unsigned int* ovf = f16 ? reinterpret_cast<unsigned int*>(mx->wscale + 2) : nullptr;
    if (f16) {
        // weight planes in FP16 (power-of-two scale from max|W_aug|), the initial operand and the constant-one column of
        // both operand buffers re-split into FP16 planes
        unsigned int* amax = reinterpret_cast<unsigned int*>(mx->wscale + 1);
        if (cudaMemsetAsync(amax, 0, 2 * sizeof(unsigned int), s) != cudaSuccess) return ODECOL_E_CUDA;      // amax, ovf
        k_absmax<<<148, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, amax);
        k_split16_w<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, static_cast<__half*>(mx->W16[0]), static_cast<__half*>(mx->W16[1]),
                                        Np, mx->KP16, amax, mx->wscale);
        for (int i = 0; i < 2; ++i) k_r16_from32<<<592, 256, 0, s>>>(Rhi[i], Rlo[i], Bp, KPa, mx->R16[i], mx->KP16, ovf);
        count_launch(4);
    }
    if (cudaMemsetAsync(done, 0, sizeof(unsigned int) * tsh.NT, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (!ck && cudaMemcpyAsync(y_out, y0, sizeof(float) * st, cudaMemcpyDeviceToDevice, s) != cudaSuccess) return ODECOL_E_CUDA;
    CUtensorMap mWhi, mWlo, mR[2][2], m32[6];
    bool ok = make_map(&m32[0], Whi, Np, KPa, KPa, BM) && make_map(&m32[1], Wlo, Np, KPa, KPa, BM);
    for (int i = 0; i < 2; ++i)
        ok = ok && make_map(&m32[2 + 2 * i], Rhi[i], Bp, KPa, KPa, TN) && make_map(&m32[3 + 2 * i], Rlo[i], Bp, KPa, KPa, TN);
    if (f16) {
        const size_t plane = (size_t)Bp * mx->KP16;
        ok = ok && make_map16(&mWhi, mx->W16[0], Np, mx->KP16, mx->KP16, BM, false) && make_map16(&mWlo, mx->W16[1], Np, mx->KP16, mx->KP16, BM, false);
        for (int i = 0; i < 2; ++i)
            for (int c = 0; c < 2; ++c)
                ok = ok && make_map16(&mR[i][c], mx->R16[i] + c * plane, Bp, mx->KP16, mx->KP16, TN, false);
    }
    if (!ok) return ODECOL_E_CUDA;

    PersistArgs a;
    a.p = p; a.tg = tg; a.ts = tsh; a.t = t_dev; a.T = T; a.out_every = out_every; a.KPa = KPa; a.y_out = y_out;
    for (int i = 0; i < 2; ++i) { a.YT[i] = YT[i]; a.Rhi[i] = Rhi[i]; a.Rlo[i] = Rlo[i]; a.R16[i] = f16 ? mx->R16[i] : nullptr; }
    a.r16_plane = f16 ? (size_t)Bp * mx->KP16 : 0; a.KP16 = f16 ? mx->KP16 : 0; a.wscale = f16 ? mx->wscale : nullptr;
    a.ovf = ovf; a.run_if = nullptr;
    for (int i = 0; i < 3; ++i) a.KT[i] = KT[i];
    a.done = done;
    if (ck) a.ck = *ck; else a.ck = CkptView{nullptr, nullptr, nullptr, nullptr, 0};
    a.inv_tm = 1.0f / p.c.tau_m; a.inv_ta = 1.0f / p.c.tau_a; a.inv_ts = 1.0f / p.c.tau_s;
    const size_t smem = (size_t)STAGES * (2 * BM * BK * 4 + 2 * (size_t)TN * BK * 4) + 1024;
    for (int v = 0; v < 2; ++v) {
        const void* kern = v ? (const void*)k_tc_rk4_fwd_persistent<true> : (const void*)k_tc_rk4_fwd_persistent<false>;
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) return ODECOL_E_CUDA;
        int max_blocks = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks, kern, kThreads, smem) != cudaSuccess || max_blocks < 1)
            return ODECOL_E_CUDA;
        if (grid > max_blocks * num_sms()) grid = max_blocks * num_sms();
    }
    if (f16) {
        void* args16[] = {&mWhi, &mWlo, &mR[0][0], &mR[0][1], &mR[1][0], &mR[1][1], &a};
        if (cudaLaunchCooperativeKernel((const void*)k_tc_rk4_fwd_persistent<true>, dim3(grid), dim3(kThreads), args16, smem, s) != cudaSuccess)
            return ODECOL_E_CUDA;
        count_launch();
        // fallback: the same solve in the TF32 format, from the start -- a no-op unless the 16-bit solve raised its flag
        tc_launch_init(p, tg, y0, t_dev, Rhi[0], Rlo[0], Rhi[1], Rlo[1], V0, V0 + pl, YT[0] + 2 * pl, KPa, Bp, s);
        if (cudaMemsetAsync(done, 0, sizeof(unsigned int) * tsh.NT, s) != cudaSuccess) return ODECOL_E_CUDA;
        a.ts.KB = KPa / BK; a.run_if = ovf;
        count_launch();
    }
    void* args[] = {&m32[0], &m32[1], &m32[2], &m32[3], &m32[4], &m32[5], &a};
    if (cudaLaunchCooperativeKernel((const void*)k_tc_rk4_fwd_persistent<false>, dim3(grid), dim3(kThreads), args, smem, s) != cudaSuccess)
        return ODECOL_E_CUDA;
    count_launch();
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

}  // namespace odecol
