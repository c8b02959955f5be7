// Family T reverse sweep: the exact discrete adjoint of the staged RK4 solve with all three contractions on the
// tensor cores (3xTF32, kernels of stage_tc.cuh):
//   recompute  W_aug . r_aug           K-major operands, forward stage epilogue + phi'
//   J^T kbar   W^T . (gamma kbar_V)    K-major operands, reverse stage epilogue (Butcher-tableau transposes of the 3/8 rule)
//   dW_aug    += (gamma kbar_V)^T r_aug  over the four stages and all trials: both operands MN-major (the same buffers
//              the other two contractions read K-major), split over trials, reduced with float atomics
// All per-element bookkeeping lives in tile-major scratch (stage_tc.cuh), float4 along trials.
#include "stage_tc.cuh"

namespace odecol {
namespace tc {

// ---------------------------------------------------------------------------------------------------------------
// reverse stage epilogue.  S = 4, 3, 2, 1: the stage whose Jacobian is applied
// ---------------------------------------------------------------------------------------------------------------
// The F component never feeds back into the dynamics, so its adjoint within a step is a fixed linear chain of lambda_F:
// every stage re-derives its own kbar_F from lambda_F in registers (same expressions a stored version would use) and no
// F plane of kbar / Ybar crosses a stage boundary; kbar_V / kbar_A of stages 4, 3, 2 are re-derived the same way from
// lambda and the stored Ybar.  Bytes per (population, trial): 32 / 40 / 56 / 52 for S = 4, 3, 2, 1.
template <int S>
struct BwdEpiT {
    DevProblem p;
    TileGeom tg;
    const float* t;
    int n, NPk, G;
    float* acurT;          // [2 planes: V, A] kbar of stage 1, written by stage 2 (the other stages re-derive theirs)
    float* lamT;           // [3 planes]
    float* b4T;            // [2 planes] Ybar_4, later Ybar_4 + Ybar_3 + Ybar_2
    float* b3T;            // [2 planes]
    const float* DRT;      // [1 plane] phi'(x_s)
    float* AVhi_nxt; float* AVlo_nxt;   // [Bp][NPk] operand of the next reverse stage (and of dW)
    const float* grad_y;   // (T, B, G)
    const int* inv;        // [3N]
    float gamma, inv_tm, inv_ta, inv_ts;
    float dt, h8p;
    const float* gy_step;  // row n of grad_y
    int needF;             // 0: no F component carries a loss gradient -> lambda_F is identically zero, its plane is never touched

    ODECOL_DEVINL void prepare() {
        dt = __fsub_rn(__ldg(t + n + 1), __ldg(t + n));
        h8p = n > 0 ? __fsub_rn(__ldg(t + n), __ldg(t + n - 1)) * 0.125f : 0.f;
        needF = __ldg(inv + 3 * p.N);
        gy_step = grad_y + (size_t)n * p.B * G;
    }

    struct Group { float4 aV, aA, dr, lV, lA, lF, p4V, p4A, p3V, p3A, gv, ga, gf; };
    ODECOL_DEVINL void load_group(Group& L, size_t oq, size_t pl, int b0, int gV, int gA, int gF) const {
        L.dr = ld4s(DRT + oq);
        L.lV = ld4s(lamT + oq); L.lA = ld4s(lamT + pl + oq);
        L.lF = needF ? ld4s(lamT + 2 * pl + oq) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (S == 1) { L.aV = ld4s(acurT + oq); L.aA = ld4s(acurT + pl + oq); }
        if (S <= 3) { L.p4V = ld4s(b4T + oq); L.p4A = ld4s(b4T + pl + oq); }
        if (S == 2) { L.p3V = ld4s(b3T + oq); L.p3A = ld4s(b3T + pl + oq); }
        if (S == 1) {                       // loss gradient of the selected components at grid point n: predicated loads off
            const float* gy = gy_step + (size_t)b0 * G;      // one row address (most populations select nothing)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const bool ok = b0 + e < p.B;
                (&L.gv.x)[e] = ldg_if(gy + gV, ok && gV >= 0);
                (&L.ga.x)[e] = ldg_if(gy + gA, ok && gA >= 0);
                (&L.gf.x)[e] = ldg_if(gy + gF, ok && gF >= 0);
                gy += G;
            }
        }
    }
    // rolled, software-pipelined group loop (see FwdEpiT::rows)
    ODECOL_DEVINL void rows(int, int j, int n0, int nt, int g, int TNq, const float (&graw)[kMaxQ]) const {
        if (j >= p.N) return;
        const int N = p.N, B = p.B;
        const float kap = __ldg(p.kappa + j);
        const size_t pl = tg.plane();
        const float h8 = dt * 0.125f, h38 = 3.0f * h8, h3 = dt * kOneThirdL;
        int gV = -1, gA = -1, gF = -1;
        if (S == 1) { gV = inv[j]; gA = inv[N + j]; gF = inv[2 * N + j]; }
        const int nq = TNq >> 2;
        const size_t qstride = (size_t)tg.Np * 4;
        const size_t o0 = tg.off(nt, g, 0, j);
        const int bg = n0 + g * TNq;
        Group nxt;
        load_group(nxt, o0, pl, bg, gV, gA, gF);
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
            const size_t oq = o0 + q * qstride;
            const Group L = nxt;
            if (q + 1 < nq) load_group(nxt, oq + qstride, pl, bg + 4 * (q + 1), gV, gA, gF);
            float nV[4], nA[4], sV[4], sA[4], sF[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float d = (&L.dr.x)[e];
                const float lv = (&L.lV.x)[e], la = (&L.lA.x)[e], lf = (&L.lF.x)[e];
                // kbar_V, kbar_A of this stage: the expression the previous reverse stage fed to its operand, re-derived
                // from lambda and the stored Ybar (stage 1 reads what stage 2 stored: it only keeps the sum of Ybar)
                float av, aa;
                if (S == 4) { av = h8 * lv; aa = h8 * la; }
                if (S == 3) { av = h38 * lv + dt * (&L.p4V.x)[e]; aa = h38 * la + dt * (&L.p4A.x)[e]; }
                if (S == 2) {
                    av = h38 * lv - dt * (&L.p4V.x)[e] + dt * (&L.p3V.x)[e];
                    aa = h38 * la - dt * (&L.p4A.x)[e] + dt * (&L.p3A.x)[e];
                }
                if (S == 1) { av = (&L.aV.x)[e]; aa = (&L.aA.x)[e]; }
                // kbar_F of this stage (and, at stage 1, the sum of the F slopes' adjoints) from lambda_F
                const float bF4 = -(h8 * lf) * inv_ts;
                float af = h8 * lf, bF3 = 0.f, bF2 = 0.f;
                if (S <= 3) { af = h38 * lf + dt * bF4; bF3 = -af * inv_ts; }
                if (S <= 2) { af = h38 * lf - dt * bF4 + dt * bF3; bF2 = -af * inv_ts; }
                if (S == 1) { af = h8 * lf + dt * bF4 - h3 * bF3 + h3 * bF2; }
                const float gg = graw[4 * q + e] + kap * aa * inv_ta + af * inv_ts;
                const float bV = -av * inv_tm + d * gg;
                const float bA = -aa * inv_ta - d * gg;
                if (S == 4) {
                    sV[e] = bV; sA[e] = bA;
                    nV[e] = h38 * lv + dt * bV; nA[e] = h38 * la + dt * bA;
                }
                if (S == 3) {
                    sV[e] = bV; sA[e] = bA;
                    nV[e] = h38 * lv - dt * (&L.p4V.x)[e] + dt * bV;
                    nA[e] = h38 * la - dt * (&L.p4A.x)[e] + dt * bA;
                }
                if (S == 2) {
                    nV[e] = h8 * lv + dt * (&L.p4V.x)[e] - h3 * (&L.p3V.x)[e] + h3 * bV;
                    nA[e] = h8 * la + dt * (&L.p4A.x)[e] - h3 * (&L.p3A.x)[e] + h3 * bA;
                    sV[e] = (&L.p4V.x)[e] + (&L.p3V.x)[e] + bV; sA[e] = (&L.p4A.x)[e] + (&L.p3A.x)[e] + bA;
                }
                if (S == 1) {
                    const float bF1 = -af * inv_ts;
                    const float LV = lv + (&L.p4V.x)[e] + bV + (&L.gv.x)[e];
                    const float LA = la + (&L.p4A.x)[e] + bA + (&L.ga.x)[e];
                    const float LF = lf + (bF4 + bF3 + bF2) + bF1 + (&L.gf.x)[e];
                    sV[e] = LV; sA[e] = LA; sF[e] = LF;
                    nV[e] = h8p * LV; nA[e] = h8p * LA;
                }
            }
            float* sdst = S == 4 ? b4T : S == 3 ? b3T : S == 2 ? b4T : lamT;
            st4s(sdst + oq, make_float4(sV[0], sV[1], sV[2], sV[3]));
            st4s(sdst + pl + oq, make_float4(sA[0], sA[1], sA[2], sA[3]));
            if (S == 1 && needF) st4s(lamT + 2 * pl + oq, make_float4(sF[0], sF[1], sF[2], sF[3]));
            if (S == 2) {
                st4s(acurT + oq, make_float4(nV[0], nV[1], nV[2], nV[3]));
                st4s(acurT + pl + oq, make_float4(nA[0], nA[1], nA[2], nA[3]));
            }
            const int b0 = bg + 4 * q;
            float* ah = AVhi_nxt + (size_t)b0 * NPk + j;       // one row address per group, predicated stores (FwdEpiT::rows)
            const ptrdiff_t lo_off = AVlo_nxt - AVhi_nxt;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float v = gamma * nV[e];
                const float h = tf32_rna(v);
                float* ph = ah + (size_t)e * NPk;
                st_global_if(ph, h, b0 + e < B);
                st_global_if(ph + lo_off, tf32_rna(v - h), b0 + e < B);
            }
        }
    }
    ODECOL_DEVINL void tile_done(int, int, int, int, int) const {}
};

// ---------------------------------------------------------------------------------------------------------------
// The four reverse stages of one step (S = 4, 3, 2, 1) in ONE cooperative launch: same structure as the persistent
// forward kernel (stage_tc_persist.cu).  Stage S reads operand slot S-1 of the current operand set and writes slot
// S-2; stage 1 writes kbar_4 of the NEXT reverse step into slot 3 of the other set, so the dW contraction of this step
// (which reads all four slots of the current set) can run after the chain.  A trial tile's next contraction waits on
// a per-trial-tile counter of finished population-tile epilogues (cumulative over launches: `done_base`).
// ---------------------------------------------------------------------------------------------------------------
// (the dW contraction's shape and MN-major descriptor are defined further down, next to the stand-alone k_tc_dw; the
// chain kernel can run the dW contraction of its step as a fifth phase, see k_tc_bwd_chain)
constexpr int DW_BK = 32;        // rows (trials) per K block = four 8-row swizzle atoms
constexpr int DW_T = 128;        // output tile: 128 x 128
struct DwShape { int MT, NT, Z, rows_per_split, total_rows, N, Kaug, ld_w; float* grad_W; uint32_t lbo, sbo, major_bits, kadv;
                 float* partial; };             // [Z][N][ld_w] or NULL: row split z accumulates into its OWN copy with plain
                                          // read-modify-writes (one CTA per (tile, z) and launch, launches stream-ordered), summed
                                          // over z in a fixed order at the end of the sweep -- bit-reproducible, no float atomics
ODECOL_DEVINL uint64_t make_smem_desc_mn(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo >> 4) << 16;                  // leading byte offset: next 32-wide block along M/N
    d |= (uint64_t)(sbo >> 4) << 32;                  // stride byte offset: next 8-row group along K
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                           // SWIZZLE_128B_BASE32B: the only MN-major layout for 32-bit operands
    return d;
}

struct BwdChainArgs {
    DevProblem p;
    TileGeom tg;
    TileShape ts;              // MT, NT, TN, KB = NPk / BK
    const float* t;
    int n, NPk, G, Bp;
    float* acurT; float* lamT; float* b4T; float* b3T;
    const float* DRT[4];
    float* AVhi; float* AVlo;  // [2 sets][4 slots][Bp][NPk]
    int set;                   // operand set of this step
    const float* grad_y; const int* inv;
    float gamma, inv_tm, inv_ta, inv_ts;
    unsigned int* done; unsigned int done_base;
    DwShape ds;                // FUSE_DW: the dW contraction of this step, run as a fifth phase (maps dA_* / dB_*)
};

template <int S>
ODECOL_DEVINL void chain_epilogue(const BwdChainArgs& a, int m_tile, int row, int n0, int nt, int g, int TNq,
                                  const float (&tot)[kMaxQ]) {
    BwdEpiT<S> e;
    e.p = a.p; e.tg = a.tg; e.t = a.t; e.n = a.n; e.NPk = a.NPk; e.G = a.G;
    e.acurT = a.acurT; e.lamT = a.lamT; e.b4T = a.b4T; e.b3T = a.b3T; e.DRT = a.DRT[S - 1];
    const size_t astride = (size_t)a.Bp * a.NPk;
    const size_t nxt = S == 1 ? (size_t)((a.set ^ 1) * 4 + 3) : (size_t)(a.set * 4 + S - 2);
    e.AVhi_nxt = a.AVhi + nxt * astride; e.AVlo_nxt = a.AVlo + nxt * astride;
    e.grad_y = a.grad_y; e.inv = a.inv; e.gamma = a.gamma;
    e.inv_tm = a.inv_tm; e.inv_ta = a.inv_ta; e.inv_ts = a.inv_ts;
    e.prepare();
    e.rows(m_tile, row, n0, nt, g, TNq, tot);
}

template <bool FUSE_DW>
__global__ void __launch_bounds__(kThreads, 1)
k_tc_bwd_chain(const __grid_constant__ CUtensorMap mW_hi, const __grid_constant__ CUtensorMap mW_lo,
               const __grid_constant__ CUtensorMap mA_hi, const __grid_constant__ CUtensorMap mA_lo,
               const __grid_constant__ CUtensorMap dA_hi, const __grid_constant__ CUtensorMap dA_lo,
               const __grid_constant__ CUtensorMap dB_hi, const __grid_constant__ CUtensorMap dB_lo, BwdChainArgs a) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 2];
    __shared__ uint32_t tmem_base_slot;
    const TileShape ts = a.ts;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_bytes = BM * BK * 4, b_bytes = (uint32_t)ts.TN * BK * 4;
    const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]);
    const uint32_t tfull = smem_u32(&bars[2 * STAGES]), tempty = smem_u32(&bars[2 * STAGES + 1]);
    const int tiles = ts.MT * ts.NT;
    const uint32_t acc_stride = (uint32_t)ts.TN;
    uint32_t ncols = 32;
    while (ncols < (kMainAcc + 1) * acc_stride) ncols <<= 1;
    if (FUSE_DW) ncols = 512;                                 // the dW phase uses (kMainAcc + 1) x 128 accumulator columns
    // Fifth phase (fuse_dw): the dW contraction of this step, work item = (output tile, row split) as in k_tc_dw.  Its
    // operands are complete long before the chain ends -- slot 3 was written by the previous step, slots 2 / 1 / 0 by the
    // epilogues of stages 4 / 3 / 2 of this step -- so the MMA warp contracts dW while the stage-1 epilogues still
    // stream their bookkeeping through HBM, and the step needs one launch instead of two.
    const DwShape& ds = a.ds;
    const int dw_tiles = ds.MT * ds.NT, dw_items = FUSE_DW ? dw_tiles * ds.Z : 0;
    constexpr uint32_t dw_box = DW_BK * 128, dw_op = 4 * dw_box, dw_stage = 4 * dw_op;
    // both phases address the ring with the same stage stride, so that a ring slot means the same bytes before and after
    // the transition (the `empty` barrier of slot s then covers exactly the bytes the next load overwrites)
    const uint32_t stride = FUSE_DW ? (stage_bytes > dw_stage ? stage_bytes : dw_stage) : stage_bytes;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
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
            for (int q = 0; q < 4; ++q) {                       // q = 0..3  <->  S = 4..1, operand slot 3 - q
                const int row0 = (a.set * 4 + 3 - q) * a.Bp;
                for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                    const int nt = tile / ts.MT, m0 = (tile % ts.MT) * BM, n0 = nt * ts.TN;
                    const unsigned int need = a.done_base + (unsigned int)ts.MT * (unsigned int)q;
                    uint32_t spins = 0;
                    while ((int)(ld_acquire_u32(a.done + nt) - need) < 0) {
                        __nanosleep(64);
                        if (++spins > (1u << 26)) __trap();
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");
                    for (int kb = 0; kb < ts.KB; ++kb) {
                        mbar_wait(empty0 + 8 * stage, phase ^ 1);
                        const uint32_t base = ring + stage * stride, fb = full0 + 8 * stage;
                        mbar_expect_tx(fb, stage_bytes);
                        tma_load_2d(base, &mW_hi, fb, kb * BK, m0);
                        tma_load_2d(base + a_bytes, &mW_lo, fb, kb * BK, m0);
                        tma_load_2d(base + 2 * a_bytes, &mA_hi, fb, kb * BK, n0 + row0);
                        tma_load_2d(base + 2 * a_bytes + b_bytes, &mA_lo, fb, kb * BK, n0 + row0);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
            // ---- dW phase: rows = stacked (operand slot, trial) of this step's operand set
            for (int item = blockIdx.x; item < dw_items; item += gridDim.x) {
                const int tile = item % dw_tiles, z = ds.Z - 1 - item / dw_tiles;   // last rows (slots 3, 2: ready first) first
                const int i0 = (tile % ds.MT) * DW_T, k0 = (tile / ds.MT) * DW_T;
                const int r0 = z * ds.rows_per_split;
                int r1 = r0 + ds.rows_per_split;
                if (r1 > ds.total_rows) r1 = ds.total_rows;
                const int KBd = (r1 - r0) / DW_BK;
                // rows of slot s < 3 are written by the epilogues of stage s + 2 of this step (q = 2 - s): wait once, up
                // front, for every trial tile the item's rows touch
                for (int slot = r0 / a.Bp; slot <= (r1 - 1) / a.Bp && slot < 3 && KBd > 0; ++slot) {
                    const int lo = (r0 > slot * a.Bp ? r0 - slot * a.Bp : 0) / ts.TN;
                    const int hi = ((r1 < (slot + 1) * a.Bp ? r1 - slot * a.Bp : a.Bp) - 1) / ts.TN;
                    const unsigned int need = a.done_base + (unsigned int)ts.MT * (unsigned int)(3 - slot);
                    for (int nt = lo; nt <= hi; ++nt) {
                        uint32_t spins = 0;
                        while ((int)(ld_acquire_u32(a.done + nt) - need) < 0) {
                            __nanosleep(64);
                            if (++spins > (1u << 26)) __trap();
                        }
                    }
                }
                asm volatile("fence.proxy.async;" ::: "memory");
                for (int kb = 0; kb < KBd; ++kb) {
                    const int row = r0 + kb * DW_BK;
                    mbar_wait(empty0 + 8 * stage, phase ^ 1);
                    const uint32_t base = ring + stage * stride, fb = full0 + 8 * stage;
                    mbar_expect_tx(fb, dw_stage);
#pragma unroll
                    for (int m = 0; m < 4; ++m) {                     // dA_* are the maps of this step's operand set
                        tma_load_2d(base + m * dw_box, &dA_hi, fb, i0 + 32 * m, row);
                        tma_load_2d(base + dw_op + m * dw_box, &dA_lo, fb, i0 + 32 * m, row);
                        tma_load_2d(base + 2 * dw_op + m * dw_box, &dB_hi, fb, k0 + 32 * m, row);
                        tma_load_2d(base + 3 * dw_op + m * dw_box, &dB_lo, fb, k0 + 32 * m, row);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(ts.TN);
            const uint32_t d_small = tmem_base + kMainAcc * acc_stride;
            int stage = 0; uint32_t phase = 0, tphase = 0;
            for (int q = 0; q < 4; ++q) {
                for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                    mbar_wait(tempty, tphase ^ 1);
                    tc_fence_after();
                    int j = 0;
                    for (int kb = 0; kb < ts.KB; ++kb) {
                        mbar_wait(full0 + 8 * stage, phase);
                        tc_fence_after();
                        const uint32_t base = ring + stage * stride;
                        const uint64_t a_hi = make_smem_desc(base), a_lo = make_smem_desc(base + a_bytes);
                        const uint64_t b_hi = make_smem_desc(base + 2 * a_bytes), b_lo = make_smem_desc(base + 2 * a_bytes + b_bytes);
#pragma unroll
                        for (int k = 0; k < BK / 8; ++k, ++j) {
                            const uint64_t adv = (uint64_t)(k * 32 >> 4);
                            umma_tf32(d_small, a_lo + adv, b_hi + adv, idesc, j != 0);
                            umma_tf32(d_small, a_hi + adv, b_lo + adv, idesc, 1);
                            umma_tf32(tmem_base + (uint32_t)(j % kMainAcc) * acc_stride, a_hi + adv, b_hi + adv, idesc, j >= kMainAcc);
                        }
                        umma_commit(empty0 + 8 * stage);
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(tfull);
                    tphase ^= 1;
                }
            }
            // ---- dW phase: both operands MN-major, 128 x 128 accumulators
            const uint32_t idesc_dw = (1u << 4) | (2u << 7) | (2u << 10) | ds.major_bits |
                                      ((uint32_t)(DW_T >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t d_small_dw = tmem_base + kMainAcc * DW_T;
            for (int item = blockIdx.x; item < dw_items; item += gridDim.x) {
                const int z = ds.Z - 1 - item / dw_tiles;
                const int r0 = z * ds.rows_per_split;
                int r1 = r0 + ds.rows_per_split;
                if (r1 > ds.total_rows) r1 = ds.total_rows;
                const int KBd = (r1 - r0) / DW_BK;
                mbar_wait(tempty, tphase ^ 1);
                tc_fence_after();
                int j = 0;
                for (int kb = 0; kb < KBd; ++kb) {
                    mbar_wait(full0 + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t base = ring + stage * stride;
                    const uint64_t a_hi = make_smem_desc_mn(base, ds.lbo, ds.sbo), a_lo = make_smem_desc_mn(base + dw_op, ds.lbo, ds.sbo);
                    const uint64_t b_hi = make_smem_desc_mn(base + 2 * dw_op, ds.lbo, ds.sbo), b_lo = make_smem_desc_mn(base + 3 * dw_op, ds.lbo, ds.sbo);
#pragma unroll
                    for (int k = 0; k < DW_BK / 8; ++k, ++j) {
                        const uint64_t adv = (uint64_t)((k * ds.kadv) >> 4);
                        umma_tf32(d_small_dw, a_lo + adv, b_hi + adv, idesc_dw, j != 0);
                        umma_tf32(d_small_dw, a_hi + adv, b_lo + adv, idesc_dw, 1);
                        umma_tf32(tmem_base + (uint32_t)(j % kMainAcc) * DW_T, a_hi + adv, b_hi + adv, idesc_dw, j >= kMainAcc);
                    }
                    umma_commit(empty0 + 8 * stage);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(tfull);
                tphase ^= 1;
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
        for (int q = 0; q < 4; ++q) {
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
                switch (q) {
                    case 0: chain_epilogue<4>(a, m_tile, row, n0, nt, g, TNq, tot); break;
                    case 1: chain_epilogue<3>(a, m_tile, row, n0, nt, g, TNq, tot); break;
                    case 2: chain_epilogue<2>(a, m_tile, row, n0, nt, g, TNq, tot); break;
                    default: chain_epilogue<1>(a, m_tile, row, n0, nt, g, TNq, tot); break;
                }
                __threadfence();
                asm volatile("bar.sync 1, %0;" ::"r"(kEpiWarps * 32) : "memory");
                if (etid == 0) atomicAdd(a.done + nt, 1u);
            }
        }
        // ---- dW phase: accumulate the finished 128 x 128 tile into grad_W (float atomics), as k_tc_dw does
        for (int item = blockIdx.x; item < dw_items; item += gridDim.x) {
            const int tile = item % dw_tiles, z = ds.Z - 1 - item / dw_tiles;   // last rows (slots 3, 2: ready first) first
            const int i0 = (tile % ds.MT) * DW_T, k0 = (tile / ds.MT) * DW_T;
            const int r0 = z * ds.rows_per_split;
            int r1 = r0 + ds.rows_per_split;
            if (r1 > ds.total_rows) r1 = ds.total_rows;
            const bool any = (r1 - r0) / DW_BK > 0;
            const int i = i0 + quarter * 32 + lane;
            mbar_wait(tfull, tphase);
            tc_fence_after();
            const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(g * 32);
#pragma unroll
            for (int qq = 0; qq < 8; ++qq) {
                uint32_t u[kMainAcc + 1][4];
#pragma unroll
                for (int c = 0; c <= kMainAcc; ++c) tmem_ld4_issue(lane_base + c * DW_T + 4 * qq, u[c]);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    float sum = __uint_as_float(u[kMainAcc][e]);
#pragma unroll
                    for (int c = 0; c < kMainAcc; ++c) sum += __uint_as_float(u[c][e]);
                    const int k = k0 + g * 32 + 4 * qq + e;
                    if (any && i < ds.N && k < ds.Kaug) atomicAdd(ds.grad_W + (size_t)i * ds.ld_w + k, sum);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
            tphase ^= 1;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// per-step operand setup: y_traj[n] (API layout) -> tile-major Y0T, phi' of stage 1, split operand with stimulus
// One CTA per group of four trials (one float4 of the tile-major layout), threads over populations.
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_tc_step_begin(DevProblem p, TileGeom tg, const float* __restrict__ y, const float* __restrict__ t_ptr,
                                float* __restrict__ hi0, float* __restrict__ lo0, float* __restrict__ Y0T,
                                float* __restrict__ DRT, int KPa) {
    const int b4 = blockIdx.x * 4, N = p.N;
    const int nt = b4 / tg.TN, g = (b4 % tg.TN) / tg.TNq, q = ((b4 % tg.TN) % tg.TNq) >> 2;
    const size_t pl = tg.plane();
    for (int i = threadIdx.x; i < tg.Np; i += blockDim.x) {
        float V[4], A[4], F[4], R[4], D[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int b = b4 + e;
            const bool in = i < N && b < p.B;
            const float* yb = y + (size_t)b * 3 * N;
            V[e] = in ? yb[i] : 0.f; A[e] = in ? yb[N + i] : 0.f; F[e] = in ? yb[2 * N + i] : 0.f;
            R[e] = 0.f; D[e] = 0.f;
            if (in) {
                phi_dphi_fast(V[e] - A[e], R[e], D[e]);
                const float h = tf32_rna(R[e]);
                hi0[(size_t)b * KPa + i] = h;
                lo0[(size_t)b * KPa + i] = tf32_rna(R[e] - h);
            }
        }
        const size_t o = tg.off(nt, g, q, i);
        st4(Y0T + o, make_float4(V[0], V[1], V[2], V[3]));
        st4(Y0T + pl + o, make_float4(A[0], A[1], A[2], A[3]));
        st4(Y0T + 2 * pl + o, make_float4(F[0], F[1], F[2], F[3]));
        if (DRT) st4(DRT + o, make_float4(D[0], D[1], D[2], D[3]));
    }
    // stimulus channels, constant-one column
    int idx = 1;
    const float tcl = knot_locate(p.knot_t, p.K, __ldg(t_ptr), idx);
    for (int e = threadIdx.x; e < 4 * (p.n_in + 1); e += blockDim.x) {
        const int b = b4 + e / (p.n_in + 1), ch = e % (p.n_in + 1);
        if (b >= p.B) continue;
        float v = 1.0f;
        if (ch < p.n_in) v = knot_value(p.knot_t, p.knot_u + (size_t)b * p.knot_stride_b, p.n_in, idx, tcl, ch);
        const float h = tf32_rna(v);
        hi0[(size_t)b * KPa + N + ch] = h;
        lo0[(size_t)b * KPa + N + ch] = tf32_rna(v - h);
    }
}

// checkpoint mode: every stage operand and phi' of step n from the saved V/A state and V slopes -- the forward stage
// recurrences of FwdEpiT, elementwise, no contraction.  Work unit = (group of four trials, slice of 128 populations), done by
// 128 threads; one CTA walks all slices of one trial group.
struct ReplayJob {
    DevProblem p; TileGeom tg;
    const float* VA; const float* KV; const float* t;
    int n, KPa, slices;                      // step, operand row length, population slices (Np / 128)
    float* Rhi; float* Rlo; size_t rstride;  // the four stacked operand buffers
    float* D[4];                             // the four phi' planes
};

ODECOL_DEVINL void replay_unit(const ReplayJob& j, int blk, int slice, int tid) {
    const DevProblem& p = j.p;
    const TileGeom& tg = j.tg;
    const int b4 = blk * 4, N = p.N;
    const float t0 = __ldg(j.t + j.n), t1 = __ldg(j.t + j.n + 1), dt = __fsub_rn(t1, t0);
    const float third = kOneThirdL, inv_ta = 1.0f / p.c.tau_a;
    const int i = slice * 128 + tid;
    if (i < N) {
        const size_t o = tg.off(b4 / tg.TN, (b4 % tg.TN) / tg.TNq, ((b4 % tg.TN) % tg.TNq) >> 2, i), pl = tg.plane();
        const float4 V0 = ld4s(j.VA + o), A0 = ld4s(j.VA + pl + o);
        const float4 k1V = ld4s(j.KV + o), k2V = ld4s(j.KV + pl + o), k3V = ld4s(j.KV + 2 * pl + o);
        const float kap = __ldg(p.kappa + i);
        float R[4][4], D[4][4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float v0 = (&V0.x)[e], a0 = (&A0.x)[e];
            phi_dphi_fast(v0 - a0, R[0][e], D[0][e]);
            const float k1A = (kap * R[0][e] - a0) * inv_ta;
            float nV = v0 + dt * (&k1V.x)[e] * third, nA = a0 + dt * k1A * third;
            phi_dphi_fast(nV - nA, R[1][e], D[1][e]);
            const float k2A = (kap * R[1][e] - nA) * inv_ta;
            nV = v0 + dt * ((&k2V.x)[e] - (&k1V.x)[e] * third); nA = a0 + dt * (k2A - k1A * third);
            phi_dphi_fast(nV - nA, R[2][e], D[2][e]);
            const float k3A = (kap * R[2][e] - nA) * inv_ta;
            nV = v0 + dt * ((&k1V.x)[e] - (&k2V.x)[e] + (&k3V.x)[e]); nA = a0 + dt * (k1A - k2A + k3A);
            phi_dphi_fast(nV - nA, R[3][e], D[3][e]);
        }
#pragma unroll
        for (int s = 0; s < 4; ++s) st4s(j.D[s] + o, make_float4(D[s][0], D[s][1], D[s][2], D[s][3]));
        float* rh = j.Rhi + (size_t)b4 * j.KPa + i;               // one row address per unit, predicated stores
        const ptrdiff_t lo_off = j.Rlo - j.Rhi;
#pragma unroll
        for (int s = 0; s < 4; ++s)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float h = tf32_rna(R[s][e]);
                float* ph = rh + s * j.rstride + (size_t)e * j.KPa;
                st_global_if(ph, h, b4 + e < p.B);
                st_global_if(ph + lo_off, tf32_rna(R[s][e] - h), b4 + e < p.B);
            }
    }
    if (slice != 0) return;
    // stimulus channels at the four stage times (the constant-one column is set once per sweep): warp s of the unit's four
    // warps writes the columns of stage s (one knot lookup per warp, four channels per lane and trip)
    if (p.n_in == 0) return;
    const int s = tid >> 5;
    const float ts = s == 0 ? t0 : s == 1 ? __fadd_rn(t0, __fmul_rn(dt, kOneThirdL)) : s == 2 ? __fadd_rn(t0, __fmul_rn(dt, kTwoThirdsL)) : t1;
    int idx = 1;
    const float tcl = knot_locate(p.knot_t, p.K, ts, idx);
    stimulus_columns(p, j.KPa, idx, tcl, b4, 4, 0, 1, tid & 31, 32, j.Rhi + s * j.rstride, j.Rlo + s * j.rstride);
}

// one CTA of 128 threads per group of four trials
__global__ void __launch_bounds__(128, 8) k_tc_replay(ReplayJob j) {
    for (int slice = 0; slice < j.slices; ++slice) replay_unit(j, blockIdx.x, slice, threadIdx.x);
}

// lam = dL/dy_out[T-1] (tile-major), kbar_4 of the last step, its operand
__global__ void k_tc_bwd_begin(DevProblem p, TileGeom tg, const float* __restrict__ grad_y, const int* __restrict__ inv,
                               int G, const float* __restrict__ t, int T, float gamma, float* __restrict__ lamT,
                               float* __restrict__ acurT, float* __restrict__ AVhi, float* __restrict__ AVlo, int NPk) {
    const int b4 = blockIdx.x * 4, N = p.N;
    const int nt = b4 / tg.TN, g = (b4 % tg.TN) / tg.TNq, q = ((b4 % tg.TN) % tg.TNq) >> 2;
    const size_t pl = tg.plane();
    const float h8 = __fsub_rn(__ldg(t + T - 1), __ldg(t + T - 2)) * 0.125f;
    for (int i = threadIdx.x; i < tg.Np; i += blockDim.x) {
        float L[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int b = b4 + e;
                float v = 0.f;
                if (i < N && b < p.B) {
                    const int gi = inv[c * N + i];
                    if (gi >= 0) v = grad_y[((size_t)(T - 1) * p.B + b) * G + gi];
                }
                L[c][e] = v;
            }
        const size_t o = tg.off(nt, g, q, i);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            st4(lamT + c * pl + o, make_float4(L[c][0], L[c][1], L[c][2], L[c][3]));
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int b = b4 + e;
            if (i < N && b < p.B) {
                const float v = gamma * h8 * L[0][e];
                const float h = tf32_rna(v);
                AVhi[(size_t)b * NPk + i] = h;
                AVlo[(size_t)b * NPk + i] = tf32_rna(v - h);
            }
        }
    }
}

// grad_y0 (API layout) from the tile-major adjoint
__global__ void k_tc_untile(DevProblem p, TileGeom tg, const float* __restrict__ srcT, float* __restrict__ dst) {
    const int b4 = blockIdx.x * 4, N = p.N;
    const int nt = b4 / tg.TN, g = (b4 % tg.TN) / tg.TNq, q = ((b4 % tg.TN) % tg.TNq) >> 2;
    const size_t pl = tg.plane();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const size_t o = tg.off(nt, g, q, i);
        for (int c = 0; c < 3; ++c) {
            const float4 v = ld4(srcT + c * pl + o);
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (b4 + e < p.B) dst[(size_t)(b4 + e) * 3 * N + c * N + i] = (&v.x)[e];
        }
    }
}

// constant-one column (the bias input) of the four stacked operand buffers
__global__ void k_tc_set_one(float* __restrict__ Rhi, int Bp, int B, int KPa, int col, int nslots) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nslots * B) return;
    const int s = e / B, b = e % B;
    Rhi[((size_t)s * Bp + b) * KPa + col] = 1.0f;
}


// ---------------------------------------------------------------------------------------------------------------
// dW contraction: C[i][k] += sum_rows A[row][i] * B[row][k], rows = stacked (stage, trial); both operands MN-major.
// For 32-bit operands the tensor core reads MN-major tiles only in the "128-byte swizzle with 32-byte atoms" layout:
// TMA boxes of 32 rows x 32 floats with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; in the descriptor a K atom is 4 rows
// (512 bytes, the stride byte offset), the next 32-wide block along M/N is one box further (leading byte offset),
// and one tcgen05.mma (K = 8) consumes two atoms, i.e. 1024 bytes.
// Same warp roles as k_tc_contract; one output tile and one slice of the rows per CTA; epilogue = float atomics.
// ---------------------------------------------------------------------------------------------------------------

// Accumulation is CHUNKED: the tensor core truncates every accumulation into TMEM (round toward zero), which shrinks a
// long sum of mostly same-signed terms by ~5e-8 per accumulation (measured on dW_aug of the C4 workload: -3e-6 with three
// rotating accumulators over 1504 rows, -1e-5 over 4736 rows).  So an accumulator only ever sees DW_CHUNK K blocks
// (32 MMA steps): the epilogue warps drain it into FP32 round-to-nearest registers and the MMA warp carries on in the
// second of two TMEM accumulator sets (main + cross terms, 2 x 256 columns) -- which makes the bias independent of the
// rows per work item, so one wave of long items (a third of the float atomics of the former three waves) is accurate.
#ifndef ODECOL_DW_CHUNK
#define ODECOL_DW_CHUNK 8
#endif
constexpr int DW_CHUNK = ODECOL_DW_CHUNK;

__global__ void __launch_bounds__(kThreads, 1)
k_tc_dw(const __grid_constant__ CUtensorMap mA_hi, const __grid_constant__ CUtensorMap mA_lo,
        const __grid_constant__ CUtensorMap mB_hi, const __grid_constant__ CUtensorMap mB_lo, DwShape ds) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 4];
    __shared__ uint32_t tmem_base_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
    constexpr uint32_t box_bytes = DW_BK * 128;                 // 32 rows x 32 floats
    constexpr uint32_t op_bytes = 4 * box_bytes;                // 128 columns
    constexpr uint32_t stage_bytes = 4 * op_bytes;              // A hi, A lo, B hi, B lo
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]);
    const uint32_t tfull0 = smem_u32(&bars[2 * STAGES]), tempty0 = smem_u32(&bars[2 * STAGES + 2]);
    constexpr uint32_t ncols = 512;                             // two sets of (main, cross) x 128 columns
    const int tile = blockIdx.x % (ds.MT * ds.NT), z = blockIdx.x / (ds.MT * ds.NT);
    const int i0 = (tile % ds.MT) * DW_T, k0 = (tile / ds.MT) * DW_T;
    const int r0 = z * ds.rows_per_split;
    int r1 = r0 + ds.rows_per_split;
    if (r1 > ds.total_rows) r1 = ds.total_rows;
    const int KB = (r1 - r0) / DW_BK;
    const int nchunks = (KB + DW_CHUNK - 1) / DW_CHUNK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull0 + 8 * s, 1); mbar_init(tempty0 + 8 * s, kEpiWarps); }
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

    if (warp == kTmaWarp) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(empty0 + 8 * stage, phase ^ 1);
                const uint32_t base = ring + stage * stage_bytes, fb = full0 + 8 * stage;
                mbar_expect_tx(fb, stage_bytes);
                const int row = r0 + kb * DW_BK;
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    tma_load_2d(base + m * box_bytes, &mA_hi, fb, i0 + 32 * m, row);
                    tma_load_2d(base + op_bytes + m * box_bytes, &mA_lo, fb, i0 + 32 * m, row);
                    tma_load_2d(base + 2 * op_bytes + m * box_bytes, &mB_hi, fb, k0 + 32 * m, row);
                    tma_load_2d(base + 3 * op_bytes + m * box_bytes, &mB_lo, fb, k0 + 32 * m, row);
                }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0) {
            // c=F32, a=b=TF32, both MN-major (bits 15, 16), N = 128, M = 128
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ds.major_bits |
                                   ((uint32_t)(DW_T >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            int stage = 0; uint32_t phase = 0;
            int c = 0, jj = 0;
            uint32_t d_main = tmem_base, d_cross = tmem_base + DW_T;
            for (int kb = 0; kb < KB; ++kb) {
                if (kb % DW_CHUNK == 0) {                       // next accumulator set, once the epilogue has drained it
                    const int set = c & 1;
                    mbar_wait(tempty0 + 8 * set, (uint32_t)((c >> 1) & 1) ^ 1u);
                    tc_fence_after();
                    d_main = tmem_base + (uint32_t)set * 2 * DW_T;
                    d_cross = d_main + DW_T;
                    jj = 0;
                }
                mbar_wait(full0 + 8 * stage, phase);
                tc_fence_after();
                const uint32_t base = ring + stage * stage_bytes;
                const uint64_t a_hi = make_smem_desc_mn(base, ds.lbo, ds.sbo), a_lo = make_smem_desc_mn(base + op_bytes, ds.lbo, ds.sbo);
                const uint64_t b_hi = make_smem_desc_mn(base + 2 * op_bytes, ds.lbo, ds.sbo), b_lo = make_smem_desc_mn(base + 3 * op_bytes, ds.lbo, ds.sbo);
#pragma unroll
                for (int k = 0; k < DW_BK / 8; ++k, ++jj) {
                    const uint64_t adv = (uint64_t)((k * ds.kadv) >> 4);   // next 8-row swizzle atom
                    umma_tf32(d_cross, a_lo + adv, b_hi + adv, idesc, jj != 0);
                    umma_tf32(d_cross, a_hi + adv, b_lo + adv, idesc, 1);
                    umma_tf32(d_main, a_hi + adv, b_hi + adv, idesc, jj != 0);
                }
                umma_commit(empty0 + 8 * stage);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                if (kb % DW_CHUNK == DW_CHUNK - 1 || kb == KB - 1) { umma_commit(tfull0 + 8 * (c & 1)); ++c; }
            }
        }
    } else if (warp >= kEpiWarp0) {
        const int ew = warp - kEpiWarp0, quarter = warp & 3, g = ew >> 2;
        const int i = i0 + quarter * 32 + lane;
        float acc[32];
        // fixed-order reduction: the running sum of this (tile, split) is fetched up front -- its latency hides behind the
        // contraction -- and stored back with the new contribution at the end (no read-modify-write in the kernel's tail)
        float* dst = ds.partial ? ds.partial + (size_t)z * ds.N * ds.ld_w : nullptr;
#pragma unroll
        for (int q = 0; q < 32; ++q) {
            const int k = k0 + g * 32 + q;
            acc[q] = (dst && i < ds.N && k < ds.Kaug) ? __ldcg(dst + (size_t)i * ds.ld_w + k) : 0.f;
        }
        for (int c = 0; c < nchunks; ++c) {
            const int set = c & 1;
            mbar_wait(tfull0 + 8 * set, (uint32_t)((c >> 1) & 1));
            tc_fence_after();
            const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(set * 2 * DW_T + g * 32);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                uint32_t um[4], ux[4];
                tmem_ld4_issue(lane_base + 4 * q, um);
                tmem_ld4_issue(lane_base + DW_T + 4 * q, ux);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[4 * q + e] += __uint_as_float(ux[e]) + __uint_as_float(um[e]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * set);
        }
        if (dst) {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int k = k0 + g * 32 + q;
                if (i < ds.N && k < ds.Kaug) dst[(size_t)i * ds.ld_w + k] = acc[q];
            }
        } else {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int k = k0 + g * 32 + q;
                if (i < ds.N && k < ds.Kaug) atomicAdd(ds.grad_W + (size_t)i * ds.ld_w + k, acc[q]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// grad_W[e] = sum_z partial[z][e] in the fixed order z = 0, 1, ... (the deterministic end of the dW reduction)
__global__ void k_dw_reduce_partials(const float* __restrict__ partial, int Z, size_t n, float* __restrict__ grad_W) {
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int z = 0; z < Z; ++z) s += partial[(size_t)z * n + e];
        grad_W[e] = s;
    }
}

static int launch_dw(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                     const DwShape& ds, cudaStream_t s) {
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(k_tc_dw, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
            return ODECOL_E_CUDA;
        configured = true;
    }
    k_tc_dw<<<ds.MT * ds.NT * ds.Z, kThreads, (size_t)STAGES * 4 * 4 * DW_BK * 128 + 1024, s>>>(a_hi, a_lo, b_hi, b_lo, ds);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

// rows x cols float32 matrix, box = box_rows x 32 floats (MN-major operand boxes reuse make_map with box_rows = 32)

__global__ void k_split_pad_T(const float* __restrict__ src, int n, int ld, float* __restrict__ hi, float* __restrict__ lo,
                              int rows_p, int cols_p) {
    // hi/lo of the transpose of the leading n x n block
    const size_t total = (size_t)rows_p * cols_p;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols_p), c = (int)(e % cols_p);
        const float x = (r < n && c < n) ? src[(size_t)c * ld + r] : 0.0f;
        const float h = tf32_rna(x);
        hi[e] = h;
        lo[e] = tf32_rna(x - h);
    }
}

struct TcBwdLayout {
    int Np, Bp, KPa, NPk, TN;
    size_t off_Whi, off_Wlo, off_WThi, off_WTlo, off_Rhi, off_Rlo, off_AVhi, off_AVlo;   // stacked x4 operand buffers
    size_t off_K[3], off_Y, off_DRT[4], off_lam, off_b4, off_b3, off_acur, off_inv, off_done, off_dwpart, total;
    int dwZ;
};

static TcBwdLayout tc_bwd_layout(const DevProblem& p) {
    TcBwdLayout L;
    L.Np = round_up(p.N, BM);
    L.NPk = L.Np;
    L.KPa = round_up(p.N + p.n_in + 1, BK);
    L.TN = pick_tile_n(L.Np / BM, p.B);
    L.Bp = round_up(p.B, L.TN);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t r = o; o += (bytes + 1023) / 1024 * 1024; return r; };
    L.off_Whi = take(4ull * L.Np * L.KPa); L.off_Wlo = take(4ull * L.Np * L.KPa);
    L.off_WThi = take(4ull * L.Np * L.NPk); L.off_WTlo = take(4ull * L.Np * L.NPk);
    L.off_Rhi = take(16ull * L.Bp * L.KPa); L.off_Rlo = take(16ull * L.Bp * L.KPa);
    L.off_AVhi = take(32ull * L.Bp * L.NPk); L.off_AVlo = take(32ull * L.Bp * L.NPk);     // two sets of four slots
    const size_t plane = 4ull * L.Np * L.Bp;
    for (int i = 0; i < 3; ++i) L.off_K[i] = take(plane);
    L.off_Y = take(3 * plane);
    for (int i = 0; i < 4; ++i) L.off_DRT[i] = take(plane);
    L.off_lam = take(3 * plane); L.off_b4 = take(2 * plane); L.off_b3 = take(2 * plane); L.off_acur = take(2 * plane);
    L.off_inv = take(sizeof(int) * (3ull * p.N + 4));      // + the "an F component is selected" flag
    L.off_done = take(sizeof(unsigned int) * (size_t)(L.Bp / L.TN) + 256);
    // per-row-split copies of grad_W_aug (deterministic dW reduction): the split count of the one-wave dW launch
    {
        const int tiles = (L.Np / DW_T) * ((L.KPa + DW_T - 1) / DW_T);
        int z = num_sms() / tiles;
        if (z < 1) z = 1;
        L.dwZ = z;
        L.off_dwpart = take(4ull * (size_t)z * p.N * p.ld_w);
    }
    L.total = o;
    return L;
}

}  // namespace tc

// diagnostic: C[m][n] += sum_k A[k][m] * B[k][n] with the MN-major contraction the dW accumulation uses
size_t tc_contract_tn_workspace_bytes(int M, int N, int K) {
    const size_t Mp = round_up(M, 128), Np = round_up(N, 32), Kp = round_up(K, 64);
    return 4 * (2 * Kp * Mp + 2 * Kp * Np) + 4096;
}

int tc_contract_tn(const float* A, const float* B, float* C, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const int Mp = round_up(M, 128), Np = round_up(N, 32), Kp = round_up(K, 64);
    if (!ws || ws_bytes < tc_contract_tn_workspace_bytes(M, N, K)) return ODECOL_E_WORKSPACE;
    float* Ahi = static_cast<float*>(ws);
    float* Alo = Ahi + (size_t)Kp * Mp;
    float* Bhi = Alo + (size_t)Kp * Mp;
    float* Blo = Bhi + (size_t)Kp * Np;
    k_split_pad<<<296, 256, 0, s>>>(A, K, M, M, Ahi, Alo, Kp, Mp);
    k_split_pad<<<296, 256, 0, s>>>(B, K, N, N, Bhi, Blo, Kp, Np);
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    if (!make_map(&a_hi, Ahi, Kp, Mp, Mp, DW_BK, sw) || !make_map(&a_lo, Alo, Kp, Mp, Mp, DW_BK, sw) ||
        !make_map(&b_hi, Bhi, Kp, Np, Np, DW_BK, sw) || !make_map(&b_lo, Blo, Kp, Np, Np, DW_BK, sw))
        return ODECOL_E_CUDA;
    DwShape ds;
    ds.MT = Mp / DW_T; ds.NT = (Np + DW_T - 1) / DW_T; ds.total_rows = Kp;
    int z = 2;
    int rows = (Kp / DW_BK + z - 1) / z * DW_BK;
    ds.rows_per_split = rows; ds.Z = (Kp + rows - 1) / rows;
    ds.N = M; ds.Kaug = N; ds.ld_w = N; ds.grad_W = C; ds.partial = nullptr;
    ds.lbo = DW_BK * 128; ds.sbo = 512; ds.major_bits = (1u << 15) | (1u << 16); ds.kadv = 1024;
    if (cudaMemsetAsync(C, 0, sizeof(float) * (size_t)M * N, s) != cudaSuccess) return ODECOL_E_CUDA;
    count_launch(2);
    return launch_dw(a_hi, a_lo, b_hi, b_lo, ds, s);
}

// grad_W[i][k] += sum_rows A[row][i] * B[row][k] for split operands A (rows x Np) and B (rows x KPa), rows % 32 == 0:
// the dW accumulation as a stand-alone step for the staged Euler-Maruyama / srk adjoints (stage_em.cu)
int tc_dw_accumulate(const float* Ahi, const float* Alo, const float* Bhi, const float* Blo, int rows, int Np, int KPa, int N,
                     int Kaug, int ld_w, float* grad_W, cudaStream_t s) {
    using namespace tc;
    if (rows % DW_BK) return ODECOL_E_SHAPE;
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    if (!make_map(&a_hi, Ahi, rows, Np, Np, DW_BK, sw) || !make_map(&a_lo, Alo, rows, Np, Np, DW_BK, sw) ||
        !make_map(&b_hi, Bhi, rows, KPa, KPa, DW_BK, sw) || !make_map(&b_lo, Blo, rows, KPa, KPa, DW_BK, sw))
        return ODECOL_E_CUDA;
    DwShape ds;
    ds.MT = Np / DW_T; ds.NT = (KPa + DW_T - 1) / DW_T; ds.total_rows = rows;
    int z = num_sms() / (ds.MT * ds.NT);
    if (z < 1) z = 1;
    int rps = (rows / DW_BK + z - 1) / z * DW_BK;
    if (rps < DW_BK) rps = DW_BK;
    ds.rows_per_split = rps; ds.Z = (rows + rps - 1) / rps;
    ds.N = N; ds.Kaug = Kaug; ds.ld_w = ld_w; ds.grad_W = grad_W; ds.partial = nullptr;
    ds.lbo = DW_BK * 128; ds.sbo = 512; ds.major_bits = (1u << 15) | (1u << 16); ds.kadv = 1024;
    return launch_dw(a_hi, a_lo, b_hi, b_lo, ds, s);
}

size_t tc_rk4_bwd_workspace_bytes(const DevProblem& p, int) { return tc::tc_bwd_layout(p).total; }

static int tc_rk4_bwd_impl(const DevProblem& p, const float* t_dev, int T, const float* y_traj, const float* ckVA,
                           const float* ckK, const float* grad_y, const int* sel, int G, float* grad_y0, float* grad_W,
                           void* ws, size_t ws_bytes, cudaStream_t s) {
    using namespace tc;
    const TcBwdLayout L = tc_bwd_layout(p);
    if (!ws || ws_bytes < L.total) return ODECOL_E_WORKSPACE;
    if (p.N % 4 != 0) return ODECOL_E_UNSUPPORTED;
    char* w = static_cast<char*>(ws);
    auto F = [&](size_t off) { return reinterpret_cast<float*>(w + off); };
    float *Whi = F(L.off_Whi), *Wlo = F(L.off_Wlo), *WThi = F(L.off_WThi), *WTlo = F(L.off_WTlo);
    float *Rhi = F(L.off_Rhi), *Rlo = F(L.off_Rlo), *AVhi = F(L.off_AVhi), *AVlo = F(L.off_AVlo);
    float* KT[3] = {F(L.off_K[0]), F(L.off_K[1]), F(L.off_K[2])};
    float* YT = F(L.off_Y);
    float* DRT[4];
    for (int k = 0; k < 4; ++k) DRT[k] = F(L.off_DRT[k]);
    float *lamT = F(L.off_lam), *b4T = F(L.off_b4), *b3T = F(L.off_b3), *acurT = F(L.off_acur);
    int* inv = reinterpret_cast<int*>(w + L.off_inv);
    const int Kaug = p.N + p.n_in + 1;
    const size_t st = (size_t)p.B * 3 * p.N;
    const float gamma = p.c.tau_s * p.c.R / p.c.tau_m;
    const TileGeom tg{L.Bp / L.TN, L.Np, L.TN, L.TN / 4};
    const size_t rstride = (size_t)L.Bp * L.KPa, astride = (size_t)L.Bp * L.NPk;

    // zero the stacked operand buffers once: padding rows / columns must stay zero
    if (cudaMemsetAsync(w + L.off_Rhi, 0, L.off_K[0] - L.off_Rhi, s) != cudaSuccess) return ODECOL_E_CUDA;
    k_split_pad<<<296, 256, 0, s>>>(p.W_aug, p.N, Kaug, p.ld_w, Whi, Wlo, L.Np, L.KPa);
    k_split_pad_T<<<296, 256, 0, s>>>(p.W_aug, p.N, p.ld_w, WThi, WTlo, L.Np, L.NPk);
    k_tc_set_one<<<(4 * p.B + 255) / 256, 256, 0, s>>>(Rhi, L.Bp, p.B, L.KPa, Kaug - 1, 4);
    k_tc_build_inv<<<1, 256, 0, s>>>(sel, G, 3 * p.N, inv);
    const size_t first = (size_t)(((T - 2) & 1) * 4 + 3);       // operand sets alternate per step: step n uses set n & 1
    k_tc_bwd_begin<<<L.Bp / 4, 128, 0, s>>>(p, tg, grad_y, inv, G, t_dev, T, gamma, lamT, acurT, AVhi + first * astride,
                                           AVlo + first * astride, L.NPk);
    unsigned int* done = reinterpret_cast<unsigned int*>(w + L.off_done);
    if (cudaMemsetAsync(done, 0, sizeof(unsigned int) * (size_t)(L.Bp / L.TN), s) != cudaSuccess) return ODECOL_E_CUDA;
    count_launch(5);

    CUtensorMap mWhi, mWlo, mWThi, mWTlo, mRhi, mRlo, mAVhi, mAVlo, dAhi[2], dAlo[2], dBhi, dBlo;
    bool ok = make_map(&mWhi, Whi, L.Np, L.KPa, L.KPa, BM) && make_map(&mWlo, Wlo, L.Np, L.KPa, L.KPa, BM) &&
              make_map(&mWThi, WThi, L.Np, L.NPk, L.NPk, BM) && make_map(&mWTlo, WTlo, L.Np, L.NPk, L.NPk, BM) &&
              make_map(&mRhi, Rhi, 4ull * L.Bp, L.KPa, L.KPa, L.TN) && make_map(&mRlo, Rlo, 4ull * L.Bp, L.KPa, L.KPa, L.TN) &&
              make_map(&mAVhi, AVhi, 8ull * L.Bp, L.NPk, L.NPk, L.TN) && make_map(&mAVlo, AVlo, 8ull * L.Bp, L.NPk, L.NPk, L.TN) &&
              make_map(&dAhi[0], AVhi, 4ull * L.Bp, L.NPk, L.NPk, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) &&
              make_map(&dAlo[0], AVlo, 4ull * L.Bp, L.NPk, L.NPk, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) &&
              make_map(&dAhi[1], AVhi + 4 * astride, 4ull * L.Bp, L.NPk, L.NPk, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) &&
              make_map(&dAlo[1], AVlo + 4 * astride, 4ull * L.Bp, L.NPk, L.NPk, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) &&
              make_map(&dBhi, Rhi, 4ull * L.Bp, L.KPa, L.KPa, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) &&
              make_map(&dBlo, Rlo, 4ull * L.Bp, L.KPa, L.KPa, DW_BK, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (!ok) return ODECOL_E_CUDA;

    // dW launch shape: output tiles x splits of the stacked rows, one wave of CTAs (chunked accumulation: long items are
    // accurate)
    DwShape ds;
    ds.MT = L.Np / DW_T; ds.NT = (L.KPa + DW_T - 1) / DW_T;
    ds.total_rows = 4 * L.Bp;
    int z = num_sms() / (ds.MT * ds.NT);
    if (z < 1) z = 1;
    int rows = (ds.total_rows / DW_BK + z - 1) / z * DW_BK;
    if (rows < DW_BK) rows = DW_BK;
    ds.rows_per_split = rows; ds.Z = (ds.total_rows + rows - 1) / rows;
    ds.N = p.N; ds.Kaug = Kaug; ds.ld_w = p.ld_w; ds.grad_W = grad_W;
    ds.lbo = DW_BK * 128; ds.sbo = 512; ds.major_bits = (1u << 15) | (1u << 16); ds.kadv = 1024;
    ds.partial = nullptr;

    const int MT = L.Np / BM, NT = L.Bp / L.TN;
    // the four reverse stages of a step as one cooperative launch (ODECOL_PERSISTENT=0: one launch per stage)
    const char* pe = getenv("ODECOL_PERSISTENT");
    bool use_chain = (pe ? atoi(pe) != 0 : true) && L.NPk / BK <= kChunkMin && L.KPa / BK <= kChunkMin;   // long K: chunked k_tc_contract
    // The dW contraction runs as a fifth phase of the chain launch (its operands are complete long before the chain ends, so
    // the MMA warp contracts dW while the stage-1 epilogues still stream): two launches per reverse step instead of three.
    // Round 1 measured it on par with a launch of its own; since the epilogues got leaner it is 2.6 % of the sweep
    // (577 against 592 ms, profiles/r2_session3_ab.md).  ODECOL_FUSE_DW=0: separate launch (always so for the fixed-order
    // reduction, whose per-split copies live in the stand-alone kernel).
    const char* fe = getenv("ODECOL_FUSE_DW");
    const bool dw_fixed_order = (p.flags & ODECOL_FLAG_DETERMINISTIC) != 0;     // default: float atomics (2 % faster sweep)
    const bool fuse_dw = use_chain && !dw_fixed_order && (fe ? atoi(fe) != 0 : true);
    // ODECOL_FLAG_DETERMINISTIC: every (output tile, row split) accumulates into its own copy of grad_W_aug across the whole
    // sweep (one CTA per (tile, split) and launch, launches ordered on the stream; the running sum is fetched at kernel start
    // and stored back at the end), the copies are summed in a fixed order after the last step -- the gradient is
    // bit-reproducible.  Measured: reverse sweep 633-639 ms against 621-625 ms with float atomics (A/B on one box).
    float* dw_partial = nullptr;
    if (dw_fixed_order && ds.Z <= L.dwZ) {
        dw_partial = reinterpret_cast<float*>(w + L.off_dwpart);
        if (cudaMemsetAsync(dw_partial, 0, sizeof(float) * (size_t)ds.Z * p.N * p.ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
        ds.partial = dw_partial;
    }
    const size_t chain_stage = 2 * BM * BK * 4 + 2 * (size_t)L.TN * BK * 4, dw_stage_b = 4 * 4 * DW_BK * 128;
    const size_t chain_smem = (size_t)STAGES * (fuse_dw && dw_stage_b > chain_stage ? dw_stage_b : chain_stage) + 1024;
    int chain_grid = MT * NT < num_sms() ? MT * NT : num_sms();
    if (use_chain) {
        int max_blocks = 0;
        if (cudaFuncSetAttribute(k_tc_bwd_chain<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(k_tc_bwd_chain<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks, k_tc_bwd_chain<true>, kThreads, chain_smem) != cudaSuccess || max_blocks < 1)
            use_chain = false;
    }
    // Checkpoint mode: every step's operands and phi' planes are replayed from the checkpoints by a launch of their own.
    // (Handing the replay to the idle epilogue warps of the previous step's dW contraction measured slower, DESIGN.md
    // section 7: the epilogue warps' arithmetic delays the contraction's two single-thread issue loops.)
    const size_t ckpl = (size_t)L.Np * L.Bp;
    auto replay = [&](int n) {
        ReplayJob j;
        j.p = p; j.tg = tg;
        j.VA = ckVA + 2 * ckpl * (size_t)n; j.KV = ckK + 3 * ckpl * (size_t)n; j.t = t_dev;
        j.n = n; j.KPa = L.KPa; j.slices = L.Np / 128;
        j.Rhi = Rhi; j.Rlo = Rlo; j.rstride = rstride;
        for (int k = 0; k < 4; ++k) j.D[k] = DRT[k];
        k_tc_replay<<<L.Bp / 4, 128, 0, s>>>(j);
        count_launch();
    };
    for (int n = T - 2; n >= 0; --n) {
        int rc = ODECOL_OK;
        if (ckVA) {
            replay(n);
        } else {
        const float* yn = y_traj + (size_t)n * st;
        k_tc_step_begin<<<L.Bp / 4, 128, 0, s>>>(p, tg, yn, t_dev + n, Rhi, Rlo, YT, DRT[0], L.KPa);
        count_launch();
        // recompute stages 1..3: operand s -> operand s+1, r and phi' of the next stage state
        auto fill_f = [&](auto& e, int S) {
            e.p = p; e.tg = tg; e.t = t_dev; e.n = n; e.KPa = L.KPa;
            e.V0T = YT; e.A0T = YT + tg.plane(); e.F0T = nullptr;       // stages 1..3 never touch F
            e.V1T = e.A1T = e.F1T = nullptr; e.traj_row = nullptr; e.ysel_row = nullptr; e.inv = nullptr; e.G = 0;
            e.K1T = KT[0]; e.K2T = KT[1]; e.K3T = KT[2];
            e.Rhi_nxt = Rhi + S * rstride; e.Rlo_nxt = Rlo + S * rstride; e.DRT_nxt = DRT[S];
            e.inv_tm = 1.0f / p.c.tau_m; e.inv_ta = 1.0f / p.c.tau_a; e.inv_ts = 1.0f / p.c.tau_s;
            e.t0 = e.t1 = e.dt = 0.f;
        };
        { FwdEpiT<1> e; fill_f(e, 1); rc = launch_contract(mWhi, mWlo, mRhi, mRlo, TileShape{MT, NT, L.TN, L.KPa / BK, 0 * L.Bp}, e, s); if (rc) return rc; }
        { FwdEpiT<2> e; fill_f(e, 2); rc = launch_contract(mWhi, mWlo, mRhi, mRlo, TileShape{MT, NT, L.TN, L.KPa / BK, 1 * L.Bp}, e, s); if (rc) return rc; }
        { FwdEpiT<3> e; fill_f(e, 3); rc = launch_contract(mWhi, mWlo, mRhi, mRlo, TileShape{MT, NT, L.TN, L.KPa / BK, 2 * L.Bp}, e, s); if (rc) return rc; }
        }
        // reverse stages 4, 3, 2, 1 (stage 1 writes kbar_4 of the next step into the OTHER operand set), then dW
        const int set = n & 1;
        if (use_chain) {
            BwdChainArgs a;
            a.p = p; a.tg = tg; a.ts = TileShape{MT, NT, L.TN, L.NPk / BK, 0}; a.t = t_dev; a.n = n; a.NPk = L.NPk; a.G = G;
            a.Bp = L.Bp; a.acurT = acurT; a.lamT = lamT; a.b4T = b4T; a.b3T = b3T;
            for (int k = 0; k < 4; ++k) a.DRT[k] = DRT[k];
            a.AVhi = AVhi; a.AVlo = AVlo; a.set = set; a.grad_y = grad_y; a.inv = inv; a.gamma = gamma;
            a.inv_tm = 1.0f / p.c.tau_m; a.inv_ta = 1.0f / p.c.tau_a; a.inv_ts = 1.0f / p.c.tau_s;
            a.done = done; a.done_base = (unsigned int)MT * 4u * (unsigned int)(T - 2 - n);
            a.ds = ds;
            void* args[] = {&mWThi, &mWTlo, &mAVhi, &mAVlo, &dAhi[set], &dAlo[set], &dBhi, &dBlo, &a};
            const void* chain_fn = fuse_dw ? (const void*)k_tc_bwd_chain<true> : (const void*)k_tc_bwd_chain<false>;
            if (cudaLaunchCooperativeKernel(chain_fn, dim3(chain_grid), dim3(kThreads), args, chain_smem, s) != cudaSuccess)
                return ODECOL_E_CUDA;
            count_launch();
        } else {
            auto fill_b = [&](auto& e, int S) {
                e.p = p; e.tg = tg; e.t = t_dev; e.n = n; e.NPk = L.NPk; e.G = G;
                e.acurT = acurT; e.lamT = lamT; e.b4T = b4T; e.b3T = b3T; e.DRT = DRT[S - 1];
                const size_t nxt = S == 1 ? (size_t)((set ^ 1) * 4 + 3) : (size_t)(set * 4 + S - 2);   // slot the epilogue writes
                e.AVhi_nxt = AVhi + nxt * astride; e.AVlo_nxt = AVlo + nxt * astride;
                e.grad_y = grad_y; e.inv = inv; e.gamma = gamma;
                e.inv_tm = 1.0f / p.c.tau_m; e.inv_ta = 1.0f / p.c.tau_a; e.inv_ts = 1.0f / p.c.tau_s;
                e.dt = e.h8p = 0.f;
            };
            const int r0 = set * 4 * L.Bp;
            { BwdEpiT<4> e; fill_b(e, 4); rc = launch_contract(mWThi, mWTlo, mAVhi, mAVlo, TileShape{MT, NT, L.TN, L.NPk / BK, r0 + 3 * L.Bp}, e, s); if (rc) return rc; }
            { BwdEpiT<3> e; fill_b(e, 3); rc = launch_contract(mWThi, mWTlo, mAVhi, mAVlo, TileShape{MT, NT, L.TN, L.NPk / BK, r0 + 2 * L.Bp}, e, s); if (rc) return rc; }
            { BwdEpiT<2> e; fill_b(e, 2); rc = launch_contract(mWThi, mWTlo, mAVhi, mAVlo, TileShape{MT, NT, L.TN, L.NPk / BK, r0 + 1 * L.Bp}, e, s); if (rc) return rc; }
            { BwdEpiT<1> e; fill_b(e, 1); rc = launch_contract(mWThi, mWTlo, mAVhi, mAVlo, TileShape{MT, NT, L.TN, L.NPk / BK, r0 + 0 * L.Bp}, e, s); if (rc) return rc; }
        }
        if (!(use_chain && fuse_dw)) {
            const int rcd = launch_dw(dAhi[set], dAlo[set], dBhi, dBlo, ds, s);
            if (rcd) return rcd;
        }
    }
    if (dw_partial) {
        k_dw_reduce_partials<<<296, 256, 0, s>>>(dw_partial, ds.Z, (size_t)p.N * p.ld_w, grad_W);
        count_launch();
    }
    if (grad_y0) {
        k_tc_untile<<<L.Bp / 4, 128, 0, s>>>(p, tg, lamT, grad_y0);
        count_launch();
    }
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

int tc_rk4_bwd(const DevProblem& p, const float* t_dev, int T, const float* y_traj, const float* grad_y, const int* sel,
               int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s) {
    return tc_rk4_bwd_impl(p, t_dev, T, y_traj, nullptr, nullptr, grad_y, sel, G, grad_y0, grad_W, ws, ws_bytes, s);
}

// reverse sweep from the checkpoints of tc_rk4_fwd_ckpt (layout: tc::CkptView)
int tc_rk4_bwd_ckpt(const DevProblem& p, const float* t_dev, int T, const void* ckpt, size_t ckpt_bytes, const float* grad_y,
                    const int* sel, int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s) {
    const tc::TcBwdLayout L = tc::tc_bwd_layout(p);
    const size_t plane = (size_t)L.Np * L.Bp;
    if (!ckpt || ckpt_bytes < 4 * plane * (2ull * T + 3ull * (T - 1))) return ODECOL_E_WORKSPACE;
    const float* VA = static_cast<const float*>(ckpt);
    return tc_rk4_bwd_impl(p, t_dev, T, nullptr, VA, VA + 2 * plane * (size_t)T, grad_y, sel, G, grad_y0, grad_W, ws, ws_bytes, s);
}

}  // namespace odecol
