// Kernel family T ("tensor"): the staged solver's contraction on the 5th-generation tensor cores.
//
//   C[i][b] = sum_k W_aug[i][k] * R_aug[b][k]   as   3xTF32:  W = Whi + Wlo, R = Rhi + Rlo (each rounded to TF32),
//   C = Wlo.Rhi + Whi.Rlo + Whi.Rhi accumulated in FP32 in tensor memory -- FP32-level accuracy at tensor-core rate.
//
// One persistent CTA per SM, warp specialised:
//   warp 0      TMA producer: cp.async.bulk.tensor (128-byte swizzle) of the four operand tiles of a 32-wide K block into
//               a 3-stage shared-memory ring, completion on mbarriers
//   warp 1      tcgen05.mma issuer (one elected thread; M = 128 populations x N = tile of trials x K = 8 per instruction).
//               The tensor core truncates (round-toward-zero) every accumulation into TMEM, which biases long sums of
//               same-signed terms (measured: -3.8e-6 relative at K = 608).  So the Whi.Rhi products rotate over THREE
//               accumulators (a third of the truncations each) and the two small cross terms go to a fourth; the epilogue
//               adds the four in FP32 round-to-nearest.  tcgen05.commit releases ring slots and publishes finished tiles
//   warps 2..17 epilogue: tcgen05.ld this thread's accumulator row segment (TMEM lane = population) into registers, hand
//               TMEM back to warp 1 (which starts contracting the next tile), then the fused RK-stage epilogue -- drift,
//               next stage state, phi, next operand already split into hi/lo -- on tile-major scratch (float4 along trials)
// The trial tile is chosen so that the number of tiles is a multiple of the SM count (148) where possible.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include "odecol_common.cuh"

namespace odecol {

constexpr float kOneThirdL = 0.3333333333333333f;
constexpr float kTwoThirdsL = 0.6666666666666666f;

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

ODECOL_DEVINL float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
ODECOL_DEVINL void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// scratch that is streamed once per launch: L2 only.  (With ~200 KB of the SM's array carved out as shared memory the
// remaining L1 is too small to hold a line for every outstanding load, and allocating loads stall on it.)
ODECOL_DEVINL float4 ld4s(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
ODECOL_DEVINL void st4s(float* p, float4 v) { __stcg(reinterpret_cast<float4*>(p), v); }

namespace tc {

constexpr int BM = 128;          // populations per tile = TMEM lanes
constexpr int BK = 32;           // floats per K block = one 128-byte swizzle row
#ifndef ODECOL_TC_STAGES
#define ODECOL_TC_STAGES 3
#endif
constexpr int STAGES = ODECOL_TC_STAGES;      // operand ring depth (stages of 2 x (128 + TN) x 128 bytes)
constexpr int kEpiWarps = 16;
constexpr int kMainAcc = 3;      // Whi.Rhi accumulators (rotated), plus one for the cross terms
// -DODECOL_EPI_REGS=n (experiment): the TMA producer and the MMA issuer get a warpgroup of their own (with two idle warps),
// release most of their registers (setmaxnreg.dec) and the sixteen epilogue warps grow to n registers (setmaxnreg.inc):
// 18 warps at 96 registers is what the register file allows at launch (five warps on one SM sub-partition x 96 <= 512),
// and the reverse epilogues spill at 96.
#ifndef ODECOL_EPI_REGS
#define ODECOL_EPI_REGS 0
#endif
constexpr int kEpiRegs = ODECOL_EPI_REGS;
constexpr int kThreads = 32 * ((kEpiRegs ? 4 : 2) + kEpiWarps);
// warp roles.  -DODECOL_ROLES_HIGH puts the TMA producer and the MMA issuer in the two HIGHEST warps of the CTA (the SM's
// arbiter prefers higher warp ids among eligible warps, B300_MICROARCH.md): an experiment on whether the sixteen epilogue
// warps delay the two single-thread issue loops.
#ifdef ODECOL_ROLES_HIGH
constexpr int kEpiWarp0 = 0, kTmaWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;
#else
constexpr int kTmaWarp = 0, kMmaWarp = 1, kEpiWarp0 = kEpiRegs ? 4 : 2;
#endif
// register reallocation between the role warpgroups: the low warpgroup (TMA, MMA, two idle warps) calls dec before its roles
// split, the epilogue warps call inc at the top of their branch (ptxas sizes a branch by the setmaxnreg that dominates it)
template <int N> ODECOL_DEVINL void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> ODECOL_DEVINL void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
constexpr uint32_t kSpinLimit = 1u << 24;
constexpr int kChunkKB = 16;     // chunked accumulation (long contractions): K blocks per accumulator chunk
constexpr int kChunkMin = 24;    // contractions of more than this many K blocks (K > 768) run chunked

ODECOL_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

ODECOL_DEVINL void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
ODECOL_DEVINL void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
ODECOL_DEVINL void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// bounded wait: a protocol bug must trap, never hang the GPU
ODECOL_DEVINL void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0, spins = 0;
    while (true) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        if (++spins > kSpinLimit) __trap();
    }
}
ODECOL_DEVINL void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
ODECOL_DEVINL void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
ODECOL_DEVINL void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
ODECOL_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
ODECOL_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
ODECOL_DEVINL void tmem_ld4_issue(uint32_t taddr, uint32_t (&u)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "r"(taddr));
}
ODECOL_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows of 128 bytes, 8-row swizzle atoms 1024 bytes apart
ODECOL_DEVINL uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);     // start address            bits [0,14)
    d |= (uint64_t)1 << 16;                           // leading byte offset      bits [16,30)  (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                 // stride byte offset       bits [32,46)
    d |= (uint64_t)1 << 46;                           // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                           // SWIZZLE_128B
    return d;
}
ODECOL_DEVINL uint32_t make_idesc(int tile_n) {
    // c=F32 (1<<4), a=b=TF32 (2<<7, 2<<10), both K-major, N>>3 at [17,23), M>>4 at [24,29)
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(tile_n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// float32 -> TF32, round to nearest with ties away from zero (what cvt.rna.tf32.f32 does): on the sign-magnitude bit
// pattern that is "add half of the dropped field, clear it" -- two integer instructions; ptxas expands the cvt into more.
// Exact for every finite value whose rounding does not overflow (|x| < 3.4e38 (1 - 2^-11)); NaN stays NaN.
ODECOL_DEVINL float tf32_rna(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

// predicated read-only load: 0 when the predicate is false (no branch, the address is never formed into an access then)
ODECOL_DEVINL float ldg_if(const float* p, bool ok) {
    float v;
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\tmov.f32 %0, 0f00000000;\n\t@q ld.global.nc.f32 %0, [%1];\n\t}"
                 : "=f"(v) : "l"(p), "r"((int)ok));
    return v;
}

// ---- 16-bit operand format of the persistent forward solve: every operand as two FP16 planes, x s = xh + xl / 2048
//   xh = fp16(x s), xl = fp16((x s - xh) 2048): 11 + 11 mantissa bits like the TF32 split, the low plane kept in FP16's normal
//   range by its 2^11 (Ootomo & Yokota's error-corrected tensor-core product).  s is a power of two: for W_aug the one
//   that puts max|W_aug| into [2^13, 2^14) (found on the device, undone by the epilogues); for the trial operand s = 1.
//   C s = wh.rh (rotating main accumulators) + 2^-11 [wl.rh + wh.rl] (cross accumulator); dropped: wl.rl ~ 2^-22.
// Three kind::f16 products of K = 16 per 32 operand bytes against three kind::tf32 products of K = 8: half the tensor-core
// instructions and half the operand bytes (4 + 4 against 8 + 8 per (row, k)).  The stage passes are bound by the bytes
// that cross the L2 <-> SM port (operand tiles + epilogue planes), so bytes are what count.  (kind::f16 wants A and B
// of ONE type -- FP16 weights against BF16 rates is an illegal instruction -- hence FP16 for the trial operand as well.)
// FP16's range is the price: an operand value beyond +-6e4 (a firing rate of 60 kHz, a stimulus of that size) cannot be
// represented.  The epilogues raise a device flag when they meet one, and the launch sequence then repeats the solve in
// the TF32 format (a kernel that returns at once when the flag is clear): same results as before wherever the 16-bit
// format cannot hold the data, no host synchronisation either way.
constexpr int BK16 = 64;         // 16-bit elements per K block = one 128-byte swizzle row
constexpr float kF16Limit = 6.0e4f;
struct F16x2 { unsigned short h, l; };
ODECOL_DEVINL F16x2 f16_split2(float x) {
    const __half h = __float2half_rn(x);
    const __half l = __float2half_rn((x - __half2float(h)) * 2048.0f);
    return {__half_as_ushort(h), __half_as_ushort(l)};
}
// predicated 16-bit store
ODECOL_DEVINL void st_global_u16_if(uint16_t* p, unsigned short v, bool ok) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.b16 [%0], %1;\n\t}" ::"l"(p), "h"(v), "r"((int)ok) : "memory");
}
ODECOL_DEVINL void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
ODECOL_DEVINL uint32_t make_idesc16(int tile_n) {
    // c=F32 (1<<4), a=b=F16 (0<<7, 0<<10), both K-major, N>>3 at [17,23), M>>4 at [24,29)
    return (1u << 4) | ((uint32_t)(tile_n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

// buffers of the 16-bit operand format (host side view; carved out of the forward workspace)
struct Mixed16 {
    void* W16[2];          // [Np][KP16] FP16: wh, wl
    uint16_t* R16[2];      // two operand buffers of [2 planes][Bp][KP16] FP16
    float* wscale;         // [0] = 1 / weight scale, [1] = scratch of the max reduction, [2] = overflow flag (uint32)
    int KP16;
};

struct TileShape {
    int MT, NT, TN, KB;      // m tiles, trial tiles, trials per tile (multiple of 16, <= 128), K blocks of 32
    int b_row0;              // first row of the B operand inside its tensor map (stacked per-stage operand buffers)
};

ODECOL_DEVINL unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

ODECOL_DEVINL void st_global(float* p, float v) { asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }
// predicated store: no branch around it (the ragged last trial tile is the only place where the predicate is ever false)
ODECOL_DEVINL void st_global_if(float* p, float v, bool ok) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v), "r"((int)ok) : "memory");
}
constexpr int kMaxQ = 32;    // accumulator columns per epilogue thread = TN / 4 <= 32

// ---------------------------------------------------------------------------------------------------------------
// the persistent warp-specialised contraction.  Epi supplies
//   prepare()                                             once per epilogue thread
//   rows(m_tile, i, n0, nt, g, tot)                       population i, trials n0 + g*TN/4 + [0, TN/4): tot[] = W_aug.r_aug
//   tile_done(m_tile, n0, tile_n, etid, nthreads)         per tile, all epilogue threads
// ---------------------------------------------------------------------------------------------------------------
// tile -> (population tile, trial tile).  Population tiles are taken in groups of kTileGroupM: consecutive tiles (= the
// CTAs of a wave) walk the trial tiles of ONE group, so a wave touches kTileGroupM W_aug panels and ~148 / kTileGroupM
// trial panels instead of all of W_aug (at N = 8192 every wave streamed the whole 539 MB of W_aug from HBM: 19 GB of DRAM
// reads per drift evaluation), and the group's panels stay in L2 for the following waves.  With MT <= kTileGroupM this is
// the plain "population tile fastest" order.
constexpr int kTileGroupM = 12;
ODECOL_DEVINL void tile_coords(int tile, int MT, int NT, int& m, int& nt) {
    const int per_group = kTileGroupM * NT;
    const int grp = tile / per_group, within = tile - grp * per_group;
    const int gm = min(kTileGroupM, MT - grp * kTileGroupM);          // the last group may be smaller
    nt = within / gm;
    m = grp * kTileGroupM + (within - nt * gm);
}

// F16: both operands as FP16 pairs (see "16-bit operand format" above): K blocks of 64 elements, kind::f16 products, the
// cross sums scaled by 2^-11 on the way out of tensor memory; ts.KB counts 64-element blocks then.
template <class Epi, bool CHUNKED, bool F16 = false>
__global__ void __launch_bounds__(kThreads, 1)
k_tc_contract(const __grid_constant__ CUtensorMap mA_hi, const __grid_constant__ CUtensorMap mA_lo,
              const __grid_constant__ CUtensorMap mB_hi, const __grid_constant__ CUtensorMap mB_lo, TileShape ts, Epi epi) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES + 4];
    __shared__ uint32_t tmem_base_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
    constexpr int KEL = F16 ? BK16 : BK;               // operand elements per K block (one 128-byte row either way)
    constexpr int CKB = F16 ? kChunkKB / 2 : kChunkKB; // K blocks per accumulator chunk (512 elements of K)
    constexpr float XS = F16 ? 4.8828125e-4f : 1.0f;   // scale of the cross sums (the low FP16 planes carry 2^11)
    const uint32_t a_bytes = BM * 128, b_bytes = (uint32_t)ts.TN * 128;
    const uint32_t stage_bytes = 2 * a_bytes + 2 * b_bytes;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[STAGES]);
    const uint32_t tfull = smem_u32(&bars[2 * STAGES]), tempty = smem_u32(&bars[2 * STAGES + 1]);
    // Long contractions (K > 32 * kChunkMin) accumulate in CHUNKS: the tensor core truncates every accumulation into TMEM,
    // which biases a long sum of mostly same-signed terms (measured on the N = 8192 sheet's W_aug: 1.4e-5 of sum|a||b|
    // with three rotating accumulators over 258 K blocks).  In chunked mode the four accumulator planes are two SETS of
    // (main, cross terms); a set sees kChunkKB K blocks, then the epilogue warps drain it into FP32 round-to-nearest
    // registers while the MMA warp fills the other set -- the error no longer grows with K.
    constexpr bool chunked = CHUNKED;                      // compile-time: each variant keeps a tight MMA issue loop
    const uint32_t cfull0 = tfull, cempty0 = smem_u32(&bars[2 * STAGES + 2]);        // chunked: [set] = +8 * set; cfull[1] = bars[2S+1]

    const int tiles = ts.MT * ts.NT;
    const uint32_t acc_stride = (uint32_t)ts.TN;
    uint32_t ncols = 32;
    while (ncols < (kMainAcc + 1) * acc_stride) ncols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, chunked ? 1 : kEpiWarps);           // chunked mode: bars[2S], bars[2S+1] are the two `full` barriers
        mbar_init(cempty0, kEpiWarps);
        mbar_init(cempty0 + 8, kEpiWarps);
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
            for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                int mt_, nt_;
                tile_coords(tile, ts.MT, ts.NT, mt_, nt_);
                const int m0 = mt_ * BM, n0 = nt_ * ts.TN;
                for (int kb = 0; kb < ts.KB; ++kb) {
                    mbar_wait(empty0 + 8 * stage, phase ^ 1);
                    const uint32_t base = ring + stage * stage_bytes, fb = full0 + 8 * stage;
                    mbar_expect_tx(fb, stage_bytes);
                    tma_load_2d(base, &mA_hi, fb, kb * KEL, m0);
                    tma_load_2d(base + a_bytes, &mA_lo, fb, kb * KEL, m0);
                    tma_load_2d(base + 2 * a_bytes, &mB_hi, fb, kb * KEL, n0 + ts.b_row0);
                    tma_load_2d(base + 2 * a_bytes + b_bytes, &mB_lo, fb, kb * KEL, n0 + ts.b_row0);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0) {
            const uint32_t idesc = F16 ? make_idesc16(ts.TN) : make_idesc(ts.TN);
            const uint32_t d_small = tmem_base + kMainAcc * acc_stride;
            int stage = 0; uint32_t phase = 0, tphase = 0;
            int c = 0;                                    // chunk counter (chunked mode), runs on across tiles
            for (int tile = blockIdx.x; chunked && tile < tiles; tile += gridDim.x) {
                int jj = 0;
                uint32_t d_main = tmem_base, d_cross = tmem_base + acc_stride;
                for (int kb = 0; kb < ts.KB; ++kb) {
                    if (kb % CKB == 0) {
                        const int set = c & 1;
                        mbar_wait(cempty0 + 8 * set, (uint32_t)((c >> 1) & 1) ^ 1u);
                        tc_fence_after();
                        d_main = tmem_base + (uint32_t)set * 2 * acc_stride;
                        d_cross = d_main + acc_stride;
                        jj = 0;
                    }
                    mbar_wait(full0 + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t base = ring + stage * stage_bytes;
                    const uint64_t a_hi = make_smem_desc(base), a_lo = make_smem_desc(base + a_bytes);
                    const uint64_t b_hi = make_smem_desc(base + 2 * a_bytes), b_lo = make_smem_desc(base + 2 * a_bytes + b_bytes);
#pragma unroll
                    for (int k = 0; k < 4; ++k, ++jj) {
                        const uint64_t adv = (uint64_t)(k * 32 >> 4);
                        if (F16) {
                            umma_f16(d_cross, a_lo + adv, b_hi + adv, idesc, jj != 0);
                            umma_f16(d_cross, a_hi + adv, b_lo + adv, idesc, 1);
                            umma_f16(d_main, a_hi + adv, b_hi + adv, idesc, jj != 0);
                        } else {
                            umma_tf32(d_cross, a_lo + adv, b_hi + adv, idesc, jj != 0);
                            umma_tf32(d_cross, a_hi + adv, b_lo + adv, idesc, 1);
                            umma_tf32(d_main, a_hi + adv, b_hi + adv, idesc, jj != 0);
                        }
                    }
                    umma_commit(empty0 + 8 * stage);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    if (kb % CKB == CKB - 1 || kb == ts.KB - 1) { umma_commit(cfull0 + 8 * (c & 1)); ++c; }
                }
            }
            for (int tile = blockIdx.x; !chunked && tile < tiles; tile += gridDim.x) {
                mbar_wait(tempty, tphase ^ 1);            // epilogue has drained the accumulators of the previous tile
                tc_fence_after();
                int j = 0;
                for (int kb = 0; kb < ts.KB; ++kb) {
                    mbar_wait(full0 + 8 * stage, phase);
                    tc_fence_after();
                    const uint32_t base = ring + stage * stage_bytes;
                    const uint64_t a_hi = make_smem_desc(base), a_lo = make_smem_desc(base + a_bytes);
                    const uint64_t b_hi = make_smem_desc(base + 2 * a_bytes), b_lo = make_smem_desc(base + 2 * a_bytes + b_bytes);
#pragma unroll
                    for (int k = 0; k < 4; ++k, ++j) {
                        const uint64_t adv = (uint64_t)(k * 32 >> 4);       // 8 TF32 / 16 FP16 = 32 bytes along the swizzled row
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
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(tfull);
                tphase ^= 1;
            }
        }
    } else if (warp >= kEpiWarp0) {
        const int ew = warp - kEpiWarp0;
        const int quarter = warp & 3;                 // a warp may only read TMEM lanes [32*(warpid%4), +32)
        const int g = ew >> 2;                        // which quarter of the tile's trials this warp owns
        const int etid = ew * 32 + lane;
        const int TNq = ts.TN >> 2;
        epi.prepare();
        uint32_t tphase = 0;
        int cchunk = 0;                               // chunk counter (chunked mode), runs on across tiles
        for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
            int m_tile, nt;
            tile_coords(tile, ts.MT, ts.NT, m_tile, nt);
            const int n0 = nt * ts.TN;
            const int row = m_tile * BM + quarter * 32 + lane;
            float tot[kMaxQ];
            if (chunked) {
                const uint32_t lb = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(g * TNq);
#pragma unroll
                for (int q = 0; q < kMaxQ; ++q) tot[q] = 0.f;
                const int nchunks = (ts.KB + CKB - 1) / CKB;
                for (int cc = 0; cc < nchunks; ++cc, ++cchunk) {
                    const int set = cchunk & 1;
                    mbar_wait(cfull0 + 8 * set, (uint32_t)((cchunk >> 1) & 1));
                    tc_fence_after();
                    // four float4 groups per round trip (the drain has to stay shorter than the MMA time of a chunk)
#pragma unroll
                    for (int q0 = 0; q0 < kMaxQ / 4; q0 += 4) {
                        uint32_t um[4][4], ux[4][4];
#pragma unroll
                        for (int d = 0; d < 4; ++d) {
                            if (4 * (q0 + d) < TNq) {
                                tmem_ld4_issue(lb + (uint32_t)set * 2 * acc_stride + 4 * (q0 + d), um[d]);
                                tmem_ld4_issue(lb + (uint32_t)set * 2 * acc_stride + acc_stride + 4 * (q0 + d), ux[d]);
                            }
                        }
                        tmem_ld_wait();
#pragma unroll
                        for (int d = 0; d < 4; ++d) {
                            if (4 * (q0 + d) < TNq) {
#pragma unroll
                                for (int e = 0; e < 4; ++e) tot[4 * (q0 + d) + e] += __uint_as_float(ux[d][e]) * XS + __uint_as_float(um[d][e]);
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(cempty0 + 8 * set);
                }
                epi.rows(m_tile, row, n0, nt, g, TNq, tot);
                epi.tile_done(m_tile, n0, ts.TN, etid, kEpiWarps * 32);
                continue;
            }
            mbar_wait(tfull, tphase);
            tc_fence_after();
            const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(g * TNq);
#pragma unroll
            for (int q = 0; q < kMaxQ / 4; ++q) {
                if (4 * q < TNq) {
                    uint32_t u[kMainAcc + 1][4];
#pragma unroll
                    for (int a = 0; a <= kMainAcc; ++a) tmem_ld4_issue(lane_base + a * acc_stride + 4 * q, u[a]);
                    tmem_ld_wait();
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        float sum = __uint_as_float(u[kMainAcc][e]) * XS;            // cross terms first (small)
#pragma unroll
                        for (int a = 0; a < kMainAcc; ++a) sum += __uint_as_float(u[a][e]);
                        tot[4 * q + e] = sum;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);        // TMEM is free again: warp 1 may start the next tile
            tphase ^= 1;
            epi.rows(m_tile, row, n0, nt, g, TNq, tot);
            epi.tile_done(m_tile, n0, ts.TN, etid, kEpiWarps * 32);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host side: tensor maps, tile shape, launch
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// rows x cols float32 matrix, row-major with `ld` floats per row; box = box_rows x 32 floats, 128-byte swizzle
inline bool make_map(CUtensorMap* map, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * sizeof(float)};
    const cuuint32_t box[2] = {BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rows x cols matrix of 16-bit elements (FP16 or BF16), `ld` elements per row; box = box_rows x 64 elements, 128-byte swizzle
inline bool make_map16(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, bool bf16) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * 2};
    const cuuint32_t box[2] = {BK16, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims,
              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline int num_sms() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// trials per tile: multiple of 16, <= 128, minimising (waves x per-tile cost) -- lands on a multiple of the SM count
inline int pick_tile_n(int MT, int B) {
    const int sms = num_sms();
    int best = 16;
    double best_cost = 1e30;
    for (int tn = 16; tn <= 128; tn += 16) {
        const int nt = (B + tn - 1) / tn;
        const long tiles = (long)MT * nt;
        const long waves = (tiles + sms - 1) / sms;
        const double cost = (double)waves * (tn + 24.0);      // 24: per-tile fixed cost in "trial" units (pipeline fill)
        if (cost < best_cost - 1e-9) { best_cost = cost; best = tn; }
    }
    return best;
}

template <class Epi>
static int launch_contract(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                           const TileShape& ts, const Epi& epi, cudaStream_t s) {
    const size_t smem = (size_t)STAGES * (2 * BM * BK * 4 + 2 * (size_t)ts.TN * BK * 4) + 1024;
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(k_tc_contract<Epi, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(k_tc_contract<Epi, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
            return ODECOL_E_CUDA;
        configured = true;
    }
    const int tiles = ts.MT * ts.NT;
    const int grid = tiles < num_sms() ? tiles : num_sms();
    if (ts.KB > kChunkMin) k_tc_contract<Epi, true><<<grid, kThreads, smem, s>>>(a_hi, a_lo, b_hi, b_lo, ts, epi);
    else k_tc_contract<Epi, false><<<grid, kThreads, smem, s>>>(a_hi, a_lo, b_hi, b_lo, ts, epi);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

// the same with both operands as FP16 pairs (maps from make_map16; ts.KB = K / 64)
template <class Epi>
static int launch_contract16(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                             const TileShape& ts, const Epi& epi, cudaStream_t s) {
    const size_t smem = (size_t)STAGES * (2 * BM * 128 + 2 * (size_t)ts.TN * 128) + 1024;
    static bool configured = false;
    if (!configured) {
        if (cudaFuncSetAttribute(k_tc_contract<Epi, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess ||
            cudaFuncSetAttribute(k_tc_contract<Epi, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess)
            return ODECOL_E_CUDA;
        configured = true;
    }
    const int tiles = ts.MT * ts.NT;
    const int grid = tiles < num_sms() ? tiles : num_sms();
    if (ts.KB > kChunkMin / 2) k_tc_contract<Epi, true, true><<<grid, kThreads, smem, s>>>(a_hi, a_lo, b_hi, b_lo, ts, epi);
    else k_tc_contract<Epi, false, true><<<grid, kThreads, smem, s>>>(a_hi, a_lo, b_hi, b_lo, ts, epi);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? ODECOL_OK : ODECOL_E_CUDA;
}

// ---------------------------------------------------------------------------------------------------------------
// operand preparation
// ---------------------------------------------------------------------------------------------------------------
static __global__ void k_split_pad(const float* __restrict__ src, int rows, int cols, int ld, float* __restrict__ hi,
                            float* __restrict__ lo, int rows_p, int cols_p) {
    const size_t total = (size_t)rows_p * cols_p;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols_p), c = (int)(e % cols_p);
        const float x = (r < rows && c < cols) ? src[(size_t)r * ld + c] : 0.0f;
        const float h = tf32_rna(x);
        hi[e] = h;
        lo[e] = tf32_rna(x - h);
    }
}

// max |src| as a float bit pattern (non-negative floats order like unsigned integers); *out zeroed by the caller
static __global__ void k_absmax(const float* __restrict__ src, int rows, int cols, int ld, unsigned int* __restrict__ out) {
    unsigned int m = 0;
    const size_t total = (size_t)rows * cols;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const float x = fabsf(src[(e / cols) * ld + (e % cols)]);
        if (x == x && x < 3.0e38f) m = max(m, __float_as_uint(x));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}
// W s = wh + wl / 2048 in FP16, zero padded; s = the power of two with max|W| s in [2^13, 2^14); wscale[0] = 1 / s
static __global__ void k_split16_w(const float* __restrict__ src, int rows, int cols, int ld, __half* __restrict__ hi,
                                   __half* __restrict__ lo, int rows_p, int cols_p, const unsigned int* __restrict__ amax,
                                   float* __restrict__ wscale) {
    const float m = __uint_as_float(*amax);
    int ex = 0;
    if (m > 0.f) frexpf(m, &ex);                       // m = f 2^ex, f in [0.5, 1)
    const int sh = m > 0.f ? max(-100, min(100, 14 - ex)) : 0;      // shifts beyond +-100: weights of 1e-35 / 1e+35
    const float sc = ldexpf(1.0f, sh);
    if (blockIdx.x == 0 && threadIdx.x == 0) wscale[0] = ldexpf(1.0f, -sh);
    unsigned int* ovf = reinterpret_cast<unsigned int*>(wscale + 2);   // the format's overflow flag (Mixed16::wscale)
    const size_t total = (size_t)rows_p * cols_p;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols_p), c = (int)(e % cols_p);
        const float x = (r < rows && c < cols) ? src[(size_t)r * ld + c] * sc : 0.0f;
        if (!(fabsf(x) <= kF16Limit)) *ovf = 1u;       // non-finite weights, or a clamped shift: the TF32 repeat takes over
        const F16x2 t = f16_split2(x);
        hi[e] = __ushort_as_half(t.h);
        lo[e] = __ushort_as_half(t.l);
    }
}
// r = hi + lo (a TF32-split K-major operand buffer) re-split into two FP16 planes of KP16 columns, zero padded
static __global__ void k_r16_from32(const float* __restrict__ hi, const float* __restrict__ lo, int Bp, int KPa,
                                    uint16_t* __restrict__ R16, int KP16, unsigned int* __restrict__ ovf) {
    const size_t total = (size_t)Bp * KP16, plane = total;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / KP16), k = (int)(e % KP16);
        const float x = k < KPa ? hi[(size_t)b * KPa + k] + lo[(size_t)b * KPa + k] : 0.0f;
        if (!(fabsf(x) <= kF16Limit)) *ovf = 1u;
        const F16x2 t = f16_split2(x);
        R16[e] = t.h; R16[plane + e] = t.l;
    }
}

// component -> position in the selection (-1: not selected); sel == NULL selects everything in order
// inv[n3] = 1 iff some F component (index >= 2 n3 / 3) is selected: F never feeds back into the dynamics, so when the
// loss does not read it the forward sweep (checkpoint mode) need not advance it and its adjoint is identically zero
static __global__ void k_tc_build_inv(const int* __restrict__ sel, int G, int n3, int* __restrict__ inv) {
    for (int e = threadIdx.x; e < n3; e += blockDim.x) inv[e] = sel ? -1 : e;
    if (threadIdx.x == 0) inv[n3] = sel ? 0 : 1;
    __syncthreads();
    if (sel) for (int g = threadIdx.x; g < G; g += blockDim.x) {
        inv[sel[g]] = g;
        if (sel[g] >= 2 * (n3 / 3)) inv[n3] = 1;
    }
}

// out[b][g] = y[b][sel[g]]
static __global__ void k_tc_gather_sel(const float* __restrict__ y, const int* __restrict__ sel, int G, int B, int n3,
                                       float* __restrict__ out) {
    const size_t total = (size_t)B * G;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / G), g = (int)(e % G);
        out[e] = y[(size_t)b * n3 + (sel ? sel[g] : g)];
    }
}

// checkpoints of the forward sweep for the reverse sweep (all tile-major planes of Np x Bp floats):
//   VA: T slots x {V, A} at the grid points;  K: (T-1) slots x {k1V, k2V, k3V}, the V slopes of stages 1..3 of each step.
// With them the reverse sweep re-derives every stage state elementwise (no contraction is recomputed).
struct CkptView {
    float* VA; float* K;
    float* y_sel;          // (T, B, G) selected components of the trajectory (forward output), or NULL in the reverse sweep
    const int* inv;        // [3N]
    int G;
};

// fast, FP32-accurate elementwise math (exp_fast, tanh_small, phi_fast, phi_dphi_fast): odecol_common.cuh

// tile-major scratch: element (component c, population i, trial b) with b = nt*TN + g*TNq + 4q + e lives at
//   c*plane + ((((nt*4 + g)*(TNq/4) + q)*Np + i)*4 + e
// so the float4 a thread reads for (q, i) sits next to its lane neighbours' (i +- 1): every warp request is one fully
// used 512-byte run and no sector is ever touched twice (the first layout, row-per-thread, re-read each sector 25 us
// later and lost it from L2 in between: 6x the DRAM traffic, profiles/r1_tc_v2_ncu.txt).
struct TileGeom {
    int NT, Np, TN, TNq;
    __host__ __device__ __forceinline__ size_t plane() const { return (size_t)NT * 4 * Np * TNq; }
    ODECOL_DEVINL size_t off(int nt, int g, int q, int i) const {
        return ((((size_t)nt * 4 + g) * (TNq >> 2) + q) * Np + i) * 4;
    }
};

// Stimulus columns [N, N + n_in) of a K-major operand (hi / lo split) for the trials [n0, n0 + tile_n) at ONE query time
// (knot interval idx, clamped time tcl: knot_locate): share `part` of `parts` equal shares of the entries, walked by
// `nthr` threads.  Four consecutive channels per thread -- two 16-byte loads of the knot values, the interpolation in
// knot_value's operations and order (bit-identical), two 16-byte stores -- when the rows allow it; the entry index is
// carried incrementally (one integer division per thread instead of two per entry).
ODECOL_DEVINL void stimulus_columns(const DevProblem& p, int KPa, int idx, float tcl, int n0, int tile_n, int part, int parts,
                                    int tid, int nthr, float* __restrict__ Rhi, float* __restrict__ Rlo) {
    const int n_in = p.n_in, N = p.N;
    const float x0 = __ldg(p.knot_t + idx - 1), x1 = __ldg(p.knot_t + idx);
    const float dx = __fsub_rn(x1, x0), dtc = __fsub_rn(tcl, x0);
    const bool vec = ((n_in | N | KPa | (int)p.knot_stride_b) & 3) == 0 &&
                     ((reinterpret_cast<uintptr_t>(p.knot_u) | reinterpret_cast<uintptr_t>(Rhi) | reinterpret_cast<uintptr_t>(Rlo)) & 15) == 0;
    if (vec) {
        const int nq = n_in >> 2, total = tile_n * nq, share = (total + parts - 1) / parts;
        const int e_end = min(total, (part + 1) * share);
        int e = part * share + tid;
        if (e >= e_end) return;
        int bl = e / nq, c = e - bl * nq;                      // trial within the tile, channel quad
        const int dbl = nthr / nq, dc = nthr - dbl * nq;
        for (; e < e_end; e += nthr) {
            const int b = n0 + bl;
            if (b < p.B) {
                const float* ku = p.knot_u + (size_t)b * p.knot_stride_b + 4 * c;
                const float4 y0 = __ldg(reinterpret_cast<const float4*>(ku + (size_t)(idx - 1) * n_in));
                const float4 y1 = __ldg(reinterpret_cast<const float4*>(ku + (size_t)idx * n_in));
                float4 h, l;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float slope = __fdiv_rn(__fsub_rn((&y1.x)[k], (&y0.x)[k]), dx);
                    const float v = __fadd_rn((&y0.x)[k], __fmul_rn(slope, dtc));
                    (&h.x)[k] = tf32_rna(v);
                    (&l.x)[k] = tf32_rna(v - (&h.x)[k]);
                }
                const size_t at = (size_t)b * KPa + N + 4 * c;
                *reinterpret_cast<float4*>(Rhi + at) = h;
                *reinterpret_cast<float4*>(Rlo + at) = l;
            }
            bl += dbl; c += dc;
            if (c >= nq) { c -= nq; ++bl; }
        }
        return;
    }
    const int total = tile_n * n_in, share = (total + parts - 1) / parts;
    const int e_end = min(total, (part + 1) * share);
    for (int e = part * share + tid; e < e_end; e += nthr) {
        const int b = n0 + e / n_in, ch = e % n_in;
        if (b < p.B) {
            const float v = knot_value(p.knot_t, p.knot_u + (size_t)b * p.knot_stride_b, n_in, idx, tcl, ch);
            const float h = tf32_rna(v);
            Rhi[(size_t)b * KPa + N + ch] = h;
            Rlo[(size_t)b * KPa + N + ch] = tf32_rna(v - h);
        }
    }
}

// the same for the two-plane FP16 operand (plane stride `plane` elements, KP16 columns per row); *ovf = 1 when a value does
// not fit the format
ODECOL_DEVINL void stimulus_columns16(const DevProblem& p, int KP16, size_t plane, int idx, float tcl, int n0, int tile_n, int part,
                                      int parts, int tid, int nthr, uint16_t* __restrict__ R16, unsigned int* __restrict__ ovf) {
    const int n_in = p.n_in, N = p.N;
    const float x0 = __ldg(p.knot_t + idx - 1), x1 = __ldg(p.knot_t + idx);
    const float dx = __fsub_rn(x1, x0), dtc = __fsub_rn(tcl, x0);
    const bool vec = ((n_in | N | KP16 | (int)p.knot_stride_b) & 3) == 0 && (plane & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(p.knot_u) & 15) == 0 && (reinterpret_cast<uintptr_t>(R16) & 7) == 0;
    if (vec) {
        const int nq = n_in >> 2, total = tile_n * nq, share = (total + parts - 1) / parts;
        const int e_end = min(total, (part + 1) * share);
        int e = part * share + tid;
        if (e >= e_end) return;
        int bl = e / nq, c = e - bl * nq;
        const int dbl = nthr / nq, dc = nthr - dbl * nq;
        for (; e < e_end; e += nthr) {
            const int b = n0 + bl;
            if (b < p.B) {
                const float* ku = p.knot_u + (size_t)b * p.knot_stride_b + 4 * c;
                const float4 y0 = __ldg(reinterpret_cast<const float4*>(ku + (size_t)(idx - 1) * n_in));
                const float4 y1 = __ldg(reinterpret_cast<const float4*>(ku + (size_t)idx * n_in));
                F16x2 t[4];
                bool big = false;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float slope = __fdiv_rn(__fsub_rn((&y1.x)[k], (&y0.x)[k]), dx);
                    const float v = __fadd_rn((&y0.x)[k], __fmul_rn(slope, dtc));
                    big |= !(fabsf(v) <= kF16Limit);
                    t[k] = f16_split2(v);
                }
                if (big) *ovf = 1u;
                uint16_t* at = R16 + (size_t)b * KP16 + N + 4 * c;
                *reinterpret_cast<uint2*>(at) = make_uint2((uint32_t)t[0].h | ((uint32_t)t[1].h << 16), (uint32_t)t[2].h | ((uint32_t)t[3].h << 16));
                *reinterpret_cast<uint2*>(at + plane) = make_uint2((uint32_t)t[0].l | ((uint32_t)t[1].l << 16), (uint32_t)t[2].l | ((uint32_t)t[3].l << 16));
            }
            bl += dbl; c += dc;
            if (c >= nq) { c -= nq; ++bl; }
        }
        return;
    }
    const int total = tile_n * n_in, share = (total + parts - 1) / parts;
    const int e_end = min(total, (part + 1) * share);
    for (int e = part * share + tid; e < e_end; e += nthr) {
        const int b = n0 + e / n_in, ch = e % n_in;
        if (b < p.B) {
            const float v = knot_value(p.knot_t, p.knot_u + (size_t)b * p.knot_stride_b, n_in, idx, tcl, ch);
            if (!(fabsf(v) <= kF16Limit)) *ovf = 1u;
            const F16x2 t = f16_split2(v);
            uint16_t* at = R16 + (size_t)b * KP16 + N + ch;
            at[0] = t.h; at[plane] = t.l;
        }
    }
}

// Forward stage epilogue (3/8 rule, reference step: torchdiffeq rk_common.py rk4_alt_step_func).  Only what cannot be
// recomputed crosses a stage boundary through HBM: the V slope of each stage (it carries the contraction).  The rates
// r_1 .. r_S of the earlier stages are recomputed from the step's start state and the stored V slopes -- the recurrences
// of the checkpoint replay -- and the A and F slopes, linear in r, are re-derived in registers from A0 / F0 and r_1..r_S
// with the same expressions, in the same order, as a kernel that had stored them; F is only touched at stage 4.  A stage
// pass costs about 1.45 us per byte per element, a phi evaluation about 2 us per pass: recomputing r instead of keeping
// it in four planes takes the epilogues from 28 / 36 / 44 / 56 to 20 / 24 / 28 / 36 bytes per element (stages 1..4,
// +12 for the trajectory).
template <int S, bool F16 = false>      // F16: the next operand is written in the 16-bit format (two FP16 planes)
struct FwdEpiT {
    DevProblem p;
    TileGeom tg;
    const float* t;
    int n, KPa;
    uint16_t* R16_nxt; size_t r16_plane; int KP16;     // F16: operand of the next contraction, [2 planes][Bp][KP16]
    const float* wscale;                               // F16: [0] = 1 / (power-of-two scale of the FP16 weight planes)
    unsigned int* ovf;                                 // F16: raised when an operand value does not fit FP16
    float ws;
    const float* V0T; const float* A0T; const float* F0T;   // [1 plane each] state at the start of the step (tile-major)
    float* V1T; float* A1T; float* F1T;                      // stage 4: state at the end of the step (tile-major)
    float* traj_row;       // stage 4: (B, 3N) row of the trajectory, or NULL
    float* ysel_row;       // stage 4: (B, G) row of the selected components (checkpoint mode), or NULL
    const int* inv;        // [3N] component -> position in the selection, -1 if not selected (with ysel_row)
    int G;
    float* K1T; float* K2T; float* K3T;     // [1 plane] each: V slope of stages 1..3
    float* Rhi_nxt; float* Rlo_nxt;         // [Bp][KPa] operand of the next contraction
    float* DRT_nxt;        // optional [1 plane]: phi'(x) of the next stage state (reverse-sweep recompute)
    float inv_tm, inv_ta, inv_ts;
    float t0, t1, dt;
    int needF;             // stage 4: advance F (always, except in checkpoint mode when no F component is selected)

    ODECOL_DEVINL void prepare() {
        t0 = __ldg(t + n); t1 = __ldg(t + n + 1);
        dt = __fsub_rn(t1, t0);
        needF = (S == 4 && ysel_row && inv && !traj_row) ? __ldg(inv + 3 * p.N) : 1;
        ws = F16 ? __ldg(wscale) : 1.0f;
    }

    // One float4 group (4 trials) of population i: what stage S reads from the scratch planes.
    struct Group { float4 V0, A0, k1V, k2V, k3V, F0; };
    ODECOL_DEVINL void load_group(Group& L, size_t oq) const {
        L.V0 = ld4s(V0T + oq); L.A0 = ld4s(A0T + oq);
        if (S >= 2) L.k1V = ld4s(K1T + oq);
        if (S >= 3) L.k2V = ld4s(K2T + oq);
        if (S >= 4) { L.k3V = ld4s(K3T + oq); if (needF) L.F0 = ld4s(F0T + oq); }
    }

    // The group loop is rolled (its body is ~1000 instructions; seven unrolled copies missed the instruction cache) and
    // software-pipelined: the loads of group q+1 are issued before group q is processed, so the memory system is never
    // idle while a warp does arithmetic.  tot[] is indexed at run time and therefore lives in local memory (L1).
    ODECOL_DEVINL void rows(int, int i, int n0, int nt, int g, int TNq, const float (&tot)[kMaxQ]) const {
        if (i >= p.N) return;
        const int N = p.N, B = p.B;
        const float kap = __ldg(p.kappa + i);
        const float third = kOneThirdL;
        const int nq = TNq >> 2;
        const size_t qstride = (size_t)tg.Np * 4;
        const size_t o0 = tg.off(nt, g, 0, i);
        int gV = -1, gA = -1, gF = -1;
        if (S == 4 && ysel_row) { gV = __ldg(inv + i); gA = __ldg(inv + N + i); gF = __ldg(inv + 2 * N + i); }
        Group nxt;
        load_group(nxt, o0);
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
            const size_t oq = o0 + q * qstride;
            const Group L = nxt;
            if (q + 1 < nq) load_group(nxt, oq + qstride);
            const float4 &V0 = L.V0, &A0 = L.A0, &F0 = L.F0;
            const float4 &k1V = L.k1V, &k2V = L.k2V, &k3V = L.k3V;
            const int q4 = 4 * q;
            float oKV[4], oNV[4], oNA[4], oNF[4], oR[4], oD[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float v0 = (&V0.x)[e], a0 = (&A0.x)[e];
                // A (and at stage 4 F) slopes of the earlier stages, re-derived from the rates r_1 .. r_{S-1}; the rates
                // themselves from the stage states, which follow from V0, A0 and the V slopes
                float k1A = 0.f, k2A = 0.f, k3A = 0.f, A = a0, V = v0;
                float r2 = 0.f, r3 = 0.f;
                const float r1 = phi_fast(v0 - a0);
                float r = r1;
                if (S >= 2) {
                    k1A = (kap * r1 - a0) * inv_ta;
                    const float v2 = v0 + dt * (&k1V.x)[e] * third, a2 = a0 + dt * k1A * third;
                    r2 = phi_fast(v2 - a2);
                    if (S == 2) { V = v2; A = a2; r = r2; }
                    if (S >= 3) {
                        k2A = (kap * r2 - a2) * inv_ta;
                        const float v3 = v0 + dt * ((&k2V.x)[e] - (&k1V.x)[e] * third), a3 = a0 + dt * (k2A - k1A * third);
                        r3 = phi_fast(v3 - a3);
                        if (S == 3) { V = v3; A = a3; r = r3; }
                        if (S >= 4) {
                            k3A = (kap * r3 - a3) * inv_ta;
                            V = v0 + dt * ((&k1V.x)[e] - (&k2V.x)[e] + (&k3V.x)[e]); A = a0 + dt * (k1A - k2A + k3A);
                            r = phi_fast(V - A);
                        }
                    }
                }
                const float total = (F16 ? tot[q4 + e] * ws : tot[q4 + e]) * p.c.tau_s;
                const float dV = (total * p.c.R - V) * inv_tm;
                const float dA = (kap * r - A) * inv_ta;
                oKV[e] = dV;
                float nV, nA, nF = 0.f;
                if (S == 1) { nV = v0 + dt * dV * third; nA = a0 + dt * dA * third; }
                if (S == 2) { nV = v0 + dt * (dV - (&k1V.x)[e] * third); nA = a0 + dt * (dA - k1A * third); }
                if (S == 3) { nV = v0 + dt * ((&k1V.x)[e] - (&k2V.x)[e] + dV); nA = a0 + dt * (k1A - k2A + dA); }
                if (S == 4) {
                    nV = v0 + ((&k1V.x)[e] + 3.f * ((&k2V.x)[e] + (&k3V.x)[e]) + dV) * dt * 0.125f;
                    nA = a0 + (k1A + 3.f * (k2A + k3A) + dA) * dt * 0.125f;
                    if (needF) {
                    const float f0 = (&F0.x)[e];
                    const float k1F = (r1 - f0) * inv_ts;
                    const float f2 = f0 + dt * k1F * third;
                    const float k2F = (r2 - f2) * inv_ts;
                    const float f3 = f0 + dt * (k2F - k1F * third);
                    const float k3F = (r3 - f3) * inv_ts;
                    const float f4 = f0 + dt * (k1F - k2F + k3F);
                    const float k4F = (r - f4) * inv_ts;
                    nF = f0 + (k1F + 3.f * (k2F + k3F) + k4F) * dt * 0.125f;
                    }
                }
                oNV[e] = nV; oNA[e] = nA; oNF[e] = nF;
                if (DRT_nxt) phi_dphi_fast(nV - nA, oR[e], oD[e]);
                else oR[e] = phi_fast(nV - nA);
            }
            if (DRT_nxt) st4s(DRT_nxt + oq, make_float4(oD[0], oD[1], oD[2], oD[3]));
            const float4 kV4 = make_float4(oKV[0], oKV[1], oKV[2], oKV[3]);
            if (S == 1) st4s(K1T + oq, kV4);
            if (S == 2) st4s(K2T + oq, kV4);
            if (S == 3) st4s(K3T + oq, kV4);
            if (S == 4) {
                st4s(V1T + oq, make_float4(oNV[0], oNV[1], oNV[2], oNV[3]));
                st4s(A1T + oq, make_float4(oNA[0], oNA[1], oNA[2], oNA[3]));
                if (needF) st4s(F1T + oq, make_float4(oNF[0], oNF[1], oNF[2], oNF[3]));
            }
            // operand rows of the next contraction: one 64-bit row address per group, the other seven stores at fixed
            // offsets from it, predicated (the branchy form spent ~27 instructions per element on these two stores)
            const int b0 = n0 + g * TNq + q4;
            float* rh = Rhi_nxt + (size_t)b0 * KPa + i;
            const ptrdiff_t lo_off = Rlo_nxt - Rhi_nxt;
            float* yr = (S == 4 && traj_row) ? traj_row + (size_t)b0 * 3 * N + i : nullptr;
            uint16_t* r16 = F16 ? R16_nxt + (size_t)b0 * KP16 + i : nullptr;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const bool ok = b0 + e < B;
                if (F16) {
                    const F16x2 t2 = f16_split2(oR[e]);
                    uint16_t* ph = r16 + (size_t)e * KP16;
                    st_global_u16_if(ph, t2.h, ok);
                    st_global_u16_if(ph + r16_plane, t2.l, ok);
                    if (ok && !(fabsf(oR[e]) <= kF16Limit)) *ovf = 1u;
                } else {
                    const float h = tf32_rna(oR[e]);
                    float* ph = rh + (size_t)e * KPa;
                    st_global_if(ph, h, ok);
                    st_global_if(ph + lo_off, tf32_rna(oR[e] - h), ok);
                }
                if (S == 4 && yr && ok) {
                    float* y = yr + (size_t)e * 3 * N;
                    st_global(y, oNV[e]); st_global(y + N, oNA[e]); st_global(y + 2 * N, oNF[e]);
                }
                if (S == 4 && ysel_row) {          // selected components: predicated stores (most populations select nothing)
                    float* y = ysel_row + (size_t)(b0 + e) * G;
                    st_global_if(y + gV, oNV[e], ok && gV >= 0);
                    st_global_if(y + gA, oNA[e], ok && gA >= 0);
                    st_global_if(y + gF, oNF[e], ok && gF >= 0);
                }
            }
        }
    }

    // stimulus columns of the next operand, written once per trial tile: the population tiles of a trial tile share the
    // entries evenly (one CTA doing all of them finished 25 us after the others and set the pace of every stage)
    ODECOL_DEVINL void tile_done(int m_tile, int n0, int tile_n, int etid, int nthr) const {
        if (p.n_in == 0) return;
        const float tn = S == 1 ? __fadd_rn(t0, __fmul_rn(dt, kOneThirdL)) : S == 2 ? __fadd_rn(t0, __fmul_rn(dt, kTwoThirdsL)) : t1;
        int idx = 1;
        const float tcl = knot_locate(p.knot_t, p.K, tn, idx);
        const int MT = tg.Np / BM;
        if (F16) stimulus_columns16(p, KP16, r16_plane, idx, tcl, n0, tile_n, m_tile, MT, etid, nthr, R16_nxt, ovf);
        else stimulus_columns(p, KPa, idx, tcl, n0, tile_n, m_tile, MT, etid, nthr, Rhi_nxt, Rlo_nxt);
    }
};


}  // namespace tc
}  // namespace odecol
