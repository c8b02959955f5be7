// C-ABI shim (include/odecol.h): validates arguments, picks the kernel family, launches on the caller's stream.
// No allocation, no synchronisation, no global state that affects results (one diagnostic launch counter).
#include <atomic>
#include <cstring>
#include <cmath>
#include "odecol_internal.h"

namespace odecol {

// diagnostic only: kernels enqueued by the most recent call (autograd runs backward on its own thread, so this is a
// process-wide relaxed atomic rather than a thread-local; it never influences a computation)
static std::atomic<int64_t> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static int to_dev(const odecol_problem* p, DevProblem& d) {
    if (!p || !p->W_aug || !p->kappa || !p->knot_t || !p->knot_u) return ODECOL_E_NULL;
    if (p->N <= 0 || p->B <= 0 || p->n_in < 0 || p->K < 2) return ODECOL_E_SHAPE;
    if (p->ld_w < p->N + p->n_in + 1 || (p->ld_w & 3)) return ODECOL_E_SHAPE;
    if ((reinterpret_cast<uintptr_t>(p->W_aug) & 15) || (reinterpret_cast<uintptr_t>(p->kappa) & 15)) return ODECOL_E_ALIGN;
    d.N = p->N; d.n_in = p->n_in; d.B = p->B; d.K = p->K; d.ld_w = p->ld_w; d.flags = p->flags;
    d.W_aug = p->W_aug; d.kappa = p->kappa; d.sigma = p->sigma; d.sigma_scale = p->sigma_scale; d.lat_gain = p->lat_gain; d.W_local = p->lat_gain ? p->W_local : nullptr; d.knot_t = p->knot_t; d.knot_u = p->knot_u;
    d.knot_stride_b = p->knot_stride_b;
    d.c.tau_s = p->tau_s; d.c.tau_m = p->tau_m; d.c.tau_a = p->tau_a; d.c.R = p->resistance;
    return ODECOL_OK;
}

static bool use_small(const odecol_problem* p, const DevProblem& d) {
    return !(p->flags & (ODECOL_FLAG_FORCE_STAGED | ODECOL_FLAG_FORCE_TENSOR)) && small_kp(d) != 0;
}

// rk4 of a network that FITS the on-chip family still goes to the tensor family when the batch is large enough to fill the
// machine with 128-row tiles: measured on the reference's parity network (N = 104; bench.py --workload small, round 2) the
// two families break even at ~2048 trials (forward + adjoint 1.77e9 vs 1.67e9 population-steps/s); at 4096 trials the
// tensor family is 1.9x (3.47e9 vs 1.79e9), at 16,384 trials 3.4x (6.13e9 vs 1.82e9; forward only 1.68e10 vs 9.1e9).  Small
// networks (WTA N = 16, XOR N = 24) would waste most of a 128-row tile and stay on chip at every batch size.
static bool use_small_rk4(const odecol_problem* p, const DevProblem& d) {
    if (!use_small(p, d)) return false;
    return !(d.B >= 4096 && d.N >= 64 && d.N % 4 == 0);
}

static inline bool misaligned(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) != 0; }

struct EmScheduleLayout { size_t off_step, off_w, off_tk, total; };
static EmScheduleLayout em_schedule_layout(int T, int64_t n_steps) {
    EmScheduleLayout L;
    auto up = [](size_t x) { return (x + 255) / 256 * 256; };
    L.off_step = 0;
    L.off_w = up(sizeof(int) * (size_t)(T + 1));
    L.off_tk = L.off_w + up(sizeof(float) * 2 * (size_t)T);
    L.total = L.off_tk + up(sizeof(float) * (size_t)(n_steps + 1));
    return L;
}

}  // namespace odecol

using namespace odecol;

extern "C" {

int odecol_abi_version(void) { return ODECOL_ABI_VERSION; }

const char* odecol_strerror(int code) {
    switch (code) {
        case ODECOL_OK: return "ok";
        case ODECOL_E_NULL: return "required pointer is NULL";
        case ODECOL_E_SHAPE: return "N, B, T, K, n_in or ld_w out of range";
        case ODECOL_E_UNSUPPORTED: return "no kernel for this request";
        case ODECOL_E_WORKSPACE: return "workspace missing or too small";
        case ODECOL_E_CUDA: return "CUDA launch failed";
        case ODECOL_E_ALIGN: return "pointer not 16-byte aligned";
        default: return "unknown odecol error";
    }
}

int64_t odecol_last_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int odecol_kernel_family(const odecol_problem* p, int op) {
    DevProblem d;
    if (to_dev(p, d) != ODECOL_OK) return -1;
    // rk4 beyond the on-chip family runs in the tensor family (persistent tcgen05 forward solve, checkpoint mode, chained
    // reverse stages); the other solvers' staged paths are family 1
    const bool rk4 = op == ODECOL_OP_RK4_FWD || op == ODECOL_OP_RK4_BWD;
    if (rk4 ? use_small_rk4(p, d) : use_small(p, d)) return 0;
    return rk4 ? 2 : 1;
}

size_t odecol_workspace_bytes(const odecol_problem* p, int op, int32_t T, int64_t n_steps) {
    DevProblem d;
    if (to_dev(p, d) != ODECOL_OK) return 0;
    const bool small = use_small(p, d), small_rk4 = use_small_rk4(p, d);
    switch (op) {
        case ODECOL_OP_RK4_FWD: return small_rk4 ? (tiny_rk4_applicable(d) ? 256 : 0) : tc_rk4_fwd_workspace_bytes(d, T);
        case ODECOL_OP_RK4_BWD: return small_rk4 ? 0 : tc_rk4_bwd_workspace_bytes(d, T);
        case ODECOL_OP_EM_FWD: return small ? 0 : stage_em_fwd_workspace_bytes(d, T);
        case ODECOL_OP_DOPRI5_FWD: return small ? 0 : stage_dopri5_fwd_workspace_bytes(d, T);
        case ODECOL_OP_DOPRI5_BWD: return small ? 0 : stage_dopri5_bwd_workspace_bytes(d, T);
        case ODECOL_OP_EM_BWD: return small ? em_schedule_layout(T, n_steps).total : stage_sde_bwd_workspace_bytes(d, T);
        case ODECOL_OP_SRK_FWD: return small ? 0 : stage_srk_fwd_workspace_bytes(d, T);
        case ODECOL_OP_SRK_BWD: return small ? em_schedule_layout(T, n_steps).total : stage_sde_bwd_workspace_bytes(d, T);
        default: return 0;
    }
}

int odecol_rhs(const odecol_problem* p, const float* t, const float* y, float* f, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y || !f) return ODECOL_E_NULL;
    g_launches.store(0, std::memory_order_relaxed);
    return launch_rhs_generic(d, t, y, f, static_cast<cudaStream_t>(stream));
}

int odecol_drift_staged(const odecol_problem* p, const float* t, const float* y, float* f, void* workspace,
                        size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (!t || !y || !f) return ODECOL_E_NULL;
    if (misaligned(y) || misaligned(f) || misaligned(workspace)) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return stage_drift(d, t, y, f, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int odecol_rk4_fwd(const odecol_problem* p, const float* t, int32_t T, const float* y0, float* y_out,
                   int32_t out_every, void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y0 || !y_out) return ODECOL_E_NULL;
    if (T < 2 || out_every < 1) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (use_small_rk4(p, d)) {
        // tens of thousands of trials of a network of <= 16 populations: trials on the M axis of the tensor core (FP16 pairs),
        // followed by the on-chip kernel, which returns at once unless the 16-bit solve raised its overflow flag
        if (tiny_rk4_applicable(d) && workspace && workspace_bytes >= 256 && !misaligned(workspace)) {
            unsigned int* ovf = static_cast<unsigned int*>(workspace);
            const int rt = launch_rk4_fwd_tiny(d, t, T, y0, y_out, out_every, ovf, s);
            if (rt != ODECOL_OK) return rt;
            return launch_rk4_fwd_small(d, t, T, y0, y_out, out_every, s, ovf);
        }
        return launch_rk4_fwd_small(d, t, T, y0, y_out, out_every, s);
    }
    if (misaligned(y0) || misaligned(y_out) || misaligned(workspace)) return ODECOL_E_ALIGN;
    return tc_rk4_fwd(d, t, T, y0, y_out, out_every, workspace, workspace_bytes, s);
}

int odecol_rk4_bwd(const odecol_problem* p, const float* t, int32_t T, const float* y_traj, const float* grad_y,
                   const int32_t* sel, int32_t G, float* grad_y0, float* grad_W_aug, void* workspace,
                   size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y_traj || !grad_y || !grad_W_aug) return ODECOL_E_NULL;
    if (T < 2 || G < 1 || G > 3 * p->N) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (cudaMemsetAsync(grad_W_aug, 0, sizeof(float) * (size_t)p->N * p->ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
    if (use_small_rk4(p, d)) return launch_rk4_bwd_small(d, t, T, y_traj, grad_y, sel, G, grad_y0, grad_W_aug, s);
    if (misaligned(y_traj) || misaligned(workspace) || misaligned(grad_W_aug)) return ODECOL_E_ALIGN;
    return tc_rk4_bwd(d, t, T, y_traj, grad_y, sel, G, grad_y0, grad_W_aug, workspace, workspace_bytes, s);
}

size_t odecol_rk4_ckpt_bytes(const odecol_problem* p, int32_t T) {
    DevProblem d;
    if (to_dev(p, d) != ODECOL_OK || T < 2) return 0;
    if (use_small_rk4(p, d) || p->N % 4 != 0) return 0;
    return tc_rk4_ckpt_bytes(d, T);
}

int odecol_rk4_fwd_ckpt(const odecol_problem* p, const float* t, int32_t T, const float* y0, const int32_t* sel, int32_t G,
                        float* y_sel, void* ckpt, size_t ckpt_bytes, void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y0 || !y_sel || !ckpt) return ODECOL_E_NULL;
    if (T < 2 || G < 1 || G > 3 * p->N) return ODECOL_E_SHAPE;
    if (use_small_rk4(p, d)) return ODECOL_E_UNSUPPORTED;
    if (misaligned(y0) || misaligned(ckpt) || misaligned(workspace)) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return tc_rk4_fwd_ckpt(d, t, T, y0, sel, G, y_sel, ckpt, ckpt_bytes, workspace, workspace_bytes,
                           static_cast<cudaStream_t>(stream));
}

int odecol_rk4_bwd_ckpt(const odecol_problem* p, const float* t, int32_t T, const void* ckpt, size_t ckpt_bytes,
                        const float* grad_y_sel, const int32_t* sel, int32_t G, float* grad_y0, float* grad_W_aug,
                        void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !ckpt || !grad_y_sel || !grad_W_aug) return ODECOL_E_NULL;
    if (T < 2 || G < 1 || G > 3 * p->N) return ODECOL_E_SHAPE;
    if (use_small_rk4(p, d)) return ODECOL_E_UNSUPPORTED;
    if (misaligned(ckpt) || misaligned(workspace) || misaligned(grad_W_aug)) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (cudaMemsetAsync(grad_W_aug, 0, sizeof(float) * (size_t)p->N * p->ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
    return tc_rk4_bwd_ckpt(d, t, T, ckpt, ckpt_bytes, grad_y_sel, sel, G, grad_y0, grad_W_aug, workspace, workspace_bytes, s);
}

int odecol_dopri5_fwd(const odecol_problem* p, const float* t, int32_t T, const float* y0, float* y_out, float rtol,
                      float atol, int32_t max_steps, int32_t* n_accept, int32_t* n_reject, int32_t* status,
                      void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y0 || !y_out) return ODECOL_E_NULL;
    if (T < 2 || max_steps < 1 || !(rtol >= 0.f) || !(atol >= 0.f)) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    if (!use_small(p, d)) {                              // beyond the on-chip family (or forced): staged solver, forward only
        if (misaligned(y0) || misaligned(y_out) || misaligned(workspace)) return ODECOL_E_ALIGN;
        const Dopri5Record norec{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
        return stage_dopri5_fwd(d, t, T, y0, y_out, rtol, atol, max_steps, n_accept, n_reject, status, norec, workspace,
                                workspace_bytes, static_cast<cudaStream_t>(stream));
    }
    const Dopri5Record none{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
    return launch_dopri5_fwd_small(d, t, T, y0, y_out, rtol, atol, max_steps, n_accept, n_reject, status, none,
                                   static_cast<cudaStream_t>(stream));
}

int odecol_dopri5_fwd_record(const odecol_problem* p, const float* t, int32_t T, const float* y0, float* y_out, float rtol,
                             float atol, int32_t max_steps, int32_t* n_accept, int32_t* n_reject, int32_t* status,
                             float* rec_y, double* rec_t0, double* rec_dt, int32_t* out_step, float* out_x, int32_t cap,
                             void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!t || !y0 || !y_out || !n_accept || !rec_y || !rec_t0 || !rec_dt || !out_step || !out_x) return ODECOL_E_NULL;
    if (T < 2 || max_steps < 1 || cap < 1 || !(rtol >= 0.f) || !(atol >= 0.f)) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    const Dopri5Record rec{rec_y, rec_t0, rec_dt, out_step, out_x, cap};
    if (!use_small(p, d)) {                              // staged solver: the same record, written by its commit kernel
        if (misaligned(y0) || misaligned(y_out) || misaligned(workspace) || misaligned(rec_y)) return ODECOL_E_ALIGN;
        return stage_dopri5_fwd(d, t, T, y0, y_out, rtol, atol, max_steps, n_accept, n_reject, status, rec, workspace,
                                workspace_bytes, static_cast<cudaStream_t>(stream));
    }
    return launch_dopri5_fwd_small(d, t, T, y0, y_out, rtol, atol, max_steps, n_accept, n_reject, status, rec,
                                   static_cast<cudaStream_t>(stream));
}

int odecol_dopri5_bwd(const odecol_problem* p, int32_t T, const float* rec_y, const double* rec_t0, const double* rec_dt,
                      const int32_t* out_step, const float* out_x, int32_t cap, const int32_t* n_accept,
                      const float* grad_y, const int32_t* sel, int32_t G, float* grad_y0, float* grad_W_aug,
                      void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!rec_y || !rec_t0 || !rec_dt || !out_step || !out_x || !n_accept || !grad_y || !grad_W_aug) return ODECOL_E_NULL;
    if (T < 2 || cap < 1 || G < 1 || G > 3 * p->N) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!use_small(p, d)) {                              // staged reverse sweep in rounds (tensor-core VJPs)
        if (misaligned(workspace) || misaligned(rec_y)) return ODECOL_E_ALIGN;
        const Dopri5Record recs{const_cast<float*>(rec_y), const_cast<double*>(rec_t0), const_cast<double*>(rec_dt),
                                const_cast<int*>(out_step), const_cast<float*>(out_x), cap};
        return stage_dopri5_bwd(d, T, recs, n_accept, grad_y, sel, G, grad_y0, grad_W_aug, workspace, workspace_bytes, s);
    }
    if (cudaMemsetAsync(grad_W_aug, 0, sizeof(float) * (size_t)p->N * p->ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
    const Dopri5Record rec{const_cast<float*>(rec_y), const_cast<double*>(rec_t0), const_cast<double*>(rec_dt),
                           const_cast<int*>(out_step), const_cast<float*>(out_x), cap};
    return launch_dopri5_bwd_small(d, T, rec, n_accept, grad_y, sel, G, grad_y0, grad_W_aug, s);
}

int64_t odecol_em_num_steps(const float* ts, int32_t T, float dt) {
    if (!ts || T < 2 || !(dt > 0.f)) return -1;
    // the float32 loop of torchsde's integrate(): curr_t += dt, clipped to ts[T-1]
    volatile float curr = ts[0];
    const float t_end = ts[T - 1];
    int64_t k = 0;
    for (int j = 1; j < T; ++j) {
        const float out_t = ts[j];
        while (curr < out_t) {
            volatile float nxt = curr + dt;
            curr = nxt < t_end ? nxt : t_end;
            ++k;
            if (k > (int64_t)1 << 40) return -1;
        }
    }
    return k;
}

int odecol_em_fwd(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out, const float* dW,
                  uint64_t seed, int64_t trial_offset, float dt, int32_t adaptive, float rtol, float atol,
                  float dt_min, int32_t* n_accept, int32_t* n_reject, int32_t* status, float* y_steps,
                  void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (!ts || !y0 || !y_out) return ODECOL_E_NULL;
    if (T < 2 || !(dt > 0.f)) return ODECOL_E_SHAPE;
    if (adaptive && (dW || y_steps || !(dt_min > 0.f))) return ODECOL_E_UNSUPPORTED;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (use_small(p, d)) {
        if (d.lat_gain) return ODECOL_E_UNSUPPORTED;     // set ODECOL_FLAG_FORCE_STAGED to sweep the gain on a small network
        // attempts are bounded: a step at dt_min is always accepted
        const long long cap = adaptive ? (1LL << 34) : (1LL << 40);
        return launch_em_fwd_small(d, ts, T, y0, y_out, dW, seed, trial_offset, dt, adaptive, rtol, atol, dt_min,
                                   n_accept, n_reject, status, y_steps, cap, s);
    }
    if (misaligned(y0) || misaligned(y_out) || misaligned(workspace)) return ODECOL_E_ALIGN;
    return stage_em_fwd(d, ts, T, y0, y_out, dW, seed, trial_offset, dt, adaptive, rtol, atol, dt_min, n_accept, n_reject,
                        status, y_steps, workspace, workspace_bytes, s);
}

int odecol_em_bwd(const odecol_problem* p, const float* ts, int32_t T, const float* y_steps, int64_t n_steps,
                  const float* grad_y, const int32_t* sel, int32_t G, float dt, float* grad_y0, float* grad_W_aug,
                  void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!ts || !y_steps || !grad_y || !grad_W_aug) return ODECOL_E_NULL;
    if (T < 2 || G < 1 || G > 3 * p->N || n_steps < 1 || !(dt > 0.f)) return ODECOL_E_SHAPE;
    if (!use_small(p, d)) {                              // staged reverse sweep (tensor-core VJPs)
        if (misaligned(workspace)) return ODECOL_E_ALIGN;
        g_launches.store(0, std::memory_order_relaxed);
        return stage_sde_bwd(0, d, ts, T, y_steps, n_steps, nullptr, nullptr, 0, 0, grad_y, sel, G, dt, grad_y0, grad_W_aug,
                             workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
    }
    const EmScheduleLayout L = em_schedule_layout(T, n_steps);
    if (!workspace || workspace_bytes < L.total) return ODECOL_E_WORKSPACE;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    int* step_of = reinterpret_cast<int*>(w + L.off_step);
    float* wts = reinterpret_cast<float*>(w + L.off_w);
    float* tk = reinterpret_cast<float*>(w + L.off_tk);
    if (cudaMemsetAsync(grad_W_aug, 0, sizeof(float) * (size_t)p->N * p->ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
    int r2 = launch_em_schedule(ts, T, dt, step_of, wts, tk, s);
    if (r2) return r2;
    return launch_em_bwd_small(d, ts, T, y_steps, grad_y, sel, G, grad_y0, grad_W_aug, step_of, wts, tk, s);
}

int odecol_srk_fwd(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out, const float* dW,
                   const float* dU, uint64_t seed, int64_t trial_offset, float dt, int32_t* status, float* y_steps,
                   void* workspace, size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!ts || !y0 || !y_out) return ODECOL_E_NULL;
    if ((dW == nullptr) != (dU == nullptr)) return ODECOL_E_NULL;
    if (T < 2 || !(dt > 0.f)) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    if (!use_small(p, d)) {                              // staged solver
        if (misaligned(y0) || misaligned(y_out) || misaligned(workspace)) return ODECOL_E_ALIGN;
        return stage_srk_fwd(d, ts, T, y0, y_out, dW, dU, seed, trial_offset, dt, status, y_steps, workspace, workspace_bytes,
                             static_cast<cudaStream_t>(stream));
    }
    return launch_srk_fwd_small(d, ts, T, y0, y_out, dW, dU, seed, trial_offset, dt, status, y_steps,
                                static_cast<cudaStream_t>(stream));
}

int odecol_srk_fwd_adaptive(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out, uint64_t seed,
                            int64_t trial_offset, float dt, float rtol, float atol, float dt_min, int32_t* n_accept,
                            int32_t* n_reject, int32_t* status, void* workspace, size_t workspace_bytes, void* stream) {
    (void)workspace; (void)workspace_bytes;
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;
    if (!ts || !y0 || !y_out) return ODECOL_E_NULL;
    if (T < 2 || !(dt > 0.f) || !(dt_min > 0.f) || !(rtol >= 0.f) || !(atol >= 0.f)) return ODECOL_E_SHAPE;
    if (!use_small(p, d)) return ODECOL_E_UNSUPPORTED;   // the adaptive srk solve exists in the on-chip family (N <= 128)
    g_launches.store(0, std::memory_order_relaxed);
    return launch_srk_adaptive_small(d, ts, T, y0, y_out, seed, trial_offset, dt, rtol, atol, dt_min, n_accept, n_reject, status,
                                     1LL << 34, static_cast<cudaStream_t>(stream));
}

int odecol_brownian_levy_query(uint64_t seed, int64_t trial_offset, int32_t B, float t_begin, float t_end, const float* t,
                               int32_t M, double* w, double* iw, void* stream) {
    if (!t || !w || !iw) return ODECOL_E_NULL;
    if (B < 1 || M < 1 || !(t_end > t_begin)) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    return launch_brownian_levy_query(seed, trial_offset, B, t_begin, t_end - t_begin, t, M, w, iw, static_cast<cudaStream_t>(stream));
}

int odecol_srk_bwd(const odecol_problem* p, const float* ts, int32_t T, const float* y_steps, int64_t n_steps,
                   const float* dW, const float* dU, uint64_t seed, int64_t trial_offset, const float* grad_y,
                   const int32_t* sel, int32_t G, float dt, float* grad_y0, float* grad_W_aug, void* workspace,
                   size_t workspace_bytes, void* stream) {
    DevProblem d;
    const int rc = to_dev(p, d);
    if (rc) return rc;
    if (d.lat_gain) return ODECOL_E_UNSUPPORTED;      // the lateral-gain axis exists in the staged Euler-Maruyama path only
    if (!ts || !y_steps || !grad_y || !grad_W_aug) return ODECOL_E_NULL;
    if ((dW == nullptr) != (dU == nullptr)) return ODECOL_E_NULL;
    if (T < 2 || G < 1 || G > 3 * p->N || n_steps < 1 || !(dt > 0.f)) return ODECOL_E_SHAPE;
    if (!use_small(p, d)) {
        if (misaligned(workspace)) return ODECOL_E_ALIGN;
        g_launches.store(0, std::memory_order_relaxed);
        return stage_sde_bwd(1, d, ts, T, y_steps, n_steps, dW, dU, seed, trial_offset, grad_y, sel, G, dt, grad_y0, grad_W_aug,
                             workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
    }
    const EmScheduleLayout L = em_schedule_layout(T, n_steps);
    if (!workspace || workspace_bytes < L.total) return ODECOL_E_WORKSPACE;
    g_launches.store(0, std::memory_order_relaxed);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* w = static_cast<char*>(workspace);
    int* step_of = reinterpret_cast<int*>(w + L.off_step);
    float* wts = reinterpret_cast<float*>(w + L.off_w);
    float* tk = reinterpret_cast<float*>(w + L.off_tk);
    if (cudaMemsetAsync(grad_W_aug, 0, sizeof(float) * (size_t)p->N * p->ld_w, s) != cudaSuccess) return ODECOL_E_CUDA;
    const int r2 = launch_em_schedule(ts, T, dt, step_of, wts, tk, s);
    if (r2) return r2;
    return launch_srk_bwd_small(d, T, y_steps, dW, dU, seed, trial_offset, grad_y, sel, G, grad_y0, grad_W_aug, step_of,
                                wts, tk, s);
}

int odecol_brownian_query(uint64_t seed, int64_t trial_offset, int32_t B, float t_begin, float t_end, const float* t,
                          int32_t M, float* w, void* stream) {
    if (!t || !w) return ODECOL_E_NULL;
    if (B < 1 || M < 1 || !(t_end > t_begin)) return ODECOL_E_SHAPE;
    g_launches.store(0, std::memory_order_relaxed);
    return launch_brownian_query(seed, trial_offset, B, t_begin, t_end - t_begin, t, M, w, static_cast<cudaStream_t>(stream));
}

int odecol_ww_generate(const double* mu, const double* i_noise0, int32_t B, int32_t steps_per_phase, int32_t every,
                       int32_t time_steps, double sigma_noise, uint64_t seed, int64_t trial_offset, float* states,
                       void* stream) {
    if (!mu || !states) return ODECOL_E_NULL;
    if (B < 1 || steps_per_phase < 1 || every < 1 || time_steps < 1) return ODECOL_E_SHAPE;
    if ((int64_t)time_steps > (3LL * steps_per_phase + every - 1) / every) return ODECOL_E_SHAPE;   // more rows than recorded updates
    g_launches.store(0, std::memory_order_relaxed);
    return launch_ww_generate(mu, i_noise0, B, steps_per_phase, every, time_steps, sigma_noise, seed, trial_offset, states,
                              static_cast<cudaStream_t>(stream));
}

int odecol_huber_rate_loss(const float* y_sel, int32_t T, int32_t B, int32_t G, int32_t P, const float* w,
                           const float* target, int64_t st_t, int64_t st_b, int64_t st_g, float beta, float* loss,
                           float* grad_y_sel, void* workspace, size_t workspace_bytes, void* stream) {
    if (!y_sel || !target || !loss || !grad_y_sel) return ODECOL_E_NULL;
    if (T < 1 || B < 1 || G < 1 || P < 1 || !(beta > 0.f) || st_t < 0 || st_b < 0 || st_g < 0) return ODECOL_E_SHAPE;
    if (!workspace || workspace_bytes < sizeof(double)) return ODECOL_E_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 7) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return launch_huber_rate_loss(y_sel, T, B, G, P, w, target, st_t, st_b, st_g, beta, loss, grad_y_sel,
                                  static_cast<double*>(workspace), static_cast<cudaStream_t>(stream));
}

int odecol_window_rate_l1_loss(const float* y_sel, int32_t T, int32_t B, int32_t P, int32_t last, const float* w,
                               const float* target, float* loss, float* pred, float* grad_y_sel, float* grad_w,
                               void* workspace, size_t workspace_bytes, void* stream) {
    if (!y_sel || !target || !loss || !pred || !grad_y_sel || !grad_w) return ODECOL_E_NULL;
    if (T < 1 || B < 1 || P < 1 || last < 1 || last > T) return ODECOL_E_SHAPE;
    if (!workspace || workspace_bytes < sizeof(double)) return ODECOL_E_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace) & 7) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return launch_window_rate_l1_loss(y_sel, T, B, P, last, w, target, loss, pred, grad_y_sel, grad_w, static_cast<double*>(workspace),
                                      static_cast<cudaStream_t>(stream));
}

size_t odecol_tc_contract_workspace_bytes(int32_t M, int32_t N, int32_t K) {
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    return tc_contract_workspace_bytes(M, N, K);
}

int odecol_tc_contract(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K, void* workspace,
                       size_t workspace_bytes, void* stream) {
    if (!A || !B || !C) return ODECOL_E_NULL;
    if (M <= 0 || N <= 0 || K <= 0) return ODECOL_E_SHAPE;
    if (misaligned(workspace)) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return tc_contract(A, B, C, M, N, K, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t odecol_tc_contract_tn_workspace_bytes(int32_t M, int32_t N, int32_t K) {
    if (M <= 0 || N <= 0 || K <= 0) return 0;
    return tc_contract_tn_workspace_bytes(M, N, K);
}

int odecol_tc_contract_tn(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K, void* workspace,
                          size_t workspace_bytes, void* stream) {
    if (!A || !B || !C) return ODECOL_E_NULL;
    if (M <= 0 || N <= 0 || K <= 0) return ODECOL_E_SHAPE;
    if (misaligned(workspace)) return ODECOL_E_ALIGN;
    g_launches.store(0, std::memory_order_relaxed);
    return tc_contract_tn(A, B, C, M, N, K, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
