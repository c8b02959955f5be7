// Internal declarations shared by the kernel translation units and the C-ABI shim.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "../../include/odecol.h"

namespace odecol {

struct Consts {
    float tau_s, tau_m, tau_a, R;
};

// device-side copy of odecol_problem (passed by value to kernels)
struct DevProblem {
    int N, n_in, B, K, ld_w;
    int flags;                  // ODECOL_FLAG_* of the caller's problem
    const float* W_aug;
    const float* kappa;
    const float* sigma;
    const float* sigma_scale;   // [B] or NULL
    const float* lat_gain;      // [B] or NULL: per-trial gain on the dense recurrent input (staged Euler-Maruyama only)
    const float* W_local;       // [N][8] or NULL: within-column weights applied outside the contraction (with lat_gain)
    const float* knot_t;
    const float* knot_u;
    long long knot_stride_b;
    Consts c;
};

// optional recording of the accepted dopri5 steps (training mode): start state, t0, dt of every accepted step and, for
// every output time, the step it was interpolated in and the abscissa
struct Dopri5Record {
    float* y;          // (cap, B, 3N) or NULL
    double* t0;        // (B, cap)
    double* dt;        // (B, cap)
    int* out_step;     // (B, T)
    float* out_x;      // (B, T)
    int cap;
};

// thread-local launch counter (odecol_last_launch_count)
void count_launch(int n = 1);

// ---- family S (small_kernels.cu) ---------------------------------------------------------------------------
int small_kp(const DevProblem& p);                 // 0 if the problem does not fit family S
size_t small_bwd_smem_bytes(int N, int KP, int trials_per_cta);
int launch_rhs_generic(const DevProblem& p, const float* t, const float* y, float* f, cudaStream_t s);
int launch_rk4_fwd_small(const DevProblem& p, const float* t, int T, const float* y0, float* y_out, int out_every,
                         cudaStream_t s, const unsigned int* run_if = nullptr);      // run_if: device flag, 0 -> the kernel returns at once
// large batches of the smallest networks on the tensor cores, trials on the M axis (tiny_tc.cu); *ovf: 4 bytes of device memory
bool tiny_rk4_applicable(const DevProblem& p);
int launch_rk4_fwd_tiny(const DevProblem& p, const float* t, int T, const float* y0, float* y_out, int out_every,
                        unsigned int* ovf, cudaStream_t s);
int launch_rk4_bwd_small(const DevProblem& p, const float* t, int T, const float* y_traj, const float* grad_y,
                         const int* sel, int G, float* grad_y0, float* grad_W, cudaStream_t s);
int launch_dopri5_fwd_small(const DevProblem& p, const float* t, int T, const float* y0, float* y_out, float rtol,
                            float atol, int max_steps, int* n_accept, int* n_reject, int* status, const Dopri5Record& rec,
                            cudaStream_t s);
int launch_dopri5_bwd_small(const DevProblem& p, int T, const Dopri5Record& rec, const int* n_accept, const float* grad_y,
                            const int* sel, int G, float* grad_y0, float* grad_W, cudaStream_t s);
int launch_em_fwd_small(const DevProblem& p, const float* ts, int T, const float* y0, float* y_out, const float* dW,
                        uint64_t seed, int64_t trial_offset, float dt, int adaptive, float rtol, float atol,
                        float dt_min, int* n_accept, int* n_reject, int* status, float* y_steps,
                        long long max_attempts, cudaStream_t s);
// schedule: step_of[T+1] (last entry = n_steps), w[2T], tk[n_steps+1]
int launch_em_schedule(const float* ts, int T, float dt, int* step_of, float* w, float* tk, cudaStream_t s);
int launch_em_bwd_small(const DevProblem& p, const float* ts, int T, const float* y_steps, const float* grad_y,
                        const int* sel, int G, float* grad_y0, float* grad_W, const int* step_of, const float* w,
                        const float* tk, cudaStream_t s);
int launch_srk_fwd_small(const DevProblem& p, const float* ts, int T, const float* y0, float* y_out, const float* dW,
                         const float* dU, uint64_t seed, int64_t trial_offset, float dt, int* status, float* y_steps,
                         cudaStream_t s);
int launch_srk_bwd_small(const DevProblem& p, int T, const float* y_steps, const float* dW, const float* dU, uint64_t seed,
                         int64_t trial_offset, const float* grad_y, const int* sel, int G, float* grad_y0, float* grad_W,
                         const int* step_of, const float* w, const float* tk, cudaStream_t s);

int launch_srk_adaptive_small(const DevProblem& p, const float* ts, int T, const float* y0, float* y_out, uint64_t seed,
                              int64_t trial_offset, float dt, float rtol, float atol, float dt_min, int* n_accept,
                              int* n_reject, int* status, long long max_attempts, cudaStream_t s);
// W(t[m]) and I(t[m]) = int W of the Levy-area-consistent tree (adaptive srk), double precision, (M, B) each
int launch_brownian_levy_query(uint64_t seed, int64_t trial_offset, int B, float t_begin, float span, const float* t, int M,
                               double* w, double* iw, cudaStream_t s);

// W(t[m]) of the virtual Brownian tree of trial (trial_offset + b) on [t_begin, t_begin + span]: w[m][b]
int launch_brownian_query(uint64_t seed, int64_t trial_offset, int B, float t_begin, float span, const float* t, int M,
                          float* w, cudaStream_t s);

// ---- Wong-Wang target generator (ww_kernel.cu) -----------------------------------------------------------------
int launch_ww_generate(const double* mu, const double* i_noise0, int B, int steps_per_phase, int every, int time_steps,
                       double sigma_noise, uint64_t seed, int64_t trial_offset, float* states, cudaStream_t s);

// ---- fused read-out losses (readout_kernels.cu) ------------------------------------------------------------------
int launch_huber_rate_loss(const float* y_sel, int T, int B, int G, int P, const float* w, const float* target,
                           long long st_t, long long st_b, long long st_g, float beta, float* loss, float* grad,
                           double* acc, cudaStream_t s);

int launch_window_rate_l1_loss(const float* y_sel, int T, int B, int P, int L, const float* w, const float* target,
                               float* loss, float* pred, float* grad, float* grad_w, double* acc, cudaStream_t s);

// ---- staged Euler-Maruyama (stage_em.cu): state in global memory, the drift contraction on the tensor cores ------
size_t stage_em_fwd_workspace_bytes(const DevProblem& p, int T);
int stage_em_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                 uint64_t seed, int64_t trial_offset, float dt, int adaptive, float rtol, float atol, float dt_min,
                 int* n_accept, int* n_reject, int* status, float* y_steps, void* ws, size_t ws_bytes, cudaStream_t s);

// one drift evaluation through the staged tensor-core path (workspace of stage_em_fwd)
int stage_drift(const DevProblem& p, const float* t_trial, const float* y, float* f, void* ws, size_t ws_bytes, cudaStream_t s);

// staged Dormand-Prince 5(4), forward (stage_em.cu): per-trial control in rounds, drift on the tensor cores
size_t stage_dopri5_fwd_workspace_bytes(const DevProblem& p, int T);
int stage_dopri5_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, float rtol, float atol,
                     int max_steps, int* n_accept, int* n_reject, int* status, const Dopri5Record& rec, void* ws,
                     size_t ws_bytes, cudaStream_t s);
// staged discrete adjoint over the recorded accepted steps (rounds over the steps from each trial's last to its first)
size_t stage_dopri5_bwd_workspace_bytes(const DevProblem& p, int T);
int stage_dopri5_bwd(const DevProblem& p, int T, const Dopri5Record& rec, const int* n_accept, const float* grad_y,
                     const int* sel, int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s);

// staged torchsde srk (fixed step), forward (stage_em.cu)
size_t stage_srk_fwd_workspace_bytes(const DevProblem& p, int T);
int stage_srk_fwd(const DevProblem& p, const float* ts_dev, int T, const float* y0, float* y_out, const float* dW,
                  const float* dU, uint64_t seed, int64_t trial_offset, float dt, int* status, float* y_steps, void* ws,
                  size_t ws_bytes, cudaStream_t s);
// staged discrete adjoints of the fixed-step Euler-Maruyama (which = 0) and srk (which = 1) solves
size_t stage_sde_bwd_workspace_bytes(const DevProblem& p, int T);
int stage_sde_bwd(int which, const DevProblem& p, const float* ts_dev, int T, const float* y_steps, int64_t n_steps,
                  const float* dW, const float* dU, uint64_t seed, int64_t trial_offset, const float* grad_y, const int* sel,
                  int G, float dt, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s);

// ---- family T (stage_tc.cu): the staged contraction on tcgen05 tensor cores (3xTF32) ------------------------------
size_t tc_rk4_fwd_workspace_bytes(const DevProblem& p, int T);
int tc_rk4_fwd(const DevProblem& p, const float* t_dev, int T, const float* y0, float* y_out, int out_every, void* ws,
               size_t ws_bytes, cudaStream_t s);
size_t tc_rk4_bwd_workspace_bytes(const DevProblem& p, int T);
int tc_rk4_bwd(const DevProblem& p, const float* t_dev, int T, const float* y_traj, const float* grad_y, const int* sel,
               int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s);
// checkpoint mode (tensor family): V/A state + V slopes per step instead of the trajectory; see tc::CkptView
size_t tc_rk4_ckpt_bytes(const DevProblem& p, int T);
int tc_rk4_fwd_ckpt(const DevProblem& p, const float* t_dev, int T, const float* y0, const int* sel, int G, float* y_sel,
                    void* ckpt, size_t ckpt_bytes, void* ws, size_t ws_bytes, cudaStream_t s);
int tc_rk4_bwd_ckpt(const DevProblem& p, const float* t_dev, int T, const void* ckpt, size_t ckpt_bytes, const float* grad_y,
                    const int* sel, int G, float* grad_y0, float* grad_W, void* ws, size_t ws_bytes, cudaStream_t s);
int tc_dw_accumulate(const float* Ahi, const float* Alo, const float* Bhi, const float* Blo, int rows, int Np, int KPa, int N,
                     int Kaug, int ld_w, float* grad_W, cudaStream_t s);
size_t tc_contract_tn_workspace_bytes(int M, int N, int K);
int tc_contract_tn(const float* A, const float* B, float* C, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t s);
size_t tc_contract_workspace_bytes(int M, int N, int K);
int tc_contract(const float* A, const float* B, float* C, int M, int N, int K, void* ws, size_t ws_bytes, cudaStream_t s);

}  // namespace odecol
