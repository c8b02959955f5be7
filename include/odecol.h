/* odecol.h -- C ABI of the B200-native fused integrator for the ODE-Column hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point replaces a piece of the
 * reference's Python call stack; the citation after each declaration names what it replaces
 * (paths relative to the reference repository, ccnmaastricht/ODE-Column).
 *
 * Conventions
 *   - all data pointers are DEVICE pointers to float32 (int32 / uint8 where declared), caller-owned,
 *     never retained past the call; the library performs no hidden allocation -- scratch memory is a
 *     caller-provided workspace sized by odecol_workspace_bytes();
 *   - calls are ordered on `stream` (a cudaStream_t passed as void* so that the header needs no CUDA include) and
 *     asynchronous with respect to the host, with these documented exceptions, all in the STAGED family (N > 128 or a
 *     forced flag): the fixed-step stochastic entry points (odecol_em_fwd, odecol_srk_fwd, odecol_em_bwd, odecol_srk_bwd)
 *     replay the data-independent float32 step schedule on the host and synchronise the stream once at entry (the two
 *     forward ones once more at exit, to read the overflow flag of the FP16 operand format, see "operand formats"); the
 *     adaptive ones (odecol_em_fwd with adaptive = 1, odecol_dopri5_fwd / _fwd_record) poll an "all trials finished"
 *     counter every 16 rounds; odecol_dopri5_bwd reads the accepted-step counts once.  None of them may be captured into
 *     a CUDA graph; everything else (the on-chip family, all rk4 entry points, the read-outs) may;
 *   - forward results (trajectories, step counts, read-outs' predictions) are bit-reproducible for a given problem,
 *     library build and device.  Sums OVER TRIALS -- grad_W_aug, the scalar losses -- add per-trial contributions with
 *     float / double atomics, so repeated runs agree to rounding (~1e-7 relative), not bit for bit; the tensor family's rk4
 *     reverse sweep (N > 128, the benchmarked path) reduces in a fixed order when ODECOL_FLAG_DETERMINISTIC is set;
 *   - return value: 0 (ODECOL_OK) or a negative error code, see odecol_strerror(); nothing throws;
 *   - re-entrant across streams, no global state that affects results, one GPU per call (multi-GPU orchestration is
 *     the caller's: shard trials, then all-reduce grad_W_aug);
 *   - there is NO CPU implementation behind this ABI;
 *   - arithmetic of the tensor-core paths (the staged family, N > 128; rk4 forward of N <= 16 networks from 4096 trials,
 *     which asks for 256 bytes of workspace and falls back to the on-chip kernel without them): float32 state, contractions as error-corrected split
 *     products on tcgen05 (operand = high + low half, three products, FP32 accumulation: 2^-22 relative).  The halves are
 *     TF32 numbers, or -- in the persistent rk4 forward kernel and the drift evaluations of the staged Euler-Maruyama, srk
 *     and forward-only (no record) dopri5 forward solves -- FP16 numbers.  FP16 cannot
 *     hold an operand value (a firing rate, a stimulus) beyond +-6e4: the kernels detect that on the device and the same
 *     call then repeats the solve on TF32 halves (rk4: a second kernel of the same launch sequence that returns at once
 *     otherwise; Euler-Maruyama / dopri5: at the host polls these entry points already have; srk: one read after the last
 *     step), so results never depend on it.
 *
 * The problem integrated (all three reference networks reduce to it, SURVEY.md section 3.2):
 *
 *     r      = phi(V - A)                                  src/utils.py:13-28
 *     I      = W r + U s(t) + bias  =  W_aug . [r ; s(t) ; 1]
 *     dV/dt  = (-V + I * tau_s * R) / tau_m                src/coupled_columns.py:225-229, 402/431, 746-749/777
 *     dA/dt  = (-A + kappa * r) / tau_a                    :230-231, 433-434, 779-780
 *     dF/dt  = (-F + r) / tau_s                            :232-233, 437-438, 783-784
 *     g      = sigma (per state component, scalar noise)   :239-249, 444-454, 790-800
 *
 * State layout: y[b] = [ V(0..N) | A(0..N) | F(0..N) ], trajectories are (T, B, 3N) row-major, exactly
 * the (len(t), batch, d) tensors torchdiffeq / torchsde return.
 */
#ifndef ODECOL_H
#define ODECOL_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ODECOL_ABI_VERSION 3

enum {
    ODECOL_OK = 0,
    ODECOL_E_NULL = -1,        /* required pointer is NULL                              */
    ODECOL_E_SHAPE = -2,       /* N, B, T, K, n_in or ld_w out of range                 */
    ODECOL_E_UNSUPPORTED = -3, /* valid request the library has no kernel for           */
    ODECOL_E_WORKSPACE = -4,   /* workspace missing or smaller than workspace_bytes()   */
    ODECOL_E_CUDA = -5,        /* a CUDA runtime call or launch failed                  */
    ODECOL_E_ALIGN = -6        /* a pointer violates the 16-byte alignment contract     */
};

/* per-trial solver status written by the adaptive entry points */
enum {
    ODECOL_ST_OK = 0,
    ODECOL_ST_NONFINITE = 1,   /* state became inf/NaN (phi has a pole at V-A = 981/48) */
    ODECOL_ST_MAXSTEPS = 2,    /* step budget exhausted before t[T-1]                   */
    ODECOL_ST_UNDERFLOW = 3    /* t + dt == t                                           */
};

/* odecol_problem.flags */
enum {
    ODECOL_FLAG_FORCE_STAGED = 1,  /* skip the persistent on-chip family: use the staged (global-state) solvers even
                                      when the problem fits on chip; for testing and measurement */
    ODECOL_FLAG_FORCE_TENSOR = 2,  /* the same as ODECOL_FLAG_FORCE_STAGED (both values are kept for binary
                                      compatibility; staged rk4 always runs in the tcgen05 family) */
    ODECOL_FLAG_DETERMINISTIC = 4  /* tensor family, rk4 reverse sweep: reduce grad_W_aug over trials in a fixed order
                                      (per-split copies summed at the end) instead of float atomics: bit-reproducible
                                      gradients for ~2 % of the sweep's time                                      */
};

/* operations, for odecol_workspace_bytes() */
enum {
    ODECOL_OP_RHS = 0,
    ODECOL_OP_RK4_FWD = 1,
    ODECOL_OP_RK4_BWD = 2,
    ODECOL_OP_DOPRI5_FWD = 3,
    ODECOL_OP_EM_FWD = 4,
    ODECOL_OP_EM_BWD = 5,
    ODECOL_OP_SRK_FWD = 6,
    ODECOL_OP_SRK_BWD = 7,
    ODECOL_OP_DOPRI5_BWD = 8
};

/* The column network in linear form plus the stimulus of every trial.
 * Replaces the nn.Module attributes the reference solvers read through func(t, y):
 *   recurrent / lateral / feedforward / input weights   src/coupled_columns.py:183, 318-341, 601, 631, 665-668
 *   background_weights * background_drive               :222, 398, 743
 *   adaptation_strength (kappa), time constants, R      :28-37, 50
 *   network.time_vec / network.stim                     scripts/wta_ode.py:154,171  xor_ode.py:112,156  parity_ode.py:181,231
 */
typedef struct odecol_problem {
    int32_t N;            /* populations (8 per column)                                      */
    int32_t n_in;         /* stimulus channels                                               */
    int32_t B;            /* trials (independent solves; the reference loops over them)      */
    int32_t K;            /* stimulus knots per trial (>= 2)                                 */
    int32_t ld_w;         /* floats per row of W_aug, >= N + n_in + 1, multiple of 4         */
    int32_t flags;        /* ODECOL_FLAG_* (0 = let the library pick the kernel family)              */
    const float* W_aug;   /* [N][ld_w]: columns [0,N) = W (row target, col source),
                             [N, N+n_in) = U, column N+n_in = bias, rest zero                */
    const float* kappa;   /* [N]                                                             */
    const float* sigma;   /* [3N] diffusion per state component, may be NULL (treated as 0)  */
    const float* knot_t;  /* [K] strictly increasing knot times (the reference's time_vec)   */
    const float* knot_u;  /* [B][K][n_in] stimulus values at the knots; piecewise-linear in
                             between, held beyond the ends (src/utils.py:31-46)              */
    int64_t knot_stride_b;/* floats between consecutive trials in knot_u (0 = shared)        */
    float tau_s, tau_m, tau_a, resistance;
    const float* sigma_scale; /* [B] per-trial factor on sigma, or NULL (1): the noise-amplitude axis of a
                                 parameter sweep (each trial integrates with g = sigma_scale[b] * sigma);
                                 read by the stochastic entry points only (ABI v2)                   */
    const float* lat_gain;    /* [B] per-trial gain g_b on the dense recurrent input, or NULL (ABI v3): the "global
                                 lateral gain" axis of a parameter sweep (BASELINE.json configs[4]).  With it the
                                 input current of trial b is
                                     I_b = g_b * (W r_b) + W_local (*) r_b + U s_b(t) + bias
                                 where W = W_aug[:, :N] then holds the between-column (lateral) weights only and
                                 the within-column weights move to W_local.  g_b must be > 0.  Honoured by
                                 odecol_em_fwd (staged family) and odecol_drift_staged; every other entry point
                                 returns ODECOL_E_UNSUPPORTED when it is set                          */
    const float* W_local;     /* [N][8] within-column weights (row i, source population 8*(i/8) + j), or NULL;
                                 read only together with lat_gain                                     */
} odecol_problem;

int odecol_abi_version(void);
const char* odecol_strerror(int code);

/* Scratch requirement of `op` on this problem with T output times (bytes, 0 if none).  n_steps is the number
 * of Euler-Maruyama steps (odecol_em_num_steps) and is ignored by the other operations. */
size_t odecol_workspace_bytes(const odecol_problem* p, int op, int32_t T, int64_t n_steps);

/* f = forward(t, y) for a batch: t[B] (one time per trial), y[B][3N] -> f[B][3N].
 * Replaces ColumnAreaWTA.forward / ColumnNetworkXOR.forward / ColumnNetwork.forward
 * (src/coupled_columns.py:204-237, 407-442, 753-788) incl. compute_firing_rate and torch_interp
 * (src/utils.py:13-46). */
int odecol_rhs(const odecol_problem* p, const float* t, const float* y, float* f, void* stream);

/* The same evaluation through the staged tensor-core path the large-network solvers use (operand split, tcgen05
 * contraction with chunked accumulation for long rows, fast FP32-accurate phi), always in TF32 operand pairs (3xTF32).
 * The solvers' forward solves, among them the N = 8192 sweep (BASELINE.json configs[4]), evaluate the same drift in
 * FP16 operand pairs unless ODECOL_EM16 / ODECOL_DP16 / ODECOL_SRK16 is 0; sdeint(method='euler', dt=1, ts=[0, 1]) with
 * zero increments returns y0 + f in that format.  Any N that is a multiple of 4; workspace:
 * odecol_workspace_bytes(p, ODECOL_OP_EM_FWD, 0, 0) sized for the STAGED family (set ODECOL_FLAG_FORCE_STAGED or
 * ODECOL_FLAG_FORCE_TENSOR on problems that would otherwise pick the on-chip family). */
int odecol_drift_staged(const odecol_problem* p, const float* t, const float* y, float* f,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Fixed-grid RK4 (3/8 rule) on the grid t[0..T): y_out[0] = y0, y_out[j] = y(t[j]).
 * Replaces torchdiffeq.odeint(func, y0, t, method='rk4') plus the per-trial Python loop
 * (scripts/xor_ode.py:104-117, scripts/parity_ode.py:223-236, scripts/wta_ode.py:167-176).
 * y_out may be strided in time: y_out[j] is written iff j % out_every == 0 or j == T-1; row index j / out_every
 * (last row = ceil((T-1)/out_every)).  out_every = 1 gives the torchdiffeq result (T, B, 3N). */
int odecol_rk4_fwd(const odecol_problem* p, const float* t, int32_t T, const float* y0,
                   float* y_out, int32_t out_every, void* workspace, size_t workspace_bytes, void* stream);

/* Exact discrete adjoint of odecol_rk4_fwd (discretise-then-optimise: what loss.backward() through
 * torchdiffeq's unrolled steps computes; scripts/xor_ode.py:177, scripts/parity_ode.py:250).
 *   y_traj      (T, B, 3N) the forward result with out_every = 1
 *   grad_y      (T, B, G)  dL/dy_out restricted to the state components sel[0..G); sel == NULL means
 *                          G = 3N, all components in order.  sel must hold DISTINCT components: each component reads
 *                          one column of grad_y (with a repeat, which one is unspecified); a caller whose loss reads a
 *                          component twice passes it once with the summed gradient
 *   grad_y0     (B, 3N)    out, may be NULL
 *   grad_W_aug  (N, ld_w)  out, OVERWRITTEN with sum over trials of dL/dW_aug (dW | dU | dbias) */
int odecol_rk4_bwd(const odecol_problem* p, const float* t, int32_t T, const float* y_traj,
                   const float* grad_y, const int32_t* sel, int32_t G,
                   float* grad_y0, float* grad_W_aug,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Checkpoint mode of the rk4 pair, for training on a selection of state components (the reference's losses read a few
 * firing-rate components: scripts/xor_ode.py:119-177, scripts/parity_ode.py:238-250).  The forward sweep returns only
 * y[:, :, sel] and leaves, per grid step, the V/A state and the three V slopes of the step in `ckpt` (20 bytes per
 * population, trial and step, kernel-private layout); the reverse sweep re-derives every stage from them elementwise
 * instead of recomputing three contractions per step.  Only the tensor family (every network beyond the on-chip family, N > 128) implements it: other
 * problems return ODECOL_E_UNSUPPORTED and the caller uses odecol_rk4_fwd / odecol_rk4_bwd.
 *   odecol_rk4_ckpt_bytes   size of `ckpt` for (p, T); 0 if unsupported
 *   y_sel       (T, B, G)  out: the selected components at every grid point (row 0 = y0[:, sel])
 *   grad_y_sel  (T, B, G)  dL/dy_sel;  sel, G, grad_y0, grad_W_aug as in odecol_rk4_bwd
 * Workspaces: odecol_workspace_bytes(p, ODECOL_OP_RK4_FWD / ODECOL_OP_RK4_BWD, T, 0). */
size_t odecol_rk4_ckpt_bytes(const odecol_problem* p, int32_t T);
int odecol_rk4_fwd_ckpt(const odecol_problem* p, const float* t, int32_t T, const float* y0,
                        const int32_t* sel, int32_t G, float* y_sel, void* ckpt, size_t ckpt_bytes,
                        void* workspace, size_t workspace_bytes, void* stream);
int odecol_rk4_bwd_ckpt(const odecol_problem* p, const float* t, int32_t T, const void* ckpt, size_t ckpt_bytes,
                        const float* grad_y_sel, const int32_t* sel, int32_t G,
                        float* grad_y0, float* grad_W_aug,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Adaptive Dormand-Prince 5(4) with per-trial step control and 4th-order dense output at t[0..T).
 * Replaces torchdiffeq.odeint(func, y0, t) with its default method (what the reference scripts get,
 * scripts/xor_ode.py:114, scripts/parity_ode.py:233; rtol 1e-7, atol 1e-9 are torchdiffeq's defaults).
 * n_accept / n_reject / status are per trial, any of them may be NULL.
 * Networks beyond the on-chip family (N > 128, or ODECOL_FLAG_FORCE_STAGED / _TENSOR) run the staged solver: the same
 * per-trial controller, one attempted step of every unfinished trial per round with the six stage evaluations on the
 * tensor cores; it needs odecol_workspace_bytes(p, ODECOL_OP_DOPRI5_FWD, T, 0) and synchronises the stream every 16
 * rounds (like the adaptive Euler-Maruyama).  The record / reverse pair below exists in both families (staged: the same
 * workspaces, ODECOL_OP_DOPRI5_FWD / ODECOL_OP_DOPRI5_BWD; the reverse sweep runs in rounds over the accepted steps, from
 * each trial's last to its first, with the drift evaluations and vector-Jacobian products on the tensor cores). */
int odecol_dopri5_fwd(const odecol_problem* p, const float* t, int32_t T, const float* y0, float* y_out,
                      float rtol, float atol, int32_t max_steps,
                      int32_t* n_accept, int32_t* n_reject, int32_t* status,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Training-mode variant of odecol_dopri5_fwd: additionally records every ACCEPTED step so that odecol_dopri5_bwd can
 * differentiate through them (discretise-then-optimise, what loss.backward() through torchdiffeq's adaptive steps
 * computes; reference scripts/xor_ode.py:114,177 -- rejected attempts and the step controller carry no gradient).
 *   rec_y     (cap, B, 3N)  state at the start of accepted step n
 *   rec_t0, rec_dt (B, cap) float64 start time and size of accepted step n
 *   out_step, out_x (B, T)  for every output time the accepted step it lies in and the dense-output abscissa
 * A trial that needs more than `cap` accepted steps stops with ODECOL_ST_MAXSTEPS (retry with a larger cap). */
int odecol_dopri5_fwd_record(const odecol_problem* p, const float* t, int32_t T, const float* y0, float* y_out,
                             float rtol, float atol, int32_t max_steps,
                             int32_t* n_accept, int32_t* n_reject, int32_t* status,
                             float* rec_y, double* rec_t0, double* rec_dt, int32_t* out_step, float* out_x, int32_t cap,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Reverse sweep over the recorded steps; grad_y / sel / G / grad_y0 / grad_W_aug as in odecol_rk4_bwd. */
int odecol_dopri5_bwd(const odecol_problem* p, int32_t T, const float* rec_y, const double* rec_t0, const double* rec_dt,
                      const int32_t* out_step, const float* out_x, int32_t cap, const int32_t* n_accept,
                      const float* grad_y, const int32_t* sel, int32_t G, float* grad_y0, float* grad_W_aug,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Euler-Maruyama in torchsde's integrate loop (scalar noise, Ito): steps of `dt` from ts[0], the last
 * one clipped to ts[T-1], outputs by linear interpolation between the two solver states around ts[j].
 * Replaces torchsde.sdeint(sde, y0, ts, names={'drift':'forward','diffusion':'diffusion'}, method='euler',
 * dt=, adaptive=, rtol=, atol=, dt_min=) (call sites scripts/wta_ode.py:174,200).
 *   dW       (n_steps, B) host-supplied Brownian increments in step order (bit-parity mode, fixed step
 *            only; n_steps = odecol_em_num_steps()), or NULL: increments come from the in-kernel Philox4x32-10
 *            virtual Brownian tree keyed by (seed, trial_offset + b)
 *   adaptive 0 = fixed step; 1 = step doubling with torchsde's controller, per trial
 *   y_steps  optional (n_steps+1, B, 3N): every solver state (needed by odecol_em_bwd), fixed step only */
int odecol_em_fwd(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out,
                  const float* dW, uint64_t seed, int64_t trial_offset,
                  float dt, int32_t adaptive, float rtol, float atol, float dt_min,
                  int32_t* n_accept, int32_t* n_reject, int32_t* status, float* y_steps,
                  void* workspace, size_t workspace_bytes, void* stream);

/* The Brownian path the adaptive solvers integrate against, for reproduction and validation: W(t[m]) - W(t_begin) of
 * trial (trial_offset + b) on the virtual Brownian tree spanning [t_begin, t_end] (Philox4x32-10 keyed by seed; the
 * solve over ts uses t_begin = ts[0], t_end = ts[T-1]).  Stands in for torchsde's BrownianInterval object, which a
 * caller can query after sdeint returns (torchsde.sdeint(..., bm=bm); reference call sites scripts/wta_ode.py:174,200
 * pass none and get a fresh one).  t[M] device pointer, w (M, B) out. */
int odecol_brownian_query(uint64_t seed, int64_t trial_offset, int32_t B, float t_begin, float t_end, const float* t,
                          int32_t M, float* w, void* stream);

/* Number of fixed steps odecol_em_fwd takes for (ts, dt): the float32 time loop is data independent.
 * ts is a HOST pointer here. */
int64_t odecol_em_num_steps(const float* ts_host, int32_t T, float dt);

/* Discrete adjoint of the fixed-step Euler-Maruyama solve (additive noise: dW does not enter the Jacobian).
 *   y_steps (n_steps+1, B, 3N) from odecol_em_fwd, grad_y (T, B, G) as in odecol_rk4_bwd. */
int odecol_em_bwd(const odecol_problem* p, const float* ts, int32_t T, const float* y_steps, int64_t n_steps,
                  const float* grad_y, const int32_t* sel, int32_t G, float dt,
                  float* grad_y0, float* grad_W_aug,
                  void* workspace, size_t workspace_bytes, void* stream);

/* torchsde's method='srk' for scalar noise, fixed step: Roessler's SRI2 scheme ("SRID2" tableau, strong order 1.5) in
 * the same integrate loop as odecol_em_fwd.  Replaces
 *   torchsde.sdeint(sde, y0, ts, names={'drift':'forward','diffusion':'diffusion'}, method='srk')
 * the call every committed SDE solve of the reference makes (scripts/wta_ode.py:174,200;
 * scripts/plotting_results.py:391,506,594).  Per step the scheme consumes the Brownian increment W and the space-time
 * Levy area U = int_{t0}^{t1} (W_r - W_{t0}) dr (torchsde: bm(t0, t1, return_U=True)):
 *   dW, dU   (n_steps, B) host-supplied, both or neither (n_steps = odecol_em_num_steps()); NULL: in-kernel
 *            Philox4x32-10, U | W ~ N(h W / 2, h^3 / 12); the W stream is the one odecol_em_fwd draws (fixed step)
 *   status   per trial, may be NULL: ODECOL_ST_NONFINITE if the final state is not finite
 *   y_steps  optional (n_steps+1, B, 3N): every solver state (needed by odecol_srk_bwd)
 * Networks beyond the on-chip family (N > 128 or a forced staged family) run the staged solver: three tensor-core drift
 * evaluations per step, workspace odecol_workspace_bytes(p, ODECOL_OP_SRK_FWD, T, 0) (and ODECOL_OP_SRK_BWD for the reverse sweep);
 * like the staged Euler-Maruyama it replays the step schedule on the host (one stream synchronisation at entry). */
int odecol_srk_fwd(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out,
                   const float* dW, const float* dU, uint64_t seed, int64_t trial_offset, float dt,
                   int32_t* status, float* y_steps, void* workspace, size_t workspace_bytes, void* stream);

/* torchsde.sdeint(..., method='srk', adaptive=True, rtol=, atol=, dt_min=): step doubling with the SRI2 step and torchsde's
 * controller, per trial -- literally the reference's "avoid the integration artefacts" option (scripts/parity_ode.py:234,
 * README.md:28-29).  Full step and half steps see one Brownian path: (W, U) of every sub-interval come from a
 * Levy-area-consistent virtual Brownian tree (Philox4x32-10 keyed by seed and trial_offset + b; see
 * odecol_brownian_levy_query).  Outputs by linear interpolation between solver states; n_accept / n_reject / status per
 * trial as in odecol_em_fwd.  On-chip family only (N <= 128: the reference's networks); larger networks return
 * ODECOL_E_UNSUPPORTED.  No workspace. */
int odecol_srk_fwd_adaptive(const odecol_problem* p, const float* ts, int32_t T, const float* y0, float* y_out,
                            uint64_t seed, int64_t trial_offset, float dt, float rtol, float atol, float dt_min,
                            int32_t* n_accept, int32_t* n_reject, int32_t* status,
                            void* workspace, size_t workspace_bytes, void* stream);

/* The path odecol_srk_fwd_adaptive integrates against: for every query time t[m] and trial b the cumulative pair
 *     w[m][b] = W(t) - W(t_begin),     iw[m][b] = int_{t_begin}^{t} (W(r) - W(t_begin)) dr         (float64)
 * of the tree spanning [t_begin, t_end].  For a step [a, b]: W = w(b) - w(a), U = iw(b) - iw(a) - (b - a) w(a) -- what
 * torchsde's bm(a, b, return_U=True) returns. */
int odecol_brownian_levy_query(uint64_t seed, int64_t trial_offset, int32_t B, float t_begin, float t_end, const float* t,
                               int32_t M, double* w, double* iw, void* stream);

/* Discrete adjoint of odecol_srk_fwd -- what loss.backward() through torchsde's unrolled srk steps computes (reference
 * scripts/wta_ode.py:174-181).  The noise is additive, but U enters the third drift stage, so the sweep needs the same
 * (dW, dU) tables or the same (seed, trial_offset) as the forward call.  Workspace:
 * odecol_workspace_bytes(p, ODECOL_OP_SRK_BWD, T, n_steps); grad_y / sel / G / grad_y0 / grad_W_aug as odecol_rk4_bwd. */
int odecol_srk_bwd(const odecol_problem* p, const float* ts, int32_t T, const float* y_steps, int64_t n_steps,
                   const float* dW, const float* dU, uint64_t seed, int64_t trial_offset,
                   const float* grad_y, const int32_t* sel, int32_t G, float dt,
                   float* grad_y0, float* grad_W_aug, void* workspace, size_t workspace_bytes, void* stream);

/* Batched Wong-Wang (2006) decision model: the training targets of the WTA task, one sample per thread, float64.
 * Replaces DM.run_sim / DM.simulate / DM.update (src/ww_model.py:92-127) inside the dataset loop make_ds_wwp
 * (scripts/wta_ode.py:56-93): three phases (mu = 0, mu = (muA, muB), mu = 0) of `steps_per_phase` updates of dt = 1e-3
 * each (the reference: int(5. / 1e-3) + 1 = 5001), firing rates recorded after every update.
 *   mu        (B, 2) float64 stimulus-phase inputs (muA, muB)
 *   i_noise0  (B, 2) float64 initial noise currents, or NULL for 0.  DM.reset() does not reset I_noise, so in the
 *             reference every sample but the first starts from the converged current (oracle/ww.py)
 *   states    (B, time_steps, 2) float32 out: r of update k for k = 0, every, 2 every, ... (first time_steps of them) --
 *             the `states` tensor of the dataset (R[:, ::10][:, :time_steps] transposed, wta_ode.py:82-87)
 *   sigma_noise  0 in the reference; otherwise the AMPA noise comes from Philox4x32-10 keyed by (seed, trial_offset + b)
 * Constants are those of DM.__init__ (src/ww_model.py:57-71). */
int odecol_ww_generate(const double* mu, const double* i_noise0, int32_t B, int32_t steps_per_phase, int32_t every,
                       int32_t time_steps, double sigma_noise, uint64_t seed, int64_t trial_offset,
                       float* states, void* stream);

/* Fused read-out loss on a trajectory restricted to read-out populations, with its gradient, in one pass:
 *     rate    = phi(V - A)                                    src/utils.py:13-25
 *     pred_g  = sum_k w[k] * rate[g*P + k]                    src/utils.py:79-84 (output_weights over the 8 populations)
 *     loss    = mean over (t, b, g) of smooth_l1(pred_g - target[t, b, g], beta)      src/utils.py:86-88
 * Replaces huber_loss_wta (src/utils.py:74-88) and loss.backward() down to the trajectory (scripts/wta_ode.py:178-179).
 *   y_sel    (T, B, 2*G*P): the V components of the G*P read-out populations, then their A components -- what
 *            odecol_rk4_fwd_ckpt returns for sel = [pops | N + pops]
 *   w        [P] or NULL (all ones);  target with element strides (st_t, st_b, st_g), 0 = broadcast along that axis
 *   loss     device scalar out;  grad_y_sel (T, B, 2*G*P) out = d loss / d y_sel (feeds odecol_*_bwd as grad_y)
 *   workspace  at least 8 bytes, 8-byte aligned */
int odecol_huber_rate_loss(const float* y_sel, int32_t T, int32_t B, int32_t G, int32_t P, const float* w,
                           const float* target, int64_t st_t, int64_t st_b, int64_t st_g, float beta,
                           float* loss, float* grad_y_sel, void* workspace, size_t workspace_bytes, void* stream);

/* Fused window read-out of the XOR and parity tasks, with its gradient, in one pass:
 *     pred_b = sum_k w[k] * mean over the last `last` grid points of phi(V_k - A_k)     k over the P read-out populations
 *     loss   = mean_b | pred_b - target[b] |
 * Replaces, down to the trajectory, compute_firing_rate + the final-point read-out of column C and
 * torch.mean(abs(final_fr_C - xor_targets)) (scripts/xor_ode.py:120-130: last = 1, w = ff_source_mask) and the mean over
 * the last 100 points times output_weights / output_scale with torch.mean(abs(final_fr_summed - parity_targets))
 * (scripts/parity_ode.py:239-249: last = 100), plus loss.backward() down to the solver output.
 *   y_sel    (T, B, 2*P): V of the P read-out populations, then their A (sel = [pops | N + pops])
 *   w        [P] or NULL (ones);  target [B];  loss device scalar out;  pred [B] out
 *   grad_y_sel (T, B, 2*P) out = d loss / d y_sel (zero outside the window)
 *   grad_w   (B, P) out: trial b's share of d loss / d w (sum over b for the gradient; the parity task trains
 *            output_weights through this read-out);  workspace >= 8 bytes, 8-byte aligned */
int odecol_window_rate_l1_loss(const float* y_sel, int32_t T, int32_t B, int32_t P, int32_t last, const float* w,
                               const float* target, float* loss, float* pred, float* grad_y_sel, float* grad_w,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Diagnostic: the tensor-core contraction core alone (3xTF32 tcgen05.mma with TMA-fed operands, FP32 accumulation in
 * tensor memory), C[n][m] = sum_k A[m][k] * B[n][k] for row-major A (M x K), B (N x K), C (N x M).  Lets the tests pin
 * the accuracy of the split-precision contraction the staged solver uses for large networks. */
size_t odecol_tc_contract_workspace_bytes(int32_t M, int32_t N, int32_t K);
int odecol_tc_contract(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Diagnostic: the MN-major variant used for the dW accumulation, C[m][n] = sum_k A[k][m] * B[k][n] for row-major
 * A (K x M), B (K x N), C (M x N). */
size_t odecol_tc_contract_tn_workspace_bytes(int32_t M, int32_t N, int32_t K);
int odecol_tc_contract_tn(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K,
                          void* workspace, size_t workspace_bytes, void* stream);

/* Which kernel family a call would use: 0 = persistent on-chip ("small", W row in registers),
 * 1 = staged dopri5 / Euler-Maruyama / srk (drift on the tensor cores), 2 = staged rk4 on the tcgen05 split-operand
 * contraction.  rk4 ops report 0 or 2, the others 0 or 1.  Diagnostic only. */
int odecol_kernel_family(const odecol_problem* p, int op);

/* Number of kernel launches the most recent entry-point call enqueued (process-wide, for bench bookkeeping). */
int64_t odecol_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* ODECOL_H */
