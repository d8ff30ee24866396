/*
 * sdcgym.h - C ABI of libsdcgym.so: the B200 (sm_100a) implementation of sdc-gym's data-parallel hot path.
 *
 * The reference (pancetta/sdc-gym) is pure Python and has no FFI boundary of its own; the seam this ABI
 * replaces is the body of the gym env methods
 *     SDC_Full_Env.reset / .step            sdc_gym/envs/sdc_env.py:316-332, 209-273   (gym id `sdc-v0`)
 *     SDC_Step_Env.step                     sdc_gym/envs/sdc_env.py:507-572            (gym id `sdc-v1`)
 *     SpectralRadiusLoss._get_spectral_radius   dp_playground.py:216-231
 *     ResidualLoss.take_step                dp_playground.py:247-258
 * executed for a whole batch ("vector") of independent envs per call.  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add; sdc_gym_b200/_lib.py is that binding.
 *
 * Conventions
 *  - Every entry point returns 0 on success, a negative SDCGYM_E* code for argument errors, or a positive
 *    cudaError_t.  Nothing throws across the ABI.
 *  - Device-pointer entry points never allocate, free or synchronise: all buffers are caller-owned device
 *    memory, work is enqueued on the caller's `stream` (a cudaStream_t passed as void*).
 *  - The host-pointer entry point (sdcgym_pipe_step) owns only its streams/events inside an opaque handle and
 *    returns when the results are in the caller's host buffers.
 *  - Batched env state is stored as planes ("struct of arrays"): plane p of env i lives at base[p*ld + i],
 *    `ld` >= N is the plane stride in elements.  Complex values are two consecutive planes (re, im).
 *      lam   : 2 planes            lambda of the running episode
 *      S     : 4*M planes          u_0.re,u_0.im,...,u_{M-1}.im, r_0.re,...,r_{M-1}.im
 *                                  (row i of the reference observation (2, M) complex128, transposed)
 *      resnorm : 1 plane           ||r||_inf of the current state (the next step's `norm_res_old`)
 *      niter, episodes, rng_ctr    int32 / int32 / uint32 planes
 *  - All arithmetic is IEEE binary64 and reproduces the reference's numpy/OpenBLAS rounding sequence
 *    (`blas_variant` selects the OpenBLAS core whose scalar tails are emulated).
 */
#ifndef SDCGYM_H
#define SDCGYM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDCGYM_ABI_VERSION 14 /* 5: sweep_mode + work buffers in sdcgym_state; 6: in-kernel peer-memory statistics exchange; 7: sdcgym_state.norm_init; 8: sdcgym_state.phase_*; 9: sdcgym_replay_*; 10: sdcgym_spectral_radius_grad_sum; 11: sdcgym_residual_sweeps; 12: sdcgym_residual_sweeps_sum; 13: sdcgym_full_solve_counts; 14: sdcgym_full_solve_counts_population, sdcgym_spectral_radius_grad_sum_population */
#define SDCGYM_MAX_M 9
#define SDCGYM_CERT_PLANES 8

/* error codes (negative); positive return values are cudaError_t */
#define SDCGYM_EINVAL (-1)       /* bad argument value */
#define SDCGYM_EUNSUPPORTED (-2) /* M / prec_type / strategy combination not compiled in */
#define SDCGYM_ENULL (-3)        /* required pointer is NULL */
#define SDCGYM_ENOMEM (-4)       /* host-pipe allocation failed */

/* env_kind: which reference env class the step reproduces */
#define SDCGYM_ENV_FULL 0 /* sdc-v0, SDC_Full_Env: iterate to convergence / max_iters / divergence */
#define SDCGYM_ENV_STEP 1 /* sdc-v1, SDC_Step_Env: one sweep per step */

/* prec_type: how the action parameterises Q_delta (dp_playground.py:194-207) or a fixed matrix
 * (prec='LU'|'min'|'EE'|'zeros', sdc_env.py:141-188; the matrix itself is supplied in `Qd_fixed`) */
#define SDCGYM_PREC_DIAG 0
#define SDCGYM_PREC_LOWER_DIAG 1
#define SDCGYM_PREC_LOWER_TRI 2
#define SDCGYM_PREC_STRICTLY_LOWER_TRI 3
#define SDCGYM_PREC_FIXED 4

/* reward_strategy (sdc_env.py:427-463) */
#define SDCGYM_REW_ITERATION_ONLY 0
#define SDCGYM_REW_RESIDUAL_CHANGE 1
#define SDCGYM_REW_GAUSS_KERNEL 2
#define SDCGYM_REW_FAST_CONVERGENCE 3
#define SDCGYM_REW_SMOOTH_FAST_CONVERGENCE 4
#define SDCGYM_REW_SMOOTHER_FAST_CONVERGENCE 5
#define SDCGYM_REW_SPECTRAL_RADIUS 6

/* flags plane written by sdcgym_step (one byte per env) */
#define SDCGYM_FLAG_DONE 1      /* episode ended (gym `done`; always set for sdc-v0) */
#define SDCGYM_FLAG_CONVERGED 2 /* ||r|| < restol */
#define SDCGYM_FLAG_ERR 4       /* NaN/Inf or residual grew > 100x (sdc_env.py:234,241,527,532) */

/* bits of sdcgym_env_desc.do_scale (0 / 1 as before; bit 1 added for use_doubles=False) */
#define SDCGYM_ACTION_SCALE 1 /* do_scale: map real actions [-1,1] -> [0,1] (sdc_env.py:125-132) */
#define SDCGYM_ACTION_F32 2   /* use_doubles=False: Q_delta entries are stored in the float32/complex64 action
                               * dtype (sdc_env.py:100,109,138-140): the scaled action is rounded to float32 */

/* sweep_mode: how the sdc-v0 full solve iterates (sdc_env.py:224-247)
 *   EXACT      the reference's numpy/OpenBLAS rounding sequence, operation for operation: every output bit-equal.
 *   CERTIFIED  substitution sweeps  u+ = u + Pinv r,  r+ = u0 - u+ + z (Q u+)  with the real collocation matrix (the
 *              node-by-node form of sdc_env_nonlinear.py:248-264; about half the FP64 instructions, and no
 *              np.linalg.inv emulation).  Each `nr > 100 nr_old` / `nr < restol` decision is taken with a rigorous
 *              running bound on |nr - nr_reference| (csrc/certify.cuh); envs that meet a decision inside the bound are
 *              re-run by the exact kernel.  niter / done / converged / err are bit-equal to the reference for EVERY env;
 *              u, r, ||r||, reward agree within rounding (<= 1e-12 relative).  Applies to sdc-v0 steps that start from
 *              an exact state (after reset / auto-reset); combinations without a certificate (sdc-v1, collect_states)
 *              run the exact kernel.  Needs the work buffers of sdcgym_state. */
#define SDCGYM_PHASE_COUNTERS 8
#define SDCGYM_SWEEP_EXACT 0
#define SDCGYM_SWEEP_CERTIFIED 1

/* OpenBLAS core whose rounding sequence is reproduced */
#define SDCGYM_BLAS_SKYLAKEX 0
#define SDCGYM_BLAS_HASWELL 1

/* Static description of a batch of envs = the reference constructor arguments (sdc_env.py:27-46). */
typedef struct sdcgym_env_desc {
    int32_t M;                 /* collocation nodes, 2..SDCGYM_MAX_M */
    int32_t env_kind;          /* SDCGYM_ENV_* */
    int32_t prec_type;         /* SDCGYM_PREC_* */
    int32_t action_is_complex; /* free_action_space: actions are (re, im) pairs */
    int32_t do_scale;          /* SDCGYM_ACTION_* bits: scale real actions [-1,1] -> [0,1]; float32 Q_delta */
    int32_t max_iters;         /* 50 (sdc_env.py:25) */
    int32_t reward_strategy;   /* SDCGYM_REW_* */
    int32_t blas_variant;      /* SDCGYM_BLAS_* */
    int32_t autoreset;         /* DummyVecEnv semantics: a finished env is reset inside the step */
    int32_t curriculum;        /* lambda_real_interpolation_interval given (sdc_env.py:287-292) */
    int32_t sweep_mode;        /* SDCGYM_SWEEP_* */
    int32_t reserved0;
    double dt, restol, step_penalty, residual_weight, norm_factor;
    double lam_re_lo, lam_re_hi, lam_im_lo, lam_im_hi; /* lambda sampling box */
    double interp_x0, interp_x1;                       /* curriculum episode interval */
    uint64_t seed;                                     /* Philox key */
    int64_t env_offset;                                /* global index of local env 0 (multi-GPU shard) */
    double Q[SDCGYM_MAX_M * SDCGYM_MAX_M];             /* collocation matrix, row-major M x M (leading entries) */
    double Qd_fixed[SDCGYM_MAX_M * SDCGYM_MAX_M];      /* SDCGYM_PREC_FIXED: real Q_delta, row-major M x M */
} sdcgym_env_desc;

/* Device-resident state of N envs (planes, see above). */
typedef struct sdcgym_state {
    int64_t N, ld;
    double* lam;       /* [2][ld] */
    double* S;         /* [4M][ld] */
    double* resnorm;   /* [ld] */
    int32_t* niter;    /* [ld] */
    int32_t* episodes; /* [ld]  num_episodes (sdc_env.py:81,276) */
    uint32_t* rng_ctr; /* [ld]  number of lambda draws made so far */
    double* norm_init; /* [ld] or NULL: ||initial residual of the running episode||_inf (scaled by norm_factor), written by
                        * every reset / auto-reset.  The `residual_change` reward divides by its logarithm
                        * (sdc_env.py:337-350); with the plane the step reads 8 bytes instead of re-deriving the initial
                        * state and its norm (~250 FP64 instructions per env-step).  Same bits either way.  Used by
                        * sdc-v1 (SDCGYM_ENV_STEP) only: the sdc-v0 step kernels neither read nor refresh it. */
    /* work buffers of SDCGYM_SWEEP_CERTIFIED (NULL otherwise): */
    float* cert;            /* [SDCGYM_CERT_PLANES][ld] per-env certificate constants, rewritten by every step */
    int32_t* fallback_list; /* [N] indices of the envs the exact kernel re-ran in the last step */
    int32_t* fallback_count; /* [2]: length of fallback_list for the last step, cumulative count over all steps */
    /* optional work buffers of the PHASED full solve (all three or none; NULL = single-launch kernels).  sdc-v0 with a
     * non-diagonal Q_delta, M <= 7, large batches: the envs of a warp stop after very different sweep counts, so the
     * solve is cut at fixed sweep counts and every later pass runs over the compacted list of the envs still
     * iterating (csrc/step_kernels.cuh, step_one PHASE).  Same sweep sequence per env, every output bit-identical. */
    int32_t* phase_list;  /* [2][N] ping-pong lists of suspended envs (indices local to this state) */
    int32_t* phase_count; /* [SDCGYM_PHASE_COUNTERS] list length per pass of the last step */
    double* phase_pinv;   /* [2 M^2][ld] inverse of I - z Q_delta of the suspended envs */
} sdcgym_state;

/* Per-step inputs/outputs (device pointers; NULL outputs are skipped). */
typedef struct sdcgym_step_io {
    const double* action;      /* element (env i, component k): action[i*env_stride + k*comp_stride] (+1 = imag) */
    int64_t action_env_stride; /* in doubles */
    int64_t action_comp_stride;
    double* reward;        /* [N] */
    uint8_t* flags;        /* [N] SDCGYM_FLAG_* */
    double* info_residual; /* [N]  info['residual'] */
    int32_t* info_niter;   /* [N]  info['niter'] */
    double* info_lam;      /* [N][2] info['lam'] (the lambda the step ran with), interleaved complex128 */
    double* terminal_obs;  /* [4M][ld] state at episode end; written for envs whose DONE flag is set */
    double* old_states;    /* collect_states: (N, 2M, max_iters) complex128, env-major (reference layout) or NULL */
} sdcgym_step_io;

int sdcgym_abi_version(void);

/* number of action components for (M, prec_type): M, M-1, M(M+1)/2, M(M-1)/2, 0 */
int sdcgym_num_actions(int M, int prec_type);

/* 1 if the (M, prec_type) combination has a compiled kernel */
int sdcgym_supported(int M, int prec_type);

/*
 * reset (sdc_env.py:316-332) of the envs with mask[i] != 0 (all envs when mask == NULL):
 * episodes += 1, niter = 0, lambda drawn from the Philox stream (or taken from lam_in[2][ld] when non-NULL),
 * u = 1, r = u0 - C u, resnorm = ||r||_inf.  With old_states != NULL column 0 is set and the rest zeroed.
 */
int sdcgym_reset(const sdcgym_env_desc* desc, const sdcgym_state* st, const double* lam_in, const uint8_t* mask,
                 double* old_states, void* stream);

/* env.step(action) for all N envs (sdc_env.py:209-273 / 507-572), plus the DummyVecEnv auto-reset when
 * desc->autoreset != 0. */
int sdcgym_step(const sdcgym_env_desc* desc, const sdcgym_state* st, const sdcgym_step_io* io, void* stream);

/*
 * The sdc-v0 full solve (sdc_env.py:209-273) of N nodes from the reset state, without any env state: what
 * sdcgym_reset(lam_in) followed by sdcgym_step gives for each node, bit for bit, but nothing is read or written besides
 * lambda, the action rows and the outputs below.  The evaluation of a Q_delta by its iteration counts
 * (rl_playground.py:147-156, dp_playground.py:844-957).
 *   desc     env_kind SDCGYM_ENV_FULL; M, prec_type, Q, Qd_fixed, dt, restol, max_iters, action_is_complex, do_scale and
 *            blas_variant as for sdcgym_step (the reward, seed and sampling fields are not used)
 *   grid     NULL: node i has lambda lam[2i] + i lam[2i+1].  Else node i is grid node first + i of the (n_re x n_im)
 *            tensor grid over [re_lo, re_hi] x [im_lo, im_hi], row-major over (re, im), end points included: the same
 *            bits as the nodes of sdcgym_spectral_radius / sdcgym_residual_sweeps_sum in grid mode.
 *   action   element (node i, component k) at action[i*a_es + k*a_cs] (+1 = imag), a_es = 0 for one row shared by
 *            every node; NULL with SDCGYM_PREC_FIXED
 *   outputs  each optional (NULL: not written): niter_out [N] int32 (info['niter']), residual_out [N] (info['residual']),
 *            flags_out [N] SDCGYM_FLAG_*, lam_out [N][2] (the lambda each node ran with)
 *   hist     optional, int64 [max_iters + 3], zeroed by the call: [0, max_iters] the niter of the converged nodes,
 *            [max_iters + 1] the number of err nodes, [max_iters + 2] the nodes that ran out of sweeps unconverged
 * Refusals, all before any CUDA call: NULL desc: SDCGYM_ENULL; env_kind != SDCGYM_ENV_FULL, or an unsupported M,
 * prec_type or blas_variant: SDCGYM_EUNSUPPORTED; N > 0 without actions for a learned prec_type, or without lam in list
 * mode: SDCGYM_ENULL; actions with SDCGYM_PREC_FIXED, per-node rows (a_es != 0) in grid mode, N < 0, max_iters outside
 * 0..16384, or a grid range outside the grid: SDCGYM_EINVAL.  N = 0 only zeroes hist.  No host synchronisation: the
 * call can be captured in a CUDA graph.
 */
typedef struct sdcgym_lambda_grid {
    int64_t n_re, n_im, first;
    double re_lo, re_hi, im_lo, im_hi;
} sdcgym_lambda_grid;
int sdcgym_full_solve_counts(const sdcgym_env_desc* desc, const sdcgym_lambda_grid* grid, int64_t N, const double* lam,
                             const double* action, int64_t a_es, int64_t a_cs, int32_t* niter_out, double* residual_out,
                             uint8_t* flags_out, double* lam_out, int64_t* hist, void* stream);

/*
 * sdcgym_full_solve_counts' histogram for each of P action rows, every row shared by all N nodes: hist int64
 * [P][max_iters + 3], row p at action + p*a_rs (component k at + k*a_cs, +1 = imag).  hist[p] equals, bit for bit,
 * the histogram of sdcgym_full_solve_counts(desc, grid, N, lam, action + p*a_rs, a_es = 0, a_cs) (one launch, row p =
 * blockIdx.y; P above 65535 takes several launches).  No per-node outputs.
 * Refusals, all before any CUDA call: NULL desc, hist or action, or N > 0 without lam in list mode: SDCGYM_ENULL;
 * env_kind != SDCGYM_ENV_FULL, SDCGYM_PREC_FIXED, or an unsupported M, prec_type or blas_variant: SDCGYM_EUNSUPPORTED;
 * P < 1, N < 0, max_iters outside 0..16384, or a grid range outside the grid: SDCGYM_EINVAL.  N = 0 only zeroes hist.
 * No host synchronisation: the call can be captured in a CUDA graph.
 */
int sdcgym_full_solve_counts_population(const sdcgym_env_desc* desc, const sdcgym_lambda_grid* grid, int64_t N,
                                        const double* lam, int64_t P, const double* action, int64_t a_rs,
                                        int64_t a_cs, int64_t* hist, void* stream);

/* planes S[4M][ld] -> reference observation layout obs[N][2][M] complex128 (interleaved re, im) and back */
int sdcgym_export_obs(int M, int64_t N, int64_t ld, const double* S, double* obs, void* stream);
int sdcgym_import_obs(int M, int64_t N, int64_t ld, const double* obs, double* S, void* stream);

/* `P` consecutive planes X[P][ld] -> rows out[N][P] (env-major).  With X = S + 2M*ld and P = 2M this is the residual
 * half of the observation, obs[:, 1, :] as [N][M] complex128; with X = S the u half, obs[:, 0, :]. */
int sdcgym_export_rows(int P, int64_t N, int64_t ld, const double* X, double* out, void* stream);

/* recompute resnorm = ||r||_inf from S (after a state injection) */
int sdcgym_refresh_resnorm(int M, int64_t N, int64_t ld, const double* S, double* resnorm, void* stream);

/*
 * Spectral radius rho(lam*dt * inv(I - lam*dt*Qd) (Q - Qd)) for N (lambda, Q_delta-parameter) pairs
 * (dp_playground.py:216-228; sdc_env.py:421-425).  lam: [N] complex128 interleaved.  qd: [N][A] real or
 * complex (interleaved) parameters in get_qdmat's layout (dp_playground.py:194-207); for SDCGYM_PREC_FIXED
 * `qd` is ignored and Qd_fixed (real M x M) is used.  rho: [N].
 * If lam == NULL, lambdas are the nodes of a (grid_re x grid_im) tensor grid over [re_lo,re_hi] x [im_lo,im_hi]
 * (row-major over re then im, end points included) and qd, if given, has a single row.  The call evaluates the N
 * nodes with flat indices grid_first .. grid_first+N-1 (grid_first = 0, N = grid_re*grid_im: the whole grid), so that
 * ranks can shard the grid by rows and all-reduce one scalar for the mean loss.
 */
typedef struct sdcgym_rho_desc {
    int32_t M, prec_type, qd_is_complex, qd_broadcast;
    double dt;
    double Q[SDCGYM_MAX_M * SDCGYM_MAX_M];
    double Qd_fixed[SDCGYM_MAX_M * SDCGYM_MAX_M];
    int64_t grid_re, grid_im, grid_first;
    double re_lo, re_hi, im_lo, im_hi;
} sdcgym_rho_desc;
int sdcgym_spectral_radius(const sdcgym_rho_desc* desc, int64_t N, const double* lam, const double* qd, double* rho,
                           void* stream);

/*
 * rho and its gradient with respect to the Q_delta parameters (what jax.value_and_grad(loss) evaluates,
 * dp_playground.py:1073, for the spectral-radius loss): grad[N][A][2] receives g (complex, interleaved) with
 * d rho = Re(sum_k g_k d theta_k); for real parameters d rho / d theta_k = Re g_k.  lam / qd as in
 * sdcgym_spectral_radius (no grid / broadcast mode).  Valid where the dominant eigenvalue is simple.
 */
int sdcgym_spectral_radius_grad(const sdcgym_rho_desc* desc, int64_t N, const double* lam, const double* qd, double* rho,
                                double* grad, void* stream);

/*
 * Sum over N samples of rho and of d rho / d theta for ONE shared parameter row (desc->qd_broadcast must be 1):
 * sums[0] = sum rho, sums[1 + 2k], sums[2 + 2k] = sum Re g_k, sum Im g_k (g as in sdcgym_spectral_radius_grad).
 * lam [N][2], or NULL for grid mode (grid_re/grid_im/grid_first/box as in sdcgym_spectral_radius).  rho [N] is
 * optional (NULL: not written).  scratch: caller-owned device memory of
 * sdcgym_spectral_radius_grad_sum_scratch_doubles(M, prec_type, N) doubles.  Deterministic: every sum is a balanced
 * binary tree whose shape depends on N only.  A failed sample (rho NaN) makes sums[0] NaN; lambda = 0 adds zeros.
 * N = 0 writes zeros to sums.  SDCGYM_PREC_FIXED has nothing to differentiate: SDCGYM_EUNSUPPORTED.
 */
int64_t sdcgym_spectral_radius_grad_sum_scratch_doubles(int M, int prec_type, int64_t N);
int sdcgym_spectral_radius_grad_sum(const sdcgym_rho_desc* desc, int64_t N, const double* lam, const double* qd,
                                    double* rho, double* scratch, double* sums, void* stream);

/*
 * sdcgym_spectral_radius_grad_sum for each of P parameter rows, every row shared by all N samples: row p at
 * qd + p*qd_rs doubles (desc->qd_broadcast must be 1, qd_is_complex as for the single row), sums [P][1 + 2A].
 * sums[p] equals, bit for bit, the sums of sdcgym_spectral_radius_grad_sum on row p: per row, the same tile tree
 * and fold tree.  scratch: caller-owned device memory of P * sdcgym_spectral_radius_grad_sum_scratch_doubles(M,
 * prec_type, N) doubles.  P above 65535 / (1 + 2A) rows takes several launches.
 * Refusals, all before any CUDA call: NULL desc, qd, scratch or sums: SDCGYM_ENULL; unsupported M / prec_type, or
 * SDCGYM_PREC_FIXED: SDCGYM_EUNSUPPORTED; qd_broadcast != 1, P < 1, N < 0, or in grid mode a node range outside the
 * grid: SDCGYM_EINVAL.  N = 0 writes zeros to sums.  No host synchronisation.
 */
int sdcgym_spectral_radius_grad_sum_population(const sdcgym_rho_desc* desc, int64_t N, const double* lam, int64_t P,
                                               const double* qd, int64_t qd_rs, double* scratch, double* sums,
                                               void* stream);

/*
 * ResidualLoss.take_step (dp_playground.py:247-258) for N samples: u' = u + inv(I - lam*dt*Qd) r_old,
 * r' = u0 - C u', norm = ||r'||_inf.  lam [N], u0/u/r_old/u_out/r_out [N][M] complex128 interleaved,
 * qd as in sdcgym_spectral_radius, Cs [N][M][M] complex128 or NULL (then C = I - lam*dt*Q is formed on the fly).
 * JAX arithmetic in the reference: agreement is to rounding level (1e-12 relative), not bit-exact.
 * grad (optional, [N][A][2]): d norm / d theta_k as complex g with d norm = Re(sum_k g_k d theta_k) - the
 * per-sample gradient jax.value_and_grad(loss) needs for the residual loss (dp_playground.py:1073).
 */
int sdcgym_residual_step(const sdcgym_rho_desc* desc, int64_t N, const double* lam, const double* qd, const double* Cs,
                         const double* u0, const double* u, const double* r_old, double* u_out, double* r_out,
                         double* norm_out, double* grad, void* stream);

/*
 * ||r_K||_inf after exactly K = `sweeps` (1..50) sweeps of the iteration take_step runs, for N samples, and its gradient
 * through all K sweeps (SDC_Fix_Env's fixed sweep count, no early stop at restol and no divergence test):
 *     delta_k = inv(I - lam*dt*Qd) r_k,   u_{k+1} = u_k + delta_k,   r_{k+1} = u0 - (I - lam*dt*Q) u_{k+1}.
 * lam [N] complex128 interleaved; qd as in sdcgym_spectral_radius, one row shared by every sample with
 * desc->qd_broadcast (read in place, not expanded); u0/u/r [N][M] complex128 interleaved, or all three NULL for the
 * envs' reset state u0 = u = 1, r = u0 - C 1 (then only lam and qd are read).  u_out/r_out [N][M] (u_K, r_K) and
 * grad [N][A][2] are optional.  grad receives g with d norm = Re(sum_k g_k d theta_k), the derivative with respect to
 * theta through every sweep (u0 and the incoming u, r constant); K = 1 is sdcgym_residual_step's gradient.
 * norm_out [N]: +inf where the iteration overflowed, NaN where any component of r_K is NaN.  A norm that is 0, +inf or
 * NaN gives g = 0.  Agreement with the reference is to rounding level, not bit-exact.
 * Refusals, all before any CUDA call: NULL desc, lam or norm_out, or only some of u0/u/r: SDCGYM_ENULL; unsupported
 * M / prec_type, or grad with SDCGYM_PREC_FIXED: SDCGYM_EUNSUPPORTED; N < 0 or sweeps outside 1..50: SDCGYM_EINVAL.
 * N = 0 is a no-op.
 */
int sdcgym_residual_sweeps(const sdcgym_rho_desc* desc, int64_t N, int sweeps, const double* lam, const double* qd,
                           const double* u0, const double* u, const double* r, double* u_out, double* r_out,
                           double* norm_out, double* grad, void* stream);

/*
 * Sum over N samples of a loss of ||r_K||_inf (sdcgym_residual_sweeps) and of its gradient, for ONE shared parameter
 * row (desc->qd_broadcast must be 1, the row is read in place).  With n_K = ||r_K||_inf, n_0 = ||r_0||_inf of the
 * starting residual (same hypot / max / NaN rule) and g the per-sample gradient of sdcgym_residual_sweeps (g = 0 where
 * n_K is 0, +inf or NaN), each sample contributes a value f and a weighted gradient:
 *     SDCGYM_SWEEPS_MEAN       f = n_K                g
 *     SDCGYM_SWEEPS_LOG_RATIO  f = log(n_K / n_0)     g / n_K
 * log_ratio: a sample with n_0 = 0 (lambda = 0 from the reset state, e.g. the corner node of a grid whose box ends at
 * 0) contributes exact zeros to f and to the gradient; any other non-finite f (n_K = 0 gives -inf; NaN) reaches
 * sums[0] unchanged.  sums[0] = sum f, sums[1 + 2k], sums[2 + 2k] = sum Re, sum Im of the weighted g_k: the layout of
 * sdcgym_spectral_radius_grad_sum's sums, so the mean divides every entry by N.
 * lam [N][2], or NULL for grid mode (grid_re/grid_im/grid_first/box as in sdcgym_spectral_radius).  u0/u/r [N][M]
 * complex128 interleaved (list mode only), or all three NULL for the envs' reset state.  norm_out [N] (n_K) is
 * optional.  scratch: caller-owned device memory of exactly sdcgym_spectral_radius_grad_sum_scratch_doubles(M,
 * prec_type, N) doubles (the same tile and fold tree).  Deterministic: every sum is a balanced binary tree whose shape
 * depends on N only.
 * Refusals, all before any CUDA call: NULL desc, qd, scratch or sums, or only some of u0/u/r: SDCGYM_ENULL;
 * unsupported M / prec_type, or SDCGYM_PREC_FIXED: SDCGYM_EUNSUPPORTED; qd_broadcast != 1, N < 0, sweeps outside
 * 1..50, an unknown reduction, or in grid mode a node range outside the grid or u0/u/r given: SDCGYM_EINVAL.
 * N = 0 writes zeros to sums.
 */
#define SDCGYM_SWEEPS_MEAN 0
#define SDCGYM_SWEEPS_LOG_RATIO 1
int sdcgym_residual_sweeps_sum(const sdcgym_rho_desc* desc, int64_t N, int sweeps, int reduction, const double* lam,
                               const double* qd, const double* u0, const double* u, const double* r, double* norm_out,
                               double* scratch, double* sums, void* stream);

/*
 * Device-side VecNormalize building blocks (SB3 RunningMeanStd semantics; utils/utils.py:295-312).
 * Planes X[P][ld] (observation planes S, or a single reward/return plane with P = 1).
 *   accumulate : sums[p] = sum_i (x_pi - shift_p), sums[P+p] = sum_i (x_pi - shift_p)^2   (deterministic tree;
 *                scratch needs sdcgym_vecnorm_scratch_doubles(P) doubles).  `sums` of several ranks may be
 *                all-reduced before the merge; shift must then be identical on all ranks (use the running mean).
 *   merge      : Chan update of (mean[P], var[P], count) with a batch of `batch_count` samples described by
 *                `sums` taken with shift == mean.  count2 = {count, scratch}.
 *   apply      : Y = clip((X - mean) / sqrt(var + eps), -clip, clip)
 *   returns    : ret = ret * gamma + reward
 *   reward     : out = normalize ? clip(reward / sqrt(ret_var + eps), +-clip) : reward; ret = 0 where DONE
 */
int sdcgym_vecnorm_scratch_doubles(int P);
int sdcgym_vecnorm_accumulate(int P, int64_t N, int64_t ld, const double* X, const double* shift, double* scratch,
                              double* sums, void* stream);
int sdcgym_vecnorm_merge(int P, double batch_count, const double* sums, double* mean, double* var, double* count2,
                         void* stream);
/* Single-rank fast path: accumulate + merge (+ commit) in ONE launch, bit-identical to the sequence above (the last
 * block folds the partial sums in index order).  `scratch` must be zero-initialised once (it holds a ticket word the
 * kernel resets itself) and `sdcgym_vecnorm_scratch_doubles(P)` doubles long.  `_update_returns` also advances the
 * discounted returns in the same pass: returns <- returns * gamma + reward, then updates the return statistics
 * (mean/var/count2 of ONE plane; scratch sized for P = 1). */
int sdcgym_vecnorm_update(int P, int64_t N, int64_t ld, const double* X, double* mean, double* var, double* count2,
                          double* scratch, double* sums, void* stream);
int sdcgym_vecnorm_update_returns(int64_t N, const double* reward, double gamma, double* returns, double* mean,
                                  double* var, double* count2, double* scratch, double* sums, void* stream);
/*
 * Several ranks (one process per GPU, envs sharded, SURVEY 8e): the same single launch, with the all-reduce of the
 * moment sums done INSIDE the kernel over peer memory (NVLink / NVSwitch P2P stores and flags) instead of
 * accumulate -> ncclAllReduce -> merge.  Every rank owns an exchange region of sdcgym_xchg_bytes(world, slot_doubles)
 * bytes (slot_doubles >= 2P + 1), allocated with sdcgym_ipc_alloc and opened by the other ranks' processes with
 * sdcgym_ipc_open (the 64-byte handles travel over the host-side process group); `peers[r]` is rank r's region as
 * seen from this process (`peers[rank]` the local one).  `seq` must be 1, 2, 3, ... for successive calls on one set of
 * regions, identically on all ranks; all ranks must make the call (a rank with N = 0 included).  The sums are added
 * in rank order on every rank, so the normalisers stay bit-identical across ranks.
 */
#define SDCGYM_MAX_RANKS 16
typedef struct sdcgym_xchg {
    int32_t world, rank;
    int32_t slot_doubles, reserved;
    uint64_t seq;
    void* peers[SDCGYM_MAX_RANKS];
} sdcgym_xchg;
size_t sdcgym_xchg_bytes(int world, int slot_doubles);
int sdcgym_vecnorm_update_dist(int P, int64_t N, int64_t ld, const double* X, double* mean, double* var, double* count2,
                               double* scratch, double* sums, const sdcgym_xchg* xchg, void* stream);
int sdcgym_vecnorm_update_returns_dist(int64_t N, const double* reward, double gamma, double* returns, double* mean,
                                       double* var, double* count2, double* scratch, double* sums,
                                       const sdcgym_xchg* xchg, void* stream);
/* Observation planes and the return plane in ONE launch (what a normalised training step needs): equivalent, bit for
 * bit, to sdcgym_vecnorm_update followed by sdcgym_vecnorm_update_returns.  `scratch`: sdcgym_vecnorm_scratch_doubles(P + 1)
 * doubles, zero-initialised once.  `xchg` == NULL: single rank; else the in-kernel exchange with slot_doubles >= 2P + 3. */
int sdcgym_vecnorm_update_both(int P, int64_t N, int64_t ld, const double* X, const double* reward, double gamma,
                               double* returns, double* obs_mean, double* obs_var, double* obs_count2, double* ret_mean,
                               double* ret_var, double* ret_count2, double* scratch, double* sums_obs, double* sums_ret,
                               const sdcgym_xchg* xchg, void* stream);
/* device memory that other processes can map: cudaMalloc + zero fill + cudaIpcGetMemHandle / cudaIpcOpenMemHandle
 * (with peer access enabled lazily) / close / free */
int sdcgym_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64);
int sdcgym_ipc_open(const unsigned char* handle64, void** dev_ptr);
int sdcgym_ipc_close(void* dev_ptr);
int sdcgym_ipc_free(void* dev_ptr);
int sdcgym_vecnorm_apply(int P, int64_t N, int64_t ld, const double* X, const double* mean, const double* var, double eps,
                         double clip, double* Y, void* stream);
int sdcgym_vecnorm_returns(int64_t N, const double* reward, double gamma, double* returns, void* stream);
int sdcgym_vecnorm_reward(int64_t N, const double* reward, const uint8_t* flags, const double* ret_var, double eps,
                          double clip, int normalize, double* out, double* returns, void* stream);

/*
 * Generalised advantage estimation over a device rollout of T steps x N envs (arrays [T][N], env index fastest):
 * SB3 RolloutBuffer.compute_returns_and_advantage, the consumer of the rollouts rl_playground.py collects through
 * model.learn (rl_playground.py:286).  episode_starts[t][i] != 0 marks that step t begins a new episode of env i.
 */
int sdcgym_gae(int T, int64_t N, const double* rewards, const double* values, const uint8_t* episode_starts,
               const double* last_values, const uint8_t* last_dones, double gamma, double gae_lambda,
               double* advantages, double* returns, void* stream);

/*
 * Replay buffer of an off-policy learner (SB3 ReplayBuffer + OffPolicyAlgorithm._store_transition; csrc/replay.cu).
 * A ring of `rows` rows x N envs, every array caller-owned device memory:
 *     obs, next_obs  [rows][P][ld]   observation planes (P = 4M, the layout of S), raw (un-normalised)
 *     actions        [rows][N][A]    doubles; complex actions are A = 2 n_act interleaved (re, im)
 *     rewards        [rows][N]       raw reward
 *     dones          [rows][N]       flags & SDCGYM_FLAG_DONE
 *     counters       [3]             pos, full (0/1), number of sample calls so far; zero-initialised by the caller
 * The counters are read and advanced on the device only, so the calls below can be captured in a CUDA graph.
 *   store_obs : obs[pos] = S                          (before the step: the observation the action is taken on)
 *   store     : next_obs[pos] = DONE ? terminal : S, actions / rewards / dones[pos]; then pos += 1, wrapping to 0
 *               and setting full.  `terminal` may be NULL when the envs are not auto-reset.  action: element (i, k)
 *               at action[i*action_stride + k].
 *   sample    : B transitions drawn with replacement (rows below pos, or all rows once full; envs uniformly) from the
 *               Philox stream keyed by `seed` (csrc/replay_index.cuh), gathered as obs / next_obs planes [P][B],
 *               actions [B][A], rewards [B], dones [B] (0.0 / 1.0), then the call counter advances.  obs_mean/obs_var
 *               non-NULL: observations normalised as sdcgym_vecnorm_apply does; ret_var non-NULL: rewards as
 *               sdcgym_vecnorm_reward does (same bits).  Sampling an empty buffer reads row 0.
 */
typedef struct sdcgym_replay {
    int32_t P, A;
    int64_t rows, N, ld; /* rows, N < 2^32 */
    uint64_t seed;
    double* obs;
    double* next_obs;
    double* actions;
    double* rewards;
    uint8_t* dones;
    int64_t* counters;
} sdcgym_replay;
int sdcgym_replay_store_obs(const sdcgym_replay* rb, const double* S, int64_t s_ld, void* stream);
int sdcgym_replay_store(const sdcgym_replay* rb, const double* S, const double* terminal, int64_t s_ld,
                        const uint8_t* flags, const double* reward, const double* action, int64_t action_stride,
                        void* stream);
int sdcgym_replay_sample(const sdcgym_replay* rb, int64_t B, const double* obs_mean, const double* obs_var,
                         const double* ret_var, double eps, double clip_obs, double clip_reward, double* obs,
                         double* next_obs, double* actions, double* rewards, double* dones, void* stream);

/*
 * Host-buffer step: `DummyVecEnv.step(actions)` with numpy-style HOST arrays on both sides, as one call.
 * Device buffers (state, staging for actions `dev->action` [N][A], outputs in `dev`, `obs_dev` [N][2][M] complex128)
 * stay caller-owned; the pipe owns its streams, events and a 256 kB staging block.  The batch is cut into `chunks`
 * pieces (boundaries grow like c^1.5) and H2D(actions) | step + export kernels | D2H(results) are overlapped; the call
 * returns when the host arrays are filled.  Batches whose results fit the staging block are instead packed on the
 * device and leave in one transfer on `caller_stream` (`obs_dev` is not written then).  Page-locked host memory
 * (sdcgym_host_alloc, cudaHostAlloc, torch pin_memory) makes the copies asynchronous; pageable memory works but
 * serialises them.  NULL host outputs are skipped.
 */
typedef struct sdcgym_pipe sdcgym_pipe;
typedef struct sdcgym_host_io {
    const double* action; /* [N][A] (complex: [N][A][2]) */
    double* obs;          /* [N][2][M] complex128 (reference observation layout) */
    double* reward;       /* [N] */
    uint8_t* flags;       /* [N] */
    int32_t* niter;       /* [N] */
    double* residual;     /* [N] */
    double* lam;          /* [N][2] */
} sdcgym_host_io;
int sdcgym_pipe_create(int max_chunks, sdcgym_pipe** out);
int sdcgym_pipe_destroy(sdcgym_pipe* pipe);
int sdcgym_pipe_step(sdcgym_pipe* pipe, const sdcgym_env_desc* desc, const sdcgym_state* st, const sdcgym_step_io* dev,
                     double* obs_dev, const sdcgym_host_io* host, int chunks, void* caller_stream);
/*
 * The same host-buffer step through a device-side VecNormalize (utils/utils.py:295-312: DummyVecEnv wrapped in
 * VecNormalize is how the reference trains): step -> statistics update (training) -> normalised observation planes
 * -> discounted returns / return statistics -> normalised reward -> host, in one call and, for small batches, one
 * D2H transfer.  `host->obs` and `host->reward` receive the NORMALISED observation / reward; the raw reward stays
 * in `dev->reward`.  Single-rank statistics only (a multi-rank normaliser needs the all-reduce between
 * sdcgym_vecnorm_accumulate and _merge).  All pointers are device memory owned by the caller.
 */
typedef struct sdcgym_vecnorm {
    int32_t norm_obs, norm_reward, training, reserved;
    double gamma, epsilon, clip_obs, clip_reward;
    double* obs_mean;    /* [4M] */
    double* obs_var;     /* [4M] */
    double* obs_count2;  /* [2] */
    double* ret_mean;    /* [1] */
    double* ret_var;     /* [1] */
    double* ret_count2;  /* [2] */
    double* returns;     /* [N] discounted returns */
    double* scratch_obs; /* sdcgym_vecnorm_scratch_doubles(4M), zero-initialised once */
    double* scratch_ret; /* sdcgym_vecnorm_scratch_doubles(1), zero-initialised once */
    double* sums_obs;    /* [2*4M + 1] */
    double* sums_ret;    /* [3] */
    double* out_planes;  /* [4M][ld] normalised observation planes (output) */
    double* out_reward;  /* [N] normalised reward (output; the raw reward if !norm_reward) */
} sdcgym_vecnorm;
int sdcgym_pipe_step_vecnorm(sdcgym_pipe* pipe, const sdcgym_env_desc* desc, const sdcgym_state* st,
                             const sdcgym_step_io* dev, double* obs_dev, const sdcgym_host_io* host,
                             const sdcgym_vecnorm* vn, void* caller_stream);
/*
 * Result blocks: ONE contiguous buffer per side (device block, page-locked host block, same layout) holding everything a
 * `DummyVecEnv.step` returns for N envs, so that a whole step's results leave the GPU in a single transfer (or, for large
 * batches, in a few large chunked ones) and land where the host-side arrays already live - no pack kernel, no scatter:
 *     obs_u    [N][M] complex128   observation row 0 (u)          obs[i, 0, :]
 *     reward   [N] f64,  residual [N] f64,  lam [N][2] f64,  niter [N] i32,  flags [N] u8
 *     obs_r    [N][M] complex128   observation row 1 (residual)   obs[i, 1, :]
 * The reference observation (N, 2, M) complex128 is the strided view (strides 16M, obs_r - obs_u, 16 bytes) based at
 * obs_u.  `skip_u`: for sdc-v0 with auto-reset the returned u row is identically 1 (sdc_env.py:306-314: every step ends
 * the episode and the observation is the reset state), so the caller fills the host u rows ONCE and the step neither
 * exports nor transfers them (117 instead of 197 bytes per env at M = 5).  All offsets are multiples of 256 bytes.
 */
typedef struct sdcgym_block_layout {
    int64_t N;
    int32_t M, reserved;
    uint64_t obs_u, reward, residual, lam, niter, flags, obs_r, total; /* byte offsets; total = block size */
} sdcgym_block_layout;
int sdcgym_block_layout_init(int M, int64_t N, sdcgym_block_layout* out);

typedef struct sdcgym_block_io {
    unsigned char* dev_block;  /* device memory, layout.total bytes; the step writes its results here */
    unsigned char* host_block; /* page-locked host memory, layout.total bytes */
    double* action_dev;        /* device staging [N][A] ([N][A][2] complex) */
    const double* action_host; /* host actions, same shape (page-locked for asynchronous upload) */
    double* terminal_obs;      /* device planes [4M][ld] or NULL (terminal observations not kept) */
    int32_t skip_u;            /* bit 0: u rows are constant, neither exported nor transferred;
                                * bit 1: info arrays (niter, residual, lam: 28 of 117 bytes per env) stay in the device
                                *        block when the batch is large enough to be pipelined in chunks - the caller
                                *        copies [layout.residual, layout.flags) on demand (info dicts are read lazily) */
    int32_t chunks;            /* <= 0: chosen by the library from the batch size */
} sdcgym_block_io;
/* env.step with host actions in, host results out (see sdcgym_pipe_step); returns when the host block is filled.
 * `vn` may be NULL.  With `vn` (see sdcgym_pipe_step_vecnorm) the host block receives the NORMALISED observation rows
 * and reward; the device block keeps the raw reward, the observation rows of the device block are the normalised ones. */
int sdcgym_pipe_step_block(sdcgym_pipe* pipe, const sdcgym_env_desc* desc, const sdcgym_state* st,
                           const sdcgym_block_layout* layout, const sdcgym_block_io* bio, const sdcgym_vecnorm* vn,
                           void* caller_stream);

int sdcgym_host_alloc(size_t bytes, void** out); /* page-locked host memory */
int sdcgym_host_free(void* p);

/* sum of x[0..N) in fp64 with a fixed (N-independent, deterministic) reduction tree -> out[0].  `scratch` is
 * caller-owned device memory of sdcgym_sum_scratch_doubles() doubles (so concurrent calls on different streams
 * do not share state). */
int sdcgym_sum_scratch_doubles(void);
int sdcgym_sum_f64(int64_t N, const double* x, double* scratch, double* out, void* stream);

/* Measured-peak helper: runs a dependent-free DFMA chain kernel and returns its FLOP count; time it with
 * events on `stream`.  flops_out may be NULL. */
int sdcgym_fp64_peak_probe(int64_t iters, double* sink, double* flops_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDCGYM_H */
