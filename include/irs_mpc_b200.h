/* irs_mpc_b200 — C ABI of the B200-native iRS-MPC hot path.
 *
 * The reference (hjsuh94/irs_mpc) is pure Python and has no FFI of its own; these entry points
 * are what a ctypes binding placed behind the reference's Python call surface binds (see
 * INTEGRATION.md).  Each function cites the reference interface it replaces (paths relative to
 * the reference tree).
 *
 * Conventions
 *   - every pointer named in a signature is a DEVICE pointer unless it says "host";
 *   - matrices are dense row-major; state/input dims (n, m) are fixed by `system`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - calls enqueue work on `stream` and return without synchronising;
 *   - return value 0 = ok, non-zero = error, message via irs_last_error();
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef IRS_MPC_B200_H
#define IRS_MPC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define IRS_ABI_VERSION 4

/* system ids — the reference's four analytic DynamicalSystem subclasses
 * (examples/pendulum/pendulum_dynamics.py:8, examples/bicycle/bicycle_dynamics.py:8,
 *  examples/quadrotor/quadrotor_dynamics.py:15, examples/three_cart/three_cart_dynamics.py:8).
 * `params` (host, doubles): pendulum [h]; bicycle [h];
 *   quadrotor [h, mass, L, g, Ixx, Iyy, Izz, kF, kM]; three_cart [h, d].
 * IRS_MLP_2_1: learned dynamics of a 2-state / 1-input system, x+ = net([x, u]) — the reference's
 *   PendulumNN (examples/pendulum/pendulum_nn.py:19-33 network, :66-90 DynamicalSystem wrapper);
 *   params [h, handle] with `handle` from irs_mlp_register. */
enum { IRS_PENDULUM = 0, IRS_BICYCLE = 1, IRS_QUADROTOR = 2, IRS_THREE_CART = 3, IRS_MLP_2_1 = 4 };

/* Registers a network Linear(dim_x + dim_u, h1) ReLU Linear(h1, h2) ReLU Linear(h2, dim_x) (the architecture of
 * examples/pendulum/pendulum_nn.py:23-29; torch.nn.Linear layout: W [out, in] row-major, float32 HOST arrays)
 * on the current device and returns its handle; h1, h2 <= 128.  The network is evaluated in float32, as the
 * reference does (pendulum_nn.py:72-76: torch.Tensor inputs, float32 module).  irs_mlp_release frees it
 * (after synchronising with the device). */
int irs_mlp_register(int dim_x, int dim_u, int h1, int h2, const float* W1, const float* b1, const float* W2,
                     const float* b2, const float* W3, const float* b3, int* handle);
int irs_mlp_release(int handle);

/* smoothing flags */
enum {
  IRS_SAMPLES_BATCH_VARIANT = 1, /* samples use dynamics_batch semantics (irs_lqr_zero_order.py:51);
                                    only three_cart distinguishes (three_cart_dynamics.py:109-194) */
  IRS_PROJECT_ABSOLUTE = 2,      /* three_cart_zero_order.py:43: sampling returns projection(...) =
                                    absolute points (three_cart_dynamics.py:196-264), reproduced literally */
  IRS_PROJECT_DELTA = 4,         /* corrected variant: projected point minus nominal */
  IRS_ANTITHETIC = 8,            /* in-kernel Philox noise in antithetic pairs: sample 2q is xbar + z_q, sample
                                    2q+1 is xbar - z_q, one counter (and one Box-Muller draw) per pair.  The
                                    reference draws independent normals (e.g. pendulum_zero_order.py:38-43);
                                    each sample keeps the same marginal N(0, sigma^2), the even-order terms of
                                    f cancel in Z^T dF, and the fused kernel needs one operand row per pair.
                                    Ignored when deltas are replayed.  i0 must be even. */
  IRS_CENTERED = 16              /* three_cart: the regressors handed to the fit are ABSOLUTE points near the
                                    nominal (replayed output of the reference's projecting closure,
                                    three_cart_zero_order.py:43).  They are accumulated relative to (xbar, ubar)
                                    together with their first moments and shifted back in fp64 by
                                    irs_smooth_finalize(centered = 1); an fp32 Gram of the absolute points loses
                                    the sample spread once |xbar| >> sigma.  IRS_PROJECT_ABSOLUTE (in-kernel
                                    projection of in-kernel noise) implies it. */
};

int irs_abi_version(void);
const char* irs_last_error(void);

/* Selects where the zero-order kernel accumulates the Gram blocks [dx du]^T[dx du | dF]:
 * -1 auto (default: tcgen05 tensor cores for quadrotor and three_cart, CUDA cores otherwise), 0 CUDA cores
 * (packed FFMA2), 1 tcgen05 (bf16x2-split operands, fp32 accumulation in TMEM).  Both engines
 * implement irs_lqr/irs_lqr_zero_order.py:54-57 and are parity-tested against each other. */
int irs_set_gram_engine(int engine);

/* DynamicalSystem.dim_x / dim_u (irs_lqr/dynamical_system.py:8-10); nj = varying Jacobian scalars */
int irs_system_dims(int system, int* n, int* m, int* nj);

/* Number of fp32 accumulators per (nominal point, chunk): order 0 = zero-order Gram
 * d(d+1)/2 + d*n (three_cart: + d + n first moments of the centred accumulation, IRS_CENTERED),
 * order 1 = first-order nj. */
int irs_partial_width(int system, int order);

/* Chunking plan for P nominal points x N samples: C chunks of S samples each (S a multiple of 256).
 * chunk_samples = 0: default target (4096 samples); > 0: the caller's target — smaller chunks give more
 * work items per launch (launches that would not fill the GPU otherwise) at the price of more partial
 * blocks.  The plan depends on (N, chunk_samples) only, never on P. */
int irs_smooth_plan(int system, int order, int P, long long N, long long chunk_samples, int* C, long long* S);

/* IrsLqrZeroOrder.get_TV_matrices sampling + fit, accumulation stage
 * (irs_lqr/irs_lqr_zero_order.py:49-57): for each nominal point p and sample i
 *   (dx,du) = noise[p,i,:]                     if noise != NULL   (replay / parity mode)
 *           = sigma * Philox-normal(seed; i0+i, p0+p, iter, stream)   otherwise
 *   dF      = f(xbar+dx, ubar+du) - f(xbar, ubar)
 * and accumulates [dx du]^T [dx du | dF] into partials[P, C, irs_partial_width(system,0)].
 * x_nom [P,n] f64, u_nom [P,m] f64, sigma_host [n+m] f32 (HOST array, may be NULL in replay mode),
 * noise [P,N,n+m] f32 or NULL.  The Philox stream is Philox4x32-7 (see csrc/common.cuh). */
int irs_smooth_zero_order_accumulate(int system, const double* params_host, int nparams, int flags,
                                     const double* x_nom, const double* u_nom, int P, long long N,
                                     const float* sigma_host, const float* noise,
                                     unsigned long long seed, unsigned iter, unsigned stream_id,
                                     unsigned p0, unsigned long long i0,
                                     int C, long long S, float* partials, void* stream);

/* IrsLqrFirstOrder.get_TV_matrices sampling + Jacobian averaging, accumulation stage
 * (irs_lqr/irs_lqr_first_order.py:42-48; Jacobians of pendulum_dynamics.py:110-127,
 * bicycle_dynamics.py:115-132, quadrotor_dynamics.py:132-148).  partials [P, C, nj]. */
int irs_smooth_first_order_accumulate(int system, const double* params_host, int nparams, int flags,
                                      const double* x_nom, const double* u_nom, int P, long long N,
                                      const float* sigma_host, const float* noise,
                                      unsigned long long seed, unsigned iter, unsigned stream_id,
                                      unsigned p0, unsigned long long i0,
                                      int C, long long S, float* partials, void* stream);

/* Chunk reduction of the accumulation stage: partials [P,C,width] fp32 -> reduced [P,width] fp64,
 * fixed chunk order.  This is the block one rank contributes when the SAMPLE axis is sharded
 * across GPUs (the per-point blocks are then all-gathered and summed in rank order). */
int irs_smooth_reduce_chunks(int system, int order, const float* partials, int P, int C,
                             double* reduced, void* stream);

/* Fit / mean + affine offset (irs_lqr_zero_order.py:27-36,:59-62; irs_lqr_first_order.py:48-53).
 * Input is EITHER `partials` (fp32 [nranks][P,C,width], other NULL) OR `reduced` (fp64
 * [nranks][P,width]); the `nranks` buffers lie `rank_stride` elements apart (peer-mapped pointers
 * are fine) and are summed in rank order, then chunk order — deterministic.  Solves the normal
 * equations (order 0; identical to lstsq for full column rank) or divides by n_total (order 1);
 * centered != 0 (three_cart, accumulate flags IRS_PROJECT_ABSOLUTE / IRS_CENTERED): the blocks hold the
 * Gram of regressors relative to the nominal point plus their first moments, and the shift
 * Z^T Z = Z'^T Z' + s m'^T + m' s^T + N s s^T, Z^T dF = Z'^T dF + s g^T (s = (xbar, ubar)) is undone in fp64;
 * writes At [P,n,n], Bt [P,n,m], ct [P,n] (f64) and status [P] (0 ok, 1 rank deficient, 2 peer
 * exchange timed out — irs_smooth_finalize_peer only). */
int irs_smooth_finalize(int system, const double* params_host, int nparams, int order,
                        const double* x_nom, const double* u_nom, int P, int C,
                        const float* partials, const double* reduced, int nranks,
                        long long rank_stride, double n_total, int centered,
                        double* At, double* Bt, double* ct, int* status, void* stream);

/* irs_smooth_finalize for a SAMPLE-SHARDED run (one process per GPU), with the exchange of the per-point
 * fp64 blocks fused into the kernel over peer memory (NVLink / NVSwitch) — replaces reduce_chunks +
 * ncclAllGather + finalize of that path (the reference's only distributed reduction is the ZeroMQ
 * task farm of irs_lqr/irs_lqr_quasistatic.py:228-273).  The block of point p reduces this rank's
 * partials [P,C,width] of p in chunk order, stores the fp64 values into slot (epoch & 1, rank) of EVERY
 * rank's exchange buffer (peer_bufs_dev: device array of `world` peer-mapped base pointers, each
 * buffer [2][world][slot_stride] doubles), raises flag (rank, p) on every rank to `epoch`
 * (peer_flags_dev: device array of `world` peer-mapped int[world][flag_stride] arrays, zero before the
 * first call), waits for the `world` flags of p, sums the blocks in rank order and fits.  The epoch
 * lives in *epoch_dev (zero-initialised local device word, advanced by the kernel itself, so the call
 * is CUDA-graph replayable); done_counter: zero-initialised local device word.  A peer that does
 * not deliver within timeout_s sets status[p] = 2 instead of hanging the GPU.  Every rank must
 * issue the same sequence of calls on the same exchange; P may change from call to call.  All P
 * blocks must be co-resident: P <= irs_smooth_finalize_peer_capacity (error otherwise). */
int irs_smooth_finalize_peer(int system, const double* params_host, int nparams, int order,
                             const double* x_nom, const double* u_nom, int P, int C, const float* partials,
                             const void* peer_bufs_dev, const void* peer_flags_dev, int* epoch_dev,
                             unsigned int* done_counter, long long slot_stride, int flag_stride,
                             int rank, int world, double timeout_s, double n_total, int centered,
                             double* At, double* Bt, double* ct, int* status, void* stream);
int irs_smooth_finalize_peer_capacity(int system, int order, int* max_points);

/* irs_smooth_finalize for a TIMESTEP-SHARDED run (one process per GPU; BASELINE north star: "the T x N
 * sample rollouts shard along the time axis, with an all-gather of the small per-step (A_t, B_t, c_t)
 * blocks"), with that all-gather fused into the kernel over peer memory.  This rank owns the global
 * points p0 .. p0 + P - 1 of P_total (x_nom, u_nom, partials: its local slice; P = 0 allowed).  The block of
 * a point writes its result into EVERY rank's output buffer (peer_out_bufs_dev: device array of `world`
 * peer-mapped base pointers, each buffer [2 parities][At: P_total n n | Bt: P_total n m | ct: P_total n |
 * status: P_total] doubles, out_stride doubles per parity) and raises flag [point] on every rank
 * (peer_flags_dev: `world` peer-mapped int[P_total] arrays, zero before the first call); the last block
 * waits for all P_total flags, so on completion the full linearization of step `epoch` lies in the local
 * buffer at parity (epoch & 1).  epoch_dev / done_counter / timeout_s as for irs_smooth_finalize_peer (a
 * missing point gets status 2).  ct_scratch: P*n doubles of local scratch. */
int irs_smooth_finalize_gather(int system, const double* params_host, int nparams, int order,
                               const double* x_nom, const double* u_nom, int P, int C, const float* partials,
                               const void* peer_out_bufs_dev, const void* peer_flags_dev, int* epoch_dev,
                               unsigned int* done_counter, long long out_stride, int p0, int P_total,
                               int rank, int world, double timeout_s, double n_total, int centered,
                               double* ct_scratch, void* stream);

/* IrsLqrExact.get_TV_matrices (irs_lqr/irs_lqr_exact.py:15-31), all fp64: [A|B] = jacobian_xu at
 * the nominal points, c = f(xbar,ubar) - A xbar - B ubar.  x_nom [P,n], u_nom [P,m]. */
int irs_exact_linearize(int system, const double* params_host, int nparams,
                        const double* x_nom, const double* u_nom, int P,
                        double* At, double* Bt, double* ct, void* stream);

/* The Philox words / deltas exactly as the fused kernels draw them (bookkeeping tests).
 * words [P,N,ceil(d/4),4] u32 or NULL; deltas [P,N,d] f32 or NULL; sigma_host: HOST array [d];
 * antithetic != 0: the IRS_ANTITHETIC stream (samples 2q, 2q+1 share the words of counter q). */
int irs_philox_dump(int P, long long N, int d, const float* sigma_host, unsigned long long seed,
                    unsigned iter, unsigned stream_id, unsigned p0, unsigned long long i0, int antithetic,
                    unsigned* words, float* deltas, void* stream);

/* DynamicalSystem.dynamics_batch (irs_lqr/dynamical_system.py:24-37). batch_variant != 0 selects
 * the reference's dynamics_batch semantics, 0 the scalar dynamics semantics (three_cart differs).
 * x [B,n], u [B,m], out [B,n]; *_f32 in float, *_f64 in double. */
int irs_dynamics_batch_f32(int system, const double* params_host, int nparams, int batch_variant,
                           const float* x, const float* u, float* out, long long B, void* stream);
int irs_dynamics_batch_f64(int system, const double* params_host, int nparams, int batch_variant,
                           const double* x, const double* u, double* out, long long B, void* stream);

/* DynamicalSystem.jacobian_xu_batch (irs_lqr/dynamical_system.py:53-66): J [B,n,n+m]. */
int irs_jacobian_xu_batch_f32(int system, const double* params_host, int nparams,
                              const float* x, const float* u, float* J, long long B, void* stream);
int irs_jacobian_xu_batch_f64(int system, const double* params_host, int nparams,
                              const double* x, const double* u, double* J, long long B, void* stream);

/* ThreeCartDynamics.projection (examples/three_cart/three_cart_dynamics.py:196-264) applied to
 * absolute states x [B,n] in place (non-penetration projection, half-depth push-out).
 * A no-op for systems without a projection. */
int irs_project_batch_f64(int system, const double* params_host, int nparams, double* x,
                          long long B, void* stream);

/* solve_tvlqr backward pass (irs_lqr/tv_lqr.py:30-145, inactive bounds): affine Riccati recursion
 * for I independent instances.  At [I,T,n,n], Bt [I,T,n,m], ct [I,T,n], Q/Qd [n,n], R [m,m]
 * (full R; the QP's 1/2 u'Ru of tv_lqr.py:110 is applied inside), xd [I,T+1,n] (xd_stride =
 * (T+1)*n) or one shared trajectory (xd_stride = 0).  The weights need not be symmetric: the cost
 * only sees their symmetric parts, and those are what the recursion uses.  Outputs K [I,T,m,n], k [I,T,m],
 * status [I] (1 = an H not SPD, or a K_t / k_t not finite -> the caller raises the reference's ValueError,
 * tv_lqr.py:139). */
int irs_tvlqr_riccati(int n, int m, const double* At, const double* Bt, const double* ct,
                      const double* Q, const double* Qd, const double* R,
                      const double* xd, long long xd_stride, int I, int T,
                      double* K, double* k, int* status, void* stream);

/* The same recursion restricted to the steps t_hi-1 .. t_lo (even n, m only).  A segment that does
 * not start at T reads (P, p) of step t_hi from carry [I, n*n + n]; one that does not end at 0 writes
 * (P, p) of step t_lo there.  Chaining the segments [t1,T), [t2,t1), ..., [0,tk) on one stream
 * reproduces irs_tvlqr_riccati bit for bit; IrsLqr.local_descent uses it to solve the late timesteps
 * while the early ones are still being linearized on another stream.  status: the segment from T
 * sets it, later segments can only raise it. */
int irs_tvlqr_riccati_segment(int n, int m, const double* At, const double* Bt, const double* ct,
                              const double* Q, const double* Qd, const double* R,
                              const double* xd, long long xd_stride, int I, int T, int t_lo, int t_hi,
                              double* carry, double* K, double* k, int* status, void* stream);

/* Box-constrained solve_tvlqr / local_descent (irs_lqr/tv_lqr.py:113-118,:132-134 absolute bounds;
 * irs_lqr/irs_lqr.py:160-184 re-solve at every timestep).  Three pieces:
 *  - irs_tvlqr_riccati_ex: irs_tvlqr_riccati that also returns Hinv [I,T,m,m] = (R/2 + B'PB)^-1 and
 *    P [I,T+1,n,n]; called with the penalty-augmented weights (Q + diag(dx)/2, Qd + diag(dx)/2,
 *    R + diag(du)) it yields the matrix part of the ADMM's equality-constrained step;
 *  - irs_tvlqr_plan_check: for every start time t0 rolls the affine model forward from the actual
 *    state x_trj[t0] under the unconstrained gains (K, k) (scratch: I*T*(n+m)*(n+1) doubles of device
 *    workspace for the closed-loop rows) and sets violated[i] = 1 if any planned
 *    state (t0 < t <= T) or input leaves [lo - tol, hi + tol].  violated == 0 means every QP of the
 *    reference's loop had inactive bounds, i.e. the one-pass Riccati descent is its exact result;
 *    irs_tvlqr_plan_rows fills `scratch` (it needs the gains only, not the trajectory: a caller can run
 *    it on a second stream beside the closed-loop rollout) and plan_check is then called with
 *    rows_ready = 1; rows_ready = 0 makes plan_check compute the rows itself;
 *  - irs_tvlqr_box_solve: ADMM on the box split.  mpc = 1: the reference's closed loop (QP over the
 *    remaining horizon at every t0 from the actual state, first input applied to the TRUE dynamics of
 *    `system`); mpc = 0: one QP from x0 (solve_tvlqr), x_trj/u_trj receive the plan.  Bounds are per
 *    coordinate: constant in time (xlo/xhi [n], ulo/uhi [m], strides 0) or one box per timestep
 *    (xlo/xhi [T+1,n] with xbox_stride = n, ulo/uhi [T,m] with ubox_stride = m; tv_lqr.py:113-116,
 *    :132-134 index their bounds by t; the box of x_0 is not used — x_0 is fixed); dx [n], du [m]
 *    are the ADMM penalties;
 *    K0 [I,T,m,n], k0 [I,T,m] (optional, mpc = 1): the UNCONSTRAINED gains; a start time whose
 *    unconstrained plan stays inside [lo - tol, hi + tol] skips its QP (its bounds are inactive, the
 *    minimiser is K0 x + k0).  A solve stops when max |y - z| and the change of z are both
 *    <= eps max(1, |z|) (units of z: invariant under a scaling of the weights).  status[i] = 1 if a
 *    solve did not reach eps within max_iter (-> the reference's ValueError).
 *    Algorithm and its check against a dense QP solve: oracle/box_tvlqr.py. */
int irs_tvlqr_riccati_ex(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* Q, const double* Qd, const double* R,
                         const double* xd, long long xd_stride, int I, int T,
                         double* K, double* k, int* status, double* Hinv_out, double* P_out, void* stream);
int irs_tvlqr_plan_rows(int n, int m, const double* At, const double* Bt, const double* ct,
                        const double* K, const double* k, int I, int T, double* scratch, void* stream);
int irs_tvlqr_plan_check(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* K, const double* k, const double* x_trj,
                         const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                         double tol, int I, int T, int rows_ready, int* violated, double* scratch, void* stream);
int irs_tvlqr_box_solve(int system, const double* params_host, int nparams, int mpc,
                        const double* At, const double* Bt, const double* ct,
                        const double* K, const double* Hinv, const double* P,
                        const double* Q, const double* Qd, const double* R,
                        const double* xd, long long xd_stride, const double* dx, const double* du,
                        const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                        long long xbox_stride, long long ubox_stride,
                        const double* x0, const double* K0, const double* k0, double tol,
                        double alpha, double eps, int max_iter, int I, int T,
                        double* x_trj, double* u_trj, double* cost, int* status, int* iters, void* stream);

/* (x*, u*) of solve_tvlqr: rollout of the affine model under u = K x + k (tv_lqr.py:142-145).
 * x0 [I,n]; xs [I,T+1,n]; us [I,T,m]. */
int irs_tvlqr_linear_rollout(int n, int m, const double* At, const double* Bt, const double* ct,
                             const double* K, const double* k, const double* x0, int I, int T,
                             double* xs, double* us, void* stream);

/* solve_tvlqr for any state and input dimension within the limits, not only those of the built-in
 * systems (irs_tvlqr_riccati and the box solve are instantiated for those alone).  Same problem, same
 * array layouts and the same conventions as the entries above; n and m are run-time arguments and every
 * pair within the limits is accepted, the built-in pairs included.  Arguments are checked on the host
 * before any launch (null pointers, n and m out of range, I < 1, T < 1, box strides, the box QP's horizon).
 *  - irs_tvlqr_any_limits: the largest n and m (32 each).  Host only.
 *  - irs_tvlqr_riccati_any: irs_tvlqr_riccati / irs_tvlqr_riccati_ex (Hinv_out [I,T,m,m] and P_out
 *    [I,T+1,n,n] may each be null).  H_t is factored by a Cholesky decomposition; status[i] = 1 if a
 *    pivot is not > 0, a K_t or k_t is not finite, or the final P holds a NaN.
 *  - irs_tvlqr_linear_rollout_any: irs_tvlqr_linear_rollout.
 *  - irs_tvlqr_box_qp_any: irs_tvlqr_box_solve with mpc = 0 (one QP from x0; no cost output).  K, Hinv,
 *    P are irs_tvlqr_riccati_any's outputs for the penalty-augmented weights (Q + diag(dx)/2,
 *    Qd + diag(dx)/2, R + diag(du)); Q, Qd, R are the problem's own weights (R is not read by the ADMM).
 *    The ADMM state lives in shared memory: 8 (5 n T + 4 m T + 7 n + m) bytes must fit in 200 KiB
 *    (T <= 88 at n = m = 32), otherwise the call fails before launch. */
int irs_tvlqr_any_limits(int* max_n, int* max_m);
int irs_tvlqr_riccati_any(int n, int m, const double* At, const double* Bt, const double* ct,
                          const double* Q, const double* Qd, const double* R,
                          const double* xd, long long xd_stride, int I, int T,
                          double* K, double* k, int* status, double* Hinv_out, double* P_out, void* stream);
int irs_tvlqr_linear_rollout_any(int n, int m, const double* At, const double* Bt, const double* ct,
                                 const double* K, const double* k, const double* x0, int I, int T,
                                 double* xs, double* us, void* stream);
int irs_tvlqr_box_qp_any(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* K, const double* Hinv, const double* P,
                         const double* Q, const double* Qd, const double* R,
                         const double* xd, long long xd_stride, const double* dx, const double* du,
                         const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                         long long xbox_stride, long long ubox_stride, const double* x0,
                         double alpha, double eps, int max_iter, int I, int T,
                         double* x_trj, double* u_trj, int* status, int* iters, void* stream);

/* IrsLqr.local_descent forward pass (irs_lqr/irs_lqr.py:169-184): u_t = K_t x_t + k_t on the TRUE
 * dynamics, plus IrsLqr.evaluate_cost (irs_lqr.py:121-137, terminal term uses Q).
 * x0 [I,n]; x_trj [I,T+1,n]; u_trj [I,T,m]; cost [I]. */
int irs_rollout_closed_loop(int system, const double* params_host, int nparams,
                            const double* K, const double* k, const double* x0,
                            const double* xd, long long xd_stride, const double* Q, const double* R,
                            int I, int T, double* x_trj, double* u_trj, double* cost, void* stream);

/* IrsLqr.rollout + evaluate_cost (irs_lqr/irs_lqr.py:105-137) for given inputs u_in [I,T,m]. */
int irs_rollout_open_loop(int system, const double* params_host, int nparams,
                          const double* u_in, const double* x0,
                          const double* xd, long long xd_stride, const double* Q, const double* R,
                          int I, int T, double* x_trj, double* cost, void* stream);

/* CrossEntropyMethod.local_descent, steps 3-4 (irs_lqr/cem.py:173-182): marks the n_elite cheapest of the
 * B candidates (elite [B] int, ties by index, NaN last) and refits mean [T,m] / std [T,m] (population
 * standard deviation) of the candidate input trajectories u_candidates [B,T,m] over them.  cost [B] is the
 * output of irs_rollout_open_loop. */
int irs_cem_refit(const double* cost, const double* u_candidates, int B, int T, int m, int n_elite,
                  int* elite, double* mean, double* std_out, void* stream);

/* IrsLqrZeroOrder.compute_least_squares (irs_lqr/irs_lqr_zero_order.py:27-36) on explicit samples: the
 * packed fp64 Gram block [Z^T Z | Z^T F] of Z = dxdu [N, n+m], F = deltaf [N, n] in the layout
 * irs_smooth_finalize reads as `reduced` (P = 1, nranks = 1). */
int irs_gram_block_f64(int n, int m, const double* Z, const double* F, long long N, double* out, void* stream);

/* Measurement aid (no reference counterpart): dependent-chain FP32 FMA microbenchmark used by
 * bench.py as the measured FP32 roofline denominator.  out: device scratch of >= 148*8*256 floats;
 * *flops_host receives the flop count of one launch. */
int irs_fp32_fma_peak(int iters, float* out, long long out_len, double* flops_host, void* stream);

/* IrsLqr.evaluate_cost (irs_lqr/irs_lqr.py:121-137) for given trajectories x_trj [I,T+1,n],
 * u_trj [I,T,m]: sum_t e'Qe + u'Ru + terminal e'Qe (Q, not Qd, :135-136).  cost [I]. */
int irs_evaluate_cost(int n, int m, const double* x_trj, const double* u_trj,
                      const double* xd, long long xd_stride, const double* Q, const double* R,
                      int I, int T, double* cost, void* stream);

/* CUDA-graph replay of a fixed call sequence (no reference counterpart; the reference's per-iteration
 * Python loop, irs_lqr/irs_lqr.py:148-186 and :188-218, re-issues the same calls every iteration).
 * Everything submitted to `stream` between irs_graph_begin and irs_graph_end — entry points of this
 * library and cudaMemcpyAsync alike — is captured into one graph instead of being executed.
 * irs_graph_update_smoothing rewrites seed / iter / stream_id / sigma (HOST array [n+m], NULL = keep)
 * of the captured accumulate kernel before a replay; pointers and shapes are fixed at capture. */
int irs_graph_begin(void* stream);
int irs_graph_end(void* stream, void** graph_out);
int irs_graph_update_smoothing(void* graph, const float* sigma_host, unsigned long long seed,
                               unsigned iter, unsigned stream_id);
int irs_graph_launch(void* graph, void* stream);
int irs_graph_destroy(void* graph);

#ifdef __cplusplus
}
#endif
#endif /* IRS_MPC_B200_H */
