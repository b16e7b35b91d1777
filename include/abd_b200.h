/* abd_b200.h -- C ABI of libabd_b200.so: the B200 (sm_100a) implementation of the abdpymc
 * inference hot path (joint log-density + gradient of the antibody-dynamics model and the
 * Gibbs sweep over its binary infection / waner indicators).
 *
 * The reference (davipatti/abdpymc, pure Python) has no FFI: its hot path is the PyTensor graph
 * built by abd.model() (abd.py:396-442) and evaluated by PyMC's two step methods inside
 * pm.sample() (abd.py:922).  Each entry point below replaces one evaluation of that graph; the
 * "replaces" note names the reference code whose result it reproduces.  INTEGRATION.md shows
 * the ctypes / PyTensor-Op / PyMC-step binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - Every function returns ABD_OK (0) or a negative ABD_ERR_* code; abd_last_error() returns a
 *    thread-local message for the last failure.  No exception crosses the boundary.
 *  - Matrices over (gap, individual) are row-major (G, N): element (t, n) at [t*N + n], the
 *    layout of the reference graph (abd.py:413-418, dims ("gap","ind") abd.py:18).  A batch of
 *    C chains is the outermost axis: i_raw[c][t][n], waner[c][n], theta[c][k].
 *  - Binary variables are int8 0/1 (any non-zero byte counts as 1).
 *  - theta13 (constrained, the 13 scalars that reach the likelihood), in this order:
 *      ab_n_perm, ab_n_temp, ab_n_rho, ab_n_init, ab_s_perm, ab_s_rho, ab_s_init,
 *      it_n_b, it_n_d, it_n_sigma, it_s_b, it_s_d, it_s_sigma
 *  - q17 (PyMC's unconstrained value variables, declaration order abd.py:424,329-340,367-388,
 *    464-467):  p_logodds__, ab_n_perm_log__, ab_n_temp_log__, ab_n_rho_logodds__, ab_n_init,
 *      ab_s_perm_log__, ab_s_rho_logodds__, ab_s_p_waner_logodds__, ab_s_tempinf_log__,
 *      ab_s_tempvac_log__, ab_s_init, it_n_b, it_n_d, it_n_sigma_log__, it_s_b, it_s_d,
 *      it_s_sigma_log__
 *  - Host-pointer functions copy inputs to the device, run, copy results back and return when
 *    the results are in the caller's buffers.  The `_dev` variants take device pointers and a
 *    cudaStream_t (as void*), enqueue work and return immediately.
 *  - i_raw / waner may be NULL in the host-pointer compute calls: the chain state already
 *    resident on the device (abd_upload_state, or left by the last abd_gibbs_sweep) is used.
 *  - Ownership: the caller owns every buffer it passes; the library owns all device memory it
 *    allocates (uploaded once in abd_create).  A handle is not re-entrant: serialise calls on
 *    it.  The CUDA context is created lazily in the calling process (fork-safe as long as the
 *    parent has not called into the library).
 *  - There is NO CPU fallback: without a CUDA device every call fails with ABD_ERR_CUDA.
 */
#ifndef ABD_B200_H
#define ABD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABD_OK 0
#define ABD_ERR_INVALID (-1) /* bad argument (shape, split, NULL pointer ...) */
#define ABD_ERR_CUDA (-2)    /* CUDA runtime error / no device */
#define ABD_ERR_ALLOC (-3)

#define ABD_N_THETA 13
#define ABD_N_Q 17
#define ABD_N_SUMS 16
#define ABD_MAX_GAPS 127 /* gap masks of 32, 64 or 128 bits; the top bit holds the waner bit */

/* abd_gibbs_sweep modes */
#define ABD_GIBBS_METROPOLIS 0 /* PyMC BinaryGibbsMetropolis semantics: propose the flip w.p.
                                  transit_p, accept w.p. min(1, exp(delta)); random order   */
#define ABD_GIBBS_HEATBATH 1   /* draw every bit from its exact full conditional            */
#define ABD_GIBBS_BLOCKED 2    /* per time chunk, redraw the chunk's raw bits TOGETHER from their
                                  exact full conditional (the position of the chunk's first raw 1
                                  is a categorical over len + 1 options; bits behind it, and all
                                  bits of a chunk overridden by PCR+, only have their Bernoulli(p)
                                  prior), then ab_s_waner as HEATBATH.  Same stationary
                                  distribution as the two single-site modes, far fewer sweeps to
                                  move an infection in time.  Needs time chunks (splits) and
                                  G <= 31; otherwise it runs as HEATBATH.  transit_p is ignored;
                                  stats = {block draws, blocks whose first 1 / waner changed}   */

typedef struct abd_handle abd_handle;

/* The cohort, as TiterData holds it (abd.py:46-126), flattened.  Per antigen a in {s, n}:
 * x = df_a["log_dilution"], od = df_a["od"] (abd.py:462,468), gap = idx_gap, ind = idx_ind
 * (abd.py:35-36).  Rows may be in any order.  pcrpos / vacs are (G, N) 0/1 bytes, i.e.
 * data.pcrpos.T / data.vacs.T (abd.py:413-418); pcrpos == NULL means ignore_pcrpos=True.
 * splits: 0, 1 or 2 ascending gap indexes (abd.py:604-622, 865-882).                       */
typedef struct abd_cohort {
  int32_t n_gaps, n_inds;
  int32_t n_splits;
  int32_t splits[2];
  const uint8_t* pcrpos;
  const uint8_t* vacs;
  int64_t n_rows_s;
  const double* x_s;
  const double* od_s;
  const int32_t* gap_s;
  const int32_t* ind_s;
  int64_t n_rows_n;
  const double* x_n;
  const double* od_n;
  const int32_t* gap_n;
  const int32_t* ind_n;
  /* Totals over ALL shards when individuals are sharded across GPUs (0 = this shard is the
   * whole cohort).  Only the joint-logp finalisation uses them.                              */
  int64_t total_inds, total_rows_s, total_rows_n;
  /* Global index of this shard's first individual (0 if not sharded): keeps the Gibbs RNG
   * stream of an individual independent of how the cohort is sharded.                       */
  int64_t ind_offset;
} abd_cohort;

const char* abd_last_error(void);
int abd_version(void);

/* Builds the device-resident cohort on CUDA device `device`.  Replaces the data side of
 * abd.model(): as_tensor(data.vacs.T), pcrpos (abd.py:413-418), make_time_chunks
 * (abd.py:865-882), the gather indices (abd.py:343,393) and check_splits (abd.py:604-622).
 * Limits: 1 <= n_gaps <= ABD_MAX_GAPS, n_inds < 2^26 (< 2^25 when n_gaps > 63).  Layout on the device: per
 * individual, the PCR+ and vaccination months as one bit mask over gaps of 32 bits (n_gaps <= 31), 64 bits
 * (<= 63) or 128 bits (<= 127); the packed resident state (abd_state_dev) holds two such masks per chain and
 * individual (8, 16 or 32 bytes).  The environment variable ABD_B200_MASK_BITS=128 selects the 128-bit layout
 * for any n_gaps (tests and measurements: same results, other kernels).                                    */
int abd_create(abd_handle** out, const abd_cohort* cohort, int device);
int abd_destroy(abd_handle* h);

/* The preprocessed cohort as ONE binary file (the device upload format): everything abd_create derives
 * from the cohort -- bit masks, per-antigen CSR row / cell tables sorted by (individual, gap), packed
 * row -> cell / dilution words, the Gibbs work order, the time chunks -- so that a later process skips
 * what TiterData.from_disk + abd.model cost on a large cohort (pd.read_csv of df.csv and np.loadtxt of
 * vacs.txt / pcrpos.txt, abd.py:171-202, then the sorts of abd_create).  abd_create_from_cache = read +
 * upload.  The file is tied to the splits / ignore_pcrpos the handle was built with (abd_cohort_info
 * tells which) and to this library version.  Replaces: TiterData.to_disk / from_disk (abd.py:149-202) as
 * the way a cohort reaches the sampler.                                                          */
int abd_save_cache(abd_handle* h, const char* path);
int abd_create_from_cache(abd_handle** out, const char* path, int device);
/* What the handle was built with: number of splits (0-2), their gap indexes, whether PCR+ data is used. */
int abd_cohort_info(const abd_handle* h, int32_t* n_splits, int32_t* splits, int32_t* has_pcrpos);

/* Sizes and algorithmic-byte accounting (SURVEY.md section 8d).  Any pointer may be NULL.   */
int abd_sizes(const abd_handle* h, int32_t* n_gaps, int32_t* n_inds, int64_t* n_rows_s,
              int64_t* n_rows_n);
int64_t abd_algorithmic_bytes_logp(const abd_handle* h, int n_chains);
int64_t abd_algorithmic_bytes_gibbs(const abd_handle* h, int n_chains);
/* Kernels launched by this handle so far (for bench.py's gpu_launches).                      */
int64_t abd_launch_count(const abd_handle* h);

/* Chain state resident on the device: i_raw[C][G][N], waner[C][N].                          */
int abd_upload_state(abd_handle* h, int n_chains, const int8_t* i_raw, const int8_t* waner);
int abd_download_state(abd_handle* h, int n_chains, int8_t* i_raw, int8_t* waner);

/* Data log-likelihood and its gradient w.r.t. the 13 constrained parameters, for C chains.
 * Replaces: the value and gradient of it_n_lik + it_s_lik (abd.py:445-469) as a function of
 * the RVs of model_n_response / model_s_response (abd.py:309-393) given i_raw, ab_s_waner --
 * i.e. constrain_infections (abd.py:640-667), perm_response (:296-306),
 * _temp_response_scalar_rho / _vector_rho (:242-274), the gather mu[idx_gap, idx_ind]
 * (:343,393) and logistic (:556-557).
 * out_counts[c] = { sum(i_raw[c]), sum(waner[c]) } (for the Bernoulli terms abd.py:373,427);
 * out_grad / out_counts may be NULL.                                                        */
int abd_loglik_grad(abd_handle* h, int n_chains, const double* theta13, const int8_t* i_raw,
                    const int8_t* waner, double* out_loglik, double* out_grad,
                    int64_t* out_counts);

/* Joint model log-density in PyMC's unconstrained space and d logp / d q17: what
 * model.logp_dlogp_function() hands NUTS on every leapfrog (abd.py:921-922).  Adds to
 * abd_loglik_grad the 17 priors (abd.py:329-340,367-388,424,464-467), the log / logodds
 * transforms with their Jacobians, and the Bernoulli terms of i_raw and ab_s_waner.          */
int abd_logp_dlogp(abd_handle* h, int n_chains, const double* q17, const int8_t* i_raw,
                   const int8_t* waner, double* out_logp, double* out_dlogp);
/* (Both host-pointer calls above return as soon as their results have arrived: the kernel writes them
 * straight into pinned host memory and the library watches them arrive instead of waiting for the end
 * of the stream -- for <= 64 chains, falling back to cudaStreamSynchronize after 150 us; the handle's
 * stream may still be draining the launch's last CTAs, which later calls on the handle are ordered
 * behind.)                                                                                           */

/* Conditional log-odds of every binary variable given all others (test hook; what "Gibbs
 * parity" means, SURVEY.md section 8a):  out_i[c][t][n] = logp(i_raw[t,n]=1 | rest) -
 * logp(i_raw[t,n]=0 | rest), out_w[c][n] likewise for ab_s_waner[n].  p, p_w: per-chain
 * constrained Bernoulli probabilities ("p", "ab_s_p_waner").                                */
int abd_cond_logodds(abd_handle* h, int n_chains, const double* theta13, const double* p,
                     const double* p_w, const int8_t* i_raw, const int8_t* waner,
                     double* out_i, double* out_w);

/* One sweep over all G*N + N binary variables of each chain.  Replaces one
 * BinaryGibbsMetropolis.astep (PyMC; assigned to i_raw and ab_s_waner by pm.sample,
 * abd.py:922).  Individuals are updated in parallel (they are conditionally independent given
 * theta, p, p_w); within an individual its G+1 bits are visited in a uniformly random order
 * drawn from a counter-based Philox4x32-10 stream keyed by (seed; sweep_idx, chain, individual).
 * i_raw / waner: in/out host buffers, or NULL to update the resident state only.
 * out_stats[c] = { proposals, accepted flips } (may be NULL).                                */
int abd_gibbs_sweep(abd_handle* h, int n_chains, const double* theta13, const double* p,
                    const double* p_w, int8_t* i_raw, int8_t* waner, uint64_t seed,
                    uint64_t sweep_idx, int mode, double transit_p, int64_t* out_stats);

/* The three Deterministics PyMC records per draw: "i" (abd.py:649,667), "ab_n_mu" (:341),
 * "ab_s_mu" (:389-391), each (C, G, N).  Any output may be NULL.                            */
int abd_deterministics(abd_handle* h, int n_chains, const double* theta13, const int8_t* i_raw,
                       const int8_t* waner, int8_t* out_i, double* out_mu_n, double* out_mu_s);

/* Pointwise log-likelihood of every OD row: out_s[c][r] / out_n[c][r] = the Normal log-density of row r of the
 * S / N antigen, in the order the rows were passed to abd_create -- what PyMC stores in the InferenceData's
 * log_likelihood group for the observed nodes it_s_lik / it_n_lik (abd.py:459-469; az.loo / az.waic read it).
 * Either output may be NULL.  abd_loglik_rows_dev: device pointers.                                      */
int abd_loglik_rows(abd_handle* h, int n_chains, const double* theta13, const int8_t* i_raw,
                    const int8_t* waner, double* out_s, double* out_n);
int abd_loglik_rows_dev(abd_handle* h, int n_chains, const double* theta13, const int8_t* i_raw,
                        const int8_t* waner, double* out_s, double* out_n, void* stream);

/* ---------------------------------------------------------------------------------------
 * Device-pointer variants: every pointer is a device pointer, `stream` is a cudaStream_t.
 * Work is enqueued on `stream`; nothing is synchronised.
 * ------------------------------------------------------------------------------------- */

/* Raw per-chain sums of this shard's individuals: sums[c][ABD_N_SUMS] =
 *   { S0,S1,S2,Qinit,Qperm,Qtemp,Qrho (N antigen), S0,S1,S2,Qinit,Qperm,Qrho (S antigen),
 *     sum(i_raw), sum(waner), 0 }  -- every entry is additive over shards, so individual-
 * sharded ranks all-reduce this (C x 16 doubles) and then call abd_finalize_*_dev.
 * theta_is_q17 != 0: `theta` holds q17 (C x 17) and is back-transformed on the device.       */
int abd_sums_dev(abd_handle* h, int n_chains, const double* theta, int theta_is_q17,
                 const int8_t* i_raw, const int8_t* waner, double* sums, void* stream);
int abd_finalize_loglik_dev(abd_handle* h, int n_chains, const double* theta13,
                            const double* sums, double* out_loglik, double* out_grad,
                            void* stream);
int abd_finalize_logp_dev(abd_handle* h, int n_chains, const double* q17, const double* sums,
                          double* out_logp, double* out_dlogp, void* stream);
/* Single-launch fused versions (sums + ordered cross-tile reduction + finalisation).        */
int abd_loglik_grad_dev(abd_handle* h, int n_chains, const double* theta13,
                        const int8_t* i_raw, const int8_t* waner, double* out_loglik,
                        double* out_grad, void* stream);
int abd_logp_dlogp_dev(abd_handle* h, int n_chains, const double* q17, const int8_t* i_raw,
                       const int8_t* waner, double* out_logp, double* out_dlogp, void* stream);
/* stats: device int64 [C][2] accumulated with atomics (caller zeroes), or NULL.  theta_is_q17:
 * `theta` holds q17 and p / p_w are taken from it (p, p_w arguments ignored).                */
int abd_gibbs_sweep_dev(abd_handle* h, int n_chains, const double* theta, int theta_is_q17,
                        const double* p, const double* p_w, int8_t* i_raw, int8_t* waner,
                        uint64_t seed, uint64_t sweep_idx, int mode, double transit_p,
                        unsigned long long* stats, void* stream);
int abd_deterministics_dev(abd_handle* h, int n_chains, const double* theta13,
                           const int8_t* i_raw, const int8_t* waner, int8_t* out_i,
                           double* out_mu_n, double* out_mu_s, void* stream);
/* Streaming posterior summaries: ADD the sum over the chains of i, ab_n_mu, ab_s_mu (each (G, N),
 * float64, gap-major like the Deterministics' dims ("gap", "ind"), abd.py:341,389-391,649,667) to
 * the caller's running totals; any of the three may be NULL.  Divide by chains x recorded draws for
 * the posterior means survival.py:68-69 / timelines.py:274 read.  theta_is_q17 as above.      */
int abd_deterministics_accum_dev(abd_handle* h, int n_chains, const double* theta, int theta_is_q17,
                                 const int8_t* i_raw, const int8_t* waner, double* sum_i,
                                 double* sum_mu_n, double* sum_mu_s, void* stream);
/* n_steps leapfrog steps of Hamiltonian dynamics over q17 for C chains with the binary state
 * fixed, in ONE persistent launch (what a NUTS / HMC trajectory of pm.sample, abd.py:922, costs
 * n_steps calls of logp_dlogp_function for).  Per step: p += eps/2 grad; q += eps inv_mass p;
 * (logp, grad) = joint logp + gradient at q; p += eps/2 grad.  q17, p17, grad17 (C x 17, in/out;
 * grad17 holds the gradient at q17 on entry), logp (C, out), eps (C), inv_mass (17 x 17 row-major,
 * symmetric).  The grid must be resident at once: C x tiles <= SMs x CTAs/SM, otherwise
 * ABD_ERR_INVALID (use abd_logp_dlogp_dev per step).  abd_leapfrog_status: synchronous check that
 * no CTA timed out in the last trajectory.                                                    */
int abd_leapfrog_dev(abd_handle* h, int n_chains, int n_steps, double* q17, double* p17,
                     double* grad17, double* logp, const double* eps, const double* inv_mass,
                     const int8_t* i_raw, const int8_t* waner, void* stream);
int abd_leapfrog_status(abd_handle* h, int n_chains);

/* The two ends of one HMC transition over q17 for C chains, on the device (what PyMC's HMC / NUTS
 * step does on the host around its leapfrogs in pm.sample, abd.py:922): momentum refresh and
 * Metropolis accept, with per-chain step-size adaptation by dual averaging (Hoffman & Gelman 2014,
 * the scheme PyMC uses).  A host-driven sampler then runs an iteration as five launches and no
 * device synchronisation: hmc_begin, leapfrog, hmc_end, gibbs_sweep, logp_dlogp.
 *   abd_hmc_begin_dev: z ~ N(0, I) (Philox4x32-10 keyed by (seed; iter, chain, component)),
 *     p = linv_t z with linv_t = (L^T)^-1, inv_mass = L L^T (17 x 17 row-major), so p ~ N(0, M);
 *     writes the work copies qw = q, gw = grad, pw = p and h0 = -logp + z.z / 2.
 *   abd_hmc_end_dev: h1 = -lpw + pw' inv_mass pw / 2; accept with probability min(1, exp(h0 - h1))
 *     (not finite => reject): q, grad, logp take the work copies; accept_out[c] = that probability.
 *     da (C x 4: mu, hbar, log_avg, t) is the dual-averaging state; when adapt != 0 it is advanced
 *     with accept_out[c] against target_accept and eps[c] = exp(log_eps) is written.          */
int abd_hmc_begin_dev(abd_handle* h, int n_chains, const double* q17, const double* grad17,
                      const double* logp, const double* linv_t, uint64_t seed, uint64_t iter,
                      double* qw, double* pw, double* gw, double* h0, void* stream);
int abd_hmc_end_dev(abd_handle* h, int n_chains, double* q17, double* grad17, double* logp,
                    const double* qw, const double* pw, const double* gw, const double* lpw,
                    const double* inv_mass, const double* h0, uint64_t seed, uint64_t iter,
                    double* accept_out, double* da, double* eps, int adapt, double target_accept,
                    void* stream);

/* The No-U-Turn sampler's tree bookkeeping on the device (what PyMC's NUTS step does on the host around
 * its leapfrogs in pm.sample, abd.py:922): multinomial sampling inside sub-trees, biased progressive
 * sampling between them, the generalised U-turn criterion on every balanced sub-tree, divergence when the
 * energy error exceeds 1000.  The C chains of a batch double in lockstep; per transition the host enqueues
 *   abd_nuts_begin_dev                                   momentum refresh, empty tree, first direction
 *   for depth j = 0 .. max_depth - 1, leaf n = 0 .. 2^j - 1:
 *       abd_leapfrog_dev(n_steps = 1, qw, pw, gw, lpw, eps_signed, ...)      one leaf for all chains
 *       abd_nuts_leaf_dev(j, n)                          fold the leaf into every chain's tree
 *     after the last leaf of a depth: any_active[j + 1] != 0 iff some chain still wants to double
 *     (ONE word read back per depth; stop when it is 0)
 *   abd_nuts_end_dev                                     move to the proposal, sample stats, step-size adaptation
 * state: C x abd_nuts_state_doubles(max_depth) doubles (device scratch owned by the caller); qw / pw / gw
 * (C x 17), lpw (C), eps_signed (C): work vectors the leapfrog integrates in place; any_active: max_depth + 1
 * ints.  Philox streams keyed by (seed; iter, global chain, purpose).  accept_out = mean acceptance statistic
 * of the tree, depth_out = tree depth, diverged_out = 0 / 1 (any may be NULL except accept_out).        */
int64_t abd_nuts_state_doubles(int max_depth);
int abd_nuts_begin_dev(abd_handle* h, int n_chains, int max_depth, const double* q17, const double* grad17,
                       const double* logp, const double* linv_t, const double* eps, uint64_t seed, uint64_t iter,
                       double* state, double* qw, double* pw, double* gw, double* eps_signed, int* any_active,
                       void* stream);
int abd_nuts_leaf_dev(abd_handle* h, int n_chains, int max_depth, int depth, int leaf, double* qw, double* pw,
                      double* gw, const double* lpw, const double* inv_mass, const double* eps, uint64_t seed,
                      uint64_t iter, double* state, double* eps_signed, int* any_active, void* stream);
/* One doubling in one call: for leaf n = 0 .. 2^depth - 1, abd_leapfrog_dev(n_steps = 1) + abd_nuts_leaf_dev (a host
 * that pays microseconds per foreign call -- Python -- would otherwise be the bottleneck of deep trees).   */
int abd_nuts_extend_dev(abd_handle* h, int n_chains, int max_depth, int depth, double* qw, double* pw, double* gw,
                        double* lpw, const double* inv_mass, const double* eps, uint64_t seed, uint64_t iter,
                        double* state, double* eps_signed, int* any_active, const int8_t* i_raw,
                        const int8_t* waner, void* stream);
int abd_nuts_end_dev(abd_handle* h, int n_chains, int max_depth, double* q17, double* grad17, double* logp,
                     const double* state, double* accept_out, double* depth_out, double* diverged_out, double* da,
                     double* eps, int adapt, double target_accept, void* stream);

/* Individual sharding over the GPUs of one node WITHOUT a separate collective: the all-reduce of
 * the C x 16 raw sums is fused into the kernel through NVLink peer memory (each rank's finishing
 * CTA stores its sums into every peer's buffer, waits for the peers' flags, adds in rank order,
 * finalises).  One process per GPU:
 *   abd_xch_alloc   allocates this rank's exchange buffer, returns its CUDA IPC handle (64 bytes);
 *   (exchange the handles between the processes, e.g. torch.distributed.all_gather)
 *   abd_xch_connect opens all peers' buffers (all_ipc_handles: world x 64 bytes, rank order);
 *   abd_logp_dlogp_sharded_dev  is then a COLLECTIVE call: every rank must make the same sequence
 *   of calls; all ranks obtain bitwise identical (logp, dlogp).  The handle must have been created
 *   with total_* / ind_offset set.  abd_xch_status: synchronous check for a timed-out wait.   */
#define ABD_IPC_HANDLE_BYTES 64
int abd_xch_alloc(abd_handle* h, int world, int rank, int max_chains, void* out_ipc_handle);
int abd_xch_connect(abd_handle* h, const void* all_ipc_handles);
int abd_logp_dlogp_sharded_dev(abd_handle* h, int n_chains, const double* q17, const int8_t* i_raw,
                               const int8_t* waner, double* out_logp, double* out_dlogp,
                               void* stream);
int abd_xch_status(abd_handle* h);
/* One leapfrog step (abd_leapfrog_dev with n_steps = 1) on an individual-sharded cohort, the all-reduce
 * fused into the launch as in abd_logp_dlogp_sharded_dev: every rank starts from the same (q, p, grad,
 * eps, inv_mass), evaluates its individuals at the new position, exchanges, and ends with bitwise
 * identical (q, p, grad, logp).  A COLLECTIVE call.  With abd_hmc_begin_dev / abd_hmc_end_dev (same
 * seed on every rank) and the local Gibbs sweeps this runs the whole compound sampler of pm.sample
 * (abd.py:922) on a sharded cohort with no other communication.                                  */
int abd_leapfrog_sharded_dev(abd_handle* h, int n_chains, double* q17, double* p17, double* grad17,
                             double* logp, const double* eps, const double* inv_mass,
                             const int8_t* i_raw, const int8_t* waner, void* stream);
/* Exchange cost kept apart from compute: out[r] (r < 8) = nanoseconds this rank's finishing CTAs have
 * spent waiting for peer r's contribution (launch skew + NVLink latency), out[8] = exchanges done
 * (one per chain and evaluation).  Synchronous; reset != 0 zeroes the counters.                   */
int abd_xch_stats(abd_handle* h, uint64_t* out, int reset);

/* Pointers to the resident chain state (valid until a call with MORE chains than any before: the
 * buffers are then reallocated -- query again).  Beside these int8 arrays the library keeps a packed
 * copy of the resident state (per chain and individual: the i_raw column as a bit mask, the waner
 * bit and the constrained infections, abd.py:640-667) that every evaluation / sweep on the resident
 * state reads instead; abd_upload_state and the Gibbs sweeps keep both in step.  A caller that
 * WRITES into the int8 arrays itself must call abd_state_touch afterwards (the packed copy is then
 * rebuilt on next use).  One stream per handle at a time: the per-handle scratch (partials, tickets,
 * work queue) is shared by every call on the handle.                                           */
int abd_state_dev(abd_handle* h, int n_chains, int8_t** i_raw, int8_t** waner);
int abd_state_touch(abd_handle* h);

/* Global index of this handle's first chain (default 0).  The Philox streams of the Gibbs sweeps
 * and of abd_hmc_begin_dev / abd_hmc_end_dev are keyed by (seed; sweep | iteration, GLOBAL chain,
 * GLOBAL individual, ...): processes that shard the CHAINS of one run over several GPUs with one
 * seed set their rank's first chain here, so that no two chains of the run share a stream
 * (the reference's chains draw from independent generators, pm.sample abd.py:922).            */
int abd_set_chain_offset(abd_handle* h, int64_t chain_offset);

/* Tuning knobs of the log-likelihood kernel (0 = automatic): target OD rows per CTA tile and
 * chains looped over inside one CTA (reusing the rows staged in shared memory).             */
int abd_set_tuning(abd_handle* h, int rows_per_tile, int chains_per_cta);
/* The grid plan of the handle's most recent log-likelihood launch: out6 = {tiles of individuals, chain groups,
 * chains per CTA, dynamic shared memory per CTA (bytes), 1 if the compact cell layout was used, resident CTAs per
 * SM}.  (Introspection for tests and measurements; nothing in the reference corresponds to it.)              */
int abd_last_plan(const abd_handle* h, int32_t* out6);

/* Test hook: out_exp[i] = the kernels' fast exp(z[i]), out_rcp[i] = their fast 1/(1 + |z[i]|)
 * (host pointers; checked against libm in tests/test_gpu_parity.py).                        */
int abd_debug_fast_math(int device, int64_t n, const double* z, double* out_exp, double* out_rcp);

#ifdef __cplusplus
}
#endif
#endif /* ABD_B200_H */
