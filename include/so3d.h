/* so3d.h -- C ABI of libso3d: sm_100a kernels for batched SO(3) manifold-diffusion math.
 *
 * Drop-in boundary for the hot path of qazwsxal/diffusion-extensions (@ f100885d):
 *   util.py (log/exp/axis-angle/scale/quaternion), distributions.py (IsotropicGaussianSO3) and
 *   diffusion.py (SO3Diffusion.q_sample / p_losses / p_sample).
 * The reference has no FFI layer of its own (it is pure Python/PyTorch); each entry point below
 * cites the reference function (file:line) whose arithmetic it replaces, and INTEGRATION.md shows
 * the ctypes binding the Python side uses.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device, float32 unless stated, dense
 *     row-major:  rotations n x 9 (3x3 row-major, 36 B), vectors n x 3, quaternions n x 4
 *     (real part first), scalars n.  Pointers need only 4-byte alignment; 16-byte aligned buffers
 *     take the vectorised path.
 *   - the caller owns all memory (inputs and outputs); the library never allocates, frees or keeps
 *     a pointer after return.
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream); it never synchronises, so calls are CUDA-graph capturable.
 *   - return value: 0 on success, >0 a cudaError_t from the launch, <0 an argument error
 *     (SO3D_EINVAL).  so3d_last_error() returns a thread-local message for the last failure.
 *   - NaN in -> NaN out; nothing traps.  n == 0 is a no-op.
 *   - `*_stride` arguments for per-row scalars: 1 = one value per row, 0 = a single value shared by
 *     all rows (the reference's scalar-eps / scalar-scale broadcasting).
 *   - random draws are counter based (Philox4x32-10): key = seed, counter = (row_offset + row,
 *     rng_offset).  Results do not depend on how a batch is sharded over GPUs when each shard passes
 *     its global row_offset.
 */
#ifndef SO3D_H_
#define SO3D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SO3D_VERSION 100
#define SO3D_EINVAL (-1)

#define SO3D_CDF_POINTS 999  /* entries per CDF row (distributions.py:15,30: 1000-point grid) */
#define SO3D_GRID_POINTS 1000
#define SO3D_GUIDE_BUCKETS 2051 /* 16-byte records per guide row */

/* evaluator for the IGSO(3) density (mode argument) */
#define SO3D_MODE_SERIES 0          /* truncated series, exactly L terms per row (SURVEY A.1); rows whose alternating sum is
                                       ill-conditioned in fp32 (omega > 4.2 eps, eps <= 1: cond > 14) take the closed form
                                       AFTER their L terms have run -- see kSeriesGuard in csrc/so3d_math.cuh              */
#define SO3D_MODE_CLOSED 1          /* 3-image closed form, distributions.py:53-72, stable rewrite         */
#define SO3D_MODE_AUTO 2            /* closed form for eps <= 1, series (live terms only) above             */
#define SO3D_MODE_SERIES_ADAPTIVE 3 /* series, skipping terms whose fp32 weight is exactly 0 (same result) */
#define SO3D_MODE_SERIES_PURE 4     /* the raw fp32 series on every row, exactly L terms, no conditioning guard            */

int so3d_version(void);
const char* so3d_last_error(void);

/* ---- L0: util.py -------------------------------------------------------------------------- */
/* util.py:164-192 log_rmat: out = 3x3 skew matrix log(R). */
int so3d_log_f32(const float* R, float* out9, int64_t n, void* stream);
/* util.py:79-84 o 164-192: vee(log R) as a 3-vector. */
int so3d_logvec_f32(const float* R, float* out3, int64_t n, void* stream);
/* util.py:208-219 rmat_to_aa: unit axis (n x 3) and angle in [0, pi] (n). */
int so3d_rmat_to_aa_f32(const float* R, float* axis3, float* angle, int64_t n, void* stream);
/* util.py:195-205 aa_to_rmat: axis is normalised inside, like the reference. */
int so3d_aa_to_rmat_f32(const float* axis3, const float* angle, float* R, int64_t n, void* stream);
/* diffusion.py:294 matrix_exp(vec2skew(v)). */
int so3d_expvec_f32(const float* v3, float* R, int64_t n, void* stream);
/* util.py:349-361 so3_scale. */
int so3d_scale_f32(const float* R, const float* s, int s_stride, float* out, int64_t n, void* stream);
/* util.py:222-252 quat_to_rmat (real-first, un-normalised input allowed). */
int so3d_quat_to_rmat_f32(const float* q4, float* R, int64_t n, void* stream);
/* no reference counterpart: unit quaternion (real-first, real part >= 0) of a rotation matrix. */
int so3d_rmat_to_quat_f32(const float* R, float* q4, int64_t n, void* stream);
/* batched 3x3 product C = op(A) op(B), op = transpose when trans* != 0 (the `@` at
 * distributions.py:50, diffusion.py:297,302,326,346).  a_stride/b_stride: 1 = per row, 0 = one
 * shared matrix. */
int so3d_compose_f32(const float* A, int a_stride, int trans_a, const float* B, int b_stride, int trans_b,
                     float* C, int64_t n, void* stream);
/* util.py:315-322 rmat_dist = |log(A^T B)|_F = sqrt(2) theta. */
int so3d_rmat_dist_f32(const float* A, const float* B, float* out, int64_t n, void* stream);
/* util.py:325-338 so3_lerp: A @ rot(axis(A^T B), w * angle(A^T B)). */
int so3d_lerp_f32(const float* A, const float* B, const float* w, int w_stride, float* out, int64_t n, void* stream);

/* backward passes (what autograd through the reference's torch ops yields; G = upstream grad) */
int so3d_log_bwd_f32(const float* R, const float* G9, float* gR, int64_t n, void* stream);
int so3d_aa_to_rmat_bwd_f32(const float* axis3, const float* angle, const float* G9, float* g_axis3,
                            float* g_angle, int64_t n, void* stream);
int so3d_expvec_bwd_f32(const float* v3, const float* G9, float* g_v3, int64_t n, void* stream);
int so3d_scale_bwd_f32(const float* R, const float* s, int s_stride, const float* G9, float* gR, float* g_s,
                       int64_t n, void* stream);

/* ---- L1: distributions.py IsotropicGaussianSO3 ------------------------------------------ */
/* distributions.py:53-72 _eps_ft: density f_eps(omega) (w.r.t. Haar measure, no (1-cos)/pi). */
int so3d_igso3_density_f32(const float* omega, const float* eps, int eps_stride, float* f, int64_t n, int mode,
                           int L, void* stream);
/* distributions.py:74-77 log_prob fused with axis-angle extraction and the score:
 *   logp[n] = log f_eps(angle(R));  score3[n x 3] = (d log f / d omega) * axis (nullable);
 *   dlogf[n] = d log f / d omega (nullable; saved for the backward). */
int so3d_igso3_logp_score_f32(const float* R, const float* eps, int eps_stride, float* logp, float* score3,
                              float* dlogf, int64_t n, int mode, int L, void* stream);
/* gradient of sum(gout * logp) w.r.t. the 9 matrix entries (SURVEY A.5; matches autograd through
 * distributions.py:74-77 + util.py:164-219). */
int so3d_igso3_logp_bwd_f32(const float* R, const float* dlogf, const float* gout, float* gR, int64_t n,
                            void* stream);
/* distributions.py:15-30: CDF rows for `rows` values of eps.  grid_loc/haar_w are the reference's
 * 1000-point float32 grid pi*linspace(0,1,1000)^3 and (1-cos(loc))/pi (host-computed, passed in so
 * the fp32 values are bit-identical to torch's).  trap_out is rows x 999 (the transpose of the
 * reference's (999, *E) layout).  quirks != 0 reproduces the reference's overflow behaviour (D5). */
int so3d_igso3_cdf_table_f32(const float* eps, int64_t rows, const float* grid_loc, const float* haar_w,
                             float* trap_out, int quirks, void* stream);
/* Search accelerator for the inverse-CDF lookup of distributions.py:38-43 (`(trap <= u).sum()`): for every CDF
 * row, SO3D_GUIDE_BUCKETS records of 16 bytes, record k = {lo | hi << 16, trap[lo-1], trap[lo], trap[lo+1]} with
 * lo = #{j : trap[j] <= a_k}, hi = #{j : trap[j] <= b_k} (trap indices clamped to [0, 998]) where [a_k, b_k] is the
 * range of u served by record k: 1/1024 steps on [1/8, 7/8], 64 steps per octave of u on [2^-13, 2^-3) and of 1 - u
 * on the mirrored range (the CDF entries crowd towards both ends), one record each for the rest of the two tails.
 * For u in that range the count lies in [lo, hi]; when hi - lo <= 1 one 16-byte load resolves the lookup,
 * otherwise a binary search restricted to [lo, hi] does: either way the index is IDENTICAL to the full search.
 * guide_out: rows x SO3D_GUIDE_BUCKETS x 4 words, 16-byte aligned. */
int so3d_igso3_cdf_guide(const float* cdf, int64_t rows, uint32_t* guide_out, void* stream);
/* distributions.py:33-51 sample: R = mean @ rot(axis, angle(u)).
 *   cdf: table rows x 999;  guide: so3d_igso3_cdf_guide(cdf) or NULL (only used with row_idx; the shared-row
 *   path builds its guide in shared memory);  loc: 999 grid angles;  row_idx: int64[n] row per sample, or NULL with
 *   `row` = the single shared row (scalar-eps path, staged in shared memory).
 *   u / axes3: optional explicit draws (u in [0,1), axes un-normalised like randn) -- when NULL
 *   they come from Philox(seed, row_offset + i, rng_offset).
 *   mean: optional 3x3 (mean_stride 0) or n x 9 (mean_stride 1) left factor.
 *   outputs: R (n x 9), and optionally the drawn angle[n] / unit axis3[n x 3]. */
int so3d_igso3_sample_f32(const float* cdf, const uint32_t* guide, const float* loc, int64_t rows, const int64_t* row_idx, int64_t row,
                          const float* u, const float* axes3, uint64_t seed, uint64_t rng_offset,
                          uint64_t row_offset, const float* mean, int mean_stride, float* R, float* angle,
                          float* axis3, int64_t n, void* stream);
/* The same draw with no table: the angle is the exact inverse CDF of the IGSO(3) angle law
 * p(w) = f_eps(w) (1 - cos w) / pi on [0, pi], found per row (|F(angle) - u| ~ 3e-7 for eps in [1e-3, 4]).
 *   eps: eps_stride 0 (one shared eps) or 1 (eps[n], one per row).  u = 0 gives angle 0; a NaN eps a NaN angle.
 *   u / axes3 / seed / rng_offset / row_offset / mean / outputs as in so3d_igso3_sample_f32, with the same Philox
 *   counter layout, so at the same seed both samplers see the same (u, axis). */
int so3d_igso3_sample_exact_f32(const float* eps, int eps_stride, const float* u, const float* axes3, uint64_t seed,
                                uint64_t rng_offset, uint64_t row_offset, const float* mean, int mean_stride, float* R,
                                float* angle, float* axis3, int64_t n, void* stream);

/* Backward of the reparameterised exact draw R = mean N, N = Rodrigues(axis3, angle), angle = F^{-1}(u; eps) at fixed
 * (u, axis), as written by so3d_igso3_sample_exact_f32 (angle and axis3 outputs).  Per row, with the upstream gradient G9:
 *   g_w = <mean^T G, hat(axis) N>,  g_eps[i] = g_w dw/deps,  g_mean9[i] = G N^T  (g_mean9 may be NULL: skipped).
 * dw/deps = -2 eps d log f / dw at the angle (the heat equation makes the implicit derivative -(dF/deps)/p exactly this):
 * the image-free closed form in x = w / (2 eps) below eps = 0.3, the density's 3-image closed form up to eps = 1 and its
 * series above.  |error| <= 8 2^-24 (|dw/deps| (1 + 4 eps^2) + [eps <= 1] angle / eps) against fp64, for eps in [1e-3, 4].
 * dw/deps is odd in eps (the law depends on eps^2) and NaN for a NaN eps.  At eps = 0 it is the eps -> 0+ limit 2 x0(u), x0
 * the Maxwell quantile: those rows read u (given) or redraw it from (seed, rng_offset, row_offset) as the sampler did.
 * Small angles need no separate form: every term left is O(w).  g_eps is per row; the caller reduces it for a shared eps
 * (eps_stride 0).  Measured on a B200 at a 1000 W power limit, 2^24 rows: 0.345 ms (shared eps 0.1) / 0.473 ms (per-row
 * eps over [4.67e-3, 1]), 0.25 / 0.17 of the forward draw, 1.7x / 2.3x its 92 / 96 B-per-row HBM floor. */
int so3d_igso3_rsample_bwd_f32(const float* eps, int eps_stride, const float* angle, const float* axis3, const float* mean,
                               int mean_stride, const float* G9, const float* u, uint64_t seed, uint64_t rng_offset,
                               uint64_t row_offset, float* g_eps, float* g_mean9, int64_t n, void* stream);

/* Entropy of IGSO(3)(eps) and its eps-derivative, per row (DESIGN.md 4.11):  H[i] = -int_0^pi p log f dw with
 * p(w) = f(w) (1 - cos w) / pi, and dH_deps[i] = 2 eps E_p[(d log f / dw)^2] (de Bruijn's identity; dH_deps may be NULL:
 * skipped).  One 16-node Gauss-Legendre pass: the image-free law in x = w / (2 eps) below eps = 0.3, the closed form up to
 * eps = 1, the cancellation-free series form -H = E_haar[(1 + delta) log1p(delta) - delta], delta = f - 1, above.
 * |error| <= 8 2^-24 (|H| + eps |dH/deps| + [eps <= 1]) for H and 8 2^-24 |dH/deps| (1 + 4 eps^2) for dH/deps, against
 * fp64, for eps in [1e-20, 6] (results below FLT_MIN, from eps ~ 4.65 on, may flush to 0).  H is even and dH/deps odd in
 * eps; eps = 0 gives -inf / +inf (the 0+ limit 3/eps), NaN gives NaN.  Runs on the persistent row engine. */
int so3d_igso3_entropy_f32(const float* eps, float* H, float* dH_deps, int64_t n, void* stream);

/* ---- L2: diffusion.py SO3Diffusion ---------------------------------------------------------- */
/* diffusion.py:339-346 q_sample + :348-355 p_losses target, fused:
 *   eps = sqrt_1m_ac[t], noise ~ IGSO3(eps) from cdf row t, x_t = so3_scale(x0, sqrt_ac[t]) @ noise,
 *   target = vee(log noise) / eps  (nullable), noise (nullable), score of the noise under
 *   IGSO3(eps) (nullable, auto evaluator).  t: int64[n] in [0, T).  guide: so3d_igso3_cdf_guide(cdf) or NULL. */
int so3d_q_sample_f32(const float* x0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac, int64_t T,
                      const float* cdf, const uint32_t* guide, const float* loc, uint64_t seed, uint64_t rng_offset,
                      uint64_t row_offset, float* x_t, float* target3, float* noise, float* score3, int64_t n, void* stream);
/* so3d_q_sample_f32 (x_t and target only) with the Philox SEED READ FROM DEVICE MEMORY when the kernel runs: a training
 * step captured in a CUDA graph (so3_train.py:70-76: loss = process(x); backward; step) draws fresh noise on every replay
 * after the caller bumps *seed_dev (a captured `seed.add_(1)`).  Draws equal so3d_q_sample_f32's at seed = *seed_dev. */
int so3d_q_sample_dseed_f32(const float* x0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac, int64_t T,
                            const float* cdf, const uint32_t* guide, const float* loc, const uint64_t* seed_dev,
                            uint64_t rng_offset, uint64_t row_offset, float* x_t, float* target3, int64_t n, void* stream);
/* q_sample with the noise supplied by the caller (diffusion.py:339-346 with noise != None). */
int so3d_q_sample_given_f32(const float* x0, const int64_t* t, const float* sqrt_ac, int64_t T, const float* noise,
                            float* x_t, int64_t n, void* stream);
/* diffusion.py:291-326 reverse step, fused:
 *   x0_hat = so3_scale(x_t, recip[t]) @ exp(hat(pred * recipm1[t]))^T          (:291-297)
 *   mean   = so3_scale(x0_hat, coef1[t]) @ so3_scale(x_t, coef2[t])            (:299-302)
 *   out    = t == 0 ? mean : mean @ noise,  noise ~ IGSO3(sigma_t) from post_cdf row t   (:315-326)
 *   t: int64[n] per row (t_stride 1) or a single shared step (t_stride 0: CDF row and guide staged in
 *   shared memory).  post_guide: so3d_igso3_cdf_guide of post_cdf (nullable; used with per-row t).
 *   post_cdf == NULL returns the mean only (p_mean_variance).  x0_hat_out nullable. */
int so3d_p_sample_f32(const float* x_t, const float* pred3, const int64_t* t, int t_stride, const float* recip,
                      const float* recipm1, const float* coef1, const float* coef2, int64_t T, const float* post_cdf,
                      const uint32_t* post_guide, const float* loc, uint64_t seed, uint64_t rng_offset, uint64_t row_offset,
                      float* out, float* x0_hat_out, int64_t n, void* stream);

/* The same step (shared t, noise on, no x0_hat) with the Philox SEED READ FROM DEVICE MEMORY at execution time:
 * a captured CUDA graph of a whole sampling loop (diffusion.py:328-337, one launch per step with rng_offset = step)
 * draws fresh noise on every replay once the caller has written a new seed to seed_dev.  Draws equal
 * so3d_p_sample_f32's at seed = *seed_dev. */
int so3d_p_sample_dseed_f32(const float* x_t, const float* pred3, const int64_t* t, const float* recip, const float* recipm1,
                            const float* coef1, const float* coef2, int64_t T, const float* post_cdf, const float* loc,
                            const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset, float* out, int64_t n,
                            void* stream);

/* diffusion.py:328-337 (p_sample_loop) with nothing but the manifold step between two steps -- no denoiser (pred3 == NULL:
 * zero prediction) or one fixed prediction per particle -- as ONE launch: the steps t_hi, t_hi - 1, ..., t_lo of
 * so3d_p_sample_f32 (shared t, rng_offset = rng_offset0 + t at step t), bit-identical to that sequence of launches.
 * Particles are independent, so a CTA keeps a chunk of them resident in shared memory for all steps: x_t is read from
 * HBM once and `out` written once (BASELINE configs[2]: 1000 steps x 2^24 particles).  post_cdf (T x 999) and its guide
 * records post_guide (T x SO3D_GUIDE_BUCKETS x 4 words, so3d_igso3_cdf_guide) are required; out may alias x_t. */
int so3d_p_sample_loop_f32(const float* x_t, const float* pred3, int64_t t_hi, int64_t t_lo, const float* recip, const float* recipm1,
                           const float* coef1, const float* coef2, int64_t T, const float* post_cdf, const uint32_t* post_guide,
                           const float* loc, uint64_t seed, uint64_t rng_offset0, uint64_t row_offset, float* out, int64_t n,
                           void* stream);

/* ---- RotPredict denoiser fused with the reverse step (SURVEY 8f-4) ------------------------------------ */
#define SO3D_ROTPREDICT_D 65              /* so3_train.py:12 d_model */
#define SO3D_ROTPREDICT_BLOB_FLOATS 39424 /* packed tf32 hi/lo weights in the tensor-core (UMMA) shared-memory layout */
/* so3_train.py:26-36 RotPredict.net (out_type "skewvec"): five nn.Linear layers, weights row-major (out x in):
 * w1..w4: 65 x 65, w5: 3 x 65, b1..b4: 65, b5: 3 (b1 is not packed: it enters through c1_table below).
 * Writes blob[SO3D_ROTPREDICT_BLOB_FLOATS] (16-byte aligned).  Re-run whenever the weights change. */
int so3d_rotpredict_pack_f32(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                             const float* b3, const float* w4, const float* b4, const float* w5, const float* b5,
                             float* blob, void* stream);
/* so3_test.py:26-31 / diffusion.py:315-337: one reverse step with the RotPredict denoiser inside the kernel,
 *   pred = RotPredict(x_t, t)  (so3_train.py:39-49, models.py:13-25);   out = p_sample(x_t, pred, t) as so3d_p_sample_f32
 * for a step index shared by the batch (t: int64[1] on the device).  The 65-wide MLP runs on the tensor cores
 * (tcgen05.mma kind::tf32, 3-term hi/lo split: fp32-level accuracy), activations stay in tensor memory.
 *   c1_table: T x 65, c1_table[t] = b1 + W1[:, 9:] @ SinusoidalPosEmb(56)(t)  -- the time embedding folded into
 *   layer 1's bias (caller-computed once per weight set).  post_cdf NULL or t == 0: no noise (posterior mean).
 *   out (n x 9) and pred_out (n x 3) are each nullable (not both).  Random draws are those of so3d_p_sample_f32
 *   at the same (seed, rng_offset, row_offset). */
int so3d_rotpredict_p_sample_f32(const float* x_t, const float* blob, const float* c1_table, const int64_t* t,
                                 const float* recip, const float* recipm1, const float* coef1, const float* coef2, int64_t T,
                                 const float* post_cdf, const float* loc, uint64_t seed, uint64_t rng_offset,
                                 uint64_t row_offset, float* out, float* pred_out, int64_t n, void* stream);

/* As above with the seed read from device memory (see so3d_p_sample_dseed_f32). */
int so3d_rotpredict_p_sample_dseed_f32(const float* x_t, const float* blob, const float* c1_table, const int64_t* t,
                                       const float* recip, const float* recipm1, const float* coef1, const float* coef2,
                                       int64_t T, const float* post_cdf, const float* loc, const uint64_t* seed_dev,
                                       uint64_t rng_offset, uint64_t row_offset, float* out, float* pred_out, int64_t n,
                                       void* stream);

/* diffusion.py:328-337 / so3_test.py:26-31: the WHOLE reverse process in one launch -- the steps t_hi, t_hi - 1, ..., t_lo
 * of so3d_rotpredict_p_sample_f32 with rng_offset = t at step t (bit-identical to that sequence of launches).  Particles
 * are independent and stay with one thread, so no grid-wide synchronisation is needed; the weights are staged once.
 * seed_dev non-NULL: the seed is read from device memory instead of `seed`.  out must not alias x_t.  post_cdf required. */
int so3d_rotpredict_p_sample_loop_f32(const float* x_t, const float* blob, const float* c1_table, int64_t t_hi, int64_t t_lo,
                                      const float* recip, const float* recipm1, const float* coef1, const float* coef2,
                                      int64_t T, const float* post_cdf, const float* loc, uint64_t seed,
                                      const uint64_t* seed_dev, uint64_t row_offset, float* out, int64_t n, void* stream);

/* ---- SE(3) arm: diffusion.py SE3Diffusion / distributions.py IGSO3xR3 (SURVEY 8f-3) --------------- */
/* diffusion.py:498-516 (SE3Diffusion.q_sample + p_losses targets), fused.  Rotation half exactly as
 * so3d_q_sample_f32 (same Philox block: identical rotation draws at the same seed / rng_offset); translation half
 *   shift_t = sqrt_ac[t] shift0 + sqrt_1m_ac[t] shift_scale z,   target_shift3 = z = noise_shift / (eps_t shift_scale)
 * with z ~ N(0, I3) from Philox(seed, row_offset + i, rng_offset | 2^63)  (distributions.py:84-110 IGSO3xR3.sample).
 * target_rot3 / target_shift3 nullable.  rng_offset < 2^63. */
int so3d_se3_q_sample_f32(const float* rot0, const float* shift0, const int64_t* t, const float* sqrt_ac,
                          const float* sqrt_1m_ac, int64_t T, const float* cdf, const uint32_t* guide, const float* loc,
                          float shift_scale, uint64_t seed, uint64_t rng_offset, uint64_t row_offset, float* rot_t,
                          float* shift_t, float* target_rot3, float* target_shift3, int64_t n, void* stream);
/* so3d_se3_q_sample_f32 with the Philox SEED READ FROM DEVICE MEMORY when the kernel runs: a captured SE(3) training
 * step draws fresh rotation and translation noise on every replay after the caller bumps *seed_dev (a captured
 * `seed.add_(1)`).  Both streams come from *seed_dev (rotation at rng_offset, translation at rng_offset | 2^63): the draws
 * equal so3d_se3_q_sample_f32's at seed = *seed_dev.  target_rot3 / target_shift3 nullable.  rng_offset < 2^63. */
int so3d_se3_q_sample_dseed_f32(const float* rot0, const float* shift0, const int64_t* t, const float* sqrt_ac,
                                const float* sqrt_1m_ac, int64_t T, const float* cdf, const uint32_t* guide, const float* loc,
                                float shift_scale, const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset,
                                float* rot_t, float* shift_t, float* target_rot3, float* target_shift3, int64_t n, void* stream);
/* diffusion.py:446-485 (SE3Diffusion.predict_start_from_noise, q_posterior, p_sample), fused.  Rotation half as
 * so3d_p_sample_f32; translation half
 *   shift0_hat = recip[t] shift_t - recipm1[t] pred_shift;  mean = coef1[t] shift0_hat + coef2[t] shift_t;
 *   shift_out = t == 0 ? mean : mean + sigma[t] shift_scale z      (sigma[t] = exp(posterior_log_variance_clipped[t]/2))
 * post_cdf == NULL returns the posterior mean only (p_mean_variance). */
int so3d_se3_p_sample_f32(const float* rot_t, const float* shift_t, const float* pred_rot3, const float* pred_shift3,
                          const int64_t* t, int t_stride, const float* recip, const float* recipm1, const float* coef1,
                          const float* coef2, const float* sigma, int64_t T, const float* post_cdf,
                          const uint32_t* post_guide, const float* loc, float shift_scale, uint64_t seed, uint64_t rng_offset,
                          uint64_t row_offset, float* rot_out, float* shift_out, int64_t n, void* stream);
/* The same step (shared t: int64[1] on the device, noise on, post_cdf required) with the Philox SEED READ FROM DEVICE
 * MEMORY at execution time: a captured CUDA graph of a whole SE(3) sampling loop (one launch per step with
 * rng_offset = step) draws fresh noise on every replay once the caller has written a new seed to seed_dev.  Draws of
 * both halves equal so3d_se3_p_sample_f32's at seed = *seed_dev.  rng_offset < 2^63. */
int so3d_se3_p_sample_dseed_f32(const float* rot_t, const float* shift_t, const float* pred_rot3, const float* pred_shift3,
                                const int64_t* t, const float* recip, const float* recipm1, const float* coef1,
                                const float* coef2, const float* sigma, int64_t T, const float* post_cdf, const float* loc,
                                float shift_scale, const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset,
                                float* rot_out, float* shift_out, int64_t n, void* stream);

/* ---- data side: distributions.py Bingham (SURVEY 8f-2) ------------------------------------------- */
/* distributions.py:113-127 Bingham.rsample (zero-mean MultivariateNormal in R^4, normalised to a unit quaternion,
 * real part first) fused with util.py:222-252 quat_to_rmat (bingham_train.py:88-90):
 *   q = L z / |L z|,  L = scale_tril16 (DEVICE pointer, 4x4 row-major, lower triangle used),
 *   z = z4[n x 4] when given (parity with explicit draws), else 4 Box-Muller normals from
 *   Philox(seed, row_offset + i, rng_offset).   Outputs (each nullable, not both): q4 (n x 4, 16-byte aligned),
 *   R (n x 9). */
int so3d_bingham_sample_f32(const float* scale_tril16, const float* z4, uint64_t seed, uint64_t rng_offset,
                            uint64_t row_offset, float* q4, float* R, int64_t n, void* stream);

/* ---- evaluation: util.py MMD (SURVEY 8f-1) ---------------------------------------------------- */
#define SO3D_PAIR_GAUSSIAN 0 /* util.py:128-134 rmat_gaussian_kernel: exp(-rmat_dist) = exp(-sqrt(2) theta(A^T B)) */
#define SO3D_PAIR_COSINE 1   /* util.py:136-150 rmat_cosine_kernel: (tr(B^T A) - 1)/2 = cos theta                 */
/* util.py:254-285 MMD: the three all-pairs kernel sums it needs, in one launch and without materialising the
 * pair matrices:   out3[0] = sum_{i,j < nx} k(X_i, X_j),  out3[1] = sum_{i,j < ny} k(Y_i, Y_j),
 *                  out3[2] = sum_{i < nx, j < ny} k(X_i, Y_j)            (doubles; Y may be NULL with ny = 0).
 * MMD = out3[0]/nx^2 + out3[1]/ny^2 - 2 out3[2]/(nx ny).  The work is a flat list of 256 x 256 tile pairs dealt
 * round-robin to `nshards` shards; this call computes shard `shard` only (multi-GPU: every rank calls with its
 * own shard and the caller adds the out3 of all ranks).  ws: scratch of ws_len doubles (>= 3; three per resident
 * CTA, 3 * 8 * #SMs lets the launch fill the device).  Deterministic for fixed (shard, nshards, ws_len). */
int so3d_pair_kernel_sums_f32(const float* X, int64_t nx, const float* Y, int64_t ny, int kernel, int64_t shard,
                              int64_t nshards, double* ws, int64_t ws_len, double* out3, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SO3D_H_ */
