/* sdfb200.h - C ABI of libsdfb200.so: the B200-native shape-SDF decoder and
 * latent-DDPM sampler hot path.
 *
 * Reference interface replaced: there is none to cite beyond the title line
 * /root/reference/README.md:1 (the mounted reference has no source).  The
 * entry points below are the C-level boundary underneath the Python API that
 * BASELINE.json's north_star names - Decoder(latent, xyz) -> sdf,
 * decode_grid(z, res), sample_latents(n) - and that SURVEY.md section 8(b)
 * proposes.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *  - every function returns 0 on success and a negative SDFB_E_* code on
 *    failure; sdfb_last_error() gives a thread-local human-readable message.
 *    Nothing throws across the boundary.
 *  - pointers named *_dev are device pointers on the context's device,
 *    *_host are host pointers.  `stream` is a cudaStream_t passed as void*
 *    (NULL = the legacy default stream).  Calls are asynchronous on `stream`
 *    unless the name ends in _host.
 *  - a context belongs to one device; calls on one context must be issued
 *    from one thread at a time and on one stream at a time (the per-latent
 *    constant block lives in the context).  The *_host calls run on streams
 *    the context owns; they order themselves after every device-path call
 *    issued on the context before them, and they return synchronised.
 *  - asynchronous calls return before their kernels run.  A kernel whose
 *    watchdog trips (a wait bounded by a wall-clock timeout) leaves invalid
 *    outputs and records the failure in the context: the NEXT call on that
 *    context - or sdfb_decoder_check / sdfb_ddpm_check, which synchronise the
 *    stream first - returns SDFB_E_KERNEL once and clears it.  Results of an
 *    asynchronous call are valid once a later call or *_check has returned 0.
 *  - no CPU fallback exists: without a CUDA device of compute capability
 *    10.x the create calls fail with SDFB_E_DEVICE.
 */
#ifndef SDFB200_H_
#define SDFB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDFB_OK 0
#define SDFB_E_INVALID (-1)   /* bad argument / unsupported shape            */
#define SDFB_E_DEVICE (-2)    /* no usable sm_100 device                     */
#define SDFB_E_CUDA (-3)      /* a CUDA runtime call failed                  */
#define SDFB_E_KERNEL (-4)    /* in-kernel watchdog or self-check tripped    */
#define SDFB_E_NOMEM (-5)

/* arithmetic of the matrix products */
#define SDFB_PREC_FP32 0 /* FFMA SIMT kernels: carries the 1e-5 / 1e-4 criteria          */
#define SDFB_PREC_BF16 1 /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM    */
#define SDFB_PREC_FP16 2 /* same kernel, fp16 operands (meets the 2e-3 bound vs fp32)    */

/* decoder parameter blob: W0,b0,W1,b1,...,W8,b8 (row-major W[out][in], fp32) */
#define SDFB_DECODER_PARAM_FLOATS 1839358
/* denoiser parameter blob: W0,b0,...,W4,b4                                   */
#define SDFB_DDPM_PARAM_FLOATS 3936512
#define SDFB_LATENT_DIM 256
#define SDFB_DDPM_STEPS 1000

typedef struct sdfb_decoder sdfb_decoder;
typedef struct sdfb_ddpm sdfb_ddpm;
typedef struct sdfb_comm sdfb_comm;
typedef struct sdfb_ddpm_trainer sdfb_ddpm_trainer;
typedef struct sdfb_decoder_trainer sdfb_decoder_trainer;

int sdfb_version(void);
const char* sdfb_last_error(void);

/* ---- SDF auto-decoder (SURVEY.md 8a rows A1-A4) -------------------------- */

/* Copies the fp32 parameters to `device`, packs the bf16 and fp16 tensor-core
 * weight streams and allocates the context workspace. */
int sdfb_decoder_create(const float* params_host, size_t n_floats, int device, sdfb_decoder** out);
int sdfb_decoder_destroy(sdfb_decoder* dec);

/* decode_grid(z, res) restricted to planes [z0, z1): writes
 * sdf_dev[(z1-z0)*res*res] (C order z,y,x).  Node (iz,iy,ix) sits at
 * c_i = float(2i-(res-1))/float(res-1) on each axis (bit-exact rule A1).
 * If mask_dev != NULL the sign-change mask (A4; built from sign bit-planes that the decoder
 * kernel emits together with the values) of the cell layers
 * [z0, min(z1,res-1)) is written as uint8 [(layers)*(res-1)*(res-1)]; when
 * z1 < res this needs the halo plane z1, which is then decoded too and stored
 * after the slab, so sdf_dev must hold (z1-z0+1)*res*res floats in that case. */
int sdfb_decode_grid(sdfb_decoder* dec, const float* latent_dev, int res, int z0, int z1,
                     float* sdf_dev, uint8_t* mask_dev, int precision, void* stream);

/* Packed variant: besides the sdf, the SIGN BIT-PLANES of the decoded planes (bit (q & 31) of word
 * q >> 5 = sdf[q] < 0, q = query index within the call, halo plane included; ceil(M / 32) words) and,
 * if mask_bits_dev != NULL, the sign-change mask PACKED one bit per cell (cell c -> bit c & 31 of
 * word c >> 5; ceil(cells / 32) words; same halo rule and sdf_dev size as sdfb_decode_grid).  The
 * tensor-core kernel writes the sign words itself, next to the values. */
int sdfb_decode_grid_bits(sdfb_decoder* dec, const float* latent_dev, int res, int z0, int z1, float* sdf_dev,
                          uint32_t* sign_bits_dev, uint32_t* mask_bits_dev, int precision, void* stream);

/* A batch of shapes (BASELINE configs 3 and 4): latents_dev [batch][256] -> sdf_dev [batch][res^3]. */
int sdfb_decode_grid_batch(sdfb_decoder* dec, const float* latents_dev, int batch, int res, float* sdf_dev,
                           int precision, void* stream);

/* Decoder(latent, xyz) -> sdf for M arbitrary points, xyz_dev [M][3]. */
int sdfb_decode_points(sdfb_decoder* dec, const float* latent_dev, const float* xyz_dev, int64_t M,
                       float* sdf_dev, int precision, void* stream);

/* Vector-Jacobian product w.r.t. the latent (SURVEY.md 8f row N4, what auto-decoder latent fitting
 * needs): grad_latent_dev[256] = sum_m dLdy_dev[m] * d sdf(latent, xyz_m) / d latent, fp32 FFMA path
 * (forward with stored activations + backward, deterministic reduction).  sdf_dev (optional, [M])
 * receives the forward values. */
int sdfb_decoder_vjp_latent(sdfb_decoder* dec, const float* latent_dev, const float* xyz_dev, int64_t M,
                            const float* dLdy_dev, float* grad_latent_dev, float* sdf_dev, void* stream);

/* The same product on the tensor pipe (precision SDFB_PREC_BF16 or SDFB_PREC_FP16): one launch of the
 * forward + backward instance of the fused decoder kernel - 16-bit operands, fp32 accumulation, the
 * column sums the latent sees kept in fp32 (oracle: decoder_vjp_latent_lowp).  sdf_dev (optional)
 * receives exactly what sdfb_decode_points returns at that precision. */
int sdfb_decoder_vjp_latent_tc(sdfb_decoder* dec, const float* latent_dev, const float* xyz_dev, int64_t M,
                               const float* dLdy_dev, float* grad_latent_dev, float* sdf_dev, int precision,
                               void* stream);

/* One step's worth of auto-decoder latent fitting (DeepSDF's inference-time reconstruction) in ONE launch of the
 * same instance: loss_dev[0] = mean_m |clamp(sdf_m) - clamp(target_dev[m])|, clamping to [-clamp_dist, clamp_dist],
 * and grad_latent_dev[256] = d loss / d latent; the upstream gradient is formed inside the kernel.
 * precision SDFB_PREC_BF16 or SDFB_PREC_FP16; sdf_dev optional. */
int sdfb_decoder_fit_loss_grad(sdfb_decoder* dec, const float* latent_dev, const float* xyz_dev, int64_t M,
                               const float* target_dev, float clamp_dist, float* grad_latent_dev,
                               float* loss_dev, float* sdf_dev, int precision, void* stream);

/* The same for a batch of shapes (reconstructing a test set): latents_dev [batch][256], xyz_dev
 * [batch][points_per_shape][3], target_dev [batch][points_per_shape] -> grad_latents_dev [batch][256], loss_dev [batch]. */
int sdfb_decoder_fit_loss_grad_batch(sdfb_decoder* dec, const float* latents_dev, const float* xyz_dev, int batch,
                                     int64_t points_per_shape, const float* target_dev, float clamp_dist,
                                     float* grad_latents_dev, float* loss_dev, int precision, void* stream);
/* The optimiser step of that fit: Adam on latents_dev [batch][256] with the gradient of the data term in grad_dev and the
 * regulariser reg |z|^2 added here (g = grad + 2 reg z); m_dev / v_dev [batch][256] are the moments (zero before step 1),
 * step = 1, 2, ... enters the bias correction.  loss_dev (optional, [batch]) receives += reg |z|^2 of the latents BEFORE the
 * update, i.e. the full loss at the point the gradient was taken.  One launch; every operation individually rounded
 * (betas are doubles so that 1 - beta and 1 - beta^step are formed the way the host expression they replace forms them). */
int sdfb_latent_adam_step(float* latents_dev, float* m_dev, float* v_dev, const float* grad_dev, float* loss_dev, int batch,
                          float lr, float reg, double beta1, double beta2, float adam_eps, int step, void* stream);

/* Host-buffer forms (what a plugin caller with CPU arrays uses): stage through
 * pinned memory owned by the context, run, copy back, synchronise. */
int sdfb_decode_grid_host(sdfb_decoder* dec, const float* latent_host, int res, int z0, int z1,
                          float* sdf_host, uint8_t* mask_host, int precision);
int sdfb_decode_points_host(sdfb_decoder* dec, const float* latent_host, const float* xyz_host,
                            int64_t M, float* sdf_host, int precision);

/* xyz of planes [z0,z1) of the res^3 grid -> xyz_dev [(z1-z0)*res*res][3] */
int sdfb_grid_points(int res, int z0, int z1, float* xyz_dev, void* stream);
/* A4 on an arbitrary [nz][ny][nx] field -> uint8 [(nz-1)(ny-1)(nx-1)] */
int sdfb_sign_change_mask(const float* sdf_dev, int nz, int ny, int nx, uint8_t* mask_dev,
                          void* stream);

/* ---- isosurface extraction (SURVEY.md 8f row N1): marching cubes over the sign-change cells ------
 * Field sdf_dev [nz][ny][nx] (C order), e.g. a decoded slab with ny = nx = res whose first plane is
 * plane z0 of the res^3 grid.  Output: a triangle soup [n][3 vertices][x, y, z] in cell order,
 * normals pointing from inside (sdf < 0) to outside; vertices interpolated from an edge's lower corner to
 * its upper corner, so cells sharing an edge emit identical bits (watertight, and bit-exact against
 * oracle/marching.py).  Two calls: count (classifies cells from the sign bit-planes - pass the words
 * sdfb_decode_grid_bits produced, or NULL to have them computed - scans, synchronises the stream and
 * returns the number of triangles), then generate into a caller-allocated buffer.  The workspace
 * (sdfb_mc_workspace_bytes) carries the classification from count to generate. */
int sdfb_mc_workspace_bytes(int nz, int ny, int nx, size_t* bytes);
int sdfb_mc_count(const float* sdf_dev, const uint32_t* sign_bits_dev, int nz, int ny, int nx, void* workspace_dev,
                  size_t workspace_bytes, int64_t* n_triangles_host, void* stream);
/* edge_keys_dev (optional, int64 [n][3]): the grid edge each vertex sits on, ((z*res + y)*res + x)*3 + axis of
 * the edge's lower node - equal for every cell sharing the edge, so unique(keys) welds the soup into an indexed mesh. */
int sdfb_mc_generate(const float* sdf_dev, int nz, int ny, int nx, int res, int z0, const void* workspace_dev,
                     float* triangles_dev, int64_t* edge_keys_dev, void* stream);

/* Welding the soup into an indexed mesh: a bitmap over the 3 res^3 grid edges marks the keys that occur, a scan ranks them,
 * and every triangle corner gets the rank of its key - vertices come out in ascending key order, each once.
 * count (synchronises): number of distinct vertices; fill: vertices_dev [n_vertices][3] and faces_dev [n_triangles][3] (int64). */
int sdfb_mc_weld_workspace_bytes(int res, size_t* bytes);
int sdfb_mc_weld_count(const int64_t* edge_keys_dev, int64_t n_triangles, int res, void* workspace_dev, size_t workspace_bytes,
                       int64_t* n_vertices_host, void* stream);
int sdfb_mc_weld_fill(const float* triangles_dev, const int64_t* edge_keys_dev, int64_t n_triangles, int res, const void* workspace_dev,
                      float* vertices_dev, int64_t* faces_dev, void* stream);

/* Synchronises `stream` and reports (once) a watchdog trip of any launch made on this context. */
int sdfb_decoder_check(sdfb_decoder* dec, void* stream);
/* Per-wait timeout of the in-kernel watchdog (default 2 s).  Test hook: a few nanoseconds make the next launch fail. */
int sdfb_decoder_set_timeout_ns(sdfb_decoder* dec, uint64_t timeout_ns);

/* Hierarchical sparse decode (SURVEY.md 8f row N2): decodes only where the surface can be and leaves what the dense
 * marching-cubes calls above consume - sdf_dense_dev [res^3] valid at every node of every cell the surface crosses
 * (elsewhere untouched), and sign_bits_dev, the COMPLETE sign bit-planes of the grid (ceil(res^3 / 32) + 1 words).
 * Two levels: corners of 8^3-cell blocks, kept if they differ in sign or come within L 8h sqrt(3)/2 of zero; inside the
 * kept blocks the lattice of 2^3-cell sub-blocks, same test with 2h; then the remaining nodes of the kept sub-blocks.
 * Every node is decoded at most once (node bitmaps compacted into query lists).  A node never decoded lies only in
 * discarded (sub-)blocks and inherits their constant sign.  lipschitz > 0: the bound L (field units per unit length);
 * 0: estimated - the largest difference quotient on the level-1 lattice times safety1 (e.g. 2), and the largest one
 * seen on either lattice times safety2 (e.g. 1.25) for level 2.  local_floor in (0, 1]: level 2 uses each 8^3 block's OWN
 * largest quotient (125 lattice samples per block) instead of the global one, but never less than local_floor times the
 * global one - a tighter, less conservative band (the field's steepest spot no longer widens the band everywhere);
 * 0 = global.  With a valid bound the marching-cubes output equals
 * the dense extraction's bit for bit, order included.  Synchronises `stream` (three counts are read back).
 * stats_host (optional, int64[8]): level-1 corners, kept blocks, level-2 lattice nodes, kept sub-blocks, remaining
 * nodes, total queries, and the two difference quotients x 1e6.  res <= 1024. */
int sdfb_decode_sparse_field(sdfb_decoder* dec, const float* latent_dev, int res, float lipschitz, float safety1, float safety2,
                             float local_floor, float* sdf_dense_dev, uint32_t* sign_bits_dev, int precision, int64_t* stats_host,
                             void* stream);

/* Debug/diagnostic: pre-activation (accumulator + bias, before ReLU) of
 * tensor-core pass `pass` (0..12) for the first 128 queries of a grid decode,
 * 128 x 256 floats.  Used by the parity tests to localise a failing layer. */
int sdfb_decode_debug_pass(sdfb_decoder* dec, const float* latent_dev, int res, int pass,
                           float* dump_dev, int precision, void* stream);
/* Elapsed device time of the last fused-decoder launch on this context, in
 * milliseconds, measured with CUDA events on the launching stream (blocks
 * until that launch has finished). */
int sdfb_decoder_last_kernel_ms(sdfb_decoder* dec, float* ms);

/* ---- latent DDPM (SURVEY.md 8a rows A5-A7) ------------------------------- */

int sdfb_ddpm_create(const float* params_host, size_t n_floats, int device, sdfb_ddpm** out);
int sdfb_ddpm_destroy(sdfb_ddpm* ddpm);

/* precision: SDFB_PREC_FP32 runs the FFMA kernels (one launch per layer and step); BF16 / FP16 run
 * ALL steps in one persistent tcgen05 kernel (all CTAs resident) (time embedding folded into a per-step
 * bias, denoiser MLP and posterior update fused; x stays fp32 and enters layer 0 as an exact
 * two-way 16-bit split).
 *
 * sample_latents(n): x_dev [n][256] holds x_T on entry and x_0 on return.
 * noise_dev [steps][n][256] is the explicit noise stream (noise[t] is consumed
 * at step t, noise[0] is ignored).  Runs t = steps-1 .. 0 of the 1000-step
 * linear-beta schedule with the x0-clipped posterior-mean update.
 * steps < 1000 TRUNCATES that schedule (it is not respaced: the coefficients stay those of the 1000-step
 * chain), which is what the short parity tests and the profilers want; samples of the trained distribution
 * need steps = 1000, or a respaced schedule (sdfb_ddpm_sample_ddim below).  1 <= steps <= 1000, anything else
 * is SDFB_E_INVALID. */
int sdfb_ddpm_sample(sdfb_ddpm* ddpm, float* x_dev, const float* noise_dev, int n, int steps,
                     int precision, void* stream);
/* one denoiser evaluation eps_hat(x, t) -> eps_dev [n][256] */
int sdfb_ddpm_denoise(sdfb_ddpm* ddpm, const float* x_dev, int t, int n, float* eps_dev,
                      int precision, void* stream);
int sdfb_ddpm_sample_host(sdfb_ddpm* ddpm, float* x_host, const float* noise_host, int n, int steps,
                          int precision);
/* Seeded sampling with IN-KERNEL noise (no [steps][n][256] stream in memory or over PCIe):
 * noise[t] = Philox4x32-10 normals, counter (column / 4, first_latent + latent, t, 0x53444642),
 * key = seed (csrc/philox.cuh; oracle/philox.py reproduces the stream on the CPU).  first_latent is
 * the global index of this call's latent 0: ranks that each sample a share of one batch draw exactly the
 * numbers a single call over the whole batch would.  gen_xT != 0: x_T is
 * generated too (row t = steps of the same stream) and x_dev is output only; otherwise x_dev holds
 * x_T on entry.  bf16/fp16: generated inside the fused kernel's update epilogue; fp32: the same
 * stream is materialised on the device first, then the FFMA sampler runs on it. */
int sdfb_ddpm_sample_philox(sdfb_ddpm* ddpm, float* x_dev, uint64_t seed, int64_t first_latent, int n, int steps,
                            int gen_xT, int precision, void* stream);
int sdfb_ddpm_sample_philox_host(sdfb_ddpm* ddpm, float* x_host, uint64_t seed, int64_t first_latent, int n, int steps,
                                 int gen_xT, int precision);
/* ---- respaced schedules: DDIM sampling and deterministic DDIM inversion ----
 * abar_t is the 1000-step linear-beta schedule above (fp64).  S steps visit tau_i = floor(i 1000 / S), i = 0 .. S-1
 * (S = 1000: every t).  Each step evaluates eps_hat at its timestep and applies
 *   x0 = clamp(sra x - srm1 eps_hat, -clamp, clamp);  x <- c1 x0 + c2 x [+ c3 eps_hat] [+ sigma z]
 * (products and sums rounded one by one in that order; the c3 term only when c3 != 0, the noise term only when sigma != 0).
 * Sampling, i = S-1 .. 0 from x at tau_i, with a = abar_{tau_i}, a' = abar_{tau_{i-1}} (1 for i = 0):
 *   sigma = eta sqrt((1 - a') / (1 - a)) sqrt(1 - a / a'),  c2 = sqrt(max(0, 1 - a' - sigma^2)) / sqrt(1 - a),
 *   c1 = sqrt(a') - c2 sqrt(a), c3 = 0, clamp = 1; eta = 1 at S = 1000 is the DDPM posterior of sdfb_ddpm_sample,
 *   eta = 0 is deterministic.  The last step (i = 0) has c1 = 1, c2 = sigma = 0.
 * Inversion, i = 0 .. S-1 from a clean x0 to x at tau_{S-1}, with a = abar_{tau_{i-1}} (1 for i = 0), a' = abar_{tau_i}:
 *   sra, srm1 of a, c1 = sqrt(a'), c2 = 0, c3 = sqrt(1 - a'), sigma = 0, clamp = +inf (x0 is not clamped).
 *
 * sdfb_ddim_schedule: host only, no device.  timesteps_host [steps] and coef_host [steps][8] = (sra, srm1, c1, c2, c3, sigma,
 * clamp, 0) receive the rows in execution order.  1 <= steps <= 1000 and 0 <= eta <= 1 (finite), else SDFB_E_INVALID
 * (inverse != 0: eta is checked but unused).  The entry points below run exactly these rows.
 *
 * Noise.  Explicit: noise_dev [steps][n][256], noise[i] is consumed at the step from tau_i (noise[0] is never read); it may be
 * NULL when eta = 0 (a NULL stream with eta > 0 is SDFB_E_INVALID).  Seeded: the Philox counter's step field is tau_i, so
 * DDIM at S = 1000, eta = 1 draws the numbers of sdfb_ddpm_sample_philox; gen_xT != 0 takes x_T from row t = 1000 of the
 * stream whatever S is (the same seed starts DDIM-S and the full 1000-step chain from the same x_T).  A step with sigma = 0
 * (every step at eta = 0) reads and generates no noise.
 * precision, the watchdog, the status mirror and sdfb_ddpm_last_kernel_ms behave as for sdfb_ddpm_sample; bf16 / fp16 run
 * all S steps in one launch of the same fused kernel.  x_dev holds x_T on entry and x_0 on return (invert: x0 on entry,
 * x at tau_{S-1} on return, in place). */
int sdfb_ddim_schedule(int steps, float eta, int inverse, int32_t* timesteps_host, float* coef_host);
int sdfb_ddpm_sample_ddim(sdfb_ddpm* ddpm, float* x_dev, const float* noise_dev, int n, int steps, float eta, int precision,
                          void* stream);
int sdfb_ddpm_sample_ddim_philox(sdfb_ddpm* ddpm, float* x_dev, uint64_t seed, int64_t first_latent, int n, int steps, float eta,
                                 int gen_xT, int precision, void* stream);
int sdfb_ddpm_invert_ddim(sdfb_ddpm* ddpm, float* x_dev, int n, int steps, int precision, void* stream);
/* The stream itself: normals of steps [t0, t1) for latents [first_latent, first_latent + n)
 * -> out_dev [(t1-t0)][n][256]. */
int sdfb_philox_normal(uint64_t seed, int64_t first_latent, int n, int t0, int t1, float* out_dev, void* stream);
/* Elapsed device time (ms) of the last fused (bf16/fp16) sampler launch on this context, CUDA
 * events on the launching stream; blocks until it has finished and reports a tripped watchdog. */
int sdfb_ddpm_last_kernel_ms(sdfb_ddpm* ddpm, float* ms);

int sdfb_ddpm_check(sdfb_ddpm* ddpm, void* stream);
int sdfb_ddpm_set_timeout_ns(sdfb_ddpm* ddpm, uint64_t timeout_ns);

/* ---- multi-GPU (SURVEY.md 8b row sdf_allgather_slabs, 8e): one process per GPU of one node -------------------
 * The path shards with no data-path collective (queries are independent); what is left is assembling the slabs of
 * BASELINE configs[4] on every rank.  A communicator wraps NCCL (resolved at run time: the libnccl.so.2 already in
 * the process, else the system's) and, for the overlapped path, a symmetric device buffer mapped into every rank
 * through CUDA IPC.
 *   sdfb_comm_unique_id : rank 0 fills a 128-byte id and hands it to the others by any means (MPI, a file, torch.distributed)
 *   sdfb_comm_create    : collective; ncclCommInitRank under the hood
 *   sdfb_comm_wrap      : use an existing ncclComm_t instead (not destroyed with the context) */
int sdfb_comm_unique_id(void* id_out /* 128 bytes */);
int sdfb_comm_create(const void* id, int world, int rank, int device, sdfb_comm** out);
int sdfb_comm_wrap(void* nccl_comm, int world, int rank, int device, sdfb_comm** out);
int sdfb_comm_destroy(sdfb_comm* comm);
int sdfb_comm_barrier(sdfb_comm* comm, void* stream);
/* In-place all-gather of equal-sized slabs: rank r's bytes_per_rank bytes sit at full_dev + r * bytes_per_rank
 * (ncclAllGather with sendbuff inside recvbuff); asynchronous on `stream`. */
int sdfb_allgather_slabs(sdfb_comm* comm, void* full_dev, size_t bytes_per_rank, void* stream);
/* BASELINE configs[4] in one call per rank: rank r decodes planes [r per, min((r+1) per, res)), per = ceil(res/world),
 * in sub-slabs of `sub_planes` planes (0 = automatic) into a symmetric buffer owned by `comm`, and pushes every
 * finished sub-slab into all peers' copies with the copy engines over NVLink while the next one is being decoded;
 * a rank barrier opens and closes the call.  On return (in `stream` order) *sdf_full_dev is the whole [res][res][res]
 * field on every rank.  want_mask: the sign-change mask, packed, as `world` blocks of *mask_words_per_rank words;
 * block r holds rank r's cell layers [r per, min((r+1) per, res-1)) from bit 0 (cell c of the block -> bit c & 31
 * of word c >> 5); the halo plane a block needs is decoded locally.  When per * (res-1)^2 is a multiple of 32 the
 * blocks concatenate to the global packing of sdfb_decode_grid_bits.  The buffers stay valid until the next sharded
 * decode on this communicator.  First use (and growth) allocates and exchanges the buffer: collective, synchronising. */
int sdfb_decode_grid_sharded(sdfb_decoder* dec, sdfb_comm* comm, const float* latent_dev, int res, int want_mask,
                             int sub_planes, int precision, float** sdf_full_dev, uint32_t** mask_bits_dev,
                             size_t* mask_words_per_rank, void* stream);

/* ---- training (SURVEY.md 8f row N4, second half) ---------------------------------------------------------------
 * The inference kernels keep activations on chip; a training step needs every layer's activations and deltas for
 * the weight gradients, so it runs layer by layer on a general tensor-core product (csrc/gemm_tc.cu: 16-bit
 * operands through TMA, fp32 accumulation in TMEM; the weight gradient dW = delta^T h contracts over the batch
 * rows of two row-major arrays, i.e. with MN-major operand descriptors), activations and deltas kept in 16 bits,
 * master weights, Adam moments and all reductions in fp32.
 *
 * DDPM denoiser training step: x_t = sqrt(abar_t) x0 + sqrt(1 - abar_t) eps per row (t_dev [n] in [0, 1000)),
 * loss = mean (eps_hat(x_t, t) - eps)^2, gradients of all weights and biases, Adam with bias correction (apply != 0;
 * apply == 0 only evaluates).  loss_dev [1]; grads_dev (optional): the gradient in the parameter blob's layout.
 * A trainer owns its copy of the parameters; sdfb_ddpm_trainer_get_params downloads them (synchronising), e.g. to
 * build a sampler from them with sdfb_ddpm_create.  precision: SDFB_PREC_BF16 or SDFB_PREC_FP16. */
int sdfb_ddpm_trainer_create(const float* params_host, size_t n_floats, int device, int precision, sdfb_ddpm_trainer** out);
int sdfb_ddpm_trainer_destroy(sdfb_ddpm_trainer* trainer);
int sdfb_ddpm_trainer_step(sdfb_ddpm_trainer* trainer, const float* x0_dev, const int32_t* t_dev, const float* eps_dev, int n,
                           float lr, float beta1, float beta2, float adam_eps, int apply, float* loss_dev, float* grads_dev,
                           void* stream);
int sdfb_ddpm_trainer_get_params(sdfb_ddpm_trainer* trainer, float* params_host);
/* Auto-decoder training step (DeepSDF): a batch of shapes, latents_dev [batch][256], xyz_dev [batch][points_per_shape][3],
 * target_dev [batch][points_per_shape]; loss = mean over all points of |clamp(sdf) - clamp(target)| (clamp to
 * [-clamp_dist, clamp_dist]); gradients of all nine layers' weights and biases (dW_l = delta_l^T a_l on the tensor pipe,
 * the head in fp32) and Adam on them (apply != 0).  The products run on the dense inputs [z | xyz] and [h3 | z | xyz] as
 * the oracle does (the latents differ per row, so nothing is folded).  grads_dev (optional): the gradient in the
 * decoder blob's layout; sdf_dev (optional, [batch * points_per_shape]): the forward values.  The latents' own gradient
 * is what sdfb_decoder_fit_loss_grad_batch returns.  At most 2^21 points per step (17 KiB of workspace per point). */
int sdfb_decoder_trainer_create(const float* params_host, size_t n_floats, int device, int precision, sdfb_decoder_trainer** out);
int sdfb_decoder_trainer_destroy(sdfb_decoder_trainer* trainer);
int sdfb_decoder_trainer_step(sdfb_decoder_trainer* trainer, const float* latents_dev, const float* xyz_dev, const float* target_dev,
                              int batch, int64_t points_per_shape, float clamp_dist, float lr, float beta1, float beta2,
                              float adam_eps, int apply, float* loss_dev, float* grads_dev, float* sdf_dev, void* stream);
int sdfb_decoder_trainer_get_params(sdfb_decoder_trainer* trainer, float* params_host);
/* Unit-test hook of the general product: out_dev [ksplit][M][N] fp32 partial sums of a . b^T (tn = 0: a [M][K], b [N][K])
 * or a^T . b (tn = 1: a [K][M], b [K][N]); row-major 16-bit inputs, leading dimensions in elements (multiples of 8);
 * bn = output tile width (64, 128, 256; N % bn == 0); tn: M % 64 == 0.  Runs on the current device; synchronises. */
int sdfb_gemm_selftest(const uint16_t* a_dev, int lda, const uint16_t* b_dev, int ldb, int M, int N, int K, int tn, int ksplit,
                       int bn, int precision, float* out_dev, void* stream);

/* ---- unit-test hook for the UMMA plumbing -------------------------------- */
/* D[128][256] (fp32) = A[128][64] * B[256][64]^T with A and B given as
 * row-major 16-bit arrays on the device (bf16 or fp16 per `precision`); the
 * kernel stages them into the 128B-swizzled smem layout itself. */
int sdfb_umma_selftest(const uint16_t* a_dev, const uint16_t* b_dev, float* d_dev, int precision,
                       void* stream);

/* Diagnostic: mean SM cycles per back-to-back tcgen05.mma (kind::f16 bf16, N=256, K=16;
 * M=128 for cta_group 1, M=256 per CTA pair for cta_group 2) over `grid` CTAs. */
int sdfb_umma_rate(int cta_group, int grid, int iters, int k_per_commit, int n_acc, int flags,
                   double* cycles_per_mma);

/* Diagnostic: bytes per SM cycle one CTA receives from L2 through the TMA unit (16 KiB pieces of a [rows][cols] 16-bit
 * tensor of `mib` MiB, 8 pieces in flight), over `grid` CTAs in clusters of `cluster` (grid a multiple of it).
 * mode 0: every CTA its own boxes (128 rows x 128 bytes, 128B swizzle); 1: the CTAs of a cluster load the same boxes;
 * 2: each box loaded once and multicast to the cluster; 3: own pieces as one 1-D bulk copy each; 4: as four 4 KiB copies;
 * 5: CTA pairs (cluster 2), own boxes with the .cta_group::2 form counted on the leader CTA's barrier;
 * 6: CTA pairs, plain loads counted on each CTA's own barrier, the peer forwards every completed stage to the leader.
 * issuers: 1, 2 or 4 warps issue in turn; uniform != 0: the issuing warps run their loop warp-uniformly with one elected
 * lane executing the TMA instructions, 0: only lane 0 runs the loop.  cols: 64 (contiguous boxes) or a multiple of 64.
 * out[0] = mean bytes/cycle/CTA, out[1] = slowest CTA's, out[2] = aggregate GB/s of the launch (event-timed). */
int sdfb_tma_ingest_rate(int grid, int cluster, int mode, int issuers, int uniform, int cols, int mib, int iters, double* out3);

#ifdef __cplusplus
}
#endif
#endif /* SDFB200_H_ */
