// Internal launcher declarations shared by the translation units of libsdfb200.
// (The public C ABI is include/sdfb200.h; nothing here is exported.)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sdfb {

// ---- model constants (SURVEY.md section 8a) --------------------------------
constexpr int kLatent = 256;
constexpr int kHid = 512;
constexpr int kSkipOut = 253;          // layer-3 width: 512 - 259
constexpr int kDecIn = 259;
constexpr int kDecLayers = 9;
constexpr long long kDecParamFloats = 1835520LL + 3838LL;

constexpr int kDdpmT = 1000;
constexpr int kDdpmLatent = 256;
constexpr int kDdpmTemb = 256;
constexpr int kDdpmHid = 1024;
constexpr long long kDdpmParamFloats =
    (512LL * 1024 + 1024) + 3 * (1024LL * 1024 + 1024) + (1024LL * 256 + 256);

// ---- fused tensor-core decoder (fused_decoder.cu) --------------------------
//
// One CTA PAIR owns a tile of 256 queries (128 per CTA) and carries it through all
// layers; the activations never leave the SMs.  Per tile the tensor core runs 13 "passes"
// (a pass = one N=256 half of a layer's output, accumulated over that layer's
// K in 64-wide chunks):
//   pass  0, 1 : L1 halves      pass  5, 6 : L4 halves (K = 256: [h3 | xyz])
//   pass  2, 3 : L2 halves      pass  7.. 12 : L5, L6, L7 halves
//   pass  4    : L3 (N = 253 padded to 256)
// The weight stream is the concatenation of the 96 (pass, k-chunk) blocks in
// exactly that order; block = 256 rows x 64 k-elements, 16-bit, stored as the
// 128B-swizzled shared-memory image (row r at r*128 B, 16-byte unit u at
// position u ^ (r & 7)), so one linear bulk copy lands an MMA-ready operand.
constexpr int kTileM = 128;
constexpr int kChunkK = 64;
constexpr int kBlockRows = 256;
constexpr int kBlockBytes = kBlockRows * kChunkK * 2;   // 32 KiB
constexpr int kPasses = 13;
constexpr int kBlocksPerTile = 96;
// Forward + backward (latent gradient) kernel: 13 more passes against the TRANSPOSED weights (block rows =
// the layer's INPUT features, k = its OUTPUT features), appended to the same stream:
//   pass 13, 14 : delta6 = delta7 W7 (halves)   pass 19     : delta3 = delta4 W4[:, :253] (N = 253 -> 256)
//   pass 15, 16 : delta5 = delta6 W6            pass 20, 21 : delta2 = delta3 W3 (K = 253 -> 256: 4 chunks)
//   pass 17, 18 : delta4 = delta5 W5            pass 22, 23 : delta1;   pass 24, 25 : delta0 (column sums only)
constexpr int kPassesBwd = 26;
constexpr int kBlocksPerTileBwd = 192;
constexpr int kAChunkBytes = kTileM * kChunkK * 2;      // 16 KiB: one 64-wide slice of activations
constexpr int kAChunks = 8;

// fp32 constant block read by the epilogue warps (one per context, the two
// folded bias rows are rewritten per latent by fold_latent_kernel)
struct DecConsts {
  float4 l0[kHid];        // (W0[n][256..258], b0[n] + W0[n][:256] . z)
  float bias[7][kHid];    // layers 1..7; row 2 (L3) zero-padded past 253; row 3 (L4) = b4 + W4[n][253:509] . z
  float head[kHid];       // W8[0][:]
  float head_b[4];        // b8, pad
};

struct DecodeParams {
  const uint8_t* wstream;      // kBlocksPerTile blocks of kBlockBytes
  const DecConsts* consts;
  const float* xyz;            // points mode: [M][3]; nullptr in grid mode
  float* out;                  // [M]
  unsigned int* signs;         // optional [ceil(M / 32)]: bit (m & 31) of word m >> 5 = (out[m] < 0)
  long long M;                 // number of queries in this launch
  long long q0;                // grid mode: global index of query 0 (= z0*res*res)
  int res;
  unsigned int* status;        // watchdog status word (0 = ok)
  unsigned int* status_host;   // its mirror in mapped pinned host memory (optional)
  float* dump;                 // debug: 128x256 pre-activations of pass `dump_pass`, tile 0
  int dump_pass;
  unsigned long long timeout_ns;
  long long* prof;             // optional [grid][3 roles][8]: blocked cycles per wait class (diagnostics)
  unsigned int debug_flags;    // bit0: producer skips the weight copies (timing experiment; results are garbage)
                               // bit1: producer exits at once (test hook: every consumer wait runs into the watchdog)
                               // bit2: hidden-pass epilogues only run the barrier protocol; bit3: they convert but do not store
                               //       (timing experiments, results are garbage)
  // forward + backward kernel only (`bwd` selects it; `out` is then optional, `signs` unused)
  const float* dLdy;           // [M] upstream gradient d loss / d sdf
  const unsigned int* dLdy_amax;   // bits of max |dLdy| (launch_abs_max): the kernel works on dLdy * 2^-vjp_scale_exponent
  // loss mode (target != nullptr, dLdy unused): the kernel forms the upstream gradient of the clamped-L1 fitting loss
  // itself, dLdy[m] = sign(clamp(sdf_m) - clamp(target_m)) [|sdf_m| < clamp] (the 1 / M is applied by the finish
  // kernel), and adds up sum_m |clamp(sdf_m) - clamp(target_m)| per warp
  const float* target;         // [M]
  float clamp;
  float* loss_partial;         // [grid * 4]
  int bwd;                     // 1 selects the forward + backward instance
  uint32_t* mask_scratch;      // [grid][6 layers + 2][16 words][128 rows]: ReLU masks of the tile in flight (layers 1-6; h0's, two tiles deep)
  float* colsum;               // [grid * 4][1024]: per-warp-quadrant column sums of delta0 (512) | delta4 (512)
};

cudaError_t fused_decoder_init();   // opt in to the large dynamic shared memory carve-out
cudaError_t tc_common_init();
cudaError_t make_wstream_tensor_map(const void* wstream, void* tmap_out /* 128 B, 64-byte aligned */);
cudaError_t launch_fused_decoder(const DecodeParams& p, const void* tmap, bool fp16, int num_sms,
                                 cudaStream_t stream);

// Unit test of the UMMA plumbing: D[128][256] = A[128][64] * B[256][64]^T, row-major 16-bit inputs.
cudaError_t launch_umma_selftest(const uint16_t* a, const uint16_t* b, float* d, unsigned int* status,
                                 bool fp16, cudaStream_t stream);

// Diagnostic: cycles per back-to-back tcgen05.mma (umma_rate.cu).
cudaError_t launch_tma_ingest(const void* tensor, int cols, int rows, int grid, int csize, int mode, int issuers, int uniform, int iters,
                              long long* out_dev, cudaStream_t stream);
cudaError_t launch_umma_rate(int cg, int grid, int iters, int k_per_commit, int n_acc, int flags, long long* out_dev,
                             cudaStream_t stream);

// Per-latent fold: consts->l0[n].w and consts->bias[3][n] from the fp32 parameters and z.
cudaError_t launch_fold_latent(const float* W0, const float* b0, const float* W4, const float* b4,
                               const float* z, DecConsts* consts, cudaStream_t stream);

// ---- fused DDPM sampler (ddpm_step.cu) --------------------------------------
//
// One persistent cooperative kernel runs `steps` denoiser evaluations + posterior updates.
// Every layer is cut into pair tiles (256 latents x BN output features, cta_group::2) spread
// over all CTA pairs; a tile waits only for the CTAs that share its 256 latents.
//   weights     : [rows][64] 16-bit, 128-byte rows stored PRE-SWIZZLED (16-byte unit u of row r
//                 at u ^ (r & 7)) so an un-swizzled TMA box lands an MMA-ready K-major operand:
//                 layer 0: 4 k-chunks x 1024 rows (the latent half of W0; the [x_hi | x_lo] operand
//                 reuses chunk k & 3), layers 1-3: 16 x 1024 rows each, layer 4: 16 x 256 rows
//   activations : row-major [n_pad][kDdpmActCols] 16-bit: [x_hi | x_lo] (512), hidden buffer 0
//                 (1024), hidden buffer 1 (1024); moved with 128B-swizzling TMA boxes of 64 x 128
constexpr int kDdpmW0Rows = 4 * 1024;
constexpr int kDdpmWHidRows = 16 * 1024;
constexpr int kDdpmW4Rows = 16 * 256;
constexpr int kDdpmWRows = kDdpmW0Rows + 3 * kDdpmWHidRows + kDdpmW4Rows;   // 57,344 rows of 128 B = 7 MiB
constexpr int kDdpmMaxStages = 8;
constexpr int kDdpmActCols = 512 + 1024 + 1024;
constexpr int kDdpmOutTile = 64;          // output-layer tile width (fixed)

// One row of a sampler schedule, in execution order.  The update of a step is
//   x0 = clamp(sra x - srm1 eps, -clamp, clamp);  x <- c1 x0 + c2 x [+ c3 eps] [+ sigma noise]
// (every product and sum rounded on its own; the c3 term only when c3 != 0, the noise term only when sigma != 0).
// DDPM: c3 = 0, clamp = 1, noise plane = t.  DDIM sampling: plane = step index.  DDIM inversion: c3 != 0, sigma = 0,
// clamp = +inf.
struct DdpmStep {
  float coef[8];           // sra, srm1, c1, c2, c3, sigma, clamp, 0   (the row format of sdfb_ddim_schedule)
  int t;                   // timestep: the tb0 row and the Philox counter's step field
  int plane;               // plane of the explicit noise stream
  int pad[2];
};
static_assert(sizeof(DdpmStep) == 48, "DdpmStep is read as three 16-byte vectors");

struct DdpmParams {
  const float* tb0;        // [1000][1024]: b0 + W0[:, 256:] temb(t)
  const float* bias;       // [3][1024] (layers 1-3) then [256] (layer 4)
  const DdpmStep* sched;   // [steps]: the rows of this call, in execution order
  int eps_mode;            // 1: a single denoiser evaluation, eps_hat is stored through tm_x (no update)
  int n;
  int pair_m_tiles;        // ceil(n / 256)
  int steps;               // steps to run: sched[0], sched[1], ...
  int bn_h;                // output-tile width of the hidden layers (256, 128 or - small batches - 64)
  int nstages;
  int cluster8;            // 1: a cluster = the pair tiles of one latent group (one tile per pair and layer): the group barrier
                           // is an mbarrier in every member instead of a counter in L2
  int cluster_ctas;        // CTAs of such a cluster: 8 (four pairs, bn_h = 256) or 16 (eight pairs, bn_h = 128); 0 without
  int philox;              // 1: noise[t] is generated in the kernel (Philox4x32-10, csrc/philox.cuh) instead of read through tm_nz
  unsigned long long seed;
  unsigned int first_latent;   // global index of latent 0 of this call in the Philox counters (sharded sampling)
  unsigned int flags;      // experiments: bit0 no consumer-side proxy fence, bit1 relaxed (not release) barrier arrival
  unsigned int* counter;   // [pair_m_tiles] barrier counters, one per group of pair tiles that share 256 latents (zeroed before the launch)
  unsigned int* status;
  unsigned int* status_host;   // mirror of `status` in mapped pinned host memory (optional)
  unsigned long long timeout_ns;
  long long* prof;         // optional diagnostics: [prof_sms][3 roles][8] blocked cycles per wait class + an event trace
  int prof_sms;            // SM count the profile buffer was sized for
};

// the five tensor maps of a launch (128 B each, 64-byte aligned)
struct DdpmMaps {
  alignas(64) unsigned char act[128];   // activations, 16-bit, box 64 x 128, SWIZZLE_128B
  alignas(64) unsigned char wh[128];    // weights, box 64 x bn_h / 2, no swizzle
  alignas(64) unsigned char wo[128];    // weights, box 64 x 32
  alignas(64) unsigned char x[128];     // fp32 state [n][256] (eps_mode: the eps output), box 32 x 128, SWIZZLE_128B
  alignas(64) unsigned char nz[128];    // fp32 noise [planes][n][256], box 32 x 128 x 1, SWIZZLE_128B
};

cudaError_t ddpm_step_init();
// generic tiled tensor map: `rank` dims (innermost first), strides in bytes for dims 1.., elem_bytes 2 or 4
cudaError_t make_tensor_map(void* tmap_out, const void* base, int elem_bytes, int rank, const unsigned long long* dims,
                            const unsigned long long* strides_bytes, const unsigned* box, bool swizzle128);
// x [n][256] fp32 -> [x_hi | x_lo] columns of the activation buffer (rows >= n zero)
cudaError_t launch_ddpm_split(const float* x, int n, int n_pad, uint16_t* act, bool fp16, cudaStream_t stream);
cudaError_t launch_ddpm_sample(const DdpmParams& p, const DdpmMaps& maps, bool fp16, int num_sms, cudaStream_t stream);
// how many 8-CTA clusters of the sampler kernel can be resident at once (0 if the query fails)
int ddpm_max_clusters8(int bn_h, int nstages, bool fp16);
int ddpm_max_clusters16(int bn_h, int nstages, bool fp16);
// Philox normals of steps [t0, t1) for latents [first_latent, first_latent + n) -> out [(t1 - t0)][n][256]
cudaError_t launch_philox_normal(unsigned long long seed, unsigned int first_latent, int n, int t0, int t1, float* out,
                                 cudaStream_t stream);

// ---- general tensor-core product for the training steps (gemm_tc.cu) ---------------------------------------------
enum : int { kGemmEpiF32 = 0, kGemmEpiBiasReluLowp = 1, kGemmEpiMaskLowp = 2 };
struct GemmParams {
  int M, N, K;                 // output C[M][N]; contraction length K
  int bn;                      // output tile width: 64, 128 or 256 (N % bn == 0)
  int ksplit;                  // K is cut into `ksplit` ranges; range s accumulates into out_f32 + s * split_stride
  int epi;                     // kGemmEpi*: what happens to alpha * acc (+ bias) before it is stored
  float alpha;
  const float* bias;           // [N] or nullptr
  const uint16_t* mask_h;      // kGemmEpiMaskLowp: forward activations [M][ldh], the value is kept where they are > 0
  int ldh;
  float* out_f32;              // optional fp32 output [M][ldo_f32] (kGemmEpiBiasReluLowp: the pre-activation unless f32_post_relu)
  int ldo_f32;
  long long split_stride;      // elements between the partial outputs of consecutive k-ranges
  int f32_post_relu;
  uint16_t* out_lowp;          // optional 16-bit output [M][ldo_lowp] (rectified for kGemmEpiBiasReluLowp)
  int ldo_lowp;
  unsigned int* status;        // watchdog status word + host mirror
  unsigned int* status_host;
  unsigned long long timeout_ns;
};
cudaError_t gemm_tc_init();
cudaError_t launch_gemm_tc(const GemmParams& p, const uint16_t* a, int lda, const uint16_t* b, int ldb, bool tn, bool fp16,
                           int num_sms, cudaStream_t stream);

// ---- training helpers (train_kernels.cu) ------------------------------------------------------------------------------
// x_t = sa[t] x0 + sb[t] eps per row -> in0 [n][512] 16-bit = [x_t | temb(t_row)] (temb table [1000][256] fp32)
cudaError_t launch_ddpm_train_prep(const float* x0, const float* eps, const int* t, const float* coef_ab /* [1000][2] */,
                                   const float* temb, int n, uint16_t* in0, bool fp16, cudaStream_t st);
// residual d = eps_hat - eps -> 16-bit [n][256]; loss_partial[block] = sum d^2 (fixed order)
cudaError_t launch_ddpm_train_residual(const float* eps_hat, const float* eps, int n, uint16_t* d_lowp, float* loss_partial,
                                       int* nblocks, bool fp16, cudaStream_t st);
// out[j] = scale * sum_m D[m][j], D 16-bit [M][ld] (deterministic: row slabs in parallel, partial sums added in slab order, fp32);
// scratch: kColsumSlabs * N floats ([slab][N] partial sums; out = nullptr: left there for the caller, *nslabs_out of them)
constexpr int kColsumSlabs = 128;
cudaError_t launch_colsum_lowp(const uint16_t* D, long long M, int ld, int N, float scale, float* out, float* scratch, bool fp16,
                               cudaStream_t st, int* nslabs_out = nullptr);
// fused Adam over one parameter tensor: g = scale * sum_{s < nparts} grad[s * part_stride + i]; updates master fp32 weights and
// moments in place and refreshes the 16-bit copies W [rows][ldw] and W^T [cols][ldwt] (either may be null; rows x cols = the
// tensor's shape, cols = 1 for a bias with both copies null).  grad_out (optional): receives g.
struct AdamParams { float lr, beta1, beta2, eps, bias_corr1, bias_corr2; };
cudaError_t launch_adam_update(float* w, float* m, float* v, const float* grad, int nparts, long long part_stride, int ld_grad,
                               float scale, int rows, int cols, const AdamParams& a, uint16_t* w_lowp, int ldw, uint16_t* wt_lowp,
                               int ldwt, float* grad_out, bool fp16, bool apply, cudaStream_t st);
cudaError_t launch_latent_adam(float* z, float* m, float* v, const float* grad, float* loss, int batch, int dim, float lr, float reg,
                               double beta1, double beta2, float eps, int step, cudaStream_t st);
cudaError_t launch_sum_loss(const float* partial, int n, float scale, float* loss_out, cudaStream_t st);
// fp32 [rows][cols] (leading dimension ld) -> 16-bit copy [rows][ldw] and transposed copy [cols][ldwt] (either may be null)
cudaError_t launch_lowp_copies(const float* w, int ld, int rows, int cols, uint16_t* w_lowp, int ldw, uint16_t* wt_lowp, int ldwt,
                               bool fp16, cudaStream_t st);

// decoder training: input rows [z_shape | xyz | 0] into columns [col0, col0 + ncols) of a 16-bit matrix; head forward + loss terms +
// delta7; head gradients (out[0..511] = dW8, out[512] = db8)
cudaError_t launch_dec_train_input(const float* latents, const float* xyz, long long M, long long per_shape, int ld, int col0, int ncols,
                                   uint16_t* out, bool fp16, cudaStream_t st);
cudaError_t launch_dec_train_head(const uint16_t* a8, const float* w8, const float* b8, const float* target, float clamp, long long M,
                                  float* y, float* d8, uint16_t* delta7, float* loss_partial, int* nblocks, bool fp16, cudaStream_t st);
cudaError_t launch_dec_train_head_grad(const uint16_t* a8, const float* d8, long long M, float scale, float* out, float* scratch, bool fp16,
                                       cudaStream_t st);

// ---- fp32 SIMT kernels (fp32_kernels.cu) -----------------------------------
// C[M,N] = act(A[M,K] * W[N,K]^T + bias[N]); row-major, leading dims in elements.
cudaError_t launch_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias,
                              float* C, int ldc, long long M, int N, int K, bool relu,
                              cudaStream_t stream);
// out[m] = tanh(dot(H[m,:K], w) + b)
cudaError_t launch_head_tanh_f32(const float* H, int ldh, const float* w, const float* b, float* out,
                                 long long M, int K, cudaStream_t stream);
// backward pieces of the fp32 path (vector-Jacobian product w.r.t. the latent, SURVEY.md 8f row N4)
// C[M,K] = (A[M,N] * W[N,K]) .* (H[M,K] > 0)
cudaError_t launch_linear_bwd_f32(const float* A, int lda, const float* W, int ldw, const float* H, int ldh, float* C,
                                  int ldc, long long M, int N, int K, cudaStream_t stream);
cudaError_t launch_head_bwd_f32(const float* dLdy, const float* y, const float* w8, const float* H7, float* D, long long M,
                                cudaStream_t stream);
cudaError_t launch_colsum_f32(const float* D, long long M, float* partial, int half, cudaStream_t stream);
// (reduces the partial rows in place into row 0 first)
cudaError_t launch_vjp_finish(float* partial, int nblk, const float* W0, const float* W4, float* grad,
                              cudaStream_t stream, const unsigned int* amax_bits = nullptr,
                              const float* loss_partial = nullptr, float inv_m = 1.f, float* loss_out = nullptr);
// out[0] = bits of max |v[i]| (0 for an empty or all-zero v)
cudaError_t launch_abs_max(const float* v, long long M, unsigned int* out, cudaStream_t stream);
// Tensor-core backward: the upstream gradient is scaled by 2^-e, e = vjp_scale_exponent(max |dLdy|), so that the
// deltas sit in the same range whatever the caller's loss scale (fp16 deltas would otherwise underflow), and the
// result is scaled back by 2^e.  amax = m 2^e with m in [0.5, 1); 0 for amax = 0 or non-finite.
__host__ __device__ inline int vjp_scale_exponent(float amax) {
  if (!(amax > 0.f) || amax > 3.0e38f) return 0;
  int e = 0;
  frexpf(amax, &e);
  return e < -100 ? -100 : (e > 100 ? 100 : e);
}
// xyz of queries [q0, q0+M) of the res^3 grid -> X[M,3] and (optionally) cols 253..255 of S[M,256]
cudaError_t launch_grid_xyz(int res, long long q0, long long M, float* X, float* S,
                            cudaStream_t stream);
// copy xyz[M,3] into cols 253..255 of S[M,256]
cudaError_t launch_scatter_xyz(const float* xyz, long long M, float* S, cudaStream_t stream);
// y[j] = b[j] + sum_k W[j*ldw + col0 + k] * z[k], k < K   (one warp per output)
cudaError_t launch_fold_bias(const float* W, int ldw, int col0, const float* b, const float* z,
                             int K, int N, float* y, cudaStream_t stream);
cudaError_t launch_sign_change_mask(const float* sdf, int nz, int ny, int nx, unsigned char* mask,
                                    cudaStream_t stream);
// bits[m >> 5] bit (m & 31) = (sdf[m] < 0), m < M   (the fused decoder writes the same words itself)
cudaError_t launch_sign_bits(const float* sdf, long long M, unsigned int* bits, cudaStream_t stream);
// A4 from the sign bits of an [nz][ny][nx] field: uint8 per cell and / or packed (cell c -> bit c & 31 of word c >> 5)
// (`rowmask`: scratch of mask_rows_words() words; `bits` must be readable one word past its last word)
size_t mask_rows_words(int nz, int ny, int nx);
cudaError_t launch_mask_from_bits(const unsigned int* bits, int nz, int ny, int nx, unsigned char* mask_u8,
                                  unsigned int* mask_bits, unsigned int* rowmask, cudaStream_t stream);
// the update of one DdpmStep row (coef = its first 8 floats): noise is used only when sigma != 0
cudaError_t launch_ddpm_update(float* x, const float* eps, const float* noise, long long count, const float* coef,
                               cudaStream_t stream);

// ---- marching cubes (marching.cu) --------------------------------------------
size_t mc_weld_workspace_bytes(long long key_range);
cudaError_t launch_mc_weld_count(const long long* keys, long long n_keys, long long key_range, void* workspace, int* count_dev,
                                 cudaStream_t stream);
cudaError_t launch_mc_weld_fill(const float* tris, const long long* keys, long long n_keys, long long key_range, const void* workspace,
                                float* verts, long long* faces, cudaStream_t stream);
// A field to extract from: a dense [nz][ny][nx] slab whose first plane is plane z0 of the res^3 grid.
struct McGeom {
  int nz, ny, nx, res, z0;
  long long total_cells, total_nodes;
};
inline McGeom mc_dense_geom(int nz, int ny, int nx, int res, int z0) {
  return McGeom{nz, ny, nx, res, z0, static_cast<long long>(nz - 1) * (ny - 1) * (nx - 1), static_cast<long long>(nz) * ny * nx};
}
size_t mc_scan_temp_bytes(long long groups);
cudaError_t launch_mc_count_scan(const unsigned int* bits, const McGeom& g, unsigned int* group_tris, void* temp,
                                 size_t temp_bytes, cudaStream_t stream);
// keys (optional, [n_tri * 3]): the grid edge of every emitted vertex, ((z res + y) res + x) * 3 + axis of its lower node
cudaError_t launch_mc_generate(const float* sdf, const unsigned int* bits, const unsigned int* group_first, const McGeom& g,
                               float* tris, long long* keys, cudaStream_t stream);

// ---- hierarchical sparse decode (sparse.cu) -----------------------------------------------------------------------
cudaError_t launch_corner_nodes(int res, int B, int nb, unsigned int* idx, cudaStream_t st);
cudaError_t launch_node_points(int res, const unsigned int* idx, long long n, float* xyz, cudaStream_t st);
cudaError_t launch_scatter(const unsigned int* idx, const float* vals, long long n, float* dense, cudaStream_t st);
cudaError_t launch_corner_lipschitz(const float* cs, int res, int B, int nb, unsigned int* out_bits, cudaStream_t st);
cudaError_t launch_select_blocks_bits(const float* cs, int nb, float tau, unsigned int* keep, cudaStream_t st);
cudaError_t launch_mark_sub_corners(int res, int B1, int B2, int nb1, const int* blocks, long long nblk, unsigned int* need,
                                    cudaStream_t st);
cudaError_t launch_sub_lipschitz(int res, int B1, int B2, int nb1, const int* blocks, long long nblk, const float* dense,
                                 unsigned int* out_bits, unsigned int* per_block, cudaStream_t st);
cudaError_t launch_select_sub_blocks(int res, int B1, int B2, int nb1, const int* blocks, long long nblk, const float* dense,
                                     const unsigned int* lip_bits, float lip_given_per_node, float safety,
                                     const unsigned int* per_block, float local_floor, unsigned int* need,
                                     unsigned long long* kept, cudaStream_t st);
cudaError_t launch_andnot(unsigned int* a, const unsigned int* b, long long words, cudaStream_t st);
long long bitmap_scan_tiles(long long words);
cudaError_t launch_bitmap_count(const unsigned int* bits, long long words, unsigned int* tile_sums, cudaStream_t st);
cudaError_t launch_bitmap_emit(const unsigned int* bits, long long words, const unsigned int* tile_offsets, unsigned int* out,
                               cudaStream_t st);
cudaError_t launch_fill_signs(int res, int B1, int B2, int nb1, const float* dense, const unsigned int* need1,
                              const unsigned int* need2, const float* cs, unsigned int* signs, cudaStream_t st);

// A1: node coordinate, one correctly rounded divide of two exact integers.
__host__ __device__ inline float axis_coord_num(int i, int res) { return static_cast<float>(2 * i - (res - 1)); }

}  // namespace sdfb
