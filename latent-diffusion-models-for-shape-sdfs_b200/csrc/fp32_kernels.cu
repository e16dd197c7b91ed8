// fp32 SIMT kernels: the true-fp32 (FFMA) path that carries the 1e-5 / 1e-4
// parity criteria, plus the small HBM-bound helpers (grid coordinates,
// sign-change mask, latent fold, DDPM update).  Tensor cores are deliberately
// not used here: TF32 has a 10-bit mantissa and cannot meet 1e-5
// (SURVEY.md section 7, H2).
#include "kernels.h"

namespace sdfb {

namespace {

constexpr int BM = 64, BN = 64, BK = 16;

// C = act(A W^T + bias).  64x64 block tile, 16-deep K slab, 256 threads, 4x4 per thread.
// Plain sequential-K FMA accumulation keeps the result within ~1e-6 of fp64.
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ A, int lda,
                                                         const float* __restrict__ W, int ldw,
                                                         const float* __restrict__ bias,
                                                         float* __restrict__ C, int ldc,
                                                         long long M, int N, int K, int relu) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Ws[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = static_cast<long long>(blockIdx.x) * BM;
  const int n0 = blockIdx.y * BN;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;
      const int r = e >> 4, kk = e & 15;
      const long long m = m0 + r;
      const int k = k0 + kk;
      As[kk][r] = (m < M && k < K) ? A[m * lda + k] : 0.f;
      const int n = n0 + r;
      Ws[kk][r] = (n < N && k < K) ? W[static_cast<long long>(n) * ldw + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + (bias ? bias[n] : 0.f);
      if (relu) v = fmaxf(v, 0.f);
      C[m * ldc + n] = v;
    }
  }
}

// Backward of a linear layer w.r.t. its input, fused with the ReLU mask of the layer below:
// C[M,K] = (A[M,N] * W[N,K]) .* (H[M,K] > 0)     (W row-major [N][K], i.e. NOT transposed; H = stored activations)
__global__ void __launch_bounds__(256) linear_bwd_f32_kernel(const float* __restrict__ A, int lda,
                                                             const float* __restrict__ W, int ldw,
                                                             const float* __restrict__ H, int ldh,
                                                             float* __restrict__ C, int ldc, long long M, int N, int K) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Ws[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = static_cast<long long>(blockIdx.x) * BM;
  const int k0 = blockIdx.y * BN;
  float acc[4][4] = {};
  for (int n0 = 0; n0 < N; n0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = tid + 256 * i;
      {
        const int r = e >> 4, nn = e & 15;             // A tile: 64 rows x 16 reduction indices
        const long long m = m0 + r;
        As[nn][r] = (m < M && n0 + nn < N) ? A[m * lda + n0 + nn] : 0.f;
      }
      {
        const int nn = e >> 6, c = e & 63;             // W tile: 16 reduction indices x 64 output columns (coalesced)
        Ws[nn][c] = (n0 + nn < N && k0 + c < K) ? W[static_cast<long long>(n0 + nn) * ldw + k0 + c] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int nn = 0; nn < BK; ++nn) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[nn][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[nn][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= K) continue;
      C[m * ldc + k] = H[m * ldh + k] > 0.f ? acc[i][j] : 0.f;
    }
  }
}

// delta7[m,k] = dLdy[m] (1 - y[m]^2) w8[k] [h7[m,k] > 0]
__global__ void head_bwd_f32_kernel(const float* __restrict__ dLdy, const float* __restrict__ y,
                                    const float* __restrict__ w8, const float* __restrict__ H7, float* __restrict__ D,
                                    long long M) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M * 512) return;
  const long long m = i >> 9;
  const int k = static_cast<int>(i & 511);
  const float yy = y[m];
  const float g = dLdy[m] * (1.f - yy * yy);
  D[i] = H7[i] > 0.f ? g * w8[k] : 0.f;
}

// partial[b][half * 512 + col] = sum over the block's 256 rows of D[m][col]   (fixed order: deterministic)
__global__ void colsum_f32_kernel(const float* __restrict__ D, long long M, float* __restrict__ partial, int half) {
  const long long r0 = static_cast<long long>(blockIdx.x) * 256;
  const long long r1 = r0 + 256 < M ? r0 + 256 : M;
  float s0 = 0.f, s1 = 0.f;
  for (long long m = r0; m < r1; ++m) {
    s0 += D[m * 512 + threadIdx.x];
    s1 += D[m * 512 + 256 + threadIdx.x];
  }
  float* dst = partial + static_cast<long long>(blockIdx.x) * 1024 + half * 512;
  dst[threadIdx.x] = s0;
  dst[256 + threadIdx.x] = s1;
}

// grad[k] = sum_n s0[n] W0[n][k] + sum_n s4[n] W4[n][253 + k], s0 / s4 = column sums over all partial blocks
// max |v| as float bits (non-negative floats order like unsigned integers); `out` starts at zero
__global__ void abs_max_kernel(const float* __restrict__ v, long long M, unsigned int* __restrict__ out) {
  float a = 0.f;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < M;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    a = fmaxf(a, fabsf(v[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, o));
  if ((threadIdx.x & 31) == 0 && a > 0.f) atomicMax(out, __float_as_uint(a));
}

// Column sums of the nblk partial rows [nblk][1024], in place into row 0: block b owns columns [32 b, 32 b + 32)
// (nobody else touches them); 8 row groups per block, combined in a fixed order.
__global__ void vjp_colsum_reduce_kernel(float* __restrict__ partial, int nblk) {
  __shared__ float s[8][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), g = threadIdx.x >> 5;
  float a = 0.f;
  for (int r = g; r < nblk; r += 8) a += partial[static_cast<long long>(r) * 1024 + c];
  s[g][threadIdx.x & 31] = a;
  __syncthreads();
  if (g == 0) {
    float t = s[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += s[i][threadIdx.x];
    partial[c] = t;
  }
}

// grad[k] = sum_n cs0[n] W0[n][k] + sum_n cs4[n] W4[n][253 + k] from the reduced column sums (1024 threads: 256
// outputs x 4 quarters of n, combined in a fixed order).
// `amax_bits` (tensor-core path): the kernel ran on dLdy * 2^-e with 2^e the power of two just above
// max |dLdy| (vjp_scale_exponent): undo it here, exactly.
__global__ void __launch_bounds__(1024) vjp_finish_kernel(const float* __restrict__ reduced, int nblk, const float* __restrict__ W0,
                                                          const float* __restrict__ W4, float* __restrict__ grad,
                                                          const unsigned int* __restrict__ amax_bits,
                                                          const float* __restrict__ loss_partial, float inv_m,
                                                          float* __restrict__ loss_out) {
  __shared__ float s[1024];
  __shared__ float part[4][256];
  s[threadIdx.x] = reduced[threadIdx.x];
  __syncthreads();
  const int k = threadIdx.x & 255, q = threadIdx.x >> 8;
  float g = 0.f;
  if (q < 2) {
    for (int n = 256 * q; n < 256 * q + 256; ++n) g = fmaf(s[n], W0[n * 259 + k], g);
  } else {
    for (int n = 256 * (q - 2); n < 256 * (q - 2) + 256; ++n) g = fmaf(s[512 + n], W4[n * 512 + 253 + k], g);
  }
  part[q][k] = g;
  __syncthreads();
  if (q == 0) {
    g = ((part[0][k] + part[1][k]) + part[2][k]) + part[3][k];
    if (amax_bits != nullptr) g = ldexpf(g, vjp_scale_exponent(__uint_as_float(*amax_bits)));
    grad[k] = g * inv_m;
  }
  if (loss_out != nullptr && threadIdx.x >= 992) {   // loss mode: mean of the per-warp sums (last warp; fixed order)
    const int lane = threadIdx.x & 31;
    float l = 0.f;
    for (int b = lane; b < nblk; b += 32) l += loss_partial[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
    if (lane == 0) loss_out[0] = l * inv_m;
  }
}

// one warp per query row: out = tanh(dot + b)
__global__ void head_tanh_f32_kernel(const float* __restrict__ H, int ldh, const float* __restrict__ w,
                                     const float* __restrict__ b, float* __restrict__ out, long long M,
                                     int K) {
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s = fmaf(H[row * ldh + k], w[k], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[row] = tanhf(s + b[0]);
}

__global__ void grid_xyz_kernel(int res, long long q0, long long M, float* __restrict__ X,
                                float* __restrict__ S) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const long long q = q0 + i;
  const int ix = static_cast<int>(q % res);
  const int iy = static_cast<int>((q / res) % res);
  const int iz = static_cast<int>(q / (static_cast<long long>(res) * res));
  const float den = static_cast<float>(res - 1);
  const float x = __fdiv_rn(axis_coord_num(ix, res), den);
  const float y = __fdiv_rn(axis_coord_num(iy, res), den);
  const float z = __fdiv_rn(axis_coord_num(iz, res), den);
  X[i * 3 + 0] = x; X[i * 3 + 1] = y; X[i * 3 + 2] = z;
  if (S) { S[i * 256 + 253] = x; S[i * 256 + 254] = y; S[i * 256 + 255] = z; }
}

__global__ void scatter_xyz_kernel(const float* __restrict__ xyz, long long M, float* __restrict__ S) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= M) return;
  S[i * 256 + 253] = xyz[i * 3 + 0];
  S[i * 256 + 254] = xyz[i * 3 + 1];
  S[i * 256 + 255] = xyz[i * 3 + 2];
}

__global__ void fold_bias_kernel(const float* __restrict__ W, int ldw, int col0,
                                 const float* __restrict__ b, const float* __restrict__ z, int K, int N,
                                 float* __restrict__ y) {
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= N) return;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s = fmaf(W[static_cast<long long>(j) * ldw + col0 + k], z[k], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) y[j] = b[j] + s;
}

// A4: inside(v) := v < 0 ; cell is active iff its 8 corners are not all on one side.
__global__ void sign_change_mask_kernel(const float* __restrict__ sdf, int nz, int ny, int nx,
                                        unsigned char* __restrict__ mask) {
  const int cx = nx - 1, cy = ny - 1, cz = nz - 1;
  const long long total = static_cast<long long>(cx) * cy * cz;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(i % cx);
    const int y = static_cast<int>((i / cx) % cy);
    const int z = static_cast<int>(i / (static_cast<long long>(cx) * cy));
    const float* p = sdf + (static_cast<long long>(z) * ny + y) * nx + x;
    const long long sy = nx, sz = static_cast<long long>(nx) * ny;
    int n_in = 0;
    n_in += p[0] < 0.f;        n_in += p[1] < 0.f;
    n_in += p[sy] < 0.f;       n_in += p[sy + 1] < 0.f;
    n_in += p[sz] < 0.f;       n_in += p[sz + 1] < 0.f;
    n_in += p[sz + sy] < 0.f;  n_in += p[sz + sy + 1] < 0.f;
    mask[i] = (n_in != 0 && n_in != 8) ? 1 : 0;
  }
}

__global__ void sign_bits_kernel(const float* __restrict__ sdf, long long M, unsigned int* __restrict__ bits) {
  const long long words = (M + 31) >> 5;
  const int lane = threadIdx.x & 31;
  for (long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; w < words;
       w += (static_cast<long long>(gridDim.x) * blockDim.x) >> 5) {
    const long long m = (w << 5) + lane;
    const unsigned int b = __ballot_sync(0xffffffffu, m < M && sdf[m] < 0.f);
    if (lane == 0) bits[w] = b;
  }
}

// A4 from sign bits, word-parallel.  Pass 1: one thread per 32 consecutive cells of an x-row: the 33 node bits of
// each of the four node rows around it are pulled out with one funnel shift, any / all over the 8 corners are
// plain bitwise ops -> one word per thread in a row-aligned packed mask [(cz cy)][wpr].  Pass 2 turns that into
// the API's layouts with coalesced stores: one byte per cell, or the linear packing (cell c -> bit c & 31 of
// word c >> 5).  (The first version gathered 8 single bits per cell with 64-bit div/mod: 1.2 ms at 512^3.)
__device__ __forceinline__ unsigned long long bits33(const unsigned int* __restrict__ bits, long long q) {
  const long long w = q >> 5;
  const unsigned int sh = static_cast<unsigned int>(q & 31);
  const unsigned long long lo = bits[w], hi = bits[w + 1];     // the bit-plane buffer carries one padding word
  return ((lo | (hi << 32)) >> sh) & 0x1FFFFFFFFull;
}

__global__ void mask_rows_kernel(const unsigned int* __restrict__ bits, int nz, int ny, int nx,
                                 unsigned int* __restrict__ rowmask, int wpr) {
  const long long rows = static_cast<long long>(nz - 1) * (ny - 1);
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * wpr) return;
  const long long r = i / wpr;
  const int g = static_cast<int>(i - r * wpr);
  const int z = static_cast<int>(r / (ny - 1)), y = static_cast<int>(r - static_cast<long long>(z) * (ny - 1));
  const int x0 = g * 32;
  const int cx = nx - 1;
  unsigned int any = 0, all = 0xFFFFFFFFu;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const long long q = (static_cast<long long>(z + (k >> 1)) * ny + (y + (k & 1))) * nx + x0;
    // nodes x0 .. x0 + 32 of this node row (bits past the row's end belong to the next row: masked off below)
    const unsigned long long a = bits33(bits, q);
    const unsigned int n0 = static_cast<unsigned int>(a), n1 = static_cast<unsigned int>(a >> 1);
    any |= n0 | n1;
    all &= n0 & n1;
  }
  const int valid = cx - x0;                                       // cells of this word that exist
  const unsigned int vm = valid >= 32 ? 0xFFFFFFFFu : ((1u << valid) - 1u);
  rowmask[i] = any & ~all & vm;
}

__global__ void mask_expand_u8_kernel(const unsigned int* __restrict__ rowmask, long long total, int cx, int wpr,
                                      unsigned char* __restrict__ mask_u8) {
  for (long long c = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; c < total;
       c += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = c / cx;
    const int x = static_cast<int>(c - r * cx);
    mask_u8[c] = (rowmask[r * wpr + (x >> 5)] >> (x & 31)) & 1u;
  }
}

__global__ void mask_pack_linear_kernel(const unsigned int* __restrict__ rowmask, long long total, int cx, int wpr,
                                        unsigned int* __restrict__ mask_bits) {
  const long long words = (total + 31) >> 5;
  const int lane = threadIdx.x & 31;
  for (long long w = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; w < words;
       w += (static_cast<long long>(gridDim.x) * blockDim.x) >> 5) {
    const long long c = (w << 5) + lane;
    bool a = false;
    if (c < total) {
      const long long r = c / cx;
      const int x = static_cast<int>(c - r * cx);
      a = (rowmask[r * wpr + (x >> 5)] >> (x & 31)) & 1u;
    }
    const unsigned int v = __ballot_sync(0xffffffffu, a);
    if (lane == 0) mask_bits[w] = v;
  }
}

// A7, op-for-op as the oracle evaluates it (separately rounded multiplies and adds).
// The row format is DdpmStep::coef: sra, srm1, c1, c2, c3, sigma, clamp.
struct UpdateCoef { float sra, srm1, c1, c2, c3, sigma, clamp; };
__global__ void ddpm_update_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                   const float* __restrict__ noise, long long count, const UpdateCoef c) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float xv = x[i], ev = eps[i];
  float x0 = __fsub_rn(__fmul_rn(c.sra, xv), __fmul_rn(c.srm1, ev));
  x0 = fminf(fmaxf(x0, -c.clamp), c.clamp);
  float o = __fadd_rn(__fmul_rn(c.c1, x0), __fmul_rn(c.c2, xv));
  if (c.c3 != 0.f) o = __fadd_rn(o, __fmul_rn(c.c3, ev));
  if (c.sigma != 0.f) o = __fadd_rn(o, __fmul_rn(c.sigma, noise[i]));
  x[i] = o;
}

inline unsigned blocks_for(long long n, int per) { return static_cast<unsigned>((n + per - 1) / per); }

}  // namespace

cudaError_t launch_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias,
                              float* C, int ldc, long long M, int N, int K, bool relu,
                              cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  dim3 grid(blocks_for(M, BM), blocks_for(N, BN));
  linear_f32_kernel<<<grid, 256, 0, stream>>>(A, lda, W, ldw, bias, C, ldc, M, N, K, relu ? 1 : 0);
  return cudaGetLastError();
}

cudaError_t launch_linear_bwd_f32(const float* A, int lda, const float* W, int ldw, const float* H, int ldh, float* C,
                                  int ldc, long long M, int N, int K, cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  dim3 grid(blocks_for(M, BM), blocks_for(K, BN));
  linear_bwd_f32_kernel<<<grid, 256, 0, stream>>>(A, lda, W, ldw, H, ldh, C, ldc, M, N, K);
  return cudaGetLastError();
}

cudaError_t launch_head_bwd_f32(const float* dLdy, const float* y, const float* w8, const float* H7, float* D, long long M,
                                cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  head_bwd_f32_kernel<<<blocks_for(M * 512, 256), 256, 0, stream>>>(dLdy, y, w8, H7, D, M);
  return cudaGetLastError();
}

cudaError_t launch_colsum_f32(const float* D, long long M, float* partial, int half, cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  colsum_f32_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(D, M, partial, half);
  return cudaGetLastError();
}

cudaError_t launch_vjp_finish(float* partial, int nblk, const float* W0, const float* W4, float* grad,
                              cudaStream_t stream, const unsigned int* amax_bits, const float* loss_partial, float inv_m,
                              float* loss_out) {
  vjp_colsum_reduce_kernel<<<32, 256, 0, stream>>>(partial, nblk);
  vjp_finish_kernel<<<1, 1024, 0, stream>>>(partial, nblk, W0, W4, grad, amax_bits, loss_partial, inv_m, loss_out);
  return cudaGetLastError();
}

cudaError_t launch_abs_max(const float* v, long long M, unsigned int* out, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(unsigned int), stream);
  if (e != cudaSuccess || M <= 0) return e;
  long long blocks = (M + 1023) / 1024;
  if (blocks > 592) blocks = 592;
  abs_max_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(v, M, out);
  return cudaGetLastError();
}

cudaError_t launch_head_tanh_f32(const float* H, int ldh, const float* w, const float* b, float* out,
                                 long long M, int K, cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  head_tanh_f32_kernel<<<blocks_for(M * 32, 256), 256, 0, stream>>>(H, ldh, w, b, out, M, K);
  return cudaGetLastError();
}

cudaError_t launch_grid_xyz(int res, long long q0, long long M, float* X, float* S,
                            cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  grid_xyz_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(res, q0, M, X, S);
  return cudaGetLastError();
}

cudaError_t launch_scatter_xyz(const float* xyz, long long M, float* S, cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  scatter_xyz_kernel<<<blocks_for(M, 256), 256, 0, stream>>>(xyz, M, S);
  return cudaGetLastError();
}

cudaError_t launch_fold_bias(const float* W, int ldw, int col0, const float* b, const float* z, int K,
                             int N, float* y, cudaStream_t stream) {
  fold_bias_kernel<<<blocks_for(static_cast<long long>(N) * 32, 256), 256, 0, stream>>>(W, ldw, col0, b,
                                                                                       z, K, N, y);
  return cudaGetLastError();
}

cudaError_t launch_sign_change_mask(const float* sdf, int nz, int ny, int nx, unsigned char* mask,
                                    cudaStream_t stream) {
  const long long total = static_cast<long long>(nx - 1) * (ny - 1) * (nz - 1);
  if (total <= 0) return cudaSuccess;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  sign_change_mask_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(sdf, nz, ny, nx, mask);
  return cudaGetLastError();
}

cudaError_t launch_sign_bits(const float* sdf, long long M, unsigned int* bits, cudaStream_t stream) {
  if (M <= 0) return cudaSuccess;
  long long blocks = (((M + 31) >> 5) * 32 + 255) / 256;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  sign_bits_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(sdf, M, bits);
  return cudaGetLastError();
}

size_t mask_rows_words(int nz, int ny, int nx) {
  return static_cast<size_t>(nz - 1) * (ny - 1) * ((nx - 1 + 31) / 32);
}

// `rowmask` = scratch of mask_rows_words(nz, ny, nx) words; `bits` must be readable one word past its last word.
cudaError_t launch_mask_from_bits(const unsigned int* bits, int nz, int ny, int nx, unsigned char* mask_u8,
                                  unsigned int* mask_bits, unsigned int* rowmask, cudaStream_t stream) {
  const long long total = static_cast<long long>(nx - 1) * (ny - 1) * (nz - 1);
  if (total <= 0) return cudaSuccess;
  const int wpr = (nx - 1 + 31) / 32;
  const long long n1 = static_cast<long long>(nz - 1) * (ny - 1) * wpr;
  mask_rows_kernel<<<static_cast<unsigned>((n1 + 255) / 256), 256, 0, stream>>>(bits, nz, ny, nx, rowmask, wpr);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 64) blocks = 148LL * 64;
  if (mask_u8 != nullptr) {
    mask_expand_u8_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(rowmask, total, nx - 1, wpr, mask_u8);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (mask_bits != nullptr) {
    mask_pack_linear_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(rowmask, total, nx - 1, wpr, mask_bits);
    e = cudaGetLastError();
  }
  return e;
}

cudaError_t launch_ddpm_update(float* x, const float* eps, const float* noise, long long count, const float* coef,
                               cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  if (coef[5] != 0.f && noise == nullptr) return cudaErrorInvalidValue;
  const UpdateCoef c{coef[0], coef[1], coef[2], coef[3], coef[4], coef[5], coef[6]};
  ddpm_update_kernel<<<blocks_for(count, 256), 256, 0, stream>>>(x, eps, noise, count, c);
  return cudaGetLastError();
}

}  // namespace sdfb
