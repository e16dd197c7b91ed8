// C ABI of libsdfb200.so (declared in include/sdfb200.h): contexts, weight packing,
// argument validation and kernel launches.  No reference interface exists to mirror
// (/root/reference/README.md:1 is a title); the surface follows SURVEY.md section 8(b).
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <vector>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "../../include/sdfb200.h"
#include "comm.h"
#include "kernels.h"

using namespace sdfb;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

}  // namespace

namespace sdfb {
// the same thread-local message for the other translation units of the library (comm.cu)
int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
}  // namespace sdfb

namespace {

#define CU_TRY(expr)                                                                         \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return fail(SDFB_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int check_device(int device, int* num_sms) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    return fail(SDFB_E_DEVICE, "no CUDA device visible: libsdfb200 has no CPU path");
  if (device < 0 || device >= count) return fail(SDFB_E_INVALID, "device %d out of range (%d devices)", device, count);
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(SDFB_E_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device, prop.major,
                prop.minor);
  *num_sms = prop.multiProcessorCount;
  return SDFB_OK;
}

uint16_t to_lowp(float f, bool fp16) {
  if (fp16) {
    __half h = __float2half_rn(f);
    uint16_t u; std::memcpy(&u, &h, 2); return u;
  }
  __nv_bfloat16 b = __float2bfloat16_rn(f);
  uint16_t u; std::memcpy(&u, &b, 2); return u;
}

// decoder layer l: offsets into the parameter blob
struct LayerOff { long long w, b; int fin, fout; };
const int kFin[9] = {259, 512, 512, 512, 512, 512, 512, 512, 512};
const int kFout[9] = {512, 512, 512, 253, 512, 512, 512, 512, 1};

void decoder_offsets(LayerOff off[9]) {
  long long o = 0;
  for (int l = 0; l < 9; ++l) {
    off[l].fin = kFin[l]; off[l].fout = kFout[l];
    off[l].w = o; o += static_cast<long long>(kFin[l]) * kFout[l];
    off[l].b = o; o += kFout[l];
  }
}

// The weight stream of kernels.h (96 forward blocks, then the 96 transposed blocks of the backward
// passes), as 128B-swizzled shared-memory images.
void pack_wstream(const float* P, const LayerOff off[9], bool fp16, std::vector<uint16_t>& out) {
  out.assign(static_cast<size_t>(kBlocksPerTileBwd) * kBlockBytes / 2, 0);
  static const int pass_layer[kPasses] = {1, 1, 2, 2, 3, 4, 4, 5, 5, 6, 6, 7, 7};
  static const int pass_half[kPasses] = {0, 1, 0, 1, 0, 0, 1, 0, 1, 0, 1, 0, 1};
  size_t blk = 0;
  for (int p = 0; p < kPasses; ++p) {
    const int L = pass_layer[p], h = pass_half[p];
    const int nk = (L == 4) ? 4 : 8;
    // L4's K = 256 operand is [h3 (253) | xyz (3)]: its weight columns are W4[:, 0:253] | W4[:, 509:512]
    const float* W = P + off[L].w;
    const int fin = off[L].fin, fout = off[L].fout;
    for (int k = 0; k < nk; ++k, ++blk) {
      uint16_t* dst = out.data() + blk * (kBlockBytes / 2);
      for (int r = 0; r < kBlockRows; ++r) {
        const int n = h * 256 + r;
        for (int u = 0; u < 8; ++u) {
          uint16_t* d = dst + r * 64 + ((u ^ (r & 7)) * 8);
          for (int e = 0; e < 8; ++e) {
            const int kk = k * 64 + u * 8 + e;
            const int src = (L == 4 && kk >= kSkipOut) ? kk + kLatent : kk;
            const float v = (n < fout) ? W[static_cast<long long>(n) * fin + src] : 0.f;
            d[e] = to_lowp(v, fp16);
          }
        }
      }
    }
  }
  // backward: block rows = INPUT features n of layer L, k = its OUTPUT features: W_L[k][n]
  static const int bpass_layer[kPassesBwd - kPasses] = {7, 7, 6, 6, 5, 5, 4, 3, 3, 2, 2, 1, 1};
  static const int bpass_half[kPassesBwd - kPasses] = {0, 1, 0, 1, 0, 1, 0, 0, 1, 0, 1, 0, 1};
  for (int p = 0; p < kPassesBwd - kPasses; ++p) {
    const int L = bpass_layer[p], h = bpass_half[p];
    const int nk = (L == 3) ? 4 : 8;                       // layer 3 has 253 outputs: K = 256
    const float* W = P + off[L].w;
    const int fin = off[L].fin, fout = off[L].fout;
    const int n_valid = (L == 4) ? kSkipOut : fin;         // the skip layer hands back its 253 hidden columns only
    for (int k = 0; k < nk; ++k, ++blk) {
      uint16_t* dst = out.data() + blk * (kBlockBytes / 2);
      for (int r = 0; r < kBlockRows; ++r) {
        const int n = h * 256 + r;
        for (int u = 0; u < 8; ++u) {
          uint16_t* d = dst + r * 64 + ((u ^ (r & 7)) * 8);
          for (int e = 0; e < 8; ++e) {
            const int kk = k * 64 + u * 8 + e;
            const float v = (n < n_valid && kk < fout) ? W[static_cast<long long>(kk) * fin + n] : 0.f;
            d[e] = to_lowp(v, fp16);
          }
        }
      }
    }
  }
}

// Denoiser weights as pre-swizzled 128-byte rows (kernels.h, "fused DDPM sampler"):
// row (layer, k-chunk, feature n) holds W[n][64 kc .. 64 kc + 64), 16-byte unit u at u ^ (n & 7).
void pack_ddpm_weights(const float* P, const long long woff[5], bool fp16, std::vector<uint16_t>& out) {
  out.assign(static_cast<size_t>(kDdpmWRows) * 64, 0);
  size_t row = 0;
  for (int l = 0; l < 5; ++l) {
    const int fin = l == 0 ? 512 : 1024, fout = l == 4 ? 256 : 1024;
    const int nk = l == 0 ? 4 : 16;             // layer 0: only the latent half of W0 (the time half is folded into tb0)
    const float* W = P + woff[l];
    for (int kc = 0; kc < nk; ++kc)
      for (int n = 0; n < fout; ++n, ++row) {
        uint16_t* dst = out.data() + row * 64;
        for (int u = 0; u < 8; ++u)
          for (int e = 0; e < 8; ++e)
            dst[((u ^ (n & 7)) * 8) + e] = to_lowp(W[static_cast<long long>(n) * fin + kc * 64 + u * 8 + e], fp16);
      }
  }
}

}  // namespace

struct sdfb_decoder {
  int device = 0, num_sms = 0;
  LayerOff off[9];
  float* params = nullptr;       // fp32 blob on device
  float* w4s = nullptr;          // [512][256]: W4[:, 0:253] | W4[:, 509:512]   (fp32 path)
  uint8_t* wstream[2] = {nullptr, nullptr};   // [0] bf16, [1] fp16
  alignas(64) unsigned char tmap[2][128];     // tensor maps over the two streams (CTA-pair kernel)
  DecConsts* consts = nullptr;
  float* bias0f = nullptr;       // fp32 path folded biases
  float* bias4f = nullptr;
  unsigned int* status = nullptr;
  unsigned int* status_host = nullptr;       // mirror of `status` in mapped pinned host memory (kernels store a trip there too)
  unsigned int* status_host_dev = nullptr;   // its device-side address
  cudaEvent_t ev_user = nullptr;             // end of the last device-path call: the *_host calls order their own streams after it
  bool user_pending = false;
  unsigned int* signs = nullptr; long long sign_words = 0;   // sign bit-planes of the last masked decode (lazy)
  unsigned int* rowmask = nullptr; size_t rowmask_words = 0; // row-aligned packed mask scratch (lazy)
  // backward workspace (lazy): stored activations of one chunk, two delta buffers, column-sum partials
  float* bw_act[8] = {}; float *bw_d0 = nullptr, *bw_d1 = nullptr, *bw_y = nullptr, *bw_partial = nullptr;
  long long bw_rows = 0, bw_blocks = 0;
  uint32_t* bw_masks = nullptr;   // tensor-core backward: ReLU-mask scratch [num_sms][6 + 2][16][128]
  float* bw_colsum = nullptr;     //                       column sums [num_sms * 4][1024]
  unsigned int* bw_amax = nullptr;   //                    bits of max |dLdy|
  float* bw_loss = nullptr;          //                    loss mode: per-warp sums [num_sms * 4]
  // hierarchical sparse decode workspace (lazy): node bitmaps, scan tiles, query lists, level-1 lattice
  struct SparseWs {
    unsigned int *need1 = nullptr, *need2 = nullptr, *keep = nullptr, *tiles = nullptr, *idx = nullptr, *lip = nullptr, *qblk = nullptr;
    unsigned long long* kept = nullptr;
    float *xyz = nullptr, *vals = nullptr, *cs = nullptr;
    int* ids = nullptr;
    long long words = 0, idx_cap = 0, corners = 0, blocks = 0;
  } sp;
  // fp32 workspace (lazy)
  long long ws_rows = 0;
  float *h0 = nullptr, *h1 = nullptr, *s = nullptr, *x = nullptr;
  // host staging (lazy, pinned) + device staging for the *_host calls
  void* pin = nullptr; size_t pin_bytes = 0;
  void* dstage = nullptr; size_t dstage_bytes = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  // *_host calls: compute and copy-out streams, one event per z-chunk (the D2H copy of a chunk overlaps the next chunk's kernel)
  cudaStream_t st_compute = nullptr, st_copy = nullptr, st_in = nullptr;
  cudaEvent_t chunk_ev[17] = {}, in_ev[17] = {};
  unsigned long long timeout_ns = 2000000000ull;
  unsigned int debug_flags = 0;
  long long* prof = nullptr;     // wait profile buffer (allocated when SDFB_PROF is set)
};

// row-major activations [act_rows][kDdpmActCols] (16-bit) and one barrier counter per 256-latent group
struct DdpmLane { uint16_t* act = nullptr; int act_rows = 0; unsigned int* counter = nullptr; };

struct sdfb_ddpm {
  int device = 0, num_sms = 0;
  float* params = nullptr;
  long long woff[5], boff[5];
  float* tb0 = nullptr;          // [1000][1024]: b0 + W0[:, 256:] temb(t)
  std::vector<DdpmStep> ddpm_rows;            // the 1000-step DDPM chain in execution order (t = 999 .. 0), fp32 coefficients
  int ws_n = 0;
  float *h0 = nullptr, *h1 = nullptr, *eps = nullptr;
  void* dstage = nullptr; size_t dstage_bytes = 0;
  void* nstage = nullptr; size_t nstage_bytes = 0;   // materialised Philox stream (fp32 path of the seeded sampler)
  // tensor-core path (ddpm_step.cu)
  uint8_t* wpack[2] = {nullptr, nullptr};     // [0] bf16, [1] fp16: kDdpmWRows rows of 128 B
  float* bias_dev = nullptr;                  // [3][1024] + [256]
  DdpmStep* ddpm_rows_dev = nullptr;          // ddpm_rows on the device: a truncated chain of `steps` is its last `steps` rows
  DdpmStep* call_rows_dev = nullptr;          // [1000]: the rows of a respaced (DDIM) call, written on the caller's stream
  DdpmLane lane[2];                           // workspaces of the (at most two) concurrent launches of a call
  cudaStream_t st_b = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  unsigned int* status = nullptr;
  unsigned int* status_host = nullptr;       // mirror of `status` in mapped pinned host memory
  unsigned int* status_host_dev = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  unsigned long long timeout_ns = 4000000000ull;
  long long* prof = nullptr;                  // wait profile buffer (allocated when SDFB_PROF is set)
  int max_clusters8[2] = {-1, -1};            // resident 8-CTA clusters of the sampler kernel (queried once), [bf16, fp16]
  int max_clusters16[2] = {-1, -1};           // ... and 16-CTA clusters (128-wide tiles)
};

namespace {

int ensure_fp32_ws(sdfb_decoder* d, long long rows) {
  if (d->ws_rows >= rows) return SDFB_OK;
  cudaFree(d->h0); cudaFree(d->h1); cudaFree(d->s); cudaFree(d->x);
  d->h0 = d->h1 = d->s = d->x = nullptr; d->ws_rows = 0;
  CU_TRY(cudaMalloc(&d->h0, rows * 512 * sizeof(float)));
  CU_TRY(cudaMalloc(&d->h1, rows * 512 * sizeof(float)));
  CU_TRY(cudaMalloc(&d->s, rows * 256 * sizeof(float)));
  CU_TRY(cudaMalloc(&d->x, rows * 3 * sizeof(float)));
  d->ws_rows = rows;
  return SDFB_OK;
}

constexpr long long kFp32Chunk = 32768;

// fp32 SIMT decode of M queries; xyz == nullptr selects grid mode (global query index q0).
int decode_fp32(sdfb_decoder* d, const float* z, const float* xyz, int res, long long q0, long long M,
                float* out, cudaStream_t st) {
  const long long chunk = M < kFp32Chunk ? M : kFp32Chunk;
  int rc = ensure_fp32_ws(d, chunk);
  if (rc) return rc;
  const float* P = d->params;
  const LayerOff* o = d->off;
  CU_TRY(launch_fold_bias(P + o[0].w, kDecIn, 0, P + o[0].b, z, kLatent, kHid, d->bias0f, st));
  CU_TRY(launch_fold_bias(P + o[4].w, kHid, kSkipOut, P + o[4].b, z, kLatent, kHid, d->bias4f, st));
  for (long long m0 = 0; m0 < M; m0 += chunk) {
    const long long m = (M - m0) < chunk ? (M - m0) : chunk;
    const float* X;
    if (xyz == nullptr) {
      CU_TRY(launch_grid_xyz(res, q0 + m0, m, d->x, d->s, st));
      X = d->x;
    } else {
      X = xyz + 3 * m0;
      CU_TRY(launch_scatter_xyz(X, m, d->s, st));
    }
    CU_TRY(launch_linear_f32(X, 3, P + o[0].w + kLatent, kDecIn, d->bias0f, d->h0, 512, m, 512, 3, true, st));
    CU_TRY(launch_linear_f32(d->h0, 512, P + o[1].w, 512, P + o[1].b, d->h1, 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(d->h1, 512, P + o[2].w, 512, P + o[2].b, d->h0, 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(d->h0, 512, P + o[3].w, 512, P + o[3].b, d->s, 256, m, kSkipOut, 512, true, st));
    CU_TRY(launch_linear_f32(d->s, 256, d->w4s, 256, d->bias4f, d->h1, 512, m, 512, 256, true, st));
    CU_TRY(launch_linear_f32(d->h1, 512, P + o[5].w, 512, P + o[5].b, d->h0, 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(d->h0, 512, P + o[6].w, 512, P + o[6].b, d->h1, 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(d->h1, 512, P + o[7].w, 512, P + o[7].b, d->h0, 512, m, 512, 512, true, st));
    CU_TRY(launch_head_tanh_f32(d->h0, 512, P + o[8].w, P + o[8].b, out + m0, m, 512, st));
  }
  return SDFB_OK;
}

int decode_tc(sdfb_decoder* d, const float* z, const float* xyz, int res, long long q0, long long M, float* out,
              bool fp16, float* dump, int dump_pass, cudaStream_t st, unsigned int* signs = nullptr) {
  const float* P = d->params;
  const LayerOff* o = d->off;
  CU_TRY(launch_fold_latent(P + o[0].w, P + o[0].b, P + o[4].w, P + o[4].b, z, d->consts, st));
  DecodeParams p{};
  p.wstream = d->wstream[fp16 ? 1 : 0];
  p.consts = d->consts;
  p.xyz = xyz;
  p.out = out;
  p.signs = signs;
  p.M = M;
  p.q0 = q0;
  p.res = res;
  p.status = d->status;
  p.status_host = d->status_host_dev;
  p.dump = dump;
  p.dump_pass = dump_pass;
  p.timeout_ns = d->timeout_ns;
  p.debug_flags = d->debug_flags;
  p.prof = d->prof;
  CU_TRY(cudaEventRecord(d->ev0, st));
  CU_TRY(launch_fused_decoder(p, d->tmap[fp16 ? 1 : 0], fp16, d->num_sms, st));
  CU_TRY(cudaEventRecord(d->ev1, st));
  d->timed = true;
  return SDFB_OK;
}

// `signs` (optional): the sign bit of every output, 32 queries per word - written by the fused kernel
// itself on the tensor-core path, by a small kernel behind the FFMA chain on the fp32 path.
int decode_any(sdfb_decoder* d, const float* z, const float* xyz, int res, long long q0, long long M, float* out,
               int precision, cudaStream_t st, unsigned int* signs = nullptr) {
  if (M == 0) return SDFB_OK;
  switch (precision) {
    case SDFB_PREC_FP32: {
      int rc = decode_fp32(d, z, xyz, res, q0, M, out, st);
      if (rc) return rc;
      if (signs != nullptr) CU_TRY(launch_sign_bits(out, M, signs, st));
      return SDFB_OK;
    }
    case SDFB_PREC_BF16: return decode_tc(d, z, xyz, res, q0, M, out, false, nullptr, -1, st, signs);
    case SDFB_PREC_FP16: return decode_tc(d, z, xyz, res, q0, M, out, true, nullptr, -1, st, signs);
    default: return fail(SDFB_E_INVALID, "unknown precision %d", precision);
  }
}

int ensure_signs(sdfb_decoder* d, long long words, cudaStream_t st) {
  if (d->sign_words >= words) return SDFB_OK;
  cudaFree(d->signs); d->signs = nullptr; d->sign_words = 0;
  CU_TRY(cudaMalloc(&d->signs, static_cast<size_t>(words + 1) * sizeof(unsigned int)));   // + 1: the mask kernel reads word pairs
  // (on the caller's stream: a legacy-stream memset is not ordered with a non-blocking stream)
  CU_TRY(cudaMemsetAsync(d->signs, 0, static_cast<size_t>(words + 1) * sizeof(unsigned int), st));
  d->sign_words = words;
  return SDFB_OK;
}

int ensure_rowmask(sdfb_decoder* d, size_t words) {
  if (d->rowmask_words >= words) return SDFB_OK;
  cudaFree(d->rowmask); d->rowmask = nullptr; d->rowmask_words = 0;
  CU_TRY(cudaMalloc(&d->rowmask, words * sizeof(unsigned int)));
  d->rowmask_words = words;
  return SDFB_OK;
}

int kernel_status(sdfb_decoder* d) {
  unsigned int s = 0;
  CU_TRY(cudaMemcpy(&s, d->status, sizeof(s), cudaMemcpyDeviceToHost));
  if (s != 0) {
    cudaMemset(d->status, 0, sizeof(unsigned int));
    if (d->status_host) *reinterpret_cast<volatile unsigned int*>(d->status_host) = 0;
    return fail(SDFB_E_KERNEL, "fused decoder watchdog tripped at wait site 0x%x", s);
  }
  return SDFB_OK;
}

// Asynchronous entry points cannot know how their own launch will end, but they can refuse to build on a launch that
// already failed: a kernel whose watchdog trips also stores the code in mapped host memory, which every entry point
// looks at first (no synchronisation).  The error is reported once and cleared.
int pending_status(sdfb_decoder* d) {
  if (d->status_host == nullptr) return SDFB_OK;
  const unsigned int s = *reinterpret_cast<volatile unsigned int*>(d->status_host);
  if (s == 0) return SDFB_OK;
  *reinterpret_cast<volatile unsigned int*>(d->status_host) = 0;
  cudaMemset(d->status, 0, sizeof(unsigned int));
  return fail(SDFB_E_KERNEL, "an earlier launch on this context tripped the kernel watchdog at wait site 0x%x: its outputs are invalid", s);
}

// End of a device-path call: remember where the caller's stream stands, so that a later *_host call (which runs on the
// context's own streams and rewrites the per-latent constants) starts after it.
struct UserMark {          // records the end of a device-path call on every return path
  sdfb_decoder* d; cudaStream_t st;
  ~UserMark() { if (cudaEventRecord(d->ev_user, st) == cudaSuccess) d->user_pending = true; }
};
int order_after_user(sdfb_decoder* d, cudaStream_t st) {
  if (d->user_pending) CU_TRY(cudaStreamWaitEvent(st, d->ev_user, 0));
  return SDFB_OK;
}

int ensure_stage(void** pin, size_t* pin_bytes, void** dev, size_t* dev_bytes, size_t need_pin, size_t need_dev) {
  if (pin != nullptr && *pin_bytes < need_pin) {
    if (*pin) cudaFreeHost(*pin);
    *pin = nullptr; *pin_bytes = 0;
    CU_TRY(cudaMallocHost(pin, need_pin));
    *pin_bytes = need_pin;
  }
  if (*dev_bytes < need_dev) {
    if (*dev) cudaFree(*dev);
    *dev = nullptr; *dev_bytes = 0;
    CU_TRY(cudaMalloc(dev, need_dev));
    *dev_bytes = need_dev;
  }
  return SDFB_OK;
}

}  // namespace

extern "C" {

int sdfb_version(void) { return 100; }
const char* sdfb_last_error(void) { return g_err; }

int sdfb_decoder_create(const float* params_host, size_t n_floats, int device, sdfb_decoder** out) {
  if (out == nullptr || params_host == nullptr) return fail(SDFB_E_INVALID, "null argument");
  *out = nullptr;
  if (n_floats != static_cast<size_t>(kDecParamFloats))
    return fail(SDFB_E_INVALID, "decoder blob must hold %lld floats, got %zu", kDecParamFloats, n_floats);
  int sms = 0;
  int rc = check_device(device, &sms);
  if (rc) return rc;
  DeviceGuard g(device);
  if (!g.ok) return fail(SDFB_E_CUDA, "cudaSetDevice(%d) failed", device);
  sdfb_decoder* d = new (std::nothrow) sdfb_decoder();
  if (!d) return fail(SDFB_E_NOMEM, "out of host memory");
  d->device = device; d->num_sms = sms;
  decoder_offsets(d->off);
  if (const char* e = std::getenv("SDFB_DEBUG_FLAGS")) d->debug_flags = static_cast<unsigned int>(std::strtoul(e, nullptr, 0));
  const float* P = params_host;
  const bool want_prof = std::getenv("SDFB_PROF") != nullptr;
  auto bail = [&](int code) { sdfb_decoder_destroy(d); return code; };
#define CU_TRY_D(expr)                                                                       \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return bail(fail(SDFB_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)));       \
  } while (0)
  CU_TRY_D(fused_decoder_init());
  CU_TRY_D(tc_common_init());
  CU_TRY_D(cudaMalloc(&d->params, n_floats * sizeof(float)));
  CU_TRY_D(cudaMemcpy(d->params, P, n_floats * sizeof(float), cudaMemcpyHostToDevice));
  // fp32 path: compact skip-layer matrix
  {
    std::vector<float> w4s(512 * 256);
    const float* W4 = P + d->off[4].w;
    for (int n = 0; n < 512; ++n) {
      for (int k = 0; k < kSkipOut; ++k) w4s[n * 256 + k] = W4[n * 512 + k];
      for (int k = 0; k < 3; ++k) w4s[n * 256 + kSkipOut + k] = W4[n * 512 + kSkipOut + kLatent + k];
    }
    CU_TRY_D(cudaMalloc(&d->w4s, w4s.size() * sizeof(float)));
    CU_TRY_D(cudaMemcpy(d->w4s, w4s.data(), w4s.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  // tensor-core path: weight streams and the constant block
  for (int f = 0; f < 2; ++f) {
    std::vector<uint16_t> ws;
    pack_wstream(P, d->off, f == 1, ws);
    CU_TRY_D(cudaMalloc(&d->wstream[f], ws.size() * 2));
    CU_TRY_D(cudaMemcpy(d->wstream[f], ws.data(), ws.size() * 2, cudaMemcpyHostToDevice));
    CU_TRY_D(make_wstream_tensor_map(d->wstream[f], d->tmap[f]));
  }
  {
    std::vector<DecConsts> hc(1);
    DecConsts& c = hc[0];
    std::memset(&c, 0, sizeof(c));
    const float* W0 = P + d->off[0].w;
    for (int n = 0; n < 512; ++n) {
      c.l0[n] = make_float4(W0[n * kDecIn + 256], W0[n * kDecIn + 257], W0[n * kDecIn + 258], 0.f);
      c.head[n] = P[d->off[8].w + n];
    }
    for (int l = 1; l <= 7; ++l)
      for (int n = 0; n < d->off[l].fout; ++n) c.bias[l - 1][n] = P[d->off[l].b + n];
    c.head_b[0] = P[d->off[8].b];
    CU_TRY_D(cudaMalloc(&d->consts, sizeof(DecConsts)));
    CU_TRY_D(cudaMemcpy(d->consts, &c, sizeof(DecConsts), cudaMemcpyHostToDevice));
  }
  CU_TRY_D(cudaMalloc(&d->bias0f, 512 * sizeof(float)));
  CU_TRY_D(cudaMalloc(&d->bias4f, 512 * sizeof(float)));
  CU_TRY_D(cudaMalloc(&d->status, sizeof(unsigned int)));
  CU_TRY_D(cudaMemset(d->status, 0, sizeof(unsigned int)));
  CU_TRY_D(cudaHostAlloc(reinterpret_cast<void**>(&d->status_host), sizeof(unsigned int), cudaHostAllocMapped));
  *d->status_host = 0;
  CU_TRY_D(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d->status_host_dev), d->status_host, 0));
  CU_TRY_D(cudaEventCreateWithFlags(&d->ev_user, cudaEventDisableTiming));
  if (want_prof) {
    CU_TRY_D(cudaMalloc(&d->prof, (static_cast<size_t>(sms) * 24 + 128) * sizeof(long long)));   // + a 4 x 32 event trace
    CU_TRY_D(cudaMemset(d->prof, 0, (static_cast<size_t>(sms) * 24 + 128) * sizeof(long long)));
  }
  CU_TRY_D(cudaEventCreate(&d->ev0));
  CU_TRY_D(cudaEventCreate(&d->ev1));
  CU_TRY_D(cudaStreamCreateWithFlags(&d->st_compute, cudaStreamNonBlocking));
  CU_TRY_D(cudaStreamCreateWithFlags(&d->st_copy, cudaStreamNonBlocking));
  for (cudaEvent_t& e : d->chunk_ev) CU_TRY_D(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (cudaEvent_t& e : d->in_ev) CU_TRY_D(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CU_TRY_D(cudaDeviceSynchronize());   // the set-up copies and memsets above are done before any caller stream can touch the context
#undef CU_TRY_D
  *out = d;
  return SDFB_OK;
}

int sdfb_decoder_destroy(sdfb_decoder* d) {
  if (!d) return SDFB_OK;
  DeviceGuard g(d->device);
  cudaDeviceSynchronize();
  cudaFree(d->params); cudaFree(d->w4s); cudaFree(d->wstream[0]); cudaFree(d->wstream[1]);
  cudaFree(d->consts); cudaFree(d->bias0f); cudaFree(d->bias4f); cudaFree(d->status);
  if (d->status_host) cudaFreeHost(d->status_host);
  if (d->ev_user) cudaEventDestroy(d->ev_user);
  cudaFree(d->h0); cudaFree(d->h1); cudaFree(d->s); cudaFree(d->x); cudaFree(d->prof); cudaFree(d->signs); cudaFree(d->rowmask);
  cudaFree(d->sp.need1); cudaFree(d->sp.need2); cudaFree(d->sp.keep); cudaFree(d->sp.tiles); cudaFree(d->sp.idx); cudaFree(d->sp.lip);
  cudaFree(d->sp.kept); cudaFree(d->sp.xyz); cudaFree(d->sp.vals); cudaFree(d->sp.cs); cudaFree(d->sp.ids); cudaFree(d->sp.qblk);
  for (float* a : d->bw_act) cudaFree(a);
  cudaFree(d->bw_d0); cudaFree(d->bw_d1); cudaFree(d->bw_y); cudaFree(d->bw_partial);
  cudaFree(d->bw_masks); cudaFree(d->bw_colsum); cudaFree(d->bw_amax); cudaFree(d->bw_loss);
  if (d->pin) cudaFreeHost(d->pin);
  cudaFree(d->dstage);
  if (d->ev0) cudaEventDestroy(d->ev0);
  if (d->ev1) cudaEventDestroy(d->ev1);
  for (cudaEvent_t e : d->chunk_ev) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : d->in_ev) if (e) cudaEventDestroy(e);
  if (d->st_in) cudaStreamDestroy(d->st_in);
  if (d->st_compute) cudaStreamDestroy(d->st_compute);
  if (d->st_copy) cudaStreamDestroy(d->st_copy);
  delete d;
  return SDFB_OK;
}

int sdfb_decode_grid(sdfb_decoder* d, const float* latent_dev, int res, int z0, int z1, float* sdf_dev,
                     uint8_t* mask_dev, int precision, void* stream) {
  if (!d || !latent_dev) return fail(SDFB_E_INVALID, "null argument");
  if (res < 2 || res > 2048) return fail(SDFB_E_INVALID, "res %d outside [2, 2048]", res);
  if (z0 < 0 || z1 > res || z0 > z1) return fail(SDFB_E_INVALID, "bad plane range [%d, %d) for res %d", z0, z1, res);
  if (z0 == z1) return SDFB_OK;                      // an empty slab (the tail ranks of an uneven split): nothing to do
  if (!sdf_dev) return fail(SDFB_E_INVALID, "null argument");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long plane = static_cast<long long>(res) * res;
  int zend = z1;
  if (mask_dev != nullptr && z1 < res && z1 > z0) zend = z1 + 1;   // halo plane, recomputed locally
  const long long M = (zend - z0) * plane;
  if (mask_dev == nullptr || zend - z0 < 2) return decode_any(d, latent_dev, nullptr, res, z0 * plane, M, sdf_dev, precision, st);
  // the decoder emits the sign bit of every value it stores; the cell mask is a combine of those bit-planes
  // (1/32 of the field's bytes) instead of a second pass over the fp32 field
  int rc = ensure_signs(d, (M + 31) >> 5, st);
  if (rc) return rc;
  if (rc == SDFB_OK) rc = ensure_rowmask(d, mask_rows_words(zend - z0, res, res));
  if (rc) return rc;
  rc = decode_any(d, latent_dev, nullptr, res, z0 * plane, M, sdf_dev, precision, st, d->signs);
  if (rc) return rc;
  CU_TRY(launch_mask_from_bits(d->signs, zend - z0, res, res, mask_dev, nullptr, d->rowmask, st));
  return SDFB_OK;
}

int sdfb_decode_grid_bits(sdfb_decoder* d, const float* latent_dev, int res, int z0, int z1, float* sdf_dev,
                          uint32_t* sign_bits_dev, uint32_t* mask_bits_dev, int precision, void* stream) {
  if (!d || !latent_dev) return fail(SDFB_E_INVALID, "null argument");
  if (res < 2 || res > 2048) return fail(SDFB_E_INVALID, "res %d outside [2, 2048]", res);
  if (z0 < 0 || z1 > res || z0 > z1) return fail(SDFB_E_INVALID, "bad plane range [%d, %d) for res %d", z0, z1, res);
  if (z0 == z1) return SDFB_OK;                      // an empty slab: nothing to do
  if (!sdf_dev || !sign_bits_dev) return fail(SDFB_E_INVALID, "null argument");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long plane = static_cast<long long>(res) * res;
  int zend = z1;
  if (mask_bits_dev != nullptr && z1 < res && z1 > z0) zend = z1 + 1;
  const long long M = (zend - z0) * plane;
  // the decoder writes into the context's own bit-plane buffer (it has the padding word the mask kernel reads);
  // the caller's copy is made from it
  int rc = ensure_signs(d, (M + 31) >> 5, st);
  if (rc == SDFB_OK && mask_bits_dev != nullptr && zend - z0 >= 2) rc = ensure_rowmask(d, mask_rows_words(zend - z0, res, res));
  if (rc) return rc;
  rc = decode_any(d, latent_dev, nullptr, res, z0 * plane, M, sdf_dev, precision, st, d->signs);
  if (rc) return rc;
  CU_TRY(cudaMemcpyAsync(sign_bits_dev, d->signs, static_cast<size_t>((M + 31) >> 5) * 4, cudaMemcpyDeviceToDevice, st));
  if (mask_bits_dev != nullptr && zend - z0 >= 2)
    CU_TRY(launch_mask_from_bits(d->signs, zend - z0, res, res, nullptr, mask_bits_dev, d->rowmask, st));
  return SDFB_OK;
}

int sdfb_decode_grid_batch(sdfb_decoder* d, const float* latents_dev, int batch, int res, float* sdf_dev, int precision,
                           void* stream) {
  if (!d || (batch > 0 && (!latents_dev || !sdf_dev))) return fail(SDFB_E_INVALID, "null argument");
  if (batch < 0 || res < 2 || res > 2048) return fail(SDFB_E_INVALID, "bad batch or res");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long M = static_cast<long long>(res) * res * res;
  for (int b = 0; b < batch; ++b) {   // shapes are independent: one fold + one persistent launch each, back to back on the stream
    int rc = decode_any(d, latents_dev + static_cast<long long>(b) * kLatent, nullptr, res, 0, M, sdf_dev + b * M, precision, st);
    if (rc) return rc;
  }
  return SDFB_OK;
}

int sdfb_decode_points(sdfb_decoder* d, const float* latent_dev, const float* xyz_dev, int64_t M, float* sdf_dev,
                       int precision, void* stream) {
  if (!d || !latent_dev || (M > 0 && (!xyz_dev || !sdf_dev))) return fail(SDFB_E_INVALID, "null argument");
  if (M < 0) return fail(SDFB_E_INVALID, "negative point count");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  return decode_any(d, latent_dev, xyz_dev, 0, 0, M, sdf_dev, precision, static_cast<cudaStream_t>(stream));
}

// g = sum_m dLdy[m] d sdf_m / d latent on the fp32 path: forward with stored activations, backward with the
// FFMA kernels, deterministic column sums; chunks of 8192 points.
int sdfb_decoder_vjp_latent(sdfb_decoder* d, const float* latent_dev, const float* xyz_dev, int64_t M, const float* dLdy_dev,
                            float* grad_latent_dev, float* sdf_dev, void* stream) {
  if (!d || !latent_dev || !grad_latent_dev || (M > 0 && (!xyz_dev || !dLdy_dev))) return fail(SDFB_E_INVALID, "null argument");
  if (M < 0) return fail(SDFB_E_INVALID, "negative point count");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (M == 0) { CU_TRY(cudaMemsetAsync(grad_latent_dev, 0, kLatent * sizeof(float), st)); return SDFB_OK; }
  constexpr long long kChunkRows = 8192;
  const long long rows = M < kChunkRows ? M : kChunkRows;
  if (d->bw_rows < rows) {
    for (float*& a : d->bw_act) { cudaFree(a); a = nullptr; }
    cudaFree(d->bw_d0); cudaFree(d->bw_d1); cudaFree(d->bw_y); d->bw_d0 = d->bw_d1 = d->bw_y = nullptr; d->bw_rows = 0;
    for (int i = 0; i < 8; ++i) CU_TRY(cudaMalloc(&d->bw_act[i], rows * (i == 3 ? 256 : 512) * sizeof(float)));
    CU_TRY(cudaMalloc(&d->bw_d0, rows * 512 * sizeof(float)));
    CU_TRY(cudaMalloc(&d->bw_d1, rows * 512 * sizeof(float)));
    CU_TRY(cudaMalloc(&d->bw_y, rows * sizeof(float)));
    d->bw_rows = rows;
  }
  const long long nblk = (M + 255) / 256 + (M + rows - 1) / rows;
  if (d->bw_blocks < nblk) {
    cudaFree(d->bw_partial); d->bw_partial = nullptr; d->bw_blocks = 0;
    CU_TRY(cudaMalloc(&d->bw_partial, nblk * 1024 * sizeof(float)));
    d->bw_blocks = nblk;
  }
  const float* P = d->params;
  const LayerOff* o = d->off;
  float** a = d->bw_act;
  CU_TRY(launch_fold_bias(P + o[0].w, kDecIn, 0, P + o[0].b, latent_dev, kLatent, kHid, d->bias0f, st));
  CU_TRY(launch_fold_bias(P + o[4].w, kHid, kSkipOut, P + o[4].b, latent_dev, kLatent, kHid, d->bias4f, st));
  long long blk = 0;
  for (long long m0 = 0; m0 < M; m0 += rows) {
    const long long m = (M - m0) < rows ? (M - m0) : rows;
    const float* X = xyz_dev + 3 * m0;
    float* y = sdf_dev != nullptr ? sdf_dev + m0 : d->bw_y;
    // forward, every activation kept
    CU_TRY(launch_scatter_xyz(X, m, a[3], st));
    CU_TRY(launch_linear_f32(X, 3, P + o[0].w + kLatent, kDecIn, d->bias0f, a[0], 512, m, 512, 3, true, st));
    CU_TRY(launch_linear_f32(a[0], 512, P + o[1].w, 512, P + o[1].b, a[1], 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(a[1], 512, P + o[2].w, 512, P + o[2].b, a[2], 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(a[2], 512, P + o[3].w, 512, P + o[3].b, a[3], 256, m, kSkipOut, 512, true, st));
    CU_TRY(launch_linear_f32(a[3], 256, d->w4s, 256, d->bias4f, a[4], 512, m, 512, 256, true, st));
    CU_TRY(launch_linear_f32(a[4], 512, P + o[5].w, 512, P + o[5].b, a[5], 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(a[5], 512, P + o[6].w, 512, P + o[6].b, a[6], 512, m, 512, 512, true, st));
    CU_TRY(launch_linear_f32(a[6], 512, P + o[7].w, 512, P + o[7].b, a[7], 512, m, 512, 512, true, st));
    CU_TRY(launch_head_tanh_f32(a[7], 512, P + o[8].w, P + o[8].b, y, m, 512, st));
    // backward
    float *da = d->bw_d0, *db = d->bw_d1;
    CU_TRY(launch_head_bwd_f32(dLdy_dev + m0, y, P + o[8].w, a[7], db, m, st));                               // delta7
    CU_TRY(launch_linear_bwd_f32(db, 512, P + o[7].w, 512, a[6], 512, da, 512, m, 512, 512, st));              // delta6
    CU_TRY(launch_linear_bwd_f32(da, 512, P + o[6].w, 512, a[5], 512, db, 512, m, 512, 512, st));              // delta5
    CU_TRY(launch_linear_bwd_f32(db, 512, P + o[5].w, 512, a[4], 512, da, 512, m, 512, 512, st));              // delta4
    CU_TRY(launch_colsum_f32(da, m, d->bw_partial + blk * 1024, 1, st));
    CU_TRY(launch_linear_bwd_f32(da, 512, P + o[4].w, 512, a[3], 256, db, 512, m, 512, kSkipOut, st));         // delta3 (253 wide)
    CU_TRY(launch_linear_bwd_f32(db, 512, P + o[3].w, 512, a[2], 512, da, 512, m, kSkipOut, 512, st));         // delta2
    CU_TRY(launch_linear_bwd_f32(da, 512, P + o[2].w, 512, a[1], 512, db, 512, m, 512, 512, st));              // delta1
    CU_TRY(launch_linear_bwd_f32(db, 512, P + o[1].w, 512, a[0], 512, da, 512, m, 512, 512, st));              // delta0
    CU_TRY(launch_colsum_f32(da, m, d->bw_partial + blk * 1024, 0, st));
    blk += (m + 255) / 256;
  }
  CU_TRY(launch_vjp_finish(d->bw_partial, static_cast<int>(blk), P + o[0].w, P + o[4].w, grad_latent_dev, st));
  return SDFB_OK;
}

// The same gradient on the tensor pipe: ONE launch of the forward + backward instance of the fused kernel (every
// tile is decoded, then run backwards through the transposed weight blocks while it is still in shared memory),
// then the small contraction of the two column sums with the fp32 latent columns of W0 and W4.
// `target_dev` != nullptr: loss mode - the kernel forms the upstream gradient of mean |clamp(sdf) - clamp(target)| itself.
namespace {
int vjp_tc(sdfb_decoder* d, const float* latent_dev, const float* xyz_dev, int64_t M, const float* dLdy_dev,
           const float* target_dev, float clamp, float* grad_latent_dev, float* loss_dev, float* sdf_dev, int precision,
           cudaStream_t st) {
  if (precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "the tensor-core gradient runs in bf16 or fp16 (precision %d); fp32: sdfb_decoder_vjp_latent", precision);
  if (M == 0) {
    CU_TRY(cudaMemsetAsync(grad_latent_dev, 0, kLatent * sizeof(float), st));
    if (loss_dev != nullptr) CU_TRY(cudaMemsetAsync(loss_dev, 0, sizeof(float), st));
    return SDFB_OK;
  }
  // workspaces: allocated on first use, kept (each checked on its own: a failed allocation is retried by the next call)
  if (d->bw_masks == nullptr) CU_TRY(cudaMalloc(&d->bw_masks, static_cast<size_t>(d->num_sms) * 8 * 16 * kTileM * sizeof(uint32_t)));
  if (d->bw_colsum == nullptr) CU_TRY(cudaMalloc(&d->bw_colsum, static_cast<size_t>(d->num_sms) * 4 * 1024 * sizeof(float)));
  if (d->bw_amax == nullptr) CU_TRY(cudaMalloc(&d->bw_amax, sizeof(unsigned int)));
  if (d->bw_loss == nullptr) CU_TRY(cudaMalloc(&d->bw_loss, static_cast<size_t>(d->num_sms) * 4 * sizeof(float)));
  const bool loss_mode = target_dev != nullptr;
  if (!loss_mode) CU_TRY(launch_abs_max(dLdy_dev, M, d->bw_amax, st));
  const bool fp16 = precision == SDFB_PREC_FP16;
  const float* P = d->params;
  const LayerOff* o = d->off;
  CU_TRY(launch_fold_latent(P + o[0].w, P + o[0].b, P + o[4].w, P + o[4].b, latent_dev, d->consts, st));
  DecodeParams p{};
  p.wstream = d->wstream[fp16 ? 1 : 0];
  p.consts = d->consts;
  p.xyz = xyz_dev;
  p.out = sdf_dev;
  p.M = M;
  p.status = d->status;
  p.status_host = d->status_host_dev;
  p.dump_pass = -1;
  p.timeout_ns = d->timeout_ns;
  p.debug_flags = d->debug_flags;
  p.prof = d->prof;
  p.bwd = 1;
  p.dLdy = dLdy_dev;
  p.dLdy_amax = d->bw_amax;
  p.target = target_dev;
  p.clamp = clamp;
  p.loss_partial = loss_mode ? d->bw_loss : nullptr;
  p.mask_scratch = d->bw_masks;
  p.colsum = d->bw_colsum;
  CU_TRY(cudaEventRecord(d->ev0, st));
  CU_TRY(launch_fused_decoder(p, d->tmap[fp16 ? 1 : 0], fp16, d->num_sms, st));
  CU_TRY(cudaEventRecord(d->ev1, st));
  d->timed = true;
  const long long tiles = (M + 2 * kTileM - 1) / (2 * kTileM);
  const long long pairs = tiles < d->num_sms / 2 ? tiles : d->num_sms / 2;
  CU_TRY(launch_vjp_finish(d->bw_colsum, static_cast<int>(2 * pairs * 4), P + o[0].w, P + o[4].w, grad_latent_dev, st,
                           loss_mode ? nullptr : d->bw_amax, loss_mode ? d->bw_loss : nullptr,
                           loss_mode ? 1.f / static_cast<float>(M) : 1.f, loss_mode ? loss_dev : nullptr));
  return SDFB_OK;
}
}  // namespace

int sdfb_decoder_vjp_latent_tc(sdfb_decoder* d, const float* latent_dev, const float* xyz_dev, int64_t M, const float* dLdy_dev,
                               float* grad_latent_dev, float* sdf_dev, int precision, void* stream) {
  if (!d || !latent_dev || !grad_latent_dev || (M > 0 && (!xyz_dev || !dLdy_dev))) return fail(SDFB_E_INVALID, "null argument");
  if (M < 0) return fail(SDFB_E_INVALID, "negative point count");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  return vjp_tc(d, latent_dev, xyz_dev, M, dLdy_dev, nullptr, 0.f, grad_latent_dev, nullptr, sdf_dev, precision,
                static_cast<cudaStream_t>(stream));
}

// One step's worth of auto-decoder fitting in one launch: loss = mean_m |clamp(sdf_m) - clamp(target_m)| (clamp to
// [-clamp_dist, clamp_dist]) and its gradient w.r.t. the latent, the upstream gradient formed inside the kernel.
int sdfb_decoder_fit_loss_grad(sdfb_decoder* d, const float* latent_dev, const float* xyz_dev, int64_t M, const float* target_dev,
                               float clamp_dist, float* grad_latent_dev, float* loss_dev, float* sdf_dev, int precision,
                               void* stream) {
  if (!d || !latent_dev || !grad_latent_dev || !loss_dev || (M > 0 && (!xyz_dev || !target_dev)))
    return fail(SDFB_E_INVALID, "null argument");
  if (M < 0) return fail(SDFB_E_INVALID, "negative point count");
  if (!(clamp_dist > 0.f)) return fail(SDFB_E_INVALID, "clamp distance must be positive");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  return vjp_tc(d, latent_dev, xyz_dev, M, nullptr, target_dev, clamp_dist, grad_latent_dev, loss_dev, sdf_dev, precision,
                static_cast<cudaStream_t>(stream));
}

// A batch of shapes, each with its own latent and its own points_per_shape samples: one fold + one forward + backward
// launch + one finish per shape, back to back on the stream (the shapes are independent; nothing is synchronised).
int sdfb_latent_adam_step(float* latents_dev, float* m_dev, float* v_dev, const float* grad_dev, float* loss_dev, int batch,
                          float lr, float reg, double beta1, double beta2, float adam_eps, int step, void* stream) {
  if (batch < 0 || step < 1) return fail(SDFB_E_INVALID, "negative batch or step < 1");
  if (batch > 0 && (!latents_dev || !m_dev || !v_dev || !grad_dev)) return fail(SDFB_E_INVALID, "null argument");
  if (!(beta1 >= 0. && beta1 < 1. && beta2 >= 0. && beta2 < 1.)) return fail(SDFB_E_INVALID, "betas must be in [0, 1)");
  CU_TRY(launch_latent_adam(latents_dev, m_dev, v_dev, grad_dev, loss_dev, batch, kLatent, lr, reg, beta1, beta2, adam_eps, step,
                            static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

int sdfb_decoder_fit_loss_grad_batch(sdfb_decoder* d, const float* latents_dev, const float* xyz_dev, int batch,
                                     int64_t points_per_shape, const float* target_dev, float clamp_dist, float* grad_latents_dev,
                                     float* loss_dev, int precision, void* stream) {
  if (!d || (batch > 0 && (!latents_dev || !grad_latents_dev || !loss_dev))) return fail(SDFB_E_INVALID, "null argument");
  if (batch < 0 || points_per_shape < 0) return fail(SDFB_E_INVALID, "negative batch or point count");
  if (batch > 0 && points_per_shape > 0 && (!xyz_dev || !target_dev)) return fail(SDFB_E_INVALID, "null argument");
  if (!(clamp_dist > 0.f)) return fail(SDFB_E_INVALID, "clamp distance must be positive");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int b = 0; b < batch; ++b) {
    const long long o = static_cast<long long>(b) * points_per_shape;
    int rc = vjp_tc(d, latents_dev + static_cast<long long>(b) * kLatent, xyz_dev + 3 * o, points_per_shape, nullptr, target_dev + o,
                    clamp_dist, grad_latents_dev + static_cast<long long>(b) * kLatent, loss_dev + b, nullptr, precision, st);
    if (rc) return rc;
  }
  return SDFB_OK;
}

// BASELINE configs[4] as one call per rank (SURVEY.md section 8e): rank r of `comm` decodes planes
// [r per, min((r + 1) per, res)), per = ceil(res / world), straight into its block of the symmetric buffer, in
// sub-slabs; each finished sub-slab is PUSHED into the same place of every peer's copy by the copy engines while the
// next one is being decoded (comm.cu).  The mask's halo plane is recomputed locally; the packed mask of the rank's
// cell layers is pushed last.  A barrier at the start keeps a rank from overwriting results a slower rank is still
// reading from the previous call (everything the caller queued on `stream` before this call is ordered before it), a
// barrier at the end makes the whole grid valid on every rank in stream order.
int sdfb_decode_grid_sharded(sdfb_decoder* d, sdfb_comm* c, const float* latent_dev, int res, int want_mask, int sub_planes,
                             int precision, float** sdf_full_dev, uint32_t** mask_bits_dev, size_t* mask_words_per_rank,
                             void* stream) {
  if (!d || !c || !latent_dev || !sdf_full_dev) return fail(SDFB_E_INVALID, "null argument");
  if (res < 2 || res > 2048) return fail(SDFB_E_INVALID, "res %d outside [2, 2048]", res);
  if (want_mask && (!mask_bits_dev || !mask_words_per_rank)) return fail(SDFB_E_INVALID, "null argument");
  if (c->device != d->device) return fail(SDFB_E_INVALID, "decoder on device %d, communicator on device %d", d->device, c->device);
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long plane = static_cast<long long>(res) * res;
  const int per = (res + c->world - 1) / c->world;
  const int z0 = c->rank * per < res ? c->rank * per : res;
  const int z1 = z0 + per < res ? z0 + per : res;
  const long long cells_layer = static_cast<long long>(res - 1) * (res - 1);
  const size_t words = static_cast<size_t>((per * cells_layer + 31) >> 5);
  const size_t off_mask = (static_cast<size_t>(plane) * res * sizeof(float) + 255) / 256 * 256;
  const size_t total = off_mask + (want_mask ? words * c->world * sizeof(uint32_t) : 0);
  int rc = comm_shared_alloc(c, total);            // collective on first use / growth
  if (rc) return rc;
  float* full = static_cast<float*>(c->local);
  uint32_t* mbits = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(c->local) + off_mask);
  *sdf_full_dev = full;
  if (want_mask) { *mask_bits_dev = mbits; *mask_words_per_rank = words; }
  rc = comm_barrier(c, st);
  if (rc) return rc;
  if (z1 > z0) {
    const bool halo = want_mask && z1 < res;
    const int planes = z1 - z0 + (halo ? 1 : 0);
    const int layers = (halo ? z1 : (z1 < res - 1 ? z1 : res - 1)) - z0;
    long long sub = sub_planes > 0 ? sub_planes : (2097152 + plane - 1) / plane;     // >= 2^21 queries per launch
    if (sub * 16 < planes) sub = (planes + 15) / 16;
    if (want_mask) {                               // sign words of a sub-slab must start on a word boundary
      long long unit = 1;
      while ((unit * plane) % 32 != 0) unit *= 2;
      sub = (sub + unit - 1) / unit * unit;
      rc = ensure_signs(d, (planes * plane + 31) >> 5, st);
      if (rc == SDFB_OK && planes >= 2) rc = ensure_rowmask(d, mask_rows_words(planes, res, res));
      if (rc) return rc;
    }
    for (long long za = 0; za < z1 - z0; za += sub) {
      long long zb = za + sub < z1 - z0 ? za + sub : z1 - z0;
      const long long zpush = zb;
      if (zb == z1 - z0 && halo) zb += 1;          // the halo plane rides with the last sub-slab (it is not pushed)
      rc = decode_any(d, latent_dev, nullptr, res, (z0 + za) * plane, (zb - za) * plane, full + (z0 + za) * plane, precision, st,
                      want_mask ? d->signs + ((za * plane) >> 5) : nullptr);
      if (rc) return rc;
      rc = comm_push(c, static_cast<size_t>((z0 + za) * plane) * sizeof(float), static_cast<size_t>((zpush - za) * plane) * sizeof(float), st);
      if (rc) return rc;
    }
    if (want_mask && layers > 0) {
      uint32_t* mine = mbits + static_cast<size_t>(c->rank) * words;
      CU_TRY(launch_mask_from_bits(d->signs, planes, res, res, nullptr, mine, d->rowmask, st));
      rc = comm_push(c, off_mask + static_cast<size_t>(c->rank) * words * sizeof(uint32_t),
                     static_cast<size_t>((layers * cells_layer + 31) >> 5) * sizeof(uint32_t), st);
      if (rc) return rc;
    }
  }
  rc = comm_join_pushes(c, st);
  if (rc) return rc;
  return comm_barrier(c, st);
}

int sdfb_decode_grid_host(sdfb_decoder* d, const float* latent_host, int res, int z0, int z1, float* sdf_host,
                          uint8_t* mask_host, int precision) {
  if (!d || !latent_host || !sdf_host) return fail(SDFB_E_INVALID, "null argument");
  if (res < 2 || res > 2048 || z0 < 0 || z1 > res || z0 > z1) return fail(SDFB_E_INVALID, "bad grid arguments");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  if (int orc = order_after_user(d, d->st_compute)) return orc;
  const long long plane = static_cast<long long>(res) * res;
  const bool halo = mask_host != nullptr && z1 < res && z1 > z0;
  const long long n_sdf = (z1 - z0 + (halo ? 1 : 0)) * plane;
  const int layers = (halo ? z1 : (z1 < res - 1 ? z1 : res - 1)) - z0;
  const long long n_mask = mask_host && layers > 0 ? static_cast<long long>(layers) * (res - 1) * (res - 1) : 0;
  const size_t off_sdf = 1024, off_mask = off_sdf + ((n_sdf * 4 + 255) / 256) * 256;
  int rc = ensure_stage(&d->pin, &d->pin_bytes, &d->dstage, &d->dstage_bytes, 1024, off_mask + n_mask);
  if (rc) return rc;
  uint8_t* base = static_cast<uint8_t*>(d->dstage);
  float* lat_dev = reinterpret_cast<float*>(base);
  float* sdf_dev = reinterpret_cast<float*>(base + off_sdf);
  std::memcpy(d->pin, latent_host, kLatent * sizeof(float));
  CU_TRY(cudaMemcpyAsync(lat_dev, d->pin, kLatent * sizeof(float), cudaMemcpyHostToDevice, d->st_compute));
  // z-chunks: the copy-out of chunk c runs on the copy stream while chunk c + 1 is being decoded
  const int planes = z1 - z0 + (halo ? 1 : 0);
  long long per = (2097152 + plane - 1) / plane;                   // >= 2^21 queries per chunk keeps the persistent kernel's tail < 1 %
  if (per * 16 < planes) per = (planes + 15) / 16;
  // With a mask, every chunk's launch also writes the sign bit-planes of its queries into the context's buffer (32
  // queries per word): a chunk must then start on a word boundary, i.e. hold a multiple of 32 queries.
  const bool want_mask = n_mask > 0;
  if (want_mask) {
    long long unit = 1;
    while ((unit * plane) % 32 != 0) unit *= 2;                   // 32 / gcd(plane, 32)
    per = (per + unit - 1) / unit * unit;
    rc = ensure_signs(d, (n_sdf + 31) >> 5, d->st_compute);
    if (rc == SDFB_OK) rc = ensure_rowmask(d, mask_rows_words(planes, res, res));
    if (rc) return rc;
  }
  int nchunk = 0;
  for (long long za = 0; za < planes; za += per, ++nchunk) {
    const long long zb = za + per < planes ? za + per : planes;
    rc = decode_any(d, lat_dev, nullptr, res, (z0 + za) * plane, (zb - za) * plane, sdf_dev + za * plane, precision, d->st_compute,
                    want_mask ? d->signs + ((za * plane) >> 5) : nullptr);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(d->chunk_ev[nchunk], d->st_compute));
    CU_TRY(cudaStreamWaitEvent(d->st_copy, d->chunk_ev[nchunk], 0));
    const long long zc = zb < (z1 - z0) ? zb : (z1 - z0);           // the halo plane stays on the device
    if (zc > za)
      CU_TRY(cudaMemcpyAsync(sdf_host + za * plane, sdf_dev + za * plane, (zc - za) * plane * sizeof(float),
                             cudaMemcpyDeviceToHost, d->st_copy));
  }
  if (n_mask) {   // the same combine of the sign bit-planes as the device path (no second pass over the fp32 field)
    CU_TRY(launch_mask_from_bits(d->signs, planes, res, res, base + off_mask, nullptr, d->rowmask, d->st_compute));
    CU_TRY(cudaEventRecord(d->chunk_ev[16], d->st_compute));
    CU_TRY(cudaStreamWaitEvent(d->st_copy, d->chunk_ev[16], 0));
    CU_TRY(cudaMemcpyAsync(mask_host, base + off_mask, n_mask, cudaMemcpyDeviceToHost, d->st_copy));
  }
  CU_TRY(cudaStreamSynchronize(d->st_compute));
  CU_TRY(cudaStreamSynchronize(d->st_copy));
  return precision == SDFB_PREC_FP32 ? SDFB_OK : kernel_status(d);
}

int sdfb_decode_points_host(sdfb_decoder* d, const float* latent_host, const float* xyz_host, int64_t M,
                            float* sdf_host, int precision) {
  if (!d || !latent_host || M < 0 || (M > 0 && (!xyz_host || !sdf_host))) return fail(SDFB_E_INVALID, "bad argument");
  if (M == 0) return SDFB_OK;
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  if (int orc = order_after_user(d, d->st_compute)) return orc;
  const size_t off_xyz = 1024, off_sdf = off_xyz + ((M * 12 + 255) / 256) * 256;
  int rc = ensure_stage(&d->pin, &d->pin_bytes, &d->dstage, &d->dstage_bytes, 1024, off_sdf + M * 4);
  if (rc) return rc;
  if (d->st_in == nullptr) CU_TRY(cudaStreamCreateWithFlags(&d->st_in, cudaStreamNonBlocking));
  uint8_t* base = static_cast<uint8_t*>(d->dstage);
  float* lat_dev = reinterpret_cast<float*>(base);
  float* xyz_dev = reinterpret_cast<float*>(base + off_xyz);
  float* sdf_dev = reinterpret_cast<float*>(base + off_sdf);
  std::memcpy(d->pin, latent_host, kLatent * sizeof(float));
  CU_TRY(cudaMemcpyAsync(lat_dev, d->pin, kLatent * sizeof(float), cudaMemcpyHostToDevice, d->st_compute));
  // three-stage pipeline over chunks of points: copy-in (st_in) | decode (st_compute) | copy-out (st_copy)
  long long per = 2097152;
  if (per * 16 < M) per = (M + 15) / 16;
  int c = 0;
  for (long long m0 = 0; m0 < M; m0 += per, ++c) {
    const long long m = (M - m0) < per ? (M - m0) : per;
    CU_TRY(cudaMemcpyAsync(xyz_dev + 3 * m0, xyz_host + 3 * m0, m * 12, cudaMemcpyHostToDevice, d->st_in));
    CU_TRY(cudaEventRecord(d->in_ev[c], d->st_in));
    CU_TRY(cudaStreamWaitEvent(d->st_compute, d->in_ev[c], 0));
    rc = decode_any(d, lat_dev, xyz_dev + 3 * m0, 0, 0, m, sdf_dev + m0, precision, d->st_compute);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(d->chunk_ev[c], d->st_compute));
    CU_TRY(cudaStreamWaitEvent(d->st_copy, d->chunk_ev[c], 0));
    CU_TRY(cudaMemcpyAsync(sdf_host + m0, sdf_dev + m0, m * sizeof(float), cudaMemcpyDeviceToHost, d->st_copy));
  }
  CU_TRY(cudaStreamSynchronize(d->st_in));
  CU_TRY(cudaStreamSynchronize(d->st_compute));
  CU_TRY(cudaStreamSynchronize(d->st_copy));
  return precision == SDFB_PREC_FP32 ? SDFB_OK : kernel_status(d);
}

int sdfb_grid_points(int res, int z0, int z1, float* xyz_dev, void* stream) {
  if (!xyz_dev) return fail(SDFB_E_INVALID, "null argument");
  if (res < 2 || res > 2048 || z0 < 0 || z1 > res || z0 > z1) return fail(SDFB_E_INVALID, "bad grid arguments");
  const long long plane = static_cast<long long>(res) * res;
  CU_TRY(launch_grid_xyz(res, z0 * plane, (z1 - z0) * plane, xyz_dev, nullptr, static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

int sdfb_sign_change_mask(const float* sdf_dev, int nz, int ny, int nx, uint8_t* mask_dev, void* stream) {
  if (!sdf_dev || !mask_dev) return fail(SDFB_E_INVALID, "null argument");
  if (nz < 1 || ny < 1 || nx < 1) return fail(SDFB_E_INVALID, "bad field shape");
  CU_TRY(launch_sign_change_mask(sdf_dev, nz, ny, nx, mask_dev, static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

// ------------------------------------------------------------ marching cubes ----
namespace {
struct McLayout { size_t off_bits, off_groups, off_temp, total; long long groups, nodes; size_t temp_bytes; };
McLayout mc_layout(long long nodes, long long cells) {
  McLayout L{};
  L.nodes = nodes;
  L.groups = (cells + 31) >> 5;
  L.temp_bytes = mc_scan_temp_bytes(L.groups);
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  L.off_bits = 0;
  L.off_groups = up(static_cast<size_t>((L.nodes + 31) >> 5) * 4);
  L.off_temp = L.off_groups + up(static_cast<size_t>(L.groups + 1) * 4);
  L.total = L.off_temp + up(L.temp_bytes);
  return L;
}

}  // namespace

int sdfb_mc_workspace_bytes(int nz, int ny, int nx, size_t* bytes) {
  if (!bytes) return fail(SDFB_E_INVALID, "null argument");
  if (nz < 2 || ny < 2 || nx < 2) return fail(SDFB_E_INVALID, "the field must have at least 2 nodes per axis");
  const McGeom g = mc_dense_geom(nz, ny, nx, nx, 0);
  *bytes = mc_layout(g.total_nodes, g.total_cells).total;
  return SDFB_OK;
}

int sdfb_mc_count(const float* sdf_dev, const uint32_t* sign_bits_dev, int nz, int ny, int nx, void* workspace_dev,
                  size_t workspace_bytes, int64_t* n_triangles_host, void* stream) {
  if (!sdf_dev || !workspace_dev || !n_triangles_host) return fail(SDFB_E_INVALID, "null argument");
  if (nz < 2 || ny < 2 || nx < 2) return fail(SDFB_E_INVALID, "the field must have at least 2 nodes per axis");
  const McGeom g = mc_dense_geom(nz, ny, nx, nx, 0);
  const McLayout L = mc_layout(g.total_nodes, g.total_cells);
  if (workspace_bytes < L.total) return fail(SDFB_E_INVALID, "workspace holds %zu bytes, %zu needed", workspace_bytes, L.total);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  unsigned int* bits = reinterpret_cast<unsigned int*>(ws + L.off_bits);
  unsigned int* groups = reinterpret_cast<unsigned int*>(ws + L.off_groups);
  if (sign_bits_dev != nullptr)
    CU_TRY(cudaMemcpyAsync(bits, sign_bits_dev, static_cast<size_t>((L.nodes + 31) >> 5) * 4, cudaMemcpyDeviceToDevice, st));
  else
    CU_TRY(launch_sign_bits(sdf_dev, L.nodes, bits, st));
  CU_TRY(launch_mc_count_scan(bits, g, groups, ws + L.off_temp, L.temp_bytes, st));
  unsigned int total = 0;
  CU_TRY(cudaMemcpyAsync(&total, groups + L.groups, sizeof(total), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  *n_triangles_host = total;
  return SDFB_OK;
}

int sdfb_mc_generate(const float* sdf_dev, int nz, int ny, int nx, int res, int z0, const void* workspace_dev,
                     float* triangles_dev, int64_t* edge_keys_dev, void* stream) {
  if (!sdf_dev || !workspace_dev || !triangles_dev) return fail(SDFB_E_INVALID, "null argument");
  if (nz < 2 || ny < 2 || nx < 2 || res < 2 || z0 < 0) return fail(SDFB_E_INVALID, "bad field shape");
  const McGeom g = mc_dense_geom(nz, ny, nx, res, z0);
  const McLayout L = mc_layout(g.total_nodes, g.total_cells);
  const uint8_t* ws = static_cast<const uint8_t*>(workspace_dev);
  CU_TRY(launch_mc_generate(sdf_dev, reinterpret_cast<const unsigned int*>(ws + L.off_bits),
                            reinterpret_cast<const unsigned int*>(ws + L.off_groups), g, triangles_dev,
                            reinterpret_cast<long long*>(edge_keys_dev), static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

// ---- welding the soup into an indexed mesh ----
int sdfb_mc_weld_workspace_bytes(int res, size_t* bytes) {
  if (!bytes || res < 2) return fail(SDFB_E_INVALID, "bad argument");
  *bytes = mc_weld_workspace_bytes(3ll * res * res * res) + 256;
  return SDFB_OK;
}

int sdfb_mc_weld_count(const int64_t* edge_keys_dev, int64_t n_triangles, int res, void* workspace_dev, size_t workspace_bytes,
                       int64_t* n_vertices_host, void* stream) {
  if (!workspace_dev || !n_vertices_host || res < 2 || n_triangles < 0 || (n_triangles > 0 && !edge_keys_dev))
    return fail(SDFB_E_INVALID, "bad argument");
  const long long range = 3ll * res * res * res;
  if (workspace_bytes < mc_weld_workspace_bytes(range) + 256) return fail(SDFB_E_INVALID, "workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  int* count_dev = reinterpret_cast<int*>(ws);
  CU_TRY(launch_mc_weld_count(reinterpret_cast<const long long*>(edge_keys_dev), 3 * n_triangles, range, ws + 256, count_dev, st));
  int count = 0;
  CU_TRY(cudaMemcpyAsync(&count, count_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  *n_vertices_host = count;
  return SDFB_OK;
}

int sdfb_mc_weld_fill(const float* triangles_dev, const int64_t* edge_keys_dev, int64_t n_triangles, int res, const void* workspace_dev,
                      float* vertices_dev, int64_t* faces_dev, void* stream) {
  if (!workspace_dev || res < 2 || n_triangles < 0) return fail(SDFB_E_INVALID, "bad argument");
  if (n_triangles > 0 && (!triangles_dev || !edge_keys_dev || !vertices_dev || !faces_dev)) return fail(SDFB_E_INVALID, "null argument");
  CU_TRY(launch_mc_weld_fill(triangles_dev, reinterpret_cast<const long long*>(edge_keys_dev), 3 * n_triangles, 3ll * res * res * res,
                             static_cast<const uint8_t*>(workspace_dev) + 256, vertices_dev, reinterpret_cast<long long*>(faces_dev),
                             static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

// ---- hierarchical sparse decode (sparse.cu): decode only where the surface can be, hand the dense MC kernels a field that
// is valid around the surface and the complete sign bit-planes ----
namespace {
int sparse_reserve_queries(sdfb_decoder* d, long long n) {
  if (d->sp.idx_cap >= n) return SDFB_OK;
  cudaFree(d->sp.idx); cudaFree(d->sp.xyz); cudaFree(d->sp.vals);
  d->sp.idx = nullptr; d->sp.xyz = nullptr; d->sp.vals = nullptr; d->sp.idx_cap = 0;
  const long long cap = n + n / 8 + 1024;
  CU_TRY(cudaMalloc(&d->sp.idx, cap * sizeof(unsigned int)));
  CU_TRY(cudaMalloc(&d->sp.xyz, cap * 3 * sizeof(float)));
  CU_TRY(cudaMalloc(&d->sp.vals, cap * sizeof(float)));
  d->sp.idx_cap = cap;
  return SDFB_OK;
}
// bitmap -> ascending index list in d->sp.idx (synchronises the stream to learn the count)
int sparse_compact(sdfb_decoder* d, const unsigned int* bits, long long words, long long* n_out, cudaStream_t st) {
  const long long tiles = bitmap_scan_tiles(words);
  CU_TRY(launch_bitmap_count(bits, words, d->sp.tiles, st));
  unsigned int total = 0;
  CU_TRY(cudaMemcpyAsync(&total, d->sp.tiles + tiles, sizeof(total), cudaMemcpyDeviceToHost, st));
  CU_TRY(cudaStreamSynchronize(st));
  *n_out = total;
  int rc = sparse_reserve_queries(d, total);
  if (rc) return rc;
  if (total) CU_TRY(launch_bitmap_emit(bits, words, d->sp.tiles, d->sp.idx, st));
  return SDFB_OK;
}
// decode the listed nodes (d->sp.idx[0 .. n)) and scatter the values into the dense field
int sparse_decode_nodes(sdfb_decoder* d, const float* latent_dev, int res, long long n, float* dense, int precision, cudaStream_t st) {
  if (n == 0) return SDFB_OK;
  CU_TRY(launch_node_points(res, d->sp.idx, n, d->sp.xyz, st));
  int rc = decode_any(d, latent_dev, d->sp.xyz, 0, 0, n, d->sp.vals, precision, st);
  if (rc) return rc;
  CU_TRY(launch_scatter(d->sp.idx, d->sp.vals, n, dense, st));
  return SDFB_OK;
}
}  // namespace

int sdfb_decode_sparse_field(sdfb_decoder* d, const float* latent_dev, int res, float lipschitz, float safety1, float safety2,
                             float local_floor, float* sdf_dense_dev, uint32_t* sign_bits_dev, int precision, int64_t* stats_host,
                             void* stream) {
  if (!d || !latent_dev || !sdf_dense_dev || !sign_bits_dev) return fail(SDFB_E_INVALID, "null argument");
  if (res < 3 || res > 1024) return fail(SDFB_E_INVALID, "res %d outside [3, 1024] (node indices are 32-bit)", res);
  if (!(lipschitz >= 0.f) || !(safety1 >= 1.f) || !(safety2 >= 1.f) || !(local_floor >= 0.f) || local_floor > 1.f)
    return fail(SDFB_E_INVALID, "bad lipschitz bound, safety factor or local floor");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  constexpr int B1 = 8, B2 = 2;
  const int nb1 = (res - 1 + B1 - 1) / B1;
  const long long nodes = static_cast<long long>(res) * res * res, words = (nodes + 31) >> 5;
  const long long corners = static_cast<long long>(nb1 + 1) * (nb1 + 1) * (nb1 + 1), blocks = static_cast<long long>(nb1) * nb1 * nb1;
  const float h = 2.f / static_cast<float>(res - 1);
  auto& sp = d->sp;
  if (sp.words < words) {
    cudaFree(sp.need1); cudaFree(sp.need2); cudaFree(sp.tiles); sp.need1 = sp.need2 = sp.tiles = nullptr; sp.words = 0;
    CU_TRY(cudaMalloc(&sp.need1, words * sizeof(unsigned int)));
    CU_TRY(cudaMalloc(&sp.need2, words * sizeof(unsigned int)));
    CU_TRY(cudaMalloc(&sp.tiles, (bitmap_scan_tiles(words) + 1) * sizeof(unsigned int)));
    sp.words = words;
  }
  if (sp.corners < corners) {
    cudaFree(sp.cs); cudaFree(sp.keep); cudaFree(sp.ids); cudaFree(sp.qblk); sp.cs = nullptr; sp.keep = nullptr; sp.ids = nullptr; sp.qblk = nullptr;
    sp.corners = 0;
    CU_TRY(cudaMalloc(&sp.qblk, blocks * sizeof(unsigned int)));
    CU_TRY(cudaMalloc(&sp.cs, corners * sizeof(float)));
    CU_TRY(cudaMalloc(&sp.keep, ((blocks + 31) / 32 + 1) * sizeof(unsigned int)));
    CU_TRY(cudaMalloc(&sp.ids, blocks * sizeof(int)));
    sp.corners = corners;
  }
  if (sp.lip == nullptr) CU_TRY(cudaMalloc(&sp.lip, 4 * sizeof(unsigned int)));
  if (sp.kept == nullptr) CU_TRY(cudaMalloc(&sp.kept, sizeof(unsigned long long)));
  CU_TRY(cudaMemsetAsync(sp.need1, 0, words * sizeof(unsigned int), st));
  CU_TRY(cudaMemsetAsync(sp.need2, 0, words * sizeof(unsigned int), st));
  CU_TRY(cudaMemsetAsync(sp.keep, 0, ((blocks + 31) / 32 + 1) * sizeof(unsigned int), st));
  CU_TRY(cudaMemsetAsync(sp.lip, 0, 4 * sizeof(unsigned int), st));
  CU_TRY(cudaMemsetAsync(sp.kept, 0, sizeof(unsigned long long), st));
  // level 1: the (nb1 + 1)^3 block corners
  int rc = sparse_reserve_queries(d, corners);
  if (rc) return rc;
  CU_TRY(launch_corner_nodes(res, B1, nb1, sp.idx, st));
  CU_TRY(launch_node_points(res, sp.idx, corners, sp.xyz, st));
  rc = decode_any(d, latent_dev, sp.xyz, 0, 0, corners, sp.cs, precision, st);
  if (rc) return rc;
  CU_TRY(launch_scatter(sp.idx, sp.cs, corners, sdf_dense_dev, st));
  float lip1_node;                                     // Lipschitz bound in field units per node spacing
  float raw1 = 0.f;
  if (lipschitz > 0.f) {
    lip1_node = lipschitz * h;
  } else {
    CU_TRY(launch_corner_lipschitz(sp.cs, res, B1, nb1, sp.lip, st));
    unsigned int bits = 0;
    CU_TRY(cudaMemcpyAsync(&bits, sp.lip, sizeof(bits), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    std::memcpy(&raw1, &bits, sizeof(raw1));
    lip1_node = safety1 * raw1;
  }
  const float tau1 = lip1_node * B1 * 0.8660254f;
  CU_TRY(launch_select_blocks_bits(sp.cs, nb1, tau1, sp.keep, st));
  // kept block ids: the same compaction as for nodes (ascending ids), into sp.idx, then copied to sp.ids
  long long nA = 0;
  rc = sparse_compact(d, sp.keep, (blocks + 31) / 32, &nA, st);
  if (rc) return rc;
  if (nA) CU_TRY(cudaMemcpyAsync(sp.ids, sp.idx, nA * sizeof(int), cudaMemcpyDeviceToDevice, st));
  // level 2: the sub-block lattice inside the kept blocks, every node once
  long long n1 = 0, n2 = 0;
  unsigned long long kept_sub = 0;
  float raw2 = 0.f;
  if (nA) {
    CU_TRY(launch_mark_sub_corners(res, B1, B2, nb1, sp.ids, nA, sp.need1, st));
    rc = sparse_compact(d, sp.need1, words, &n1, st);
    if (rc) return rc;
    rc = sparse_decode_nodes(d, latent_dev, res, n1, sdf_dense_dev, precision, st);
    if (rc) return rc;
    // the finer lattice sees the field's steepest slopes better than the coarse one: L2 = safety2 * max(raw1, raw2)
    // (sp.lip[0] = level-1 quotient, sp.lip[1] = level-2 quotient; the selection kernel takes the larger)
    const bool local = local_floor > 0.f && !(lipschitz > 0.f);
    if (local) CU_TRY(cudaMemsetAsync(sp.qblk, 0, nA * sizeof(unsigned int), st));
    if (!(lipschitz > 0.f)) CU_TRY(launch_sub_lipschitz(res, B1, B2, nb1, sp.ids, nA, sdf_dense_dev, sp.lip + 1, local ? sp.qblk : nullptr, st));
    CU_TRY(launch_select_sub_blocks(res, B1, B2, nb1, sp.ids, nA, sdf_dense_dev, sp.lip, lipschitz > 0.f ? lipschitz * h : 0.f,
                                    safety2, local ? sp.qblk : nullptr, local_floor, sp.need2, sp.kept, st));
    CU_TRY(launch_andnot(sp.need2, sp.need1, words, st));
    rc = sparse_compact(d, sp.need2, words, &n2, st);
    if (rc) return rc;
    rc = sparse_decode_nodes(d, latent_dev, res, n2, sdf_dense_dev, precision, st);
    if (rc) return rc;
  }
  CU_TRY(launch_fill_signs(res, B1, B2, nb1, sdf_dense_dev, sp.need1, sp.need2, sp.cs, sign_bits_dev, st));
  if (stats_host != nullptr) {
    unsigned int bits2 = 0;
    CU_TRY(cudaMemcpyAsync(&kept_sub, sp.kept, sizeof(kept_sub), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(&bits2, sp.lip + 1, sizeof(bits2), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    std::memcpy(&raw2, &bits2, sizeof(raw2));
    stats_host[0] = corners; stats_host[1] = nA; stats_host[2] = n1; stats_host[3] = static_cast<int64_t>(kept_sub); stats_host[4] = n2;
    stats_host[5] = corners + n1 + n2;                                       // queries decoded in total
    stats_host[6] = static_cast<int64_t>(1e6f * raw1 / h);                   // level-1 difference quotient, field units per unit length, x 1e6
    stats_host[7] = static_cast<int64_t>(1e6f * raw2 / h);                   // level-2
  }
  return SDFB_OK;
}

int sdfb_decode_debug_pass(sdfb_decoder* d, const float* latent_dev, int res, int pass, float* dump_dev,
                           int precision, void* stream) {
  if (!d || !latent_dev || !dump_dev) return fail(SDFB_E_INVALID, "null argument");
  if (pass < 0 || pass >= kPasses) return fail(SDFB_E_INVALID, "pass %d outside [0, 13)", pass);
  if (precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "debug pass dump exists for the tensor-core path only");
  if (res < 2 || static_cast<long long>(res) * res * res < kTileM) return fail(SDFB_E_INVALID, "grid too small");
  DeviceGuard g(d->device);
  if (int prc = pending_status(d)) return prc;
  UserMark um{d, static_cast<cudaStream_t>(stream)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = ensure_stage(nullptr, nullptr, &d->dstage, &d->dstage_bytes, 0, kTileM * sizeof(float));
  if (rc) return rc;
  return decode_tc(d, latent_dev, nullptr, res, 0, kTileM, static_cast<float*>(d->dstage),
                   precision == SDFB_PREC_FP16, dump_dev, pass, st);
}

int sdfb_decoder_check(sdfb_decoder* d, void* stream) {
  if (!d) return fail(SDFB_E_INVALID, "null argument");
  DeviceGuard g(d->device);
  CU_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return kernel_status(d);
}

int sdfb_decoder_set_timeout_ns(sdfb_decoder* d, uint64_t timeout_ns) {
  if (!d || timeout_ns == 0) return fail(SDFB_E_INVALID, "bad argument");
  d->timeout_ns = timeout_ns;
  return SDFB_OK;
}

int sdfb_decoder_last_kernel_ms(sdfb_decoder* d, float* ms) {
  if (!d || !ms) return fail(SDFB_E_INVALID, "null argument");
  if (!d->timed) return fail(SDFB_E_INVALID, "no fused-decoder launch recorded yet");
  DeviceGuard g(d->device);
  CU_TRY(cudaEventSynchronize(d->ev1));
  CU_TRY(cudaEventElapsedTime(ms, d->ev0, d->ev1));
  if (d->prof != nullptr) {   // diagnostics: mean blocked cycles per role and wait class of the last launch
    std::vector<long long> h(static_cast<size_t>(d->num_sms) * 24);
    CU_TRY(cudaMemcpy(h.data(), d->prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    static const char* role[3] = {"epilogue", "producer", "mma"};
    static const char* cls[8] = {"total", "w_full", "w_empty", "acc_full", "acc_empty", "a_ready", "a_free", "tiles"};
    for (int r = 0; r < 3; ++r) {
      double m[8] = {0};
      int n = 0;
      for (int b = 0; b < d->num_sms; ++b) {
        const long long* v = h.data() + (static_cast<size_t>(b) * 3 + r) * 8;
        if (v[0] == 0) continue;
        ++n;
        for (int i = 0; i < 8; ++i) m[i] += static_cast<double>(v[i]);
      }
      if (n == 0) continue;
      std::fprintf(stderr, "[sdfb prof] %-8s", role[r]);
      for (int i = 0; i < 8; ++i) std::fprintf(stderr, " %s=%.0f", cls[i], m[i] / n);
      std::fprintf(stderr, " (cycles, mean over %d CTAs; %.2f ms)\n", n, *ms);
    }
    // per-pass event trace of CTA 0, tile 5 (fused_decoder.cu SDFB_K1_TRACE; written when the grid covers all SMs)
    std::vector<long long> tr(128);
    CU_TRY(cudaMemcpy(tr.data(), d->prof + static_cast<size_t>(d->num_sms) * 24, 128 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (tr[0] != 0) {
      static const char* kind[4] = {"issue_first", "issue_last", "acc_full_seen", "epi_done"};
      for (int k = 0; k < 4; ++k) {
        std::fprintf(stderr, "[sdfb trace] %-13s", kind[k]);
        for (int ps = 0; ps < 13; ++ps) std::fprintf(stderr, " %lld", tr[32 * k + ps] ? tr[32 * k + ps] - tr[0] : -1);
        std::fprintf(stderr, "\n");
      }
    }
  }
  return kernel_status(d);
}

int sdfb_umma_selftest(const uint16_t* a_dev, const uint16_t* b_dev, float* d_dev, int precision, void* stream) {
  if (!a_dev || !b_dev || !d_dev) return fail(SDFB_E_INVALID, "null argument");
  if (precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16) return fail(SDFB_E_INVALID, "bf16 or fp16 only");
  CU_TRY(tc_common_init());
  unsigned int* status = nullptr;
  CU_TRY(cudaMalloc(&status, sizeof(unsigned int)));
  CU_TRY(cudaMemset(status, 0, sizeof(unsigned int)));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = launch_umma_selftest(a_dev, b_dev, d_dev, status, precision == SDFB_PREC_FP16, st);
  unsigned int s = 0;
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaMemcpy(&s, status, sizeof(s), cudaMemcpyDeviceToHost);
  cudaFree(status);
  if (e != cudaSuccess) return fail(SDFB_E_CUDA, "umma selftest: %s", cudaGetErrorString(e));
  if (s != 0) return fail(SDFB_E_KERNEL, "umma selftest watchdog tripped (0x%x)", s);
  return SDFB_OK;
}

int sdfb_umma_rate(int cta_group, int grid, int iters, int k_per_commit, int n_acc, int flags, double* cycles_per_mma) {
  if (!cycles_per_mma || (cta_group != 1 && cta_group != 2) || grid < cta_group || iters < 1 || k_per_commit < 1 ||
      n_acc < 1 || n_acc > 2)
    return fail(SDFB_E_INVALID, "bad argument");
  // the probe's one-outstanding-group protocol (flags bit0 clear) assumes the tensor pipe is slower than the issuing thread; with
  // the N = 128 forms (bit3 without bit6, or bit8) it is not, a barrier phase is skipped and the kernel never returns
  if ((((flags & 8) && !(flags & 64)) || (flags & 256)) && !(flags & 1))
    return fail(SDFB_E_INVALID, "the N = 128 forms need flags bit0 (no intermediate waits)");
  grid -= grid % cta_group;
  long long* out = nullptr;
  CU_TRY(cudaMalloc(&out, sizeof(long long) * grid));
  CU_TRY(cudaMemset(out, 0, sizeof(long long) * grid));
  cudaError_t e = launch_umma_rate(cta_group, grid, iters, k_per_commit, n_acc, flags, out, 0);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  std::vector<long long> h(grid / cta_group);
  if (e == cudaSuccess) e = cudaMemcpy(h.data(), out, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost);
  cudaFree(out);
  if (e != cudaSuccess) return fail(SDFB_E_CUDA, "umma rate: %s", cudaGetErrorString(e));
  double s = 0;
  for (long long v : h) s += static_cast<double>(v);
  *cycles_per_mma = s / h.size() / (static_cast<double>(iters) * k_per_commit * 4);
  return SDFB_OK;
}

int sdfb_tma_ingest_rate(int grid, int cluster, int mode, int issuers, int uniform, int cols, int mib, int iters, double* out3) {
  if (!out3 || grid < 1 || cluster < 1 || cluster > 16 || (cluster & (cluster - 1)) || grid % cluster || mode < 0 || mode > 6 || (mode >= 5 && cluster != 2) ||
      (issuers != 1 && issuers != 2 && issuers != 4) || cols < 64 || cols % 64 || mib < 1 || mib > 4096 || iters < 8 || (mode == 2 && 8 % cluster))
    return fail(SDFB_E_INVALID, "bad argument");
  const long long total = static_cast<long long>(mib) << 20;
  const int rows = static_cast<int>(total / (2ll * cols)) / 128 * 128;
  if (rows < 128) return fail(SDFB_E_INVALID, "tensor smaller than one box");
  void* buf = nullptr;
  long long* out = nullptr;
  CU_TRY(cudaMalloc(&buf, static_cast<size_t>(rows) * cols * 2));
  cudaError_t e = cudaMalloc(&out, sizeof(long long) * grid);
  cudaEvent_t a = nullptr, b = nullptr;
  float ms = 0.f;
  if (e == cudaSuccess) e = cudaMemset(buf, 0, static_cast<size_t>(rows) * cols * 2);
  if (e == cudaSuccess) e = cudaEventCreate(&a);
  if (e == cudaSuccess) e = cudaEventCreate(&b);
  // one untimed pass pulls the tensor into L2, the second one is measured
  if (e == cudaSuccess) e = launch_tma_ingest(buf, cols, rows, grid, cluster, mode, issuers, uniform, iters, out, 0);
  if (e == cudaSuccess) e = cudaEventRecord(a, 0);
  if (e == cudaSuccess) e = launch_tma_ingest(buf, cols, rows, grid, cluster, mode, issuers, uniform, iters, out, 0);
  if (e == cudaSuccess) e = cudaEventRecord(b, 0);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, a, b);
  std::vector<long long> h(grid);
  if (e == cudaSuccess) e = cudaMemcpy(h.data(), out, sizeof(long long) * grid, cudaMemcpyDeviceToHost);
  if (a) cudaEventDestroy(a);
  if (b) cudaEventDestroy(b);
  cudaFree(out);
  cudaFree(buf);
  if (e != cudaSuccess) return fail(SDFB_E_CUDA, "tma ingest: %s", cudaGetErrorString(e));
  double sum = 0, worst = 0;
  for (long long v : h) { sum += static_cast<double>(v); worst = v > worst ? static_cast<double>(v) : worst; }
  const double bytes = 16384.0 * iters;
  out3[0] = bytes / (sum / grid);
  out3[1] = bytes / worst;
  out3[2] = bytes * grid / (ms * 1e-3) / 1e9;
  return SDFB_OK;
}

// ------------------------------------------------------------------ DDPM ----

int sdfb_ddpm_create(const float* params_host, size_t n_floats, int device, sdfb_ddpm** out) {
  if (out == nullptr || params_host == nullptr) return fail(SDFB_E_INVALID, "null argument");
  *out = nullptr;
  if (n_floats != static_cast<size_t>(kDdpmParamFloats))
    return fail(SDFB_E_INVALID, "denoiser blob must hold %lld floats, got %zu", kDdpmParamFloats, n_floats);
  int sms = 0;
  int rc = check_device(device, &sms);
  if (rc) return rc;
  DeviceGuard g(device);
  if (!g.ok) return fail(SDFB_E_CUDA, "cudaSetDevice(%d) failed", device);
  sdfb_ddpm* d = new (std::nothrow) sdfb_ddpm();
  if (!d) return fail(SDFB_E_NOMEM, "out of host memory");
  d->device = device; d->num_sms = sms;
  const int fin[5] = {512, 1024, 1024, 1024, 1024}, fout[5] = {1024, 1024, 1024, 1024, 256};
  long long o = 0;
  for (int l = 0; l < 5; ++l) { d->woff[l] = o; o += static_cast<long long>(fin[l]) * fout[l]; d->boff[l] = o; o += fout[l]; }
  auto bail = [&](int code) { sdfb_ddpm_destroy(d); return code; };
#define CU_TRY_D(expr)                                                                       \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return bail(fail(SDFB_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)));       \
  } while (0)
  CU_TRY_D(cudaMalloc(&d->params, n_floats * sizeof(float)));
  CU_TRY_D(cudaMemcpy(d->params, params_host, n_floats * sizeof(float), cudaMemcpyHostToDevice));
  // A5: schedule in fp64, cast to fp32 (oracle/ddpm.py ddpm_schedule), as the DDPM table: t = 999 .. 0, noise plane t,
  // no eps term, clamp bound 1
  {
    const int T = kDdpmT;
    d->ddpm_rows.assign(T, DdpmStep{});
    double abar = 1.0, abar_prev = 1.0;
    for (int t = 0; t < T; ++t) {
      const double beta = 1e-4 + (0.02 - 1e-4) * static_cast<double>(t) / (T - 1);
      const double alpha = 1.0 - beta;
      abar_prev = abar;
      abar = abar * alpha;
      DdpmStep& r = d->ddpm_rows[T - 1 - t];
      r.coef[0] = static_cast<float>(1.0 / std::sqrt(abar));
      r.coef[1] = static_cast<float>(std::sqrt(1.0 / abar - 1.0));
      r.coef[2] = static_cast<float>(beta * std::sqrt(abar_prev) / (1.0 - abar));
      r.coef[3] = static_cast<float>((1.0 - abar_prev) * std::sqrt(alpha) / (1.0 - abar));
      r.coef[5] = t == 0 ? 0.f : static_cast<float>(std::sqrt(beta * (1.0 - abar_prev) / (1.0 - abar)));
      r.coef[6] = 1.f;
      r.t = t;
      r.plane = t;
    }
  }
  // time-embedding half of layer 0 folded into a per-step bias table
  {
    const int T = kDdpmT, half = kDdpmTemb / 2;
    std::vector<float> temb(static_cast<size_t>(T) * kDdpmTemb);
    for (int t = 0; t < T; ++t)
      for (int i = 0; i < half; ++i) {
        const double f = std::exp(-std::log(10000.0) * i / half);
        temb[t * kDdpmTemb + i] = static_cast<float>(std::sin(t * f));
        temb[t * kDdpmTemb + half + i] = static_cast<float>(std::cos(t * f));
      }
    float* temb_dev = nullptr;
    CU_TRY_D(cudaMalloc(&temb_dev, temb.size() * sizeof(float)));
    CU_TRY_D(cudaMemcpy(temb_dev, temb.data(), temb.size() * sizeof(float), cudaMemcpyHostToDevice));
    CU_TRY_D(cudaMalloc(&d->tb0, static_cast<size_t>(T) * kDdpmHid * sizeof(float)));
    cudaError_t e = launch_linear_f32(temb_dev, kDdpmTemb, d->params + d->woff[0] + kDdpmLatent, 512,
                                      d->params + d->boff[0], d->tb0, kDdpmHid, T, kDdpmHid, kDdpmTemb, false, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(temb_dev);
    CU_TRY_D(e);
  }
  // tensor-core path: packed weights, bias rows, per-step coefficients, barrier and status words
  CU_TRY_D(ddpm_step_init());
  for (int f = 0; f < 2; ++f) {
    std::vector<uint16_t> wp;
    pack_ddpm_weights(params_host, d->woff, f == 1, wp);
    CU_TRY_D(cudaMalloc(&d->wpack[f], wp.size() * 2));
    CU_TRY_D(cudaMemcpy(d->wpack[f], wp.data(), wp.size() * 2, cudaMemcpyHostToDevice));
  }
  {
    std::vector<float> hb(3 * kDdpmHid + kDdpmLatent);
    for (int l = 1; l <= 3; ++l) std::memcpy(hb.data() + (l - 1) * kDdpmHid, params_host + d->boff[l], kDdpmHid * sizeof(float));
    std::memcpy(hb.data() + 3 * kDdpmHid, params_host + d->boff[4], kDdpmLatent * sizeof(float));
    CU_TRY_D(cudaMalloc(&d->bias_dev, hb.size() * sizeof(float)));
    CU_TRY_D(cudaMemcpy(d->bias_dev, hb.data(), hb.size() * sizeof(float), cudaMemcpyHostToDevice));
    CU_TRY_D(cudaMalloc(&d->ddpm_rows_dev, kDdpmT * sizeof(DdpmStep)));
    CU_TRY_D(cudaMemcpy(d->ddpm_rows_dev, d->ddpm_rows.data(), kDdpmT * sizeof(DdpmStep), cudaMemcpyHostToDevice));
    CU_TRY_D(cudaMalloc(&d->call_rows_dev, kDdpmT * sizeof(DdpmStep)));
  }
  CU_TRY_D(cudaMalloc(&d->status, sizeof(unsigned int)));
  CU_TRY_D(cudaMemset(d->status, 0, sizeof(unsigned int)));
  CU_TRY_D(cudaHostAlloc(reinterpret_cast<void**>(&d->status_host), sizeof(unsigned int), cudaHostAllocMapped));
  *d->status_host = 0;
  CU_TRY_D(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d->status_host_dev), d->status_host, 0));
  if (std::getenv("SDFB_PROF") != nullptr) {   // [num_sms][3 roles][8] wait classes + a 96-entry event trace
    CU_TRY_D(cudaMalloc(&d->prof, (static_cast<size_t>(sms) * 24 + 96) * sizeof(long long)));
    CU_TRY_D(cudaMemset(d->prof, 0, (static_cast<size_t>(sms) * 24 + 96) * sizeof(long long)));
  }
  CU_TRY_D(cudaEventCreate(&d->ev0));
  CU_TRY_D(cudaEventCreate(&d->ev1));
  CU_TRY_D(cudaDeviceSynchronize());   // the set-up copies and memsets above are done before any caller stream can touch the context
#undef CU_TRY_D
  *out = d;
  return SDFB_OK;
}

int sdfb_ddpm_destroy(sdfb_ddpm* d) {
  if (!d) return SDFB_OK;
  DeviceGuard g(d->device);
  cudaDeviceSynchronize();
  cudaFree(d->params); cudaFree(d->tb0); cudaFree(d->h0); cudaFree(d->h1); cudaFree(d->eps); cudaFree(d->dstage);
  cudaFree(d->wpack[0]); cudaFree(d->wpack[1]); cudaFree(d->bias_dev); cudaFree(d->ddpm_rows_dev); cudaFree(d->call_rows_dev);
  for (DdpmLane& L : d->lane) { cudaFree(L.act); cudaFree(L.counter); }
  if (d->st_b) cudaStreamDestroy(d->st_b);
  if (d->ev_fork) cudaEventDestroy(d->ev_fork);
  if (d->ev_join) cudaEventDestroy(d->ev_join);
  cudaFree(d->status); cudaFree(d->prof); cudaFree(d->nstage);
  if (d->status_host) cudaFreeHost(d->status_host);
  if (d->ev0) cudaEventDestroy(d->ev0);
  if (d->ev1) cudaEventDestroy(d->ev1);
  delete d;
  return SDFB_OK;
}

static int ddpm_ws(sdfb_ddpm* d, int n) {
  if (d->ws_n >= n) return SDFB_OK;
  cudaFree(d->h0); cudaFree(d->h1); cudaFree(d->eps);
  d->h0 = d->h1 = d->eps = nullptr; d->ws_n = 0;
  CU_TRY(cudaMalloc(&d->h0, static_cast<size_t>(n) * kDdpmHid * sizeof(float)));
  CU_TRY(cudaMalloc(&d->h1, static_cast<size_t>(n) * kDdpmHid * sizeof(float)));
  CU_TRY(cudaMalloc(&d->eps, static_cast<size_t>(n) * kDdpmLatent * sizeof(float)));
  d->ws_n = n;
  return SDFB_OK;
}

static int denoise_fp32(sdfb_ddpm* d, const float* x, int t, int n, float* eps, cudaStream_t st) {
  const float* P = d->params;
  CU_TRY(launch_linear_f32(x, kDdpmLatent, P + d->woff[0], 512, d->tb0 + static_cast<size_t>(t) * kDdpmHid, d->h0,
                           kDdpmHid, n, kDdpmHid, kDdpmLatent, true, st));
  CU_TRY(launch_linear_f32(d->h0, kDdpmHid, P + d->woff[1], kDdpmHid, P + d->boff[1], d->h1, kDdpmHid, n, kDdpmHid,
                           kDdpmHid, true, st));
  CU_TRY(launch_linear_f32(d->h1, kDdpmHid, P + d->woff[2], kDdpmHid, P + d->boff[2], d->h0, kDdpmHid, n, kDdpmHid,
                           kDdpmHid, true, st));
  CU_TRY(launch_linear_f32(d->h0, kDdpmHid, P + d->woff[3], kDdpmHid, P + d->boff[3], d->h1, kDdpmHid, n, kDdpmHid,
                           kDdpmHid, true, st));
  CU_TRY(launch_linear_f32(d->h1, kDdpmHid, P + d->woff[4], kDdpmHid, P + d->boff[4], eps, kDdpmLatent, n,
                           kDdpmLatent, kDdpmHid, false, st));
  return SDFB_OK;
}

// FFMA path: the schedule rows `rows` (host memory, execution order), one denoiser evaluation and one update each; the
// noise of a row is plane `plane` of the stream and is read only when its sigma != 0.
static int sample_fp32(sdfb_ddpm* d, float* x, const float* noise, int n, const DdpmStep* rows, int steps, cudaStream_t st) {
  int rc = ddpm_ws(d, n);
  if (rc) return rc;
  const long long cnt = static_cast<long long>(n) * kDdpmLatent;
  for (int s = 0; s < steps; ++s) {
    const DdpmStep& r = rows[s];
    rc = denoise_fp32(d, x, r.t, n, d->eps, st);
    if (rc) return rc;
    CU_TRY(launch_ddpm_update(x, d->eps, r.coef[5] != 0.f ? noise + static_cast<size_t>(r.plane) * cnt : nullptr, cnt, r.coef, st));
  }
  return SDFB_OK;
}

// One launch of the fused sampler over latents [0, n) of (x, noise) with workspace `lane`: the `steps` schedule rows
// `rows` (device memory, execution order), or (eps_out != nullptr) a single denoiser evaluation at rows[0].t.  The
// explicit noise stream has `steps` planes; `noise_batch` is the latent count of its plane stride (> n when this launch
// covers a share of a batch); bn_force = 0: auto.
static int ddpm_tc_lane(sdfb_ddpm* d, int lane, float* x, const float* noise, long long noise_batch, int n, const DdpmStep* rows, int steps,
                        float* eps_out, bool fp16, cudaStream_t st, bool philox, unsigned long long seed, unsigned int first_latent,
                        int bn_force, bool time_it) {
  DdpmLane& L = d->lane[lane];
  const int m_pairs = (n + 255) / 256, n_pad = 256 * m_pairs;
  if (L.act_rows < n_pad) {
    cudaFree(L.act); cudaFree(L.counter); L.act = nullptr; L.counter = nullptr; L.act_rows = 0;
    CU_TRY(cudaMalloc(&L.counter, static_cast<size_t>(m_pairs) * sizeof(unsigned int)));
    CU_TRY(cudaMalloc(&L.act, static_cast<size_t>(n_pad) * kDdpmActCols * 2));
    // on the lane's own stream: a legacy-stream memset is not ordered with a non-blocking stream and could land after
    // the kernels below have started to fill the buffer
    CU_TRY(cudaMemsetAsync(L.act, 0, static_cast<size_t>(n_pad) * kDdpmActCols * 2, st));
    L.act_rows = n_pad;
  }
  // tile width of the hidden layers: the narrowest that still leaves every CTA pair at most ONE tile per layer (more, narrower
  // tiles keep more SMs busy, but a second tile per pair and layer costs far more than it spreads: 3072 latents take 49 us per
  // step as 96 tiles of 128 on 74 pairs and 35 us as 48 tiles of 256).  n <= 1024: 64; n <= 2304: 128; else 256.
  const int max_pairs = d->num_sms / 2;
  int bn_h = m_pairs * (kDdpmHid / 64) <= max_pairs ? 64 : (m_pairs * (kDdpmHid / 128) <= max_pairs ? 128 : 256);
  if (bn_force) bn_h = bn_force;
  if (const char* e = std::getenv("SDFB_DDPM_BN")) {
    const int v = std::atoi(e);
    if (v == 64 || v == 128 || v == 256) bn_h = v;
  }
  DdpmParams p{};
  p.tb0 = d->tb0; p.bias = d->bias_dev; p.sched = rows;
  p.eps_mode = eps_out != nullptr ? 1 : 0;
  p.philox = philox ? 1 : 0; p.seed = seed; p.first_latent = first_latent;
  p.n = n; p.pair_m_tiles = m_pairs; p.steps = steps;
  p.bn_h = bn_h;
  p.nstages = bn_h == 256 ? 5 : (bn_h == 128 ? 6 : 8);   // 5 x 32 KiB, 6 x 24 KiB or 8 x 20 KiB of operand ring + 64 KiB of epilogue staging
  // the four pair tiles of a latent group as ONE cluster of 8 CTAs (cluster-scope group barrier) when every pair has
  // exactly one tile per layer and that many clusters can be resident
  if (bn_h == 256 && m_pairs * 4 <= max_pairs) {
    if (d->max_clusters8[fp16 ? 1 : 0] < 0) d->max_clusters8[fp16 ? 1 : 0] = ddpm_max_clusters8(256, p.nstages, fp16);
    p.cluster8 = m_pairs <= d->max_clusters8[fp16 ? 1 : 0] ? 1 : 0;
    p.cluster_ctas = p.cluster8 ? 8 : 0;
  }
  // ... and with 128-wide tiles the eight pair tiles of a group as ONE cluster of 16 (non-portable size; few of them fit)
  if (bn_h == 128 && lane == 0 && eps_out == nullptr && std::getenv("SDFB_DDPM_NO_C16") == nullptr) {
    if (d->max_clusters16[fp16 ? 1 : 0] < 0) d->max_clusters16[fp16 ? 1 : 0] = ddpm_max_clusters16(128, p.nstages, fp16);
    p.cluster8 = m_pairs <= d->max_clusters16[fp16 ? 1 : 0] ? 1 : 0;
    p.cluster_ctas = p.cluster8 ? 16 : 0;
  }
  if (const char* e = std::getenv("SDFB_DDPM_CLUSTER8")) p.cluster8 = (p.cluster8 && std::atoi(e) != 0) ? 1 : 0;
  if (lane != 0) p.cluster8 = 0;     // the second launch runs beside a full house of 8-CTA clusters: plain pairs only
  if (!p.cluster8) p.cluster_ctas = 0;
  if (d->prof != nullptr)
    std::fprintf(stderr, "[sdfb ddpm prof] lane %d: n=%d bn_h=%d stages=%d cluster_ctas=%d (resident 8-CTA clusters: %d, 16-CTA: %d)\n", lane, n, bn_h,
                 p.nstages, p.cluster_ctas, d->max_clusters8[fp16 ? 1 : 0], d->max_clusters16[fp16 ? 1 : 0]);
  if (const char* e = std::getenv("SDFB_DDPM_STAGES")) {   // diagnostics: a shallower ring (leaves shared memory to a profiler)
    const int v = std::atoi(e);
    if (v >= 2 && v < p.nstages) p.nstages = v;
  }
  p.counter = L.counter; p.status = d->status; p.status_host = d->status_host_dev; p.timeout_ns = d->timeout_ns; p.prof = lane == 0 ? d->prof : nullptr; p.prof_sms = d->num_sms;
  if (const char* e = std::getenv("SDFB_DDPM_FLAGS")) p.flags = static_cast<unsigned int>(std::strtoul(e, nullptr, 0));
  DdpmMaps maps;
  {
    const unsigned long long a_dims[2] = {kDdpmActCols, static_cast<unsigned long long>(L.act_rows)};
    const unsigned long long a_str[1] = {kDdpmActCols * 2ull};
    const unsigned a_box[2] = {64, 128};
    CU_TRY(make_tensor_map(maps.act, L.act, 2, 2, a_dims, a_str, a_box, true));
    const unsigned long long w_dims[2] = {64, kDdpmWRows};
    const unsigned long long w_str[1] = {128};
    const unsigned wh_box[2] = {64, static_cast<unsigned>(bn_h / 2)}, wo_box[2] = {64, kDdpmOutTile / 2};
    CU_TRY(make_tensor_map(maps.wh, d->wpack[fp16 ? 1 : 0], 2, 2, w_dims, w_str, wh_box, false));
    CU_TRY(make_tensor_map(maps.wo, d->wpack[fp16 ? 1 : 0], 2, 2, w_dims, w_str, wo_box, false));
    const unsigned long long x_dims[2] = {kDdpmLatent, static_cast<unsigned long long>(n)};
    const unsigned long long x_str[1] = {kDdpmLatent * 4ull};
    const unsigned x_box[2] = {32, 128};
    CU_TRY(make_tensor_map(maps.x, eps_out != nullptr ? eps_out : x, 4, 2, x_dims, x_str, x_box, true));
    if (noise != nullptr && eps_out == nullptr) {
      const unsigned long long n_dims[3] = {kDdpmLatent, static_cast<unsigned long long>(n), static_cast<unsigned long long>(steps)};
      const unsigned long long n_str[2] = {kDdpmLatent * 4ull, static_cast<unsigned long long>(noise_batch) * kDdpmLatent * 4ull};
      const unsigned n_box[3] = {32, 128, 1};
      CU_TRY(make_tensor_map(maps.nz, noise, 4, 3, n_dims, n_str, n_box, true));
    } else {
      std::memcpy(maps.nz, maps.x, 128);   // never dereferenced (eps_mode, seeded, or sigma = 0 in every row)
    }
  }
  CU_TRY(launch_ddpm_split(x, n, n_pad, L.act, fp16, st));
  CU_TRY(cudaMemsetAsync(L.counter, 0, static_cast<size_t>(m_pairs) * sizeof(unsigned int), st));
  if (p.prof) CU_TRY(cudaMemsetAsync(d->prof, 0, (static_cast<size_t>(d->num_sms) * 24 + 96) * sizeof(long long), st));
  if (time_it) CU_TRY(cudaEventRecord(d->ev0, st));
  CU_TRY(launch_ddpm_sample(p, maps, fp16, d->num_sms, st));
  return SDFB_OK;
}

// Tensor-core path: the `steps` schedule rows `rows` (device memory; fused denoise + update steps) in ONE cooperative launch
// (eps_out != nullptr: a single denoiser evaluation, no update) - or in TWO concurrent launches when the batch has
// one to three latent groups more than fit the 8-CTA-cluster mode: the groups that fit run in that mode (they have no
// dependency outside their cluster), the rest as plain CTA pairs on the SMs that are left, on a second stream.
static int ddpm_tc(sdfb_ddpm* d, float* x, const float* noise, int n, const DdpmStep* rows, int steps, float* eps_out,
                   bool fp16, cudaStream_t st, bool philox = false, unsigned long long seed = 0, unsigned int first_latent = 0) {
  const int m_pairs = (n + 255) / 256;
  const int f = fp16 ? 1 : 0;
  if (d->max_clusters8[f] < 0) d->max_clusters8[f] = ddpm_max_clusters8(256, 5, fp16);
  const int c8 = d->max_clusters8[f];
  bool split = eps_out == nullptr && c8 > 0 && m_pairs > c8 && m_pairs * 4 <= d->num_sms / 2 &&
               std::getenv("SDFB_DDPM_BN") == nullptr && std::getenv("SDFB_DDPM_CLUSTER8") == nullptr &&
               std::getenv("SDFB_DDPM_NO_SPLIT") == nullptr;
  int bn_b = 0;
  if (split) {
    const int groups_b = m_pairs - c8;
    bn_b = groups_b == 1 ? 128 : 256;
    if (2 * groups_b * (kDdpmHid / bn_b) > d->num_sms - 8 * c8) split = false;    // the rest must be resident beside the clusters
  }
  if (!split) {
    int rc = ddpm_tc_lane(d, 0, x, noise, n, n, rows, steps, eps_out, fp16, st, philox, seed, first_latent, 0, true);
    if (rc) return rc;
    CU_TRY(cudaEventRecord(d->ev1, st));
    d->timed = true;
    return SDFB_OK;
  }
  const int n_a = 256 * c8, n_b = n - n_a;
  if (d->st_b == nullptr) {
    CU_TRY(cudaStreamCreateWithFlags(&d->st_b, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&d->ev_fork, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&d->ev_join, cudaEventDisableTiming));
  }
  CU_TRY(cudaEventRecord(d->ev0, st));
  CU_TRY(cudaEventRecord(d->ev_fork, st));
  CU_TRY(cudaStreamWaitEvent(d->st_b, d->ev_fork, 0));
  // (both launches read the same schedule rows)
  int rc = ddpm_tc_lane(d, 0, x, noise, n, n_a, rows, steps, nullptr, fp16, st, philox, seed, first_latent, 256, false);
  if (rc) return rc;
  rc = ddpm_tc_lane(d, 1, x + static_cast<size_t>(n_a) * kDdpmLatent, noise ? noise + static_cast<size_t>(n_a) * kDdpmLatent : nullptr, n,
                    n_b, rows, steps, nullptr, fp16, d->st_b, philox, seed, first_latent + static_cast<unsigned int>(n_a), bn_b, false);
  if (rc) return rc;
  CU_TRY(cudaEventRecord(d->ev_join, d->st_b));
  CU_TRY(cudaStreamWaitEvent(st, d->ev_join, 0));
  CU_TRY(cudaEventRecord(d->ev1, st));
  d->timed = true;
  return SDFB_OK;
}

static int ddpm_status(sdfb_ddpm* d) {
  unsigned int s = 0;
  CU_TRY(cudaMemcpy(&s, d->status, sizeof(s), cudaMemcpyDeviceToHost));
  if (s != 0) {
    cudaMemset(d->status, 0, sizeof(unsigned int));
    if (d->status_host) *reinterpret_cast<volatile unsigned int*>(d->status_host) = 0;
    return fail(SDFB_E_KERNEL, "fused DDPM kernel watchdog tripped at wait site 0x%x", s);
  }
  return SDFB_OK;
}

// see pending_status(sdfb_decoder*)
static int ddpm_pending_status(sdfb_ddpm* d) {
  if (d->status_host == nullptr) return SDFB_OK;
  const unsigned int s = *reinterpret_cast<volatile unsigned int*>(d->status_host);
  if (s == 0) return SDFB_OK;
  *reinterpret_cast<volatile unsigned int*>(d->status_host) = 0;
  cudaMemset(d->status, 0, sizeof(unsigned int));
  return fail(SDFB_E_KERNEL, "an earlier launch on this context tripped the fused DDPM kernel's watchdog at wait site 0x%x: its outputs are invalid", s);
}

int sdfb_ddpm_check(sdfb_ddpm* d, void* stream) {
  if (!d) return fail(SDFB_E_INVALID, "null argument");
  DeviceGuard g(d->device);
  CU_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return ddpm_status(d);
}

int sdfb_ddpm_set_timeout_ns(sdfb_ddpm* d, uint64_t timeout_ns) {
  if (!d || timeout_ns == 0) return fail(SDFB_E_INVALID, "bad argument");
  d->timeout_ns = timeout_ns;
  return SDFB_OK;
}

int sdfb_ddpm_last_kernel_ms(sdfb_ddpm* d, float* ms) {
  if (!d || !ms) return fail(SDFB_E_INVALID, "null argument");
  if (!d->timed) return fail(SDFB_E_INVALID, "no fused DDPM launch recorded yet");
  DeviceGuard g(d->device);
  CU_TRY(cudaEventSynchronize(d->ev1));
  CU_TRY(cudaEventElapsedTime(ms, d->ev0, d->ev1));
  if (d->prof != nullptr) {   // diagnostics: mean blocked cycles per role and wait class of the last launch
    std::vector<long long> h(static_cast<size_t>(d->num_sms) * 24);
    CU_TRY(cudaMemcpy(h.data(), d->prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    static const char* role[3] = {"epilogue", "producer", "mma"};
    static const char* cls[8] = {"total", "full", "empty", "acc_full", "acc_empty", "group_barrier", "full_first", "-"};
    for (int r = 0; r < 3; ++r) {
      double m[8] = {0};
      int n = 0;
      for (int b = 0; b < d->num_sms; ++b) {
        const long long* v = h.data() + (static_cast<size_t>(b) * 3 + r) * 8;
        if (v[0] == 0) continue;
        ++n;
        for (int i = 0; i < 8; ++i) m[i] += static_cast<double>(v[i]);
      }
      if (n == 0) continue;
      std::fprintf(stderr, "[sdfb ddpm prof] %-8s", role[r]);
      for (int i = 0; i < 7; ++i) std::fprintf(stderr, " %s=%.0f", cls[i], m[i] / n);
      std::fprintf(stderr, " (cycles, mean over %d CTAs; %.2f ms)\n", n, *ms);
    }
    // event trace of CTA 0, step 5 (ddpm_step.cu SDFB_TRACE): cycles relative to layer 0's first MMA
    std::vector<long long> tr(96);
    CU_TRY(cudaMemcpy(tr.data(), d->prof + static_cast<size_t>(d->num_sms) * 24, 96 * sizeof(long long), cudaMemcpyDeviceToHost));
    static const char* ev[13] = {"mma_start", "mma_issued", "epi_acc_full", "epi_chunk0_ready", "epi_stores_issued",
                                 "epi_stores_done", "epi_arrived", "prod_at_barrier", "prod_barrier_done", "prod_A_issued",
                                 "L4_tmem_read", "L4_unit0_computed", "L4_unit0_stored"};
    if (tr[0] != 0)
      for (int l = 0; l < 6; ++l) {   // row 5 = layer 0 of the following step
        std::fprintf(stderr, "[sdfb ddpm trace] L%d", l);
        for (int e = 0; e < 13; ++e) std::fprintf(stderr, " %s=%lld", ev[e], tr[l * 16 + e] ? tr[l * 16 + e] - tr[0] : -1);
        std::fprintf(stderr, "\n");
      }
  }
  return ddpm_status(d);
}

int sdfb_ddpm_denoise(sdfb_ddpm* d, const float* x_dev, int t, int n, float* eps_dev, int precision, void* stream) {
  if (!d || !x_dev || !eps_dev) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || t < 0 || t >= kDdpmT) return fail(SDFB_E_INVALID, "bad n or t");
  if (precision != SDFB_PREC_FP32 && precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "unknown precision %d", precision);
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  if (precision != SDFB_PREC_FP32)
    return ddpm_tc(d, const_cast<float*>(x_dev), nullptr, n, d->ddpm_rows_dev + (kDdpmT - 1 - t), 1, eps_dev, precision == SDFB_PREC_FP16,
                   static_cast<cudaStream_t>(stream));
  int rc = ddpm_ws(d, n);
  if (rc) return rc;
  return denoise_fp32(d, x_dev, t, n, eps_dev, static_cast<cudaStream_t>(stream));
}

int sdfb_ddpm_sample(sdfb_ddpm* d, float* x_dev, const float* noise_dev, int n, int steps, int precision,
                     void* stream) {
  if (!d || !x_dev) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || steps < 1 || steps > kDdpmT) return fail(SDFB_E_INVALID, "bad n or steps");
  if (steps > 1 && !noise_dev) return fail(SDFB_E_INVALID, "noise stream required");
  if (precision != SDFB_PREC_FP32 && precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "unknown precision %d", precision);
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (precision != SDFB_PREC_FP32)
    return ddpm_tc(d, x_dev, noise_dev, n, d->ddpm_rows_dev + (kDdpmT - steps), steps, nullptr, precision == SDFB_PREC_FP16, st);
  return sample_fp32(d, x_dev, noise_dev, n, d->ddpm_rows.data() + (kDdpmT - steps), steps, st);
}

int sdfb_philox_normal(uint64_t seed, int64_t first_latent, int n, int t0, int t1, float* out_dev, void* stream) {
  if (!out_dev) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || t0 < 0 || t1 < t0 || first_latent < 0 || first_latent + n > 0xFFFFFFFFll)
    return fail(SDFB_E_INVALID, "bad n, latent range or step range");
  CU_TRY(launch_philox_normal(seed, static_cast<unsigned int>(first_latent), n, t0, t1, out_dev, static_cast<cudaStream_t>(stream)));
  return SDFB_OK;
}

int sdfb_ddpm_sample_philox(sdfb_ddpm* d, float* x_dev, uint64_t seed, int64_t first_latent, int n, int steps, int gen_xT,
                            int precision, void* stream) {
  if (!d || !x_dev) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || steps < 1 || steps > kDdpmT) return fail(SDFB_E_INVALID, "bad n or steps");
  if (first_latent < 0 || first_latent + n > 0xFFFFFFFFll) return fail(SDFB_E_INVALID, "latent range outside [0, 2^32)");
  const unsigned int f0 = static_cast<unsigned int>(first_latent);
  if (precision != SDFB_PREC_FP32 && precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "unknown precision %d", precision);
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (gen_xT) CU_TRY(launch_philox_normal(seed, f0, n, steps, steps + 1, x_dev, st));  // x_T = row t = steps of the stream
  if (precision != SDFB_PREC_FP32)
    return ddpm_tc(d, x_dev, nullptr, n, d->ddpm_rows_dev + (kDdpmT - steps), steps, nullptr, precision == SDFB_PREC_FP16, st, true, seed, f0);
  // fp32 path: materialise the same stream (bit for bit the in-kernel one) and run the FFMA sampler on it
  const size_t cnt = static_cast<size_t>(n) * kDdpmLatent;
  int rc = ensure_stage(nullptr, nullptr, &d->nstage, &d->nstage_bytes, 0, static_cast<size_t>(steps) * cnt * sizeof(float));
  if (rc) return rc;
  CU_TRY(launch_philox_normal(seed, f0, n, 0, steps, static_cast<float*>(d->nstage), st));
  return sdfb_ddpm_sample(d, x_dev, static_cast<float*>(d->nstage), n, steps, precision, stream);
}

int sdfb_ddpm_sample_philox_host(sdfb_ddpm* d, float* x_host, uint64_t seed, int64_t first_latent, int n, int steps, int gen_xT,
                                 int precision) {
  if (!d || !x_host) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || steps < 1 || steps > kDdpmT) return fail(SDFB_E_INVALID, "bad n or steps");
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  const size_t cnt = static_cast<size_t>(n) * kDdpmLatent;
  int rc = ensure_stage(nullptr, nullptr, &d->dstage, &d->dstage_bytes, 0, cnt * sizeof(float));
  if (rc) return rc;
  float* x = static_cast<float*>(d->dstage);
  if (!gen_xT) CU_TRY(cudaMemcpyAsync(x, x_host, cnt * sizeof(float), cudaMemcpyHostToDevice, 0));
  rc = sdfb_ddpm_sample_philox(d, x, seed, first_latent, n, steps, gen_xT, precision, nullptr);
  if (rc) return rc;
  CU_TRY(cudaMemcpyAsync(x_host, x, cnt * sizeof(float), cudaMemcpyDeviceToHost, 0));
  CU_TRY(cudaStreamSynchronize(0));
  return precision == SDFB_PREC_FP32 ? SDFB_OK : ddpm_status(d);
}

int sdfb_ddpm_sample_host(sdfb_ddpm* d, float* x_host, const float* noise_host, int n, int steps, int precision) {
  if (!d || !x_host) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0 || steps < 1 || steps > kDdpmT) return fail(SDFB_E_INVALID, "bad n or steps");
  if (steps > 1 && !noise_host) return fail(SDFB_E_INVALID, "noise stream required");
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  const size_t cnt = static_cast<size_t>(n) * kDdpmLatent;
  const size_t need = (1 + static_cast<size_t>(steps)) * cnt * sizeof(float);
  int rc = ensure_stage(nullptr, nullptr, &d->dstage, &d->dstage_bytes, 0, need);
  if (rc) return rc;
  float* x = static_cast<float*>(d->dstage);
  float* nz = x + cnt;
  CU_TRY(cudaMemcpyAsync(x, x_host, cnt * sizeof(float), cudaMemcpyHostToDevice, 0));
  if (steps > 1) CU_TRY(cudaMemcpyAsync(nz, noise_host, static_cast<size_t>(steps) * cnt * sizeof(float), cudaMemcpyHostToDevice, 0));
  rc = sdfb_ddpm_sample(d, x, nz, n, steps, precision, nullptr);
  if (rc) return rc;
  CU_TRY(cudaMemcpyAsync(x_host, x, cnt * sizeof(float), cudaMemcpyDeviceToHost, 0));
  CU_TRY(cudaStreamSynchronize(0));
  return precision == SDFB_PREC_FP32 ? SDFB_OK : ddpm_status(d);
}

// ---- respaced (DDIM) schedules ----

// The rows of sdfb_ddim_schedule as the sampler's table: the timestep selects the time-embedding bias and the Philox
// counter, the plane is the step index i (noise[i] is consumed at the step from tau_i).
static int ddim_rows(int steps, float eta, int inverse, std::vector<DdpmStep>& rows) {
  std::vector<int32_t> ts(static_cast<size_t>(steps));
  std::vector<float> coef(static_cast<size_t>(steps) * 8);
  int rc = sdfb_ddim_schedule(steps, eta, inverse, ts.data(), coef.data());
  if (rc) return rc;
  rows.assign(static_cast<size_t>(steps), DdpmStep{});
  for (int k = 0; k < steps; ++k) {
    std::memcpy(rows[k].coef, coef.data() + static_cast<size_t>(k) * 8, 8 * sizeof(float));
    rows[k].t = ts[k];
    rows[k].plane = inverse ? k : steps - 1 - k;
  }
  return SDFB_OK;
}

int sdfb_ddim_schedule(int steps, float eta, int inverse, int32_t* timesteps_host, float* coef_host) {
  if (!timesteps_host || !coef_host) return fail(SDFB_E_INVALID, "null argument");
  if (steps < 1 || steps > kDdpmT) return fail(SDFB_E_INVALID, "steps must be in [1, %d], got %d", kDdpmT, steps);
  if (!(eta >= 0.f && eta <= 1.f)) return fail(SDFB_E_INVALID, "eta must be a finite value in [0, 1]");
  // abar of the 1000-step linear-beta chain in fp64, with beta = numpy.linspace(1e-4, 0.02, 1000) to the last bit
  const int T = kDdpmT;
  std::vector<double> abar(T);
  {
    const double start = 1e-4, stop = 0.02, step = (stop - start) / (T - 1);
    double a = 1.0;
    for (int t = 0; t < T; ++t) {
      const double beta = t == T - 1 ? stop : static_cast<double>(t) * step + start;
      a = a * (1.0 - beta);
      abar[t] = a;
    }
  }
  auto tau = [&](int i) { return static_cast<int>(static_cast<long long>(i) * T / steps); };
  const double e = static_cast<double>(eta);
  const float inf = std::numeric_limits<float>::infinity();
  for (int k = 0; k < steps; ++k) {
    const int i = inverse ? k : steps - 1 - k;              // rows in execution order
    float* c = coef_host + static_cast<size_t>(k) * 8;
    timesteps_host[k] = tau(i);
    if (inverse) {
      // from x at tau_{i-1} (x0 itself for i = 0) to x at tau_i, with eps evaluated at tau_i; x0 is not clamped
      const double cur = i > 0 ? abar[tau(i - 1)] : 1.0, next = abar[tau(i)];
      const double v[8] = {1.0 / std::sqrt(cur), std::sqrt(1.0 / cur - 1.0), std::sqrt(next), 0.0, std::sqrt(1.0 - next), 0.0, 0.0, 0.0};
      for (int j = 0; j < 8; ++j) c[j] = static_cast<float>(v[j]);
      c[6] = inf;
    } else {
      const double ab = abar[tau(i)], abp = i > 0 ? abar[tau(i - 1)] : 1.0;
      const double sigma = e * std::sqrt((1.0 - abp) / (1.0 - ab)) * std::sqrt(1.0 - ab / abp);
      const double c2 = std::sqrt(std::max(0.0, 1.0 - abp - sigma * sigma)) / std::sqrt(1.0 - ab);
      const double c1 = std::sqrt(abp) - c2 * std::sqrt(ab);
      const double v[8] = {1.0 / std::sqrt(ab), std::sqrt(1.0 / ab - 1.0), c1, c2, 0.0, sigma, 1.0, 0.0};
      for (int j = 0; j < 8; ++j) c[j] = static_cast<float>(v[j]);
    }
  }
  return SDFB_OK;
}

// The checks every respaced entry point shares; on success the schedule rows are in `rows`.
static int ddim_prepare(sdfb_ddpm* d, const float* x_dev, int n, int steps, float eta, int inverse, int precision,
                        std::vector<DdpmStep>& rows) {
  if (!d || !x_dev) return fail(SDFB_E_INVALID, "null argument");
  if (n <= 0) return fail(SDFB_E_INVALID, "bad n");
  if (precision != SDFB_PREC_FP32 && precision != SDFB_PREC_BF16 && precision != SDFB_PREC_FP16)
    return fail(SDFB_E_INVALID, "unknown precision %d", precision);
  return ddim_rows(steps, eta, inverse, rows);
}

// Runs the rows: the fused kernel reads them from the context's call table, written on the caller's stream and so ordered
// with the kernel that reads it; the FFMA path takes them from the host.
static int ddim_run(sdfb_ddpm* d, float* x_dev, const float* noise, int n, const std::vector<DdpmStep>& rows, int precision, cudaStream_t st,
                    bool philox = false, unsigned long long seed = 0, unsigned int f0 = 0) {
  const int steps = static_cast<int>(rows.size());
  if (precision == SDFB_PREC_FP32) return sample_fp32(d, x_dev, noise, n, rows.data(), steps, st);
  CU_TRY(cudaMemcpyAsync(d->call_rows_dev, rows.data(), rows.size() * sizeof(DdpmStep), cudaMemcpyHostToDevice, st));
  return ddpm_tc(d, x_dev, noise, n, d->call_rows_dev, steps, nullptr, precision == SDFB_PREC_FP16, st, philox, seed, f0);
}

int sdfb_ddpm_sample_ddim(sdfb_ddpm* d, float* x_dev, const float* noise_dev, int n, int steps, float eta, int precision, void* stream) {
  std::vector<DdpmStep> rows;
  int rc = ddim_prepare(d, x_dev, n, steps, eta, 0, precision, rows);
  if (rc) return rc;
  if (eta > 0.f && !noise_dev) return fail(SDFB_E_INVALID, "noise stream required for eta > 0");
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  return ddim_run(d, x_dev, noise_dev, n, rows, precision, static_cast<cudaStream_t>(stream));
}

int sdfb_ddpm_sample_ddim_philox(sdfb_ddpm* d, float* x_dev, uint64_t seed, int64_t first_latent, int n, int steps, float eta, int gen_xT,
                                 int precision, void* stream) {
  std::vector<DdpmStep> rows;
  int rc = ddim_prepare(d, x_dev, n, steps, eta, 0, precision, rows);
  if (rc) return rc;
  if (first_latent < 0 || first_latent + n > 0xFFFFFFFFll) return fail(SDFB_E_INVALID, "latent range outside [0, 2^32)");
  const unsigned int f0 = static_cast<unsigned int>(first_latent);
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // x_T = row t = 1000 of the stream whatever the step count: DDIM and the full DDPM chain start from the same x_T
  if (gen_xT) CU_TRY(launch_philox_normal(seed, f0, n, kDdpmT, kDdpmT + 1, x_dev, st));
  if (precision != SDFB_PREC_FP32) return ddim_run(d, x_dev, nullptr, n, rows, precision, st, true, seed, f0);
  // fp32 path: materialise plane i = Philox row tau_i for the steps that draw noise, then run the FFMA sampler on it
  const size_t cnt = static_cast<size_t>(n) * kDdpmLatent;
  rc = ensure_stage(nullptr, nullptr, &d->nstage, &d->nstage_bytes, 0, static_cast<size_t>(steps) * cnt * sizeof(float));
  if (rc) return rc;
  float* nz = static_cast<float*>(d->nstage);
  for (const DdpmStep& r : rows)
    if (r.coef[5] != 0.f) CU_TRY(launch_philox_normal(seed, f0, n, r.t, r.t + 1, nz + static_cast<size_t>(r.plane) * cnt, st));
  return ddim_run(d, x_dev, nz, n, rows, precision, st);
}

int sdfb_ddpm_invert_ddim(sdfb_ddpm* d, float* x_dev, int n, int steps, int precision, void* stream) {
  std::vector<DdpmStep> rows;
  int rc = ddim_prepare(d, x_dev, n, steps, 0.f, 1, precision, rows);
  if (rc) return rc;
  DeviceGuard g(d->device);
  if (int prc = ddpm_pending_status(d)) return prc;
  return ddim_run(d, x_dev, nullptr, n, rows, precision, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
