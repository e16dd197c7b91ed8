// K2: fused latent-DDPM sampler for sm_100a (tcgen05 / TMEM / TMA, CTA pairs, one persistent
// launch - every CTA resident - for all steps of a sample_latents call).
//
// What it computes (SURVEY.md section 8a rows A5-A7; oracle: oracle/ddpm.py denoiser_forward_lowp,
// ddpm_step, sample_latents; no upstream source exists, /root/reference/README.md:1):
//   per step t:  h0 = relu([x_hi | x_lo] [W0x | W0x]^T + tb0[t])      K = 512, time embedding folded
//                h1..h3 = relu(h W^T + b)                             K = 1024
//                eps = h3 W4^T + b4                                   fp32, never rounded
//                x0 = clamp(sra x - srm1 eps, -c, c);  x <- c1 x0 + c2 x [+ c3 eps] [+ sigma noise]
//   with t, the noise plane and the coefficients read from the call's schedule table (DdpmStep, execution order):
//   DDPM, DDIM sampling and DDIM inversion are different tables
// 16-bit operands, fp32 accumulation in TMEM; the state x stays fp32 and enters layer 0 as an
// exact two-way 16-bit split.
//
// Mapping.  Every layer is cut into pair tiles of 256 latents x BN output features
// (cta_group::2: each CTA holds 128 rows of A and half of the weight rows) that are spread over
// all CTA pairs; K is streamed in 64-wide chunks through a shared-memory ring.  ALL global
// traffic of the kernel goes through the TMA unit: the epilogue warps build a tile's output in
// a swizzled shared-memory staging buffer and store it with one bulk tensor copy per 64-feature
// chunk into an L2-resident row-major activation buffer, from which the next layer's operand
// boxes are loaded (scattered per-thread stores cost 32 LSU wavefronts per instruction and a
// write-drain fence; the profile of the first version was dominated by them).  A tile waits
// only for the CTAs that share its 256 latents (one barrier counter per latent group: release-add
// by the storing thread after its bulk stores completed, acquire spin in the producer); weights
// do not depend on it and are prefetched across it.  The last layer's epilogue is the DDPM
// update: x and the step's noise plane arrive as TMA boxes, x_new, x_hi and x_lo leave as TMA boxes.
//
//   warps 0-7  epilogue   (TMEM lane quadrant = warp & 3; the two warp sets split the columns)
//   warp 8     producer   (TMA; completion counted on the LEADER's barrier)
//   warp 9     MMA issuer (leader CTA only) + TMEM allocation (both CTAs)
#include <atomic>
#include <cstdlib>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "kernels.h"
#include "philox.cuh"
#include "ptx.cuh"

namespace sdfb {

namespace {

constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreads = kEpiThreads + 64;
constexpr int kLayers = 5;
constexpr uint32_t kStagingBytes = 64 * 1024;   // four 16 KiB slots.  hidden: the tile's chunk images | last layer: x boxes in slots 0, 1,
                                                // noise boxes in slots 2, 3, later overwritten by the x_hi / x_lo images
constexpr uint32_t kChunk = 16384;

constexpr int kBarFull = 0;
constexpr int kBarEmpty = kBarFull + kDdpmMaxStages;
constexpr int kBarAccFull = kBarEmpty + kDdpmMaxStages;
constexpr int kBarAccEmpty = kBarAccFull + 2;
constexpr int kBarXn = kBarAccEmpty + 2;
constexpr int kBarOwn = kBarXn + 1;          // staging slot s holds a finished operand chunk (6 slots)
constexpr int kBarGroup = kBarOwn + 6;        // cluster8 mode: every warp set of the latent group's 8 CTAs has stored its output
constexpr int kNumBars = kBarGroup + 1;
constexpr uint32_t kBarBytes = (kNumBars * 8 + 15) & ~15u;   // keeps what follows 16-byte aligned

// wait sites (status codes); (site >> 4) & 7 is the class under which blocked cycles are profiled
enum : uint32_t { kErrFull = 0x110, kErrEmpty = 0x120, kErrAccFull = 0x130, kErrAccEmpty = 0x140, kErrGrid = 0x150,
                  kErrFullFirst = 0x160, kErrXn = 0x170, kErrOwn = 0x180 };

// Diagnostics: with profiling on, CTA 0 stamps clock64() at key events of every layer of step 5 (and
// of layer 0 of step 6, row 5) into the tail of the profile buffer ([prof_sms * 24 + row * 16 + event]).
#define SDFB_TRACE(ev)                                                                              \
  do {                                                                                              \
    if (p.prof != nullptr && blockIdx.x == 0 && (s == 5 || (s == 6 && l == 0)))                     \
      p.prof[static_cast<size_t>(p.prof_sms) * 24 + (s == 6 ? 5 : l) * 16 + (ev)] = clock64();            \
  } while (0)

struct Geo {
  int nk;          // 64-wide k-chunks
  int a_col0;      // first column of the layer's A operand in the activation buffer
  int o_col0;      // first column of the buffer the layer's epilogue writes
  int w_row0;      // first weight row of the layer
  int n_total;     // output features
  int bn;          // tile width
  int ntn;         // n-tiles
};

__device__ __forceinline__ Geo layer_geo(const DdpmParams& p, int l) {
  Geo g;
  g.nk = l == 0 ? 8 : 16;
  g.a_col0 = l == 0 ? 0 : ((l & 1) ? 512 : 1536);      // L1, L3 read buffer 0; L2, L4 read buffer 1
  g.o_col0 = l == 4 ? 0 : ((l & 1) ? 1536 : 512);      // L0, L2 write buffer 0; L1, L3 write buffer 1; L4 writes [x_hi | x_lo]
  g.w_row0 = l == 0 ? 0 : (l < 4 ? kDdpmW0Rows + (l - 1) * kDdpmWHidRows : kDdpmW0Rows + 3 * kDdpmWHidRows);
  g.n_total = l == 4 ? kDdpmLatent : kDdpmHid;
  g.bn = l == 4 ? kDdpmOutTile : p.bn_h;
  g.ntn = g.n_total / g.bn;
  return g;
}

// First tile of pair `pidx` in layer l (further tiles follow npairs apart).  With 16-CTA clusters (eight pairs of 128-wide
// hidden tiles per latent group) the last layer has only FOUR 64-wide tiles per group: pairs 0-3 of the cluster take them
// and pairs 4-7 sit the layer out, so that a group's tiles never leave its cluster.
__device__ __forceinline__ int first_tile(const DdpmParams& p, int l, int pidx, int T) {
  if (l == 4 && p.cluster_ctas == 16) return (pidx & 7) < 4 ? (pidx >> 3) * 4 + (pidx & 7) : T;
  return pidx;
}

// Own chunks.  With one tile per pair and layer, the k-chunks a pair produced in the previous layer are
// still in its staging buffer in operand layout: the next layer starts on them at once (weights come
// through the ring, A straight from staging) while the peers' chunks travel through L2.
//   layers 1-3: the bn_h / 64 chunks [j bn_h / 64, ...) in staging slots round * bn_h / 64 ..   (L4 reuses those slots for x / noise: no own chunks)
//   layer 0   : x_hi chunk j and x_lo chunk 4 + j in slots 2, 3 (needs the same tile index in L4 and L0: bn_h = 256)
struct Own { int n, kc0, kstride, slot0; };
// `rounds` = tiles per pair and hidden layer, `round` = which of them this tile is.  The four staging slots hold the
// hidden outputs of all of a pair's tiles of one layer, so own chunks need rounds * (bn_h / 64) <= 4.
__device__ __forceinline__ Own own_chunks(const DdpmParams& p, int s, int l, int j, int round, int rounds) {
  Own o{0, 0, 1, 0};
  const int nch = p.bn_h >> 6;
  if (rounds * nch > 4) return o;
  if (l == 0) {
    if (s > 0 && p.bn_h == 256) { o.n = 2; o.kc0 = j; o.kstride = 4; o.slot0 = 2; }
  } else if (l < 4) {
    o.n = nch; o.kc0 = j * nch; o.slot0 = round * nch;
  }
  return o;
}
// i-th k-chunk of a tile: own chunks first, then the rest in increasing order
__device__ __forceinline__ int kc_of(const Own& o, int i) {
  if (i < o.n) return o.kc0 + i * o.kstride;
  int idx = i - o.n;
  if (o.n == 0) return idx;
  if (o.kstride == 1) return idx < o.kc0 ? idx : idx + o.n;
  if (idx >= o.kc0) ++idx;
  if (idx >= o.kc0 + o.kstride) ++idx;
  return idx;
}

__device__ __forceinline__ uint32_t ld_acquire_gpu(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_relaxed_gpu_add(unsigned int* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_release_gpu_add(unsigned int* p, uint32_t v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// generic-proxy <-> async-proxy (TMA) ordering on global memory
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// Wait until `target` arrivals have been counted on a barrier counter (bounded).
__device__ __forceinline__ bool grid_wait(const DdpmParams& p, const unsigned int* counter, uint32_t target, const Watchdog& wd) {
  if (ld_acquire_gpu(counter) >= target) return true;
  const long long c0 = wd.wait_cycles != nullptr ? clock64() : 0;
  const uint64_t t0 = global_timer_ns();
  uint32_t spins = 0;
  while (true) {
    if (ld_acquire_gpu(counter) >= target) {
      if (wd.wait_cycles != nullptr) wd.wait_cycles[(kErrGrid >> 4) & 7u] += clock64() - c0;
      return true;
    }
    if ((++spins & 0x3Fu) == 0) {
      if (*wd.abort_flag) return false;
      if (*reinterpret_cast<volatile unsigned int*>(p.status) != 0) { *wd.abort_flag = kErrGrid; return false; }
      if (global_timer_ns() - t0 > wd.timeout_ns) {
        *wd.abort_flag = kErrGrid;
        wd_trip(wd, static_cast<unsigned int>(kErrGrid));
        return false;
      }
    }
  }
}

template <bool FP16>
__device__ __forceinline__ float lowp_to_float(uint32_t bits16) {
  if constexpr (FP16) {
    return __half2float(__ushort_as_half(static_cast<unsigned short>(bits16 & 0xFFFFu)));
  } else {
    return __uint_as_float(bits16 << 16);
  }
}
// (hi, lo) 16-bit split of two consecutive fp32 values: x = hi + lo + O(2^-16 |x|)
template <bool FP16>
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack_plain<FP16>(a, b);
  const float ra = a - lowp_to_float<FP16>(hi & 0xFFFFu);
  const float rb = b - lowp_to_float<FP16>(hi >> 16);
  lo = pack_plain<FP16>(ra, rb);
}

// ---- TMA helpers (tensor maps passed as __grid_constant__ kernel parameters) ----
// box at (c0, c1) -> local shared memory, bytes counted on the LEADER CTA's barrier
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst_smem, const void* tmap, int c0, int c1, uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3}], [%4];" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(leader_bar)
      : "memory");
}
// box -> local shared memory, bytes counted on a local barrier
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst_smem, const void* tmap, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, int c0, int c1, uint32_t src_smem) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(c0), "r"(c1), "r"(src_smem)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <bool FP16>
__global__ void __launch_bounds__(kThreads, 1)
ddpm_sample_kernel(const DdpmParams p, const __grid_constant__ CUtensorMap tm_act, const __grid_constant__ CUtensorMap tm_wh,
                   const __grid_constant__ CUtensorMap tm_wo, const __grid_constant__ CUtensorMap tm_x,
                   const __grid_constant__ CUtensorMap tm_nz) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem0 = smem_u32(smem_raw);
  if ((smem0 & 1023u) != 0) {
    if (threadIdx.x == 0) atomicCAS(p.status, 0u, 0xA12u);
    return;
  }
  const uint32_t stage_bytes = kChunk + static_cast<uint32_t>(p.bn_h) * 64u;   // A chunk + this CTA's half of a weight chunk
  const uint32_t o_stage = static_cast<uint32_t>(p.nstages) * stage_bytes;     // epilogue staging
  const uint32_t o_bar = o_stage + kStagingBytes;
  const uint32_t stg = smem0 + o_stage;
  const uint32_t bars = smem0 + o_bar;
  volatile uint32_t* misc = reinterpret_cast<volatile uint32_t*>(smem_raw + o_bar + kBarBytes);   // [0] tmem base, [1] abort
  float* sbias = reinterpret_cast<float*>(smem_raw + o_bar + kBarBytes + 16);                    // 2 x 256 floats: the tile's bias slice
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // The cluster is one CTA pair, or (cluster8 mode) the four - with 128-wide tiles eight - pairs that share 256 latents.
  const uint32_t crank = cluster_ctarank();
  const uint32_t rank = crank & 1u;                    // rank inside the pair
  const uint32_t lrank = crank & ~1u;                  // cluster rank of this pair's leader CTA
  const uint16_t pmask = static_cast<uint16_t>(3u << lrank);
  const bool leader = rank == 0;
  const int npairs = gridDim.x >> 1, pidx = blockIdx.x >> 1;
  // Barrier arithmetic: a pair tile contributes 4 arrivals (2 CTAs x 2 warp sets) to the counter of its
  // latent group pm.  A hidden layer has kDdpmHid / bn_h tiles per group, the last layer 4.
  const uint32_t arr_h = 4u * static_cast<uint32_t>(kDdpmHid / p.bn_h);
  const uint32_t arr_step = 4u * arr_h + 16u;

  if (threadIdx.x == 0) {
    misc[1] = 0;
    for (int s = 0; s < kDdpmMaxStages; ++s) {
      mbar_init(bars + 8 * (kBarFull + s), 1);
      mbar_init(bars + 8 * (kBarEmpty + s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bars + 8 * (kBarAccFull + b), 1);
      mbar_init(bars + 8 * (kBarAccEmpty + b), 2 * kEpiWarps);
    }
    mbar_init(bars + 8 * kBarXn, 1);
    for (int c = 0; c < 6; ++c) mbar_init(bars + 8 * (kBarOwn + c), kEpiWarps);   // one warp set x 2 CTAs arrive per phase
    mbar_init(bars + 8 * kBarGroup, p.cluster_ctas == 16 ? 32u : 16u);          // 8 (or 16) CTAs x 2 warp sets
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc<2>(smem0 + o_bar + kBarBytes, 512);
    tmem_relinquish<2>();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = misc[0];
  long long waited[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  Watchdog wd{misc + 1, p.status, p.timeout_ns, p.prof != nullptr ? waited : nullptr, p.status_host};
  const long long t_start = clock64();

  if (warp == 8) {
    // ===================== producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, gphase = 0;
      const uint32_t nst = static_cast<uint32_t>(p.nstages);
      for (int s = 0; s < p.steps; ++s) {
        for (int l = 0; l < kLayers; ++l) {
          const Geo g = layer_geo(p, l);
          const CUtensorMap* tmw = l == 4 ? &tm_wo : &tm_wh;
          const uint32_t tx = 2u * kChunk + static_cast<uint32_t>(g.bn) * 128u;
          const bool need_sync = !(s == 0 && l == 0);      // the operand of the very first layer was written by an earlier kernel
          const uint32_t target = static_cast<uint32_t>(s) * arr_step + static_cast<uint32_t>(l) * arr_h;
          const int T = p.pair_m_tiles * g.ntn;
          const int rounds = (p.pair_m_tiles * (kDdpmHid / p.bn_h) + npairs - 1) / npairs;
          if (p.cluster_ctas == 16 && l == 4 && first_tile(p, l, pidx, T) >= T) {
            // sitting the last layer out (see first_tile): the group barrier's phase must still be SEEN, or the next wait
            // would test a parity two phases away and pass at once
            if (!mbar_wait_cluster(bars + 8 * kBarGroup, gphase, wd, kErrGrid)) goto done;
            gphase ^= 1u;
          }
          for (int tile = first_tile(p, l, pidx, T), round = 0; tile < T; tile += npairs, ++round) {
            const int pm = tile / g.ntn, j = tile - pm * g.ntn;
            const int a_row = (2 * pm + static_cast<int>(rank)) * 128;
            const int w_row = g.w_row0 + j * g.bn + static_cast<int>(rank) * (g.bn >> 1);
            const Own o = own_chunks(p, s, l, j, round, rounds);
            int i = 0;
            // own chunks: only their weights travel
            for (; i < o.n; ++i) {
              if (!mbar_wait(bars + 8 * (kBarEmpty + stage), phase ^ 1u, wd, kErrEmpty, stage)) goto done;
              const uint32_t full = bars + 8 * (kBarFull + stage);
              if (leader) mbar_arrive_expect_tx(full, static_cast<uint32_t>(g.bn) * 128u);
              const int kc = kc_of(o, i), wk = l == 0 ? (kc & 3) : kc;
              tma_load_2d_pair(smem0 + stage * stage_bytes + kChunk, tmw, 0, w_row + wk * g.n_total, map_to_cta(full, lrank));
              if (++stage == nst) { stage = 0; phase ^= 1u; }
            }
            if (need_sync) {
              // weights first (they do not depend on the previous layer), then the group barrier, then A
              const int rest = g.nk - o.n;
              // (an odd number of own chunks: the issuer releases the last own stage only together with the first streamed one
              // - it commits per PAIR of chunks - so the prefetch must not wrap around onto that stage)
              const int room = static_cast<int>(nst) - (o.n & 1);
              const int pre = rest < room ? rest : room;
              uint32_t st = stage, ph = phase;
              for (int k = 0; k < pre; ++k) {
                if (!mbar_wait(bars + 8 * (kBarEmpty + st), ph ^ 1u, wd, kErrEmpty, st)) goto done;
                const uint32_t full = bars + 8 * (kBarFull + st);
                if (leader) mbar_arrive_expect_tx(full, tx);
                const int kc = kc_of(o, i + k), wk = l == 0 ? (kc & 3) : kc;
                tma_load_2d_pair(smem0 + st * stage_bytes + kChunk, tmw, 0, w_row + wk * g.n_total, map_to_cta(full, lrank));
                if (++st == nst) { st = 0; ph ^= 1u; }
              }
              SDFB_TRACE(7);
              if (p.cluster8) {
                if (!mbar_wait_cluster(bars + 8 * kBarGroup, gphase, wd, kErrGrid)) goto done;
                gphase ^= 1u;
              } else {
                if (!grid_wait(p, p.counter + pm, target, wd)) goto done;
              }
              SDFB_TRACE(8);
              if (!(p.flags & 1u)) fence_proxy_async_global();
              st = stage;
              for (int k = 0; k < pre; ++k) {
                tma_load_2d_pair(smem0 + st * stage_bytes, &tm_act, g.a_col0 + kc_of(o, i + k) * 64, a_row,
                                 map_to_cta(bars + 8 * (kBarFull + st), lrank));
                if (++st == nst) st = 0;
              }
              SDFB_TRACE(9);
              stage = st;
              phase = ph;
              i += pre;
            }
            for (; i < g.nk; ++i) {
              if (!mbar_wait(bars + 8 * (kBarEmpty + stage), phase ^ 1u, wd, kErrEmpty, stage)) goto done;
              const uint32_t full = bars + 8 * (kBarFull + stage);
              if (leader) mbar_arrive_expect_tx(full, tx);
              const int kc = kc_of(o, i), wk = l == 0 ? (kc & 3) : kc;
              const uint32_t full_l = map_to_cta(full, lrank);
              tma_load_2d_pair(smem0 + stage * stage_bytes + kChunk, tmw, 0, w_row + wk * g.n_total, full_l);
              tma_load_2d_pair(smem0 + stage * stage_bytes, &tm_act, g.a_col0 + kc * 64, a_row, full_l);
              if (++stage == nst) { stage = 0; phase ^= 1u; }
            }
          }
        }
      }
    }
  } else if (warp == 9) {
    // ===================== MMA issuer (leader CTA; whole warp runs the loop, see fused_decoder.cu) =====================
    if (leader) {
      const uint32_t idesc_h = umma_idesc(256, p.bn_h, FP16 ? 0 : 1);
      const uint32_t idesc_o = umma_idesc(256, kDdpmOutTile, FP16 ? 0 : 1);
      const uint64_t desc_hi = umma_desc_sw128(0) & 0xFFFFFFFF00000000ull;
      const uint32_t nst = static_cast<uint32_t>(p.nstages);
      uint32_t stage = 0, phase = 0, ephase = 0, gt = 0, own_phase = 0, own_pending = 0;
      const bool prof = p.prof != nullptr;
      const int rounds = (p.pair_m_tiles * (kDdpmHid / p.bn_h) + npairs - 1) / npairs;
      const uint32_t stg_lo = ((smem0 + o_stage) & 0x3FFFFu) >> 4;
      for (int s = 0; s < p.steps; ++s) {
        for (int l = 0; l < kLayers; ++l) {
          const int nk = l == 0 ? 8 : 16;
          const uint32_t idesc = l == 4 ? idesc_o : idesc_h;
          const int ntn = l == 4 ? kDdpmLatent / kDdpmOutTile : kDdpmHid / p.bn_h;
          const int T = p.pair_m_tiles * ntn;
          // staging slots this pair's epilogue fills in this layer (one barrier phase each per tile)
          uint32_t my_slots = 0;
          int round = 0;
          for (int tile = first_tile(p, l, pidx, T); tile < T; tile += npairs, ++gt, ++round) {
            // staging slots this tile's epilogue fills (one barrier phase each)
            my_slots |= l == 4 ? (p.eps_mode ? 0u : 0xCu) : ((((1u << (p.bn_h >> 6)) - 1u) << (round * (p.bn_h >> 6))) & 0xFu);
            const uint32_t b = gt & 1u;
            const uint32_t d_tmem = tmem_base + b * 256;
            const Own o = own_chunks(p, s, l, tile % ntn, round, rounds);
            if (!mbar_wait(bars + 8 * (kBarAccEmpty + b), ((ephase >> b) & 1u) ^ 1u, wd, kErrAccEmpty, b)) goto done;
            ephase ^= 1u << b;
            // Two chunks per trip (nk is even; one commit point per pair - see the header comment), each issued as soon as
            // its own operands are there: this warp's instructions issue ~4 cycles apart, so a trip costs its instruction count
            // times that, and with 64- or 128-wide tiles that, not the tensor pipe, paced the layer.  Outside profiling runs
            // a wait is one try_wait.
#pragma unroll 1
            for (int k = 0; k < nk; k += 2) {
              const uint32_t s0 = stage, s1 = stage + 1 == nst ? 0u : stage + 1;
              const uint32_t ph1 = s1 == 0 ? phase ^ 1u : phase;
              uint32_t a0 = (((smem0 + s0 * stage_bytes) & 0x3FFFFu) >> 4) | (1u << 16);
              uint32_t a1 = (((smem0 + s1 * stage_bytes) & 0x3FFFFu) >> 4) | (1u << 16);
              const uint32_t b0 = a0 + (kChunk >> 4), b1 = a1 + (kChunk >> 4);
              if (k < o.n) {       // own chunks: A from the staging buffer, as soon as both CTAs' epilogues have finished it
                const uint32_t slot = static_cast<uint32_t>(o.slot0 + k);
                const uint32_t ob = bars + 8 * (kBarOwn + slot), op = (own_phase >> slot) & 1u;
                if (prof || !mbar_try_wait(ob, op)) { if (!mbar_wait(ob, op, wd, kErrOwn, slot)) goto done; }
                a0 = (stg_lo + slot * (kChunk >> 4)) | (1u << 16);
                if (k + 1 < o.n) {
                  const uint32_t ob1 = ob + 8, op1 = (own_phase >> (slot + 1)) & 1u;
                  if (prof || !mbar_try_wait(ob1, op1)) { if (!mbar_wait(ob1, op1, wd, kErrOwn, slot + 1)) goto done; }
                  a1 = (stg_lo + (slot + 1) * (kChunk >> 4)) | (1u << 16);
                }
              }
              const uint32_t f0 = bars + 8 * (kBarFull + s0), f1 = bars + 8 * (kBarFull + s1);
              if (prof || !mbar_try_wait(f0, phase)) { if (!mbar_wait(f0, phase, wd, k == 0 ? kErrFullFirst : kErrFull, s0)) goto done; }
              tc_fence_after();
              if (k == 0 && lane == 0) SDFB_TRACE(0);
              if (elect_one()) {
                const uint64_t ad0 = desc_hi | a0, bd0 = desc_hi | b0;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) umma_ss<2>(d_tmem, ad0 + 2 * jj, bd0 + 2 * jj, idesc, (k | jj) != 0 ? 1u : 0u);
              }
              if (prof || !mbar_try_wait(f1, ph1)) { if (!mbar_wait(f1, ph1, wd, kErrFull, s1)) goto done; }
              tc_fence_after();
              if (elect_one()) {
                const uint64_t ad1 = desc_hi | a1, bd1 = desc_hi | b1;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) umma_ss<2>(d_tmem, ad1 + 2 * jj, bd1 + 2 * jj, idesc, 1u);
                umma_commit<2>(bars + 8 * (kBarEmpty + s0), pmask);
                umma_commit<2>(bars + 8 * (kBarEmpty + s1), pmask);
                if (k + 2 == nk) umma_commit<2>(bars + 8 * (kBarAccFull + b), pmask);
              }
              __syncwarp();
              if (k + 2 == nk && lane == 0) SDFB_TRACE(1);
              if (s1 == 0) phase ^= 1u;
              stage = s1 + 1;
              if (stage == nst) { stage = 0; phase ^= 1u; }
            }
          }
          // The phases the previous layer's epilogues completed are behind us now, whether or not they were waited
          // for.  (With more tiles per layer than staging slots, slots are rewritten within a layer and own chunks
          // are off: the tracking is then unused.)
          own_phase ^= own_pending;
          own_pending = my_slots;
        }
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int q = warp & 3, set = warp >> 2;
    const int row = q * 32 + lane;                       // row of this CTA's 128 = TMEM lane
    const uint32_t row7 = static_cast<uint32_t>(row & 7);
    const uint32_t tmem_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const bool set_leader = (q == 0 && lane == 0);
    uint32_t acc_phase = 0, gt = 0, xn_phase = 0;
    for (int s = 0; s < p.steps; ++s) {
      // this step's schedule row: the timestep here, the coefficients and the noise plane only in the last layer (kept out
      // of the registers the hidden layers' epilogues need)
      const DdpmStep* srow = p.sched + s;
      const int t = srow->t;
      for (int l = 0; l < kLayers; ++l) {
        const Geo g = layer_geo(p, l);
        const float* bias = l == 0 ? p.tb0 + static_cast<long long>(t) * kDdpmHid
                                   : (l < 4 ? p.bias + (l - 1) * kDdpmHid : p.bias + 3 * kDdpmHid);
        const int T = p.pair_m_tiles * g.ntn;
        const int rounds = (p.pair_m_tiles * (kDdpmHid / p.bn_h) + npairs - 1) / npairs;
        for (int tile = first_tile(p, l, pidx, T), round = 0; tile < T; tile += npairs, ++gt, ++round) {
          const int pm = tile / g.ntn, j = tile - pm * g.ntn;
          const int g_row = (2 * pm + static_cast<int>(rank)) * 128;             // first latent of this CTA's half tile
          // staging slots of this tile's hidden output: one set per round while they all fit (they are then the
          // next layer's own chunks), else slots 0.. are simply reused
          const int slot0 = (l < 4 && rounds * (g.bn >> 6) <= 4) ? round * (g.bn >> 6) : 0;
          const uint32_t b = gt & 1u;
          const uint32_t tbase = tmem_row + b * 256;
          // The tile's bias slice -> shared memory, off the critical path (the producer's gpu-scope
          // acquires invalidate L1, so reading it from global after the accumulator wait costs an L2
          // round trip per load).  Double-buffered by tile parity.  The barrier also orders the
          // staging buffer: every bulk store of the previous tile has completed (its issuing thread
          // waited for that before it got here).
          float* sb = sbias + (gt & 1u) * 256;
          if (static_cast<int>(threadIdx.x) < g.bn) sb[threadIdx.x] = bias[j * g.bn + threadIdx.x];
          float4 cf = make_float4(0.f, 0.f, 0.f, 0.f), cg = cf;           // sra, srm1, c1, c2 | c3, sigma, clamp
          if (l == 4) {
            cf = reinterpret_cast<const float4*>(srow->coef)[0];
            cg = reinterpret_cast<const float4*>(srow->coef)[1];
          }
          const float sigma = cg.y;
          named_bar_sync(1, kEpiThreads);
          if (l == 4 && threadIdx.x == 0 && !p.eps_mode) {
            // x and this step's noise plane of this half tile: two 32-column fp32 boxes each
            const uint32_t xn = bars + 8 * kBarXn;
            const bool nz_box = sigma != 0.f && !p.philox;
            mbar_arrive_expect_tx(xn, (nz_box ? 4u : 2u) * kChunk);
            tma_load_2d(stg, &tm_x, j * 64, g_row, xn);
            tma_load_2d(stg + kChunk, &tm_x, j * 64 + 32, g_row, xn);
            if (nz_box) {
              tma_load_3d(stg + 2 * kChunk, &tm_nz, j * 64, g_row, srow->plane, xn);
              tma_load_3d(stg + 3 * kChunk, &tm_nz, j * 64 + 32, g_row, srow->plane, xn);
            }
          }
          if (l == 4 && p.philox && !p.eps_mode && sigma != 0.f) {
            // in-kernel noise: this thread's 32 normals -> its row of the noise box (the layout the TMA box would
            // have had), generated while the tensor core is still busy with this tile
            const uint32_t nrow_w = stg + (2 + set) * kChunk + row * 128u;
            const uint2 key = make_uint2(static_cast<uint32_t>(p.seed), static_cast<uint32_t>(p.seed >> 32));
#pragma unroll 2
            for (int u = 0; u < 8; ++u)
              st_shared_f4(nrow_w + ((static_cast<uint32_t>(u) ^ row7) << 4),
                           philox_normal4(static_cast<uint32_t>(j * 16 + set * 8 + u), static_cast<uint32_t>(p.first_latent + g_row + row),
                                          static_cast<uint32_t>(t), key));
          }
          if (!mbar_wait(bars + 8 * (kBarAccFull + b), (acc_phase >> b) & 1u, wd, kErrAccFull, b)) goto done;
          acc_phase ^= 1u << b;
          __syncwarp();
          tc_fence_after();
          if (threadIdx.x == 0) SDFB_TRACE(2);
          if (l < 4 && g.bn == 64) {
            // hidden layer, 64-wide tile (small batches: more, narrower tiles keep more SMs busy): ONE chunk, the two warp
            // sets convert its two 32-column halves; set 0 publishes it once both halves are written
            uint32_t v[32];
            tmem_ld32(tbase + set * 32, v);
            const uint32_t srow = stg + slot0 * kChunk + row * 128u;
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) arrive_on_leader(bars + 8 * (kBarAccEmpty + b), 1, lrank);
            const float4* b4 = reinterpret_cast<const float4*>(sb + 32 * set);
            uint32_t pk[16];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const float4 bb = b4[e];
              pk[2 * e] = pack_relu<FP16>(__uint_as_float(v[4 * e]) + bb.x, __uint_as_float(v[4 * e + 1]) + bb.y);
              pk[2 * e + 1] = pack_relu<FP16>(__uint_as_float(v[4 * e + 2]) + bb.z, __uint_as_float(v[4 * e + 3]) + bb.w);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
              st_shared_v4(srow + (((4 * set + u) ^ row7) << 4), pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
            fence_proxy_async_smem();
            named_bar_sync(1, kEpiThreads);
            if (set == 0 && lane == 0) arrive_on_leader(bars + 8 * (kBarOwn + slot0), 1, lrank);   // 4 warps x 2 CTAs = the 8 expected
            if (threadIdx.x == 0) {
              SDFB_TRACE(3);
              tma_store_2d(&tm_act, g.o_col0 + j * 64, g_row, stg + slot0 * kChunk);
              bulk_commit_group();
              SDFB_TRACE(4);
              bulk_wait_group0();
              SDFB_TRACE(5);
              if (p.flags & 2u) {
                red_relaxed_gpu_add(p.counter + pm, 2u);
              } else {
                fence_proxy_async_global();
                red_release_gpu_add(p.counter + pm, 2u);                         // both warp sets' worth
              }
              SDFB_TRACE(6);
            }
          } else if (l < 4) {
            // hidden layer: + bias, ReLU, round to 16 bits -> swizzled operand image in the staging
            // buffer -> one TMA store per 64-feature chunk (set s owns chunks c = s, s + 2, ...)
            const int nch = g.bn >> 6;
            for (int c = set; c < nch; c += 2) {
              uint32_t v[2][32];
              tmem_ld32(tbase + c * 64, v[0]);
              tmem_ld32(tbase + c * 64 + 32, v[1]);
              const uint32_t srow = stg + (slot0 + c) * kChunk + row * 128u;
              tmem_ld_wait();
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const float4* b4 = reinterpret_cast<const float4*>(sb + c * 64 + 32 * h);
                uint32_t pk[16];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                  const float4 bb = b4[e];
                  pk[2 * e] = pack_relu<FP16>(__uint_as_float(v[h][4 * e]) + bb.x, __uint_as_float(v[h][4 * e + 1]) + bb.y);
                  pk[2 * e + 1] = pack_relu<FP16>(__uint_as_float(v[h][4 * e + 2]) + bb.z, __uint_as_float(v[h][4 * e + 3]) + bb.w);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                  st_shared_v4(srow + (((4 * h + u) ^ row7) << 4), pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
              }
              if (c + 2 >= nch) {      // every column this warp owns has been read: hand the accumulator back
                tc_fence_before();
                __syncwarp();
                if (lane == 0) arrive_on_leader(bars + 8 * (kBarAccEmpty + b), 1, lrank);
              }
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) arrive_on_leader(bars + 8 * (kBarOwn + slot0 + c), 1, lrank);   // the pair's next layer may start on this chunk
              named_bar_sync(2 + set, kEpiThreads / 2);
              if (set_leader) {
                if (c == 0) SDFB_TRACE(3);
                tma_store_2d(&tm_act, g.o_col0 + j * g.bn + c * 64, g_row, stg + (slot0 + c) * kChunk);
                bulk_commit_group();
              }
            }
            if (threadIdx.x == 0) SDFB_TRACE(4);
            if (set_leader) {          // stores complete -> arrive on the barrier of this latent group
              bulk_wait_group0();
              if (threadIdx.x == 0) SDFB_TRACE(5);
              if (p.cluster8) {
                // the latent group IS the cluster: one arrival on every member's group barrier instead of a counter in L2
                fence_proxy_async_global();
                fence_acq_rel_cluster();
                for (uint32_t r = 0; r < static_cast<uint32_t>(p.cluster_ctas); ++r) mbar_arrive_remote_relaxed(bars + 8 * kBarGroup, r, 1u);
              } else if (p.flags & 2u) {
                red_relaxed_gpu_add(p.counter + pm, 1u);
              } else {
                fence_proxy_async_global();
                red_release_gpu_add(p.counter + pm, 1u);
              }
              if (threadIdx.x == 0) SDFB_TRACE(6);
            }
          } else {
            // last layer (64 features per tile; set s owns columns [32 s, 32 s + 32)):
            // eps -> the schedule row's update, op for op as oracle/ddpm.py ddpm_step (DDPM rows) and tests/ddim_reference.py (DDIM rows)
            uint32_t v[32];
            tmem_ld32(tbase + set * 32, v);
            if (!p.eps_mode) {
              if (!mbar_wait(bars + 8 * kBarXn, xn_phase, wd, kErrXn)) goto done;
              xn_phase ^= 1u;
            }
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) arrive_on_leader(bars + 8 * (kBarAccEmpty + b), 1, lrank);
            if (threadIdx.x == 0) SDFB_TRACE(10);
            const uint32_t xrow = stg + set * kChunk + row * 128u;             // this thread's 32 floats of x (swizzled 16-byte units)
            const uint32_t nrow = xrow + 2 * kChunk;
            const uint32_t hrow = stg + 2 * kChunk + row * 128u, lrow = hrow + kChunk;   // x_hi / x_lo images: OVER the noise boxes
            // everything this thread needs from shared memory -> registers, then a barrier: after it the noise boxes
            // (read by their own warp set only) may be overwritten by the operand images (written by both sets)
            float4 xq[8], nq[8];
            if (!p.eps_mode) {
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const uint32_t off = (static_cast<uint32_t>(u) ^ row7) << 4;
                xq[u] = ld_shared_f4(xrow + off);
                nq[u] = sigma != 0.f ? ld_shared_f4(nrow + off) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
            }
            named_bar_sync(1, kEpiThreads);
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const uint32_t off = (static_cast<uint32_t>(u) ^ row7) << 4;
              const float4 bb = *reinterpret_cast<const float4*>(sb + set * 32 + 4 * u);
              const float e0 = __uint_as_float(v[4 * u]) + bb.x, e1 = __uint_as_float(v[4 * u + 1]) + bb.y;
              const float e2 = __uint_as_float(v[4 * u + 2]) + bb.z, e3 = __uint_as_float(v[4 * u + 3]) + bb.w;
              float4 o;
              if (p.eps_mode) {
                o = make_float4(e0, e1, e2, e3);
              } else {
                const float ev[4] = {e0, e1, e2, e3};
                const float xs[4] = {xq[u].x, xq[u].y, xq[u].z, xq[u].w};
                const float ns[4] = {nq[u].x, nq[u].y, nq[u].z, nq[u].w};
                float r[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float x0 = __fsub_rn(__fmul_rn(cf.x, xs[e]), __fmul_rn(cf.y, ev[e]));
                  x0 = fminf(fmaxf(x0, -cg.z), cg.z);
                  r[e] = __fadd_rn(__fmul_rn(cf.z, x0), __fmul_rn(cf.w, xs[e]));
                  if (cg.x != 0.f) r[e] = __fadd_rn(r[e], __fmul_rn(cg.x, ev[e]));
                  if (sigma != 0.f) r[e] = __fadd_rn(r[e], __fmul_rn(sigma, ns[e]));
                }
                o = make_float4(r[0], r[1], r[2], r[3]);
                split2<FP16>(r[0], r[1], hi[2 * (u & 1)], lo[2 * (u & 1)]);
                split2<FP16>(r[2], r[3], hi[2 * (u & 1) + 1], lo[2 * (u & 1) + 1]);
                if (u & 1) {   // 8 values = one 16-byte unit of the x_hi / x_lo operand images
                  const uint32_t hoff = ((static_cast<uint32_t>(4 * set + (u >> 1))) ^ row7) << 4;
                  st_shared_v4(hrow + hoff, hi[0], hi[1], hi[2], hi[3]);
                  st_shared_v4(lrow + hoff, lo[0], lo[1], lo[2], lo[3]);
                }
              }
              st_shared_f4(xrow + off, o);                                      // in place (eps_mode: the eps tile)
            }
            if (threadIdx.x == 0) SDFB_TRACE(11);
            fence_proxy_async_smem();
            named_bar_sync(1, kEpiThreads);
            // both sets wrote both images: only now are they complete.  x_hi (slot 2) / x_lo (slot 3) are the own
            // chunks of the next step's layer 0; one warp set arrives per slot, as for the hidden layers' slots.
            if (lane == 0 && !p.eps_mode) arrive_on_leader(bars + 8 * (kBarOwn + 2 + set), 1, lrank);
            if (threadIdx.x == 0) {
              tma_store_2d(&tm_x, j * 64, g_row, stg);                          // rows >= n are clipped by the TMA unit
              tma_store_2d(&tm_x, j * 64 + 32, g_row, stg + kChunk);
              if (!p.eps_mode) {
                tma_store_2d(&tm_act, j * 64, g_row, stg + 2 * kChunk);
                tma_store_2d(&tm_act, 256 + j * 64, g_row, stg + 3 * kChunk);
              }
              bulk_commit_group();
              SDFB_TRACE(4);
              bulk_wait_group0();
              SDFB_TRACE(5);
              if (p.cluster8) {
                fence_proxy_async_global();
                fence_acq_rel_cluster();
                // (four tiles per group: with 16 CTAs each of the eight arriving CTAs stands in for two)
                for (uint32_t r = 0; r < static_cast<uint32_t>(p.cluster_ctas); ++r)
                  mbar_arrive_remote_relaxed(bars + 8 * kBarGroup, r, p.cluster_ctas == 16 ? 4u : 2u);
              } else if (p.flags & 2u) {
                red_relaxed_gpu_add(p.counter + pm, 2u);
              } else {
                fence_proxy_async_global();
                red_release_gpu_add(p.counter + pm, 2u);                        // both warp sets' worth
              }
              SDFB_TRACE(6);
            }
          }
        }
      }
    }
  }
done:
  if (p.prof != nullptr && lane == 0 && (warp == 0 || warp >= 8) && (leader || warp != 9)) {
    const int role = warp == 0 ? 0 : warp - 7;            // 0 epilogue, 1 producer, 2 MMA issuer
    long long* dst = p.prof + (static_cast<long long>(blockIdx.x) * 3 + role) * 8;
#pragma unroll
    for (int i = 1; i < 8; ++i) dst[i] = waited[i];
    dst[0] = clock64() - t_start;
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 9) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<2>(tmem_base, 512);
  }
}

// x fp32 -> [x_hi | x_lo] columns (0..511) of the row-major activation buffer; rows >= n are zero.
template <bool FP16>
__global__ void ddpm_split_kernel(const float* __restrict__ x, int n, int n_pad, uint16_t* __restrict__ act) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // (row, 8-column unit)
  const long long total = static_cast<long long>(n_pad) * 32;
  if (i >= total) return;
  const long long m = i >> 5;
  const int u8 = static_cast<int>(i & 31);
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (m < n) {
    const float4* src = reinterpret_cast<const float4*>(x + m * kDdpmLatent + u8 * 8);
    const float4 a = src[0], b = src[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) split2<FP16>(v[2 * e], v[2 * e + 1], hi[e], lo[e]);
  uint16_t* rowp = act + m * kDdpmActCols + u8 * 8;
  *reinterpret_cast<uint4*>(rowp) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<uint4*>(rowp + 256) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// noise rows [t0, t1) of n latents -> out [(t1 - t0)][n][256] (what the sampler generates in-kernel)
__global__ void philox_normal_kernel(unsigned long long seed, unsigned int first_latent, int n, int t0, int t1,
                                     float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // (t, row, column group)
  const long long total = static_cast<long long>(t1 - t0) * n * 64;
  if (i >= total) return;
  const uint32_t g = static_cast<uint32_t>(i & 63);
  const long long rt = i >> 6;
  const uint32_t row = static_cast<uint32_t>(rt % n), t = static_cast<uint32_t>(t0 + rt / n);
  const float4 z = philox_normal4(g, first_latent + row, t, make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
  reinterpret_cast<float4*>(out)[i] = z;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

uint32_t smem_bytes_for(int bn_h, int nstages) {
  return static_cast<uint32_t>(nstages) * (kChunk + static_cast<uint32_t>(bn_h) * 64u) + kStagingBytes + kBarBytes + 16 + 2048;
}

}  // namespace

cudaError_t ddpm_step_init() {
  const uint32_t m1 = smem_bytes_for(256, 5), m2 = smem_bytes_for(128, 6), m3 = smem_bytes_for(64, 8);
  const int max_smem = static_cast<int>(m1 > m2 ? (m1 > m3 ? m1 : m3) : (m2 > m3 ? m2 : m3));   // ring + 64 KiB staging, largest configuration
  cudaError_t e = cudaFuncSetAttribute(ddpm_sample_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(ddpm_sample_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
  if (e != cudaSuccess) return e;
  // clusters of 16 CTAs (one latent group of eight 128-wide pair tiles) are beyond the portable size of 8
  e = cudaFuncSetAttribute(ddpm_sample_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(ddpm_sample_kernel<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
}

cudaError_t make_tensor_map(void* tmap_out, const void* base, int elem_bytes, int rank, const unsigned long long* dims,
                            const unsigned long long* strides_bytes, const unsigned* box, bool swizzle128) {
  // the driver entry point is looked up once (this runs twice per launch of the general product: ~30 times per training step)
  static std::atomic<void*> cached{nullptr};
  void* fn = cached.load(std::memory_order_acquire);
  if (fn == nullptr) {
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess) return e;
    if (fn == nullptr || qres != cudaDriverEntryPointSuccess) return cudaErrorNotSupported;
    cached.store(fn, std::memory_order_release);
  }
  cuuint64_t gdim[3], gstride[2];
  cuuint32_t bx[3], estr[3] = {1u, 1u, 1u};
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) gstride[i] = strides_bytes[i];
  CUresult r = reinterpret_cast<EncodeTiledFn>(fn)(
      static_cast<CUtensorMap*>(tmap_out), elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16,
      static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim, gstride, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
      swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

cudaError_t launch_philox_normal(unsigned long long seed, unsigned int first_latent, int n, int t0, int t1, float* out,
                                 cudaStream_t stream) {
  const long long total = static_cast<long long>(t1 - t0) * n * 64;
  if (total <= 0) return cudaSuccess;
  philox_normal_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(seed, first_latent, n, t0, t1, out);
  return cudaGetLastError();
}

// How many clusters of `csize` CTAs of the sampler kernel can be resident at once (0 if the query fails).
static int ddpm_max_clusters(int csize, int bn_h, int nstages, bool fp16) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(csize * 18);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes_for(bn_h, nstages);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  cudaError_t e = fp16 ? cudaOccupancyMaxActiveClusters(&n, ddpm_sample_kernel<true>, &cfg)
                       : cudaOccupancyMaxActiveClusters(&n, ddpm_sample_kernel<false>, &cfg);
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int ddpm_max_clusters8(int bn_h, int nstages, bool fp16) { return ddpm_max_clusters(8, bn_h, nstages, fp16); }
int ddpm_max_clusters16(int bn_h, int nstages, bool fp16) { return ddpm_max_clusters(16, bn_h, nstages, fp16); }

cudaError_t launch_ddpm_split(const float* x, int n, int n_pad, uint16_t* act, bool fp16, cudaStream_t stream) {
  const long long total = static_cast<long long>(n_pad) * 32;
  const unsigned blocks = static_cast<unsigned>((total + 255) / 256);
  if (fp16) ddpm_split_kernel<true><<<blocks, 256, 0, stream>>>(x, n, n_pad, act);
  else ddpm_split_kernel<false><<<blocks, 256, 0, stream>>>(x, n, n_pad, act);
  return cudaGetLastError();
}

cudaError_t launch_ddpm_sample(const DdpmParams& p, const DdpmMaps& maps, bool fp16, int num_sms, cudaStream_t stream) {
  const int T = p.pair_m_tiles * (kDdpmHid / p.bn_h);       // pair tiles of a hidden layer (>= those of the last layer)
  const int max_pairs = num_sms / 2;
  const int rounds = (T + max_pairs - 1) / max_pairs;       // tiles per pair and layer
  const int pairs = (T + rounds - 1) / rounds;              // balanced: no pair gets more than `rounds`, few get less
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(2 * pairs));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem_bytes_for(p.bn_h, p.nstages);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.cluster8 ? p.cluster_ctas : 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // Every CTA must be resident: pair tiles of one latent group wait on one another.  The grid never exceeds one CTA
  // per SM and is checked against the occupancy calculator here, instead of asking for a cooperative launch (which
  // profilers cannot replay together with clusters): on a GPU this process shares with nothing else the whole grid is
  // then co-resident, and if something else does hold SMs the in-kernel watchdog turns the wait into SDFB_E_KERNEL.
  // (In cluster8 mode nothing waits across clusters, and the hardware co-schedules a cluster's CTAs.)
  if (!p.cluster8) {
    static int max_pairs_cache[2][3][8] = {};     // [fp16][bn_h / 128][nstages]
    int& cached = max_pairs_cache[fp16 ? 1 : 0][p.bn_h >> 7][p.nstages & 7];
    if (cached == 0) cached = ddpm_max_clusters(2, p.bn_h, p.nstages, fp16);
    if (pairs > cached) return cudaErrorCooperativeLaunchTooLarge;
  }
  const CUtensorMap* a = reinterpret_cast<const CUtensorMap*>(maps.act);
  const CUtensorMap* wh = reinterpret_cast<const CUtensorMap*>(maps.wh);
  const CUtensorMap* wo = reinterpret_cast<const CUtensorMap*>(maps.wo);
  const CUtensorMap* x = reinterpret_cast<const CUtensorMap*>(maps.x);
  const CUtensorMap* nz = reinterpret_cast<const CUtensorMap*>(maps.nz);
  if (fp16) return cudaLaunchKernelEx(&cfg, ddpm_sample_kernel<true>, p, *a, *wh, *wo, *x, *nz);
  return cudaLaunchKernelEx(&cfg, ddpm_sample_kernel<false>, p, *a, *wh, *wo, *x, *nz);
}

}  // namespace sdfb
