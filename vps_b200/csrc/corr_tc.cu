// Correlation (cost volume) on tcgen05 tensor cores -- the FlowNetC (pad 20, d 20, s2 2 -> 441 ch) and
// LiteFlowNetCorr (pad 4, d 4, s2 1 -> 81 ch) call sites of correlation_cuda.forward
// (correlation_cuda.cc:10-87, correlation_cuda_kernel.cu:74-147), bf16 features, fp32 accumulation.
//
// Banded GEMM, transposed on purpose:  D[n, m] = sum_c f2[n, c] * f1[m, c]
//   m = one of 96 output pixels of a TH x TW tile (pixels of ONE stride2-parity class, so that every needed f2
//       pixel has the same parity and element-strided TMA boxes fetch exactly the useful pixels),
//   n = f2 pixels of the tile's displacement neighbourhood, (TH + 2R) rows x 32 columns, 4 rows (128 pixels = 128
//       TMEM lanes) per MMA block.
// With f2 on the TMEM-lane axis, a thread (lane = neighbourhood column j') that walks the accumulator columns of a
// tile row i finds in column (i, j) the value of output pixel (i, j) at displacement (tj, ti) = (i' - i, j' - j):
// consecutive lanes hold consecutive ti of the SAME output pixel, i.e. consecutive addresses of the NHWC output --
// the band is extracted with plain coalesced stores, no shuffles and no shared-memory staging.
//
//   warp 0: TMA producer (f1 tile resident & double-buffered per tile; f2 blocks streamed through a 6-stage ring)
//   warp 1: TMEM alloc + tcgen05.mma issue (M=128, N=96, K=16), accumulators double-buffered
//   warps 2-9: epilogue, warp -> neighbourhood row 4*block + (warp % 4); the two warps of a row split the output rows
#include <cudaTypedefs.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace {

constexpr int NPIX = 96;           // output pixels per tile (MMA N)
constexpr int KC = 64;             // channels per K chunk (128-byte rows, SWIZZLE_128B)
constexpr int A_BYTES = 128 * KC * 2;       // one f2 block chunk  (16 KiB)
constexpr int B_BYTES = NPIX * KC * 2;      // one f1 tile chunk   (12 KiB)
constexpr int A_STAGES = 6;
constexpr int MAX_KCH = 4;         // C <= 256

struct CorrParams {
  int H, W, C, kch;
  int tiles_x, tiles_y, total_tiles;   // total = tiles_y * tiles_x * S2*S2 * n_img
  int n_img;
  void* out; int out_cs, out_dtype;
  int act; float slope;
  float scale;        // result = accumulator * scale (1/C; the correction passes of the fp32-parity mode carry 2^-11 as well)
  int accumulate;     // 1: add to the fp32 value already in `out` before the activation
  int f16;            // 1: fp16 operands (the split planes of fp32 features), 0: bf16
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1u << 26)) {
      printf("vps corr_tc: mbarrier timeout block %d thread %d bar %u\n", blockIdx.x, threadIdx.x, bar);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t addr) {   // K-major, 128-byte rows, SWIZZLE_128B
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t* r);
template <>
__device__ __forceinline__ void tmem_ld<4>(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld<8>(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// R = max_displacement / stride2, S2 = stride2.  TW = 32 - 2R so the neighbourhood is exactly 32 columns wide.
template <int R, int S2>
__global__ void __launch_bounds__(320, 1)
corr_tc_kernel(const __grid_constant__ CUtensorMap tmF1, const __grid_constant__ CUtensorMap tmF2, const CorrParams p) {
  constexpr int D = 2 * R + 1;
  constexpr int TW = 32 - 2 * R;
  constexpr int TH = NPIX / TW;
  constexpr int NBLK = (TH + 2 * R) / 4;
  static_assert(TW * TH == NPIX && (TH + 2 * R) % 4 == 0, "tile geometry");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_ring = base;                                   // A_STAGES x 16 KiB
  const uint32_t b_buf = base + A_STAGES * A_BYTES;               // 2 x (kch x 12 KiB)
  const uint32_t b_tile_bytes = (uint32_t)p.kch * B_BYTES;
  const uint32_t bars = b_buf + 2 * MAX_KCH * B_BYTES;
  auto afull = [&](int s) { return bars + 8u * s; };
  auto aempty = [&](int s) { return bars + 8u * (A_STAGES + s); };
  auto bfull = [&](int s) { return bars + 8u * (2 * A_STAGES + s); };
  auto bempty = [&](int s) { return bars + 8u * (2 * A_STAGES + 2 + s); };
  auto tfull = [&](int s) { return bars + 8u * (2 * A_STAGES + 4 + s); };
  auto tempty = [&](int s) { return bars + 8u * (2 * A_STAGES + 6 + s); };
  const uint32_t tmem_slot = bars + 8u * (2 * A_STAGES + 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < A_STAGES; ++s) { mbar_init(afull(s), 1); mbar_init(aempty(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(bfull(s), 1); mbar_init(bempty(s), 1); mbar_init(tfull(s), 1); mbar_init(tempty(s), 256); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(256u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  const int tiles_per_par = p.tiles_y * p.tiles_x;
  auto decode = [&](int tile, int& img, int& py, int& px, int& y0, int& x0) {
    const int per_img = tiles_per_par * S2 * S2;
    img = tile / per_img;
    int t = tile - img * per_img;
    const int par = t / tiles_per_par;
    t -= par * tiles_per_par;
    py = par / S2; px = par % S2;
    y0 = (t / p.tiles_x) * TH * S2; x0 = (t % p.tiles_x) * TW * S2;
  };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int bsel = 0; uint32_t bphase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        int img, py, px, y0, x0;
        decode(tile, img, py, px, y0, x0);
        // f1 tile (MMA B operand): resident for the whole tile, double-buffered across tiles
        mbar_wait(bempty(bsel), bphase ^ 1);
        mbar_expect_tx(bfull(bsel), b_tile_bytes);
        for (int kc = 0; kc < p.kch; ++kc)
          tma_load_4d(b_buf + bsel * MAX_KCH * B_BYTES + kc * B_BYTES, &tmF1, bfull(bsel), kc * KC, x0 + px, y0 + py, img);
        // f2 neighbourhood blocks (MMA A operand): 4 rows x 32 columns of same-parity pixels each
        for (int b = 0; b < NBLK; ++b) {
          for (int kc = 0; kc < p.kch; ++kc) {
            mbar_wait(aempty(stage), phase ^ 1);
            mbar_expect_tx(afull(stage), A_BYTES);
            tma_load_4d(a_ring + stage * A_BYTES, &tmF2, afull(stage), kc * KC, x0 + px - R * S2,
                        y0 + py + (4 * b - R) * S2, img);
            if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
          }
        }
        bsel ^= 1; if (bsel == 0) bphase ^= 1;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t fmt = p.f16 ? 0u : ((1u << 7) | (1u << 10));       // A / B format: 0 = f16, 1 = bf16
      const uint32_t idesc = (1u << 4) | fmt | ((uint32_t)(NPIX >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      int stage = 0; uint32_t phase = 0;
      int bsel = 0; uint32_t bphase = 0;
      int acc = 0; uint32_t aphase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        mbar_wait(bfull(bsel), bphase);
        tc_fence_after();
        for (int b = 0; b < NBLK; ++b) {
          mbar_wait(tempty(acc), aphase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)acc * 128u;
          for (int kc = 0; kc < p.kch; ++kc) {
            mbar_wait(afull(stage), phase);
            tc_fence_after();
            const uint64_t adesc = make_desc(a_ring + stage * A_BYTES);
            const uint64_t bdesc = make_desc(b_buf + bsel * MAX_KCH * B_BYTES + kc * B_BYTES);
#pragma unroll
            for (int k = 0; k < KC / 16; ++k)
              umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (uint32_t)((kc | k) != 0));
            umma_commit(aempty(stage));
            if (++stage == A_STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit(tfull(acc));
          acc ^= 1; if (acc == 0) aphase ^= 1;
        }
        umma_commit(bempty(bsel));      // all MMAs reading this f1 tile have completed when this fires
        bsel ^= 1; if (bsel == 0) bphase ^= 1;
      }
    }
  } else {
    // 8 epilogue warps: warp -> TMEM lane quarter q (= neighbourhood row inside the block); the two warps of a quarter
    // take alternate output rows i.  The TMEM load of the next row is in flight while the current one is stored.
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    int acc = 0; uint32_t aphase = 0;
    const float inv_c = p.scale;
    auto load_row = [&](uint32_t t_row, int i, uint32_t* r) {
      if constexpr (TW == 12) { tmem_ld<8>(t_row + i * TW, r); tmem_ld<4>(t_row + i * TW + 8, r + 8); }
      else { tmem_ld<16>(t_row + i * TW, r); tmem_ld<8>(t_row + i * TW + 16, r + 16); }
    };
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      int img, py, px, y0, x0;
      decode(tile, img, py, px, y0, x0);
      for (int b = 0; b < NBLK; ++b) {
        mbar_wait(tfull(acc), aphase);
        tc_fence_after();
        const int ip = 4 * b + q;        // neighbourhood row i' of this warp; lane = neighbourhood column j'
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * 128u;
        // output rows i with 0 <= i' - i < D, split between the two warps of this quarter
        const int i_lo = max(0, ip - D + 1) + half, i_hi = min(TH - 1, ip);
        auto store_row = [&](int i, const uint32_t* r) {
          const int tj = ip - i;
          const int y = y0 + py + i * S2;
          if (y >= p.H) return;
          const int64_t rowb = ((int64_t)img * p.H + y) * p.W * p.out_cs + tj * D + lane;
#pragma unroll
          for (int j = 0; j < TW; ++j) {
            const int ti = lane - j;
            const int x = x0 + px + j * S2;
            if (ti >= 0 && ti < D && x < p.W) {
              float v = __uint_as_float(r[j]) * inv_c;
              const int64_t o = rowb + (int64_t)x * p.out_cs - j;
              if (p.accumulate) v += ((const float*)p.out)[o];
              if (p.act == VPS_ACT_LRELU) v = v > 0.f ? v : v * p.slope;
              if (p.out_dtype == VPS_BF16) ((__nv_bfloat16*)p.out)[o] = __float2bfloat16_rn(v);
              else ((float*)p.out)[o] = v;
            }
          }
        };
        uint32_t ra[TW], rb[TW];
        int i = i_lo;
        if (i <= i_hi) load_row(t_row, i, ra);
        while (i <= i_hi) {
          tmem_wait();
          if (i + 2 <= i_hi) load_row(t_row, i + 2, rb);
          store_row(i, ra);
          i += 2;
          if (i > i_hi) break;
          tmem_wait();
          if (i + 2 <= i_hi) load_row(t_row, i + 2, ra);
          store_row(i, rb);
          i += 2;
        }
        tmem_wait();
        tc_fence_before();
        mbar_arrive(tempty(acc));
        acc ^= 1; if (acc == 0) aphase ^= 1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
}

PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (PFN_cuTensorMapEncodeTiled_v12000)ptr;
  }
  return fn;
}

template <int R, int S2>
int launch(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int act, float slope, cudaStream_t st,
           float scale = 0.f, int accumulate = 0, int f16 = 0) {
  constexpr int TW = 32 - 2 * R, TH = NPIX / TW;
  auto encode = get_encode();
  if (!encode) { vps::set_error("cuTensorMapEncodeTiled unavailable"); return VPS_E_CUDA; }
  static int num_sms = 0;
  if (!num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  CorrParams p;
  p.H = f1->h; p.W = f1->w; p.C = f1->c; p.kch = f1->c / KC; p.n_img = f1->n;
  p.tiles_y = vps::cdiv(vps::cdiv(f1->h, S2), TH);
  p.tiles_x = vps::cdiv(vps::cdiv(f1->w, S2), TW);
  p.total_tiles = p.tiles_y * p.tiles_x * S2 * S2 * f1->n;
  p.out = out->ptr; p.out_cs = out->cs; p.out_dtype = out->dtype; p.act = act; p.slope = slope;
  p.scale = scale != 0.f ? scale : 1.0f / (float)f1->c; p.accumulate = accumulate; p.f16 = f16;
  CUtensorMap tm1, tm2;
  for (int which = 0; which < 2; ++which) {
    const vps_tensor* t = which == 0 ? f1 : f2;
    cuuint64_t dims[4] = {(cuuint64_t)t->c, (cuuint64_t)t->w, (cuuint64_t)t->h, (cuuint64_t)t->n};
    cuuint64_t strides[3] = {(cuuint64_t)t->cs * 2, (cuuint64_t)t->w * t->cs * 2, (cuuint64_t)t->h * t->w * t->cs * 2};
    cuuint32_t box1[4] = {KC, (cuuint32_t)(TW * S2), (cuuint32_t)(TH * S2), 1};
    cuuint32_t box2[4] = {KC, (cuuint32_t)(32 * S2), (cuuint32_t)(4 * S2), 1};
    cuuint32_t estr[4] = {1, S2, S2, 1};
    CUresult r = encode(which == 0 ? &tm1 : &tm2, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, t->ptr, dims, strides,
                        which == 0 ? box1 : box2, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { vps::set_error("correlation_tc: tensor map encode failed (%d)", (int)r); return VPS_E_CUDA; }
  }
  const int smem = A_STAGES * A_BYTES + 2 * MAX_KCH * B_BYTES + 1024 + 8 * (2 * A_STAGES + 12);
  auto kern = corr_tc_kernel<R, S2>;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
      vps::set_error("correlation_tc: smem attr: %s", cudaGetErrorString(cudaGetLastError()));
      return VPS_E_CUDA;
    }
    attr_set = true;
  }
  const int grid = p.total_tiles < num_sms ? p.total_tiles : num_sms;
  kern<<<grid, 320, smem, st>>>(tm1, tm2, p);
  VPS_CUDA_LAST("corr_tc_kernel");
  return VPS_OK;
}

// fp32 features -> two fp16 planes (dense NHWC, cs = c):  hi = fp16(v),  lo = fp16(2^11 * (v - hi))  -- the operand split of the
// fp32-parity convolutions (conv_tc32.cu): v = hi + 2^-11 * lo to ~2^-22 relative
__global__ void split_f16_planes_kernel(const float* __restrict__ x, int64_t npix, int c, int cs, __half* __restrict__ hi,
                                        __half* __restrict__ lo, unsigned int* overflow) {
  const int64_t total = npix * (c / 4);
  bool over = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pix = i / (c / 4);
    const int c4 = (int)(i - pix * (c / 4)) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + pix * cs + c4);
    const float vv[4] = {v.x, v.y, v.z, v.w};
    __half h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned short hb, lb;
      asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(hb) : "f"(vv[k]));
      over = over || !(fabsf(vv[k]) <= 65504.f);
      const float r = (vv[k] - __half2float(__ushort_as_half(hb))) * 2048.f;
      asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(lb) : "f"(r));
      h[k] = __ushort_as_half(hb); l[k] = __ushort_as_half(lb);
    }
    *reinterpret_cast<uint2*>(hi + pix * c + c4) = *reinterpret_cast<const uint2*>(h);
    *reinterpret_cast<uint2*>(lo + pix * c + c4) = *reinterpret_cast<const uint2*>(l);
  }
  if (over && overflow) atomicAdd(overflow, 1u);
}

}  // namespace

extern "C" unsigned int* vps_tc32_overflow_flag();      // conv_tc32.cu: device address of the saturation counter

extern "C" int64_t vps_correlation_tc32_ws_bytes(const vps_tensor* f1) {
  return 4 * (int64_t)f1->n * f1->h * f1->w * f1->c * 2 + 1024;
}

// Correlation of fp32 features on the tensor cores in the parity precision: both maps are split into fp16 planes
// (v = hi + 2^-11 lo) and the banded GEMM runs three times, hi.hi, then hi.lo and lo.hi scaled by 2^-11 and accumulated
// into the fp32 output (the activation is applied by the last pass).  Unlike the stacked convolutions a correlation is a
// single K = C <= 256 contraction (16 MMAs per accumulator chain) whose result is not fed through further layers of the same
// kind, so the tensor core's truncating accumulation needs no promotion here (measured on a B200 at C = 256 with
// all-positive features: mean relative error -1.2e-6, max 1.4e-6 of sum |f1 f2| / C; the promoted convolutions: -7e-8).
// `ws`: vps_correlation_tc32_ws_bytes() of scratch, 256-byte aligned.  Same supported geometries as vps_correlation_tc.
extern "C" int vps_correlation_tc32(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad, int max_disp,
                                    int stride1, int stride2, int act, float slope, void* ws, void* stream) {
  VPS_CHECK_ARG(stride1 == 1 && pad == max_disp, "correlation_tc32: only stride1=1, pad==max_displacement");
  VPS_CHECK_ARG(f1->dtype == VPS_F32 && f2->dtype == VPS_F32 && out->dtype == VPS_F32, "correlation_tc32: fp32 tensors only");
  VPS_CHECK_ARG(f1->h == f2->h && f1->w == f2->w && f1->c == f2->c && f1->n == f2->n && out->h == f1->h && out->w == f1->w,
                "correlation_tc32: shape mismatch");
  VPS_CHECK_ARG(f1->c % KC == 0 && f1->c <= KC * MAX_KCH, "correlation_tc32: C must be a multiple of 64, <= 256");
  VPS_CHECK_ARG(f1->cs % 4 == 0 && f2->cs % 4 == 0 && ((uintptr_t)f1->ptr & 15) == 0 && ((uintptr_t)f2->ptr & 15) == 0 &&
                    ws && ((uintptr_t)ws & 255) == 0, "correlation_tc32: features / scratch must be aligned");
  VPS_CHECK_ARG(act == VPS_ACT_NONE || act == VPS_ACT_LRELU, "correlation_tc32: act");
  const int R = max_disp / stride2, D = 2 * R + 1;
  VPS_CHECK_ARG(out->c == D * D, "correlation_tc32: out.c %d != %d", out->c, D * D);
  VPS_CHECK_ARG((R == 10 && stride2 == 2) || (R == 4 && stride2 == 1), "correlation_tc32: unsupported (max_disp %d, stride2 %d)",
                max_disp, stride2);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t npix = (int64_t)f1->n * f1->h * f1->w, plane = npix * f1->c;
  __half* base = (__half*)ws;
  vps_tensor t[4];      // f1 hi, f1 lo, f2 hi, f2 lo
  for (int i = 0; i < 4; ++i) {
    t[i] = *f1; t[i].ptr = base + i * plane; t[i].cs = f1->c; t[i].dtype = VPS_BF16;      // (2-byte elements; the kernel is told f16)
  }
  unsigned int* flag = vps_tc32_overflow_flag();
  const int blocks = (int)((npix * (f1->c / 4) + 255) / 256 > 8192 ? 8192 : (npix * (f1->c / 4) + 255) / 256);
  split_f16_planes_kernel<<<blocks, 256, 0, st>>>((const float*)f1->ptr, npix, f1->c, f1->cs, base, base + plane, flag);
  VPS_CUDA_LAST("split_f16_planes");
  split_f16_planes_kernel<<<blocks, 256, 0, st>>>((const float*)f2->ptr, npix, f1->c, f2->cs, base + 2 * plane, base + 3 * plane, flag);
  VPS_CUDA_LAST("split_f16_planes");
  const float s1 = 1.0f / (float)f1->c, s2 = s1 * (1.0f / 2048.0f);
  int rc;
#define CORR_PASS(A, B, SC, ACC, ACT)                                                                        \
  rc = (R == 10) ? launch<10, 2>(&t[A], &t[B], out, ACT, slope, st, SC, ACC, 1) : launch<4, 1>(&t[A], &t[B], out, ACT, slope, st, SC, ACC, 1); \
  if (rc != VPS_OK) return rc;
  CORR_PASS(0, 2, s1, 0, VPS_ACT_NONE)      // f1.hi x f2.hi
  CORR_PASS(0, 3, s2, 1, VPS_ACT_NONE)      // f1.hi x f2.lo
  CORR_PASS(1, 2, s2, 1, act)               // f1.lo x f2.hi, then the activation
#undef CORR_PASS
  return VPS_OK;
}

// Tensor-core correlation; returns VPS_E_ARG (without launching) when the geometry is not one of the two supported
// call sites -- vps_correlation then uses the CUDA-core kernel.
extern "C" int vps_correlation_tc(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad, int max_disp,
                                  int stride1, int stride2, int act, float slope, void* stream) {
  VPS_CHECK_ARG(stride1 == 1 && pad == max_disp, "correlation_tc: only stride1=1, pad==max_displacement");
  VPS_CHECK_ARG(f1->dtype == VPS_BF16 && f2->dtype == VPS_BF16, "correlation_tc: bf16 features only");
  VPS_CHECK_ARG(f1->h == f2->h && f1->w == f2->w && f1->c == f2->c && f1->n == f2->n && out->h == f1->h && out->w == f1->w,
                "correlation_tc: shape mismatch");
  VPS_CHECK_ARG(f1->c % KC == 0 && f1->c <= KC * MAX_KCH, "correlation_tc: C must be a multiple of 64, <= 256");
  VPS_CHECK_ARG(f1->cs % 8 == 0 && f2->cs % 8 == 0 && ((uintptr_t)f1->ptr & 15) == 0 && ((uintptr_t)f2->ptr & 15) == 0,
                "correlation_tc: features must be 16-byte aligned");
  VPS_CHECK_ARG(act == VPS_ACT_NONE || act == VPS_ACT_LRELU, "correlation_tc: act");
  const int R = max_disp / stride2, D = 2 * R + 1;
  VPS_CHECK_ARG(out->c == D * D, "correlation_tc: out.c %d != %d", out->c, D * D);
  cudaStream_t st = (cudaStream_t)stream;
  if (R == 10 && stride2 == 2) return launch<10, 2>(f1, f2, out, act, slope, st);
  if (R == 4 && stride2 == 1) return launch<4, 1>(f1, f2, out, act, slope, st);
  vps::set_error("correlation_tc: unsupported (max_disp %d, stride2 %d)", max_disp, stride2);
  return VPS_E_ARG;
}
