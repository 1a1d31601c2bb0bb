// Shared device code of the tcgen05 implicit-GEMM kernels (conv_tc.cu: bf16 operands; conv_tc32.cu: fp32 operands
// split on the fly into two fp16 planes, v = fp16(v) + 2^-11 fp16(2^11 (v - fp16(v)))): launch parameters, PTX wrappers (mbarrier / TMA / tcgen05),
// and the epilogue (TMEM -> bias / activation / residual -> NHWC store).
#pragma once
#include <cudaTypedefs.h>

#include "common.cuh"

namespace {

constexpr int BLOCK_M = 128;
constexpr int TMEM_COLS = 512;
constexpr int MAX_STAGES = 8;

constexpr int MAX_PROB = 4;   // stride-phase sub-convolutions of one transposed conv share a launch

struct ConvTcParams {
  int bk;                     // K elements per pipeline stage: 64 (SWIZZLE_128B rows) or 16 (SWIZZLE_32B rows)
  int nprob, tiles_per_prob;  // problems differ only in weights, padding and output pixel offset
  int ph_[MAX_PROB], pw_[MAX_PROB], oy_off_[MAX_PROB], ox_off_[MAX_PROB];
  int n_img, oh, ow;
  int th, tw, tiles_y, tiles_x;
  int n_tiles_n, block_n;
  int kh, kw, sh, sw, ph, pw;
  int cin_chunks;
  int a_stages, b_stages;     // operand rings (A: activation boxes, B: weight boxes)
  int halo;                   // 1: one (th+kh-1) x (tw+kw-1) activation box per channel chunk feeds all kh*kw taps
  int halo_w;                 // tw + kw - 1 (pixels per halo row)
  int a_stage_bytes;          // bytes of one A ring slot (multiple of 1024)
  int a_box_bytes;            // bytes one A TMA box delivers
  int rowg;                   // halo mode: 1 = one B ring slot holds the kw taps of a filter row (one barrier round per row)
  int gsub;                   // flat (non-halo) mode: K steps per ring slot (one barrier round covers gsub steps)
  int nk_last;                // K16 slabs of the last channel chunk that hold real channels (the rest is zero padding)
  int total_tiles;
  long long* stats;           // optional [grid][8] clock counters (VPS_CONV_STATS=1), else NULL
  long long* trace;           // optional [8][256] event clocks of CTA 0's first 256 K steps (VPS_CONV_TRACE=1, tc32 kernel), else NULL
  void* y;
  int y_h, y_w, y_cs, y_dtype, y_vec;
  int oy_mul, oy_off, ox_mul, ox_off;
  const void* res;
  int res_cs, res_dtype, res_after_act, res_vec;
  int epi_t;                   // tc32 kernels: coalesced (8x8-transposed) fp32 epilogue for full 32-channel chunks
  const float* bias;
  int cout;
  int act;
  float slope, out_scale;
};

#ifndef VPS_MBAR_SPIN_LOG2
#define VPS_MBAR_SPIN_LOG2 26     // debugging builds: VPS_NVCC_EXTRA=-DVPS_MBAR_SPIN_LOG2=20 python -m vps_b200.build -f
#endif
// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    ++spins;                               // a lost arrival must fail loudly, never hang the GPU box: every stuck warp reports
    if (spins == (1u << VPS_MBAR_SPIN_LOG2) && (threadIdx.x & 31) == 0)     // once, then the kernel is trapped
      printf("vps conv_tc: mbarrier timeout block %d warp %d bar %u parity %u\n", blockIdx.x, threadIdx.x >> 5, bar, parity);
    if (spins > (1u << VPS_MBAR_SPIN_LOG2) + (1u << (VPS_MBAR_SPIN_LOG2 - 2))) __trap();
  }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// true in exactly one lane of the (converged) warp -- the same lane every time for a full mask
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// K-major operand tile whose rows are bk*2 bytes: bk=64 -> 128-byte rows, SWIZZLE_128B, 8-row groups 1024 B apart;
// bk=16 -> 32-byte rows, SWIZZLE_32B, 8-row groups 256 B apart.
// sbo = byte distance between consecutive 8-row groups (8 * row bytes for a dense tile; the halo row pitch when the
// 8 rows of a group are 8 consecutive pixels of one halo row).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, int bk, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);                 // start address, bits [0,14)
  d |= (uint64_t)(sbo >> 4) << 32;                             // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                                      // descriptor version (sm_100)
  d |= (uint64_t)(bk == 64 ? 2 : 6) << 61;                     // layout type SWIZZLE_128B / SWIZZLE_32B
  return d;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]),
        "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]),
        "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]),
        "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 256-bit global accesses (sm_100: LDG.256 / STG.256): a 32-column chunk of a pixel is 2 (bf16) or 4 (fp32) of them
__device__ __forceinline__ void st_global_256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void ld_global_256(const void* p, uint32_t (&v)[8]) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]),
               "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}

// ---------------------------------------------------------------- epilogue math for one 32-column chunk of one pixel
template <int ACT>
__device__ __forceinline__ void epi_chunk(const ConvTcParams& p, const uint32_t (&r)[32], int64_t pix, int n0, int nlim) {
  const int nv = min(32, nlim - n0);      // nlim = end of this tile's channel range (N tiles may be narrower than 32)
  const bool full = nv == 32;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (p.bias) {
    if (full) {
      const float4* bp = reinterpret_cast<const float4*>(p.bias + n0);   // n0 % 32 == 0, bias 16-byte aligned (host check)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(bp + j);
        v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
      }
    } else {
      const int ng = nv >> 2;                      // float4 groups (n0 % 32 == 0 keeps them 16-byte aligned)
      const float4* bp = reinterpret_cast<const float4*>(p.bias + n0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (j < ng) {
          const float4 b = __ldg(bp + j);
          v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j >= 4 * ng && j < nv) v[j] += __ldg(p.bias + n0 + j);
    }
  }
  const bool has_res = p.res != nullptr;
  // residual added in place (no second register array); `pass` 0 = before the activation, 1 = after it
  auto add_res = [&]() {
    const int64_t ro = pix * p.res_cs + n0;
    if (p.res_dtype == VPS_BF16) {
      const __nv_bfloat16* rp = (const __nv_bfloat16*)p.res + ro;
      if (full && p.res_vec == 2) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          uint32_t raw[8];
          ld_global_256(rp + 16 * j, raw);
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw[t]));
            v[16 * j + 2 * t] += f.x; v[16 * j + 2 * t + 1] += f.y;
          }
        }
      } else if (full && p.res_vec) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 raw = *reinterpret_cast<const uint4*>(rp + 8 * j);
          const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float2 f = __bfloat1622float2(b2[t]);
            v[8 * j + 2 * t] += f.x; v[8 * j + 2 * t + 1] += f.y;
          }
        }
      } else {
        const int ng = p.res_vec ? (nv >> 3) : 0;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (g < ng) {
            const uint4 raw = *reinterpret_cast<const uint4*>(rp + 8 * g);
            const __nv_bfloat162* b2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float2 f = __bfloat1622float2(b2[t]);
              v[8 * g + 2 * t] += f.x; v[8 * g + 2 * t + 1] += f.y;
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j >= 8 * ng && j < nv) v[j] += __bfloat162float(rp[j]);
      }
    } else {
      // fp32 residual: 256-bit / 128-bit loads (a scalar load per channel touches 32 different lines per warp instruction --
      // 64 such instructions per tile cost more than the tile's MMAs: measured 17k clocks per 128x128 tile)
      const float* rp = (const float*)p.res + ro;
      if (full && p.res_vec == 2) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t raw[8];
          ld_global_256(rp + 8 * j, raw);
#pragma unroll
          for (int t = 0; t < 8; ++t) v[8 * j + t] += __uint_as_float(raw[t]);
        }
      } else if (full && p.res_vec) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 f = *reinterpret_cast<const float4*>(rp + 4 * j);
          v[4 * j] += f.x; v[4 * j + 1] += f.y; v[4 * j + 2] += f.z; v[4 * j + 3] += f.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nv) v[j] += rp[j];
      }
    }
  };
  if (has_res && !p.res_after_act) add_res();
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float t = v[j];
    const int act = ACT < 0 ? p.act : ACT;          // ACT = -1: decided at run time (instrumented debugging build only)
    if (act == VPS_ACT_RELU) t = fmaxf(t, 0.f);
    else if (act == VPS_ACT_LRELU) t = t > 0.f ? t : t * p.slope;
    else if (act == VPS_ACT_SIGMOID) t = 1.f / (1.f + __expf(-t));
    v[j] = t * p.out_scale;
  }
  if (has_res && p.res_after_act) add_res();
  const int64_t yo = pix * p.y_cs + n0;
  if (p.y_dtype == VPS_BF16) {
    __nv_bfloat16* yp = (__nv_bfloat16*)p.y + yo;
    if (p.y_vec == 2 && full) {
#pragma unroll
      for (int j = 0; j < 32; j += 16) {
        uint32_t pk[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          __nv_bfloat162 b = __floats2bfloat162_rn(v[j + 2 * t], v[j + 2 * t + 1]);
          pk[t] = *reinterpret_cast<uint32_t*>(&b);
        }
        st_global_256(yp + j, pk);
      }
    } else if (p.y_vec && full) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 pk;
        __nv_bfloat162 b0 = __floats2bfloat162_rn(v[j], v[j + 1]);
        __nv_bfloat162 b1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
        __nv_bfloat162 b2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]);
        __nv_bfloat162 b3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
        pk.x = *(uint32_t*)&b0; pk.y = *(uint32_t*)&b1; pk.z = *(uint32_t*)&b2; pk.w = *(uint32_t*)&b3;
        *(uint4*)(yp + j) = pk;
      }
    } else {
      const int ng = p.y_vec ? (nv >> 3) : 0;      // 16-byte groups of a partial chunk, then a scalar tail
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        if (g < ng) {
          const int j = 8 * g;
          uint4 pk;
          __nv_bfloat162 b0 = __floats2bfloat162_rn(v[j], v[j + 1]);
          __nv_bfloat162 b1 = __floats2bfloat162_rn(v[j + 2], v[j + 3]);
          __nv_bfloat162 b2 = __floats2bfloat162_rn(v[j + 4], v[j + 5]);
          __nv_bfloat162 b3 = __floats2bfloat162_rn(v[j + 6], v[j + 7]);
          pk.x = *(uint32_t*)&b0; pk.y = *(uint32_t*)&b1; pk.z = *(uint32_t*)&b2; pk.w = *(uint32_t*)&b3;
          *(uint4*)(yp + j) = pk;
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j >= 8 * ng && j < nv) yp[j] = __float2bfloat16_rn(v[j]);
    }
  } else {
    float* yp = (float*)p.y + yo;
    if (p.y_vec == 2 && full) {
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint32_t pk[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) pk[t] = __float_as_uint(v[j + t]);
        st_global_256(yp + j, pk);
      }
    } else if (p.y_vec && full) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) *(float4*)(yp + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
      const int ng = p.y_vec ? (nv >> 2) : 0;
#pragma unroll
      for (int g = 0; g < 8; ++g)
        if (g < ng) *(float4*)(yp + 4 * g) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j >= 4 * ng && j < nv) yp[j] = v[j];
    }
  }
}

// ---------------------------------------------------------------- epilogue role (warps 2..9)
// warp -> TMEM lane quarter q = warp % 4 (hardware restriction); the two warps of a quarter take alternate
// 32-column chunks.  Two register sets: the next chunk's tcgen05.ld is in flight while the current one is processed.
template <int ACT, int GROUPS>
__device__ __forceinline__ void epilogue_loop(const ConvTcParams& p, uint32_t tmem_base, uint32_t tfull0, uint32_t tempty0,
                                              int warp, int lane) {
  constexpr int CSTEP = 32 * GROUPS;      // the GROUPS warps of a TMEM lane quarter take alternate 32-column chunks
  const int q = warp & 3;
  const int half = (warp - 2) >> 2;
  const int row = q * 32 + lane;
  const int ty_in = row / p.tw, tx_in = row - ty_in * p.tw;
  const int tiles_per_img = p.tiles_y * p.tiles_x;
  int acc = 0;
  uint32_t acc_phase = 0;
  long long st_w = 0, st_e = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const int prob = tile / p.tiles_per_prob;
    const int t_in = tile - prob * p.tiles_per_prob;
    const int n_idx = t_in % p.n_tiles_n;
    const int m_idx = t_in / p.n_tiles_n;
    const int img = m_idx / tiles_per_img;
    const int rem = m_idx - img * tiles_per_img;
    const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
    const int oy = ty * p.th + ty_in, ox = tx * p.tw + tx_in;
    const bool valid = (oy < p.oh) && (ox < p.ow);
    const int64_t pix = ((int64_t)img * p.y_h + (oy * p.oy_mul + p.oy_off_[prob])) * p.y_w + (ox * p.ox_mul + p.ox_off_[prob]);
    const int nbase = n_idx * p.block_n;
    const int nlim = min(p.cout, nbase + p.block_n);

    const long long t0 = p.stats ? clock64() : 0;
    mbar_wait(tfull0 + 8u * acc, acc_phase);
    const long long t1 = p.stats ? clock64() : 0;
    st_w += t1 - t0;
    tc_fence_after();
    const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * 256u;
    uint32_t ra[32], rb[32];
    int c0 = half * 32;
    if (c0 < p.block_n) tmem_ld32(t_row + (uint32_t)c0, ra);
    while (c0 < p.block_n) {
      tmem_ld_wait();
      const int c1 = c0 + CSTEP;
      if (c1 < p.block_n) tmem_ld32(t_row + (uint32_t)c1, rb);
      if (valid && nbase + c0 < nlim) epi_chunk<ACT>(p, ra, pix, nbase + c0, nlim);
      if (c1 >= p.block_n) break;
      tmem_ld_wait();
      const int c2 = c1 + CSTEP;
      if (c2 < p.block_n) tmem_ld32(t_row + (uint32_t)c2, ra);
      if (valid && nbase + c1 < nlim) epi_chunk<ACT>(p, rb, pix, nbase + c1, nlim);
      c0 = c2;
    }
    tmem_ld_wait();
    tc_fence_before();
    mbar_arrive(tempty0 + 8u * acc);
    if (p.stats) st_e += clock64() - t1;
    acc ^= 1;
    if (acc == 0) acc_phase ^= 1;
  }
  if (p.stats && warp == 2 && lane == 0) { p.stats[blockIdx.x * 8 + 6] = st_w; p.stats[blockIdx.x * 8 + 7] = st_e; }
}


}  // namespace
