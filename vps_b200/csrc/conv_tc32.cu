// fp32-parity convolution on tcgen05 tensor cores (sm_100a): the "tc32" precision.
//
// The reference computes every convolution in fp32 (cuDNN, e.g. resnet.py:506-517, flownet2.py:133-198) and
// north_star asks for label maps / track ids bit-exact and logits within 1e-3 of it -- which a single bf16 pass
// (8 significant bits per operand) cannot give.  This kernel keeps activations and results fp32 in HBM and feeds the
// tensor cores three fp16 products per K slab that together carry ~23 significant bits of every operand:
//
//     a = A + 2^-11 * A2,   A = fp16(a) (round to nearest),  A2 = fp16(2^11 * (a - A))      [b = B + 2^-11 * B2 likewise]
//     a*b ~= A*B  +  2^-11 * (A2*B + A*B2)                      (all kind::f16, f16 x f16, fp32 accumulate)
//
// a - A is exact in fp32 and at most half an fp16 ulp of a, so 2^11 * (a - A) never exceeds |a| (no overflow) and stays
// a normal fp16 number whenever a is one; dropped are a_lo*b_lo <= 2^-24 |ab| and the fp16 rounding of A2 / B2 (2^-23).
// Cost: 3 tensor-core passes -- against 6 for a three-way bf16 split of the same accuracy class; a two-way bf16 split
// (bf16x3) is NOT enough: its CPU emulation through the whole FuseTrack path (tools/emulate_split.py) flips proposals /
// ids / label pixels.  fp16's narrow exponent range is harmless below (values under 2^-14 are carried by A2: the residual
// of a subnormal A is <= 2^-25, i.e. 2^-14 after scaling); values above 65504 are saturated and counted in a device
// flag the caller must check (vps_tc32_overflow) -- the result then only has fp16-saturation accuracy.
//
// tcgen05.mma adds into its fp32 accumulator with TRUNCATION towards zero (measured: tools/probe_tc_rounding.py -- a chain
// of m MMAs on same-sign data loses 0.34*m ulp, 1.3e-4 relative after 2300 MMAs; negating A gives the bit-identical
// mirrored result, i.e. sign-magnitude RZ).  A bias that compounds over ~60 stacked layers, so:
//   * the large main product accumulates in chains of only `group` K steps (2 MMAs each) on ping-pong TMEM buffers that
//     start from accumulate = 0; finished groups are promoted to per-thread register sums with round-to-nearest fp32 adds;
//   * the two correction products accumulate (un-scaled: A2*B + A*B2) for the whole tile in their own TMEM buffer and
//     are added once at the end with one fused multiply-add by 2^-11 per element.
//
// Pipeline per CTA (persistent, one 128-pixel x block_n (<= 128) tile at a time, K consumed 32 channels per step):
//   warp 0     : TMA producer: raw fp32 activation boxes {32 ch, pixels} into a staging ring; pre-split weight tiles
//                [B | B2] (vps_pack_weights_tc32) into the B ring.
//   warps 3-7  : converters: staging box -> two SWIZZLE_64B operand planes A, A2
//                (generic-proxy writes -> fence.proxy.async -> mbarrier).  In halo mode (stride 1, > 1 tap) one converted
//                (th+kh-1) x (tw+kw-1) box feeds all kh*kw taps through shifted descriptor start addresses.
//   warps 1, 2 : MMA issuers (main product / corrections): 2 + 4 tcgen05.mma.kind::f16 (M128 x N x K16) per (tap, 32-channel chunk).
//   warps 8-15 : promotion + epilogue: tcgen05.ld finished groups, RN-add into registers (setmaxnreg gives these two
//                warpgroups 200 registers), finally bias / activation / residual and the NHWC store (conv_tc.cu's epilogue).
#include <cuda_fp16.h>

#include "conv_tc_common.cuh"

namespace {

constexpr int T32_EPI_WARPS = 8;            // warps 8..15: two per TMEM lane quarter, alternating 32-column chunks
constexpr int T32_CONV_WARPS = 5;           // warps 3..7 (warp 0 = TMA, warp 1 = main-product issuer, warp 2 = correction issuer;
                                            // VPS_TC32_SPLIT=1: warp 3 issues the corrections of the odd K steps, 4 converter warps)
constexpr int T32_THREADS = 96 + 32 * (T32_EPI_WARPS + T32_CONV_WARPS);     // 512 = 4 warpgroups
// setmaxnreg: 256 * 80 + 256 * 176 = 65536.  The single-thread issue loops must not spill (every instruction of theirs is on the
// kernel's critical path: with 64 registers ptxas kept a few values in local memory); the promotion fits 176 since its
// epilogue became the TMA store (0 spill bytes in this kernel).
constexpr int T32_REGS_LOW = 80, T32_REGS_HIGH = 176;
constexpr int T32_KC = 32;                  // channels per K step: 64-byte operand rows (SWIZZLE_64B), 2 x K16
constexpr int T32_MAX_N = 128;              // TMEM: block_n <= 64: 6 main (group) + 2 correction (tile) buffers of 64 columns,
                                            //       block_n <= 128: 3 main + 1 correction buffer of 128 columns
constexpr int T32_MAX_MAIN = 8;
constexpr int T32_STAGE_SLOTS = 2;          // fp32 staging boxes (TMA -> converters)
constexpr int T32_PLANES = 2;               // operand planes: fp16(v), fp16(2^11 (v - fp16(v)))
constexpr float T32_LO_SCALE = 2048.f, T32_LO_INV = 1.f / 2048.f;
constexpr uint32_t T32_SCRATCH_BYTES = 8u * 4096u;     // TMA-store epilogue: one [32 px][32 ch] fp32 box per promotion warp

__device__ unsigned int g_tc32_overflow = 0;     // activations / weights that exceeded the fp16 range of the main product

struct Tc32Extra {
  int rows;                  // activation rows (pixels) per A item: halo_h * halo_w, or 128
  int plane_bytes;           // bytes of one operand plane of an A item (rows * 64, padded to 1024)
  int stage_bytes;           // bytes of one fp32 staging slot (rows * 128, padded to 1024)
  int b_plane_bytes;         // block_n * 64: one weight plane of one step
  int nk_last;               // K16 slabs of the last channel chunk that hold real channels
  int group;                 // K steps of the main product accumulated inside the tensor core before promotion
  int dcn;                   // 1: the operand planes are produced by the deformable-sampling warps (no activation TMA)
  int nmain, ncorr, buf_cols;   // TMEM accumulator buffers: nmain group buffers, then ncorr correction buffers, buf_cols apart
  int dbg;                      // timing experiments only (VPS_TC32_DBG): bit 0: skip A x B2, bit 1: skip A2 x B, bit 2: skip main
  int corr_split;               // 1: the correction products of even / odd K steps are issued by two warps (2 and 3)
  int sleep_ns;                 // back-off of the converter / producer waits (VPS_TC32_SLEEP, default 0 = poll)
  int split4;                   // 1 (implies corr_split; halo mode, group = 1, even nmain): the main product too is issued by two
                                //    warps (1 and 4), even / odd K steps counted over the whole CTA -> each owns the group buffers
                                //    of its parity
};

struct Dcn32Params {
  const float* x;
  const float* off;
  int x_cs, off_cs, H, W;
};
constexpr int DCN32_SETUP_BYTES = 9 * BLOCK_M * 32;      // per (tap, pixel): 4 bilinear weights + 4 element offsets
// the fused DCN kernel is bound by its sampling warps (CUDA-core issue + L1 latency: 5 warps needed ~3900 clocks per K step
// against 384 clocks of MMA time), so it runs 6 warpgroups: warps 0-2 TMA / MMA issuers, warps 3-7 and 16-23 = 13 sampling
// warps, warps 8-15 promotion + epilogue
#ifndef VPS_DCN32_THREADS
#define VPS_DCN32_THREADS 768
#endif
constexpr int DCN32_THREADS = VPS_DCN32_THREADS;
constexpr int DCN32_GATHER_WARPS = DCN32_THREADS == 768 ? 13 : 5;
constexpr int DCN32_UNITS_PER_STEP = 16;                 // 8-row x 32-channel units of one K step

struct Ring32 {
  uint32_t s_base, s_bytes;      // staging ring
  uint32_t a_base, a_bytes;      // operand-plane ring (T32_PLANES planes per slot)
  uint32_t b_base, b_bytes;      // weight ring (T32_PLANES planes per slot)
  uint32_t bar_base;
  __device__ __forceinline__ uint32_t sfull(int s) const { return bar_base + 8u * s; }
  __device__ __forceinline__ uint32_t sempty(int s) const { return bar_base + 8u * (MAX_STAGES + s); }
  __device__ __forceinline__ uint32_t pfull(int s) const { return bar_base + 8u * (2 * MAX_STAGES + s); }
  __device__ __forceinline__ uint32_t pempty(int s) const { return bar_base + 8u * (3 * MAX_STAGES + s); }
  __device__ __forceinline__ uint32_t bfull(int s) const { return bar_base + 8u * (4 * MAX_STAGES + s); }
  __device__ __forceinline__ uint32_t bempty(int s) const { return bar_base + 8u * (5 * MAX_STAGES + s); }
  __device__ __forceinline__ uint32_t gfull(int a) const { return bar_base + 8u * (6 * MAX_STAGES + a); }
  __device__ __forceinline__ uint32_t gempty(int a) const { return bar_base + 8u * (6 * MAX_STAGES + T32_MAX_MAIN + a); }
  __device__ __forceinline__ uint32_t cfull(int a) const { return bar_base + 8u * (6 * MAX_STAGES + 2 * T32_MAX_MAIN + a); }
  __device__ __forceinline__ uint32_t cempty(int a) const { return bar_base + 8u * (6 * MAX_STAGES + 2 * T32_MAX_MAIN + 2 + a); }
  __device__ __forceinline__ uint32_t tmem_slot() const { return bar_base + 8u * (6 * MAX_STAGES + 2 * T32_MAX_MAIN + 4); }
  __device__ __forceinline__ uint32_t issue_sync() const { return tmem_slot() + 8u; }     // steps issued by the main-product warp
};
constexpr int T32_NBAR = 6 * MAX_STAGES + 2 * T32_MAX_MAIN + 4;
constexpr int T32_BAR_BYTES = 8 * (T32_NBAR + 4);

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// K-major operand tile of 64-byte rows, SWIZZLE_64B (layout type 4): 8-row groups `sbo` bytes apart
__device__ __forceinline__ uint64_t desc_hi64(uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;
  return d;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// fp16 (round to nearest, saturating) of v; `over` collects |v| > 65504 (and NaN)
__device__ __forceinline__ float to_f16_sat(float v, unsigned short& bits, bool& over) {
  unsigned short h;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(h) : "f"(v));
  bits = h;
  over = over || !(fabsf(v) <= 65504.f);
  return __half2float(__ushort_as_half(h));
}

// operand split of two values at once: hi = packed fp16x2 of (v0, v1) (round to nearest, saturating), lo = packed fp16x2 of
// 2^11 * (v - fp16(v)).  Same values as two to_f16_sat() pairs with 10 instead of 14 instructions (the converter and the
// deformable sampler are bound by exactly this arithmetic).
__device__ __forceinline__ void split_pair_f16(float v0, float v1, uint32_t& hi, uint32_t& lo, bool& over) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(v1), "f"(v0));       // first source -> upper half
  over = over || !(fabsf(v0) <= 65504.f) || !(fabsf(v1) <= 65504.f);
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  const float r0 = (v0 - h.x) * T32_LO_SCALE, r1 = (v1 - h.y) * T32_LO_SCALE;          // exact in fp32
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
}

// debugging aid (VPS_CONV_TRACE=1): clock of event `ev` at K step `step` of CTA 0
__device__ __forceinline__ void trace_ev(const ConvTcParams& p, int ev, uint32_t step) {
  if (p.trace && blockIdx.x == 0 && step < 256u && (threadIdx.x & 31) == 0) p.trace[ev * 256 + step] = clock64();
}

// wait with back-off for roles with slack (converters, TMA producer): a failed poll sleeps instead of re-polling at once, so
// that the idle warps' polling does not queue in front of the latency-critical issuers' shared-memory / barrier operations
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
    if (ns) __nanosleep(ns);
    if (++spins > (1u << VPS_MBAR_SPIN_LOG2)) {
      if ((threadIdx.x & 31) == 0) printf("vps conv_tc32: mbarrier timeout (relaxed wait) block %d warp %d bar %u\n", blockIdx.x, threadIdx.x >> 5, bar);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- tile walk shared by the roles
struct TileCoord {
  int prob, n_idx, img, ty, tx;
};
__device__ __forceinline__ TileCoord tile_coord(const ConvTcParams& p, int tile) {
  TileCoord t;
  t.prob = tile / p.tiles_per_prob;
  const int t_in = tile - t.prob * p.tiles_per_prob;
  t.n_idx = t_in % p.n_tiles_n;
  const int m_idx = t_in / p.n_tiles_n;
  const int tiles_per_img = p.tiles_y * p.tiles_x;
  t.img = m_idx / tiles_per_img;
  const int rem = m_idx - t.img * tiles_per_img;
  t.ty = rem / p.tiles_x;
  t.tx = rem - t.ty * p.tiles_x;
  return t;
}

// ---------------------------------------------------------------- warp 0: TMA producer
__device__ __forceinline__ void producer32(const ConvTcParams& p, const Tc32Extra& e, const Ring32& rg, const CUtensorMap* tmA,
                                           const CUtensorMap* tmB) {
  const int ntaps = p.kh * p.kw, kw = p.kw;
  const bool halo = p.halo != 0;
  const uint32_t a_box_bytes = (uint32_t)p.a_box_bytes, b_bytes = (uint32_t)T32_PLANES * (uint32_t)e.b_plane_bytes;
  const int bn = p.block_n;
  int ss = 0, bs = 0;
  uint32_t sphase = 0, bphase = 0, pstep = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const TileCoord t = tile_coord(p, tile);
    const int x_base = t.tx * p.tw * p.sw - p.pw_[t.prob];
    const int y_base = t.ty * p.th * p.sh - p.ph_[t.prob];
    const int n0 = t.n_idx * bn;
    for (int cc = 0; cc < p.cin_chunks; ++cc) {
      int r = 0, s = 0;
      for (int tap = 0; tap < ntaps; ++tap) {
        if (!e.dcn && (!halo || tap == 0)) {
          mbar_wait_relaxed(rg.sempty(ss), sphase ^ 1, (uint32_t)e.sleep_ns);
          if (elect_one()) {
            mbar_expect_tx(rg.sfull(ss), a_box_bytes);
            tma_load_4d(rg.s_base + ss * rg.s_bytes, tmA, rg.sfull(ss), cc * T32_KC, halo ? x_base : x_base + s,
                        halo ? y_base : y_base + r, t.img);
          }
          if (++ss == T32_STAGE_SLOTS) { ss = 0; sphase ^= 1; }
        }
        mbar_wait_relaxed(rg.bempty(bs), bphase ^ 1, (uint32_t)e.sleep_ns);
        trace_ev(p, 0, pstep++);
        if (elect_one()) {     // both weight planes of this (tap, chunk) in one 5-D box
          mbar_expect_tx(rg.bfull(bs), b_bytes);
          tma_load_5d(rg.b_base + bs * rg.b_bytes, tmB, rg.bfull(bs), cc * T32_KC, n0, tap, t.prob, 0);
        }
        if (++bs == p.b_stages) { bs = 0; bphase ^= 1; }
        if (++s == kw) { s = 0; ++r; }
      }
    }
  }
}

// ---------------------------------------------------------------- warps 3..7: fp32 box -> the two fp16 operand planes
__device__ __forceinline__ void converter32(const ConvTcParams& p, const Tc32Extra& e, const Ring32& rg, int ctid, int nthreads) {
  const int ntaps = p.kh * p.kw;
  const int items_per_tile = p.cin_chunks * (p.halo ? 1 : ntaps);
  const int tasks = e.rows * 4;                       // 8 channels (two 16-byte fp32 chunks) per task
  int ss = 0, as = 0;
  uint32_t sphase = 0, aphase = 0;
  bool over = false;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    for (int it = 0; it < items_per_tile; ++it) {
      mbar_wait_relaxed(rg.sfull(ss), sphase, (uint32_t)e.sleep_ns);
      mbar_wait_relaxed(rg.pempty(as), aphase ^ 1, (uint32_t)e.sleep_ns);
      const uint32_t src = rg.s_base + ss * rg.s_bytes;
      const uint32_t dst = rg.a_base + as * rg.a_bytes;
      for (int task = ctid; task < tasks; task += nthreads) {
        const int r = task >> 2, j = task & 3;
        // staging rows are 128 bytes, SWIZZLE_128B (written by TMA): 16-byte chunk c of row r sits at chunk c ^ (r & 7)
        const uint32_t row_s = src + (uint32_t)r * 128u;
        const uint32_t sw = (uint32_t)(r & 7);
        float v[8];
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3])
                     : "r"(row_s + (((uint32_t)(2 * j) ^ sw) << 4)));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                     : "r"(row_s + (((uint32_t)(2 * j + 1) ^ sw) << 4)));
        uint32_t hp[4], lp[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split_pair_f16(v[2 * q], v[2 * q + 1], hp[q], lp[q], over);
        // operand planes: 64-byte rows, SWIZZLE_64B: 16-byte chunk j of row r sits at chunk j ^ ((r >> 1) & 3)
        const uint32_t off = (uint32_t)r * 64u + ((((uint32_t)j) ^ ((uint32_t)(r >> 1) & 3u)) << 4);
        const uint32_t pm = dst + off, pl = pm + (uint32_t)e.plane_bytes;
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(pm), "r"(hp[0]), "r"(hp[1]), "r"(hp[2]), "r"(hp[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(pl), "r"(lp[0]), "r"(lp[1]), "r"(lp[2]), "r"(lp[3]) : "memory");
      }
      mbar_arrive(rg.sempty(ss));                                        // staging slot may be refilled
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic-proxy writes -> tensor-core reads
      mbar_arrive(rg.pfull(as));
      if (++ss == T32_STAGE_SLOTS) { ss = 0; sphase ^= 1; }
      if (++as == p.a_stages) { as = 0; aphase ^= 1; }
    }
  }
  if (over) atomicAdd(&g_tc32_overflow, 1u);
}


// ---------------------------------------------------------------- DCNv1: warps 2..7 sample the operand planes (fused im2col)
// deformable_im2col (deform_conv_cuda_kernel.cu:189-242) for a 3x3 / stride 1 / pad 1 / dilation 1 kernel with one deformable
// group: column (tap k, channel c) of output pixel (y, x) = bilinear sample of x[c] at (y - 1 + k/3 + dy_k, x - 1 + k%3 + dx_k),
// zero outside (-1, H) x (-1, W), corner taps outside the image contribute 0.  The sampled fp32 value is split into the two
// fp16 planes straight into the operand ring -- the 9x column matrix (1.2 GB per P2 layer in fp32) never exists.  K steps run
// chunk-major / tap-minor: the nine taps of a 32-channel chunk re-read the same few KB of input from L1.
__device__ __forceinline__ void dcn_gather32(const ConvTcParams& p, const Tc32Extra& e, const Dcn32Params& d, const Ring32& rg,
                                             uint32_t setup_base, uint32_t ctr_addr, int gtid) {
  constexpr int NT = 32 * DCN32_GATHER_WARPS;
  const int H = d.H, W = d.W;
  const int lane = gtid & 31;
  const int j = lane & 3;                    // 8-channel group of the 32-channel chunk
  const int steps_per_tile = p.cin_chunks * 9;
  const uint32_t units_per_tile = (uint32_t)steps_per_tile * 16u;      // a unit = 8 rows (pixels) x 32 channels of one K step
  const uint32_t a_stages = (uint32_t)p.a_stages;
  uint32_t step_base = 0;                    // K steps of the tiles this CTA has finished
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const TileCoord t = tile_coord(p, tile);
    if (gtid == 0) asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(ctr_addr), "r"(0u) : "memory");
    // ---- sampling set-up of all (tap, pixel) pairs of this tile
    for (int item = gtid; item < 9 * BLOCK_M; item += NT) {
      const int k = item >> 7, r = item & (BLOCK_M - 1);
      const int ty_in = r / p.tw, tx_in = r - ty_in * p.tw;
      const int yo = t.ty * p.th + ty_in, xo = t.tx * p.tw + tx_in;
      float wts[4] = {0.f, 0.f, 0.f, 0.f};
      int offs[4] = {0, 0, 0, 0};
      if (yo < H && xo < W) {
        const float* op = d.off + ((int64_t)(t.img * H + yo) * W + xo) * d.off_cs;
        const float oh = __ldg(op + 2 * k), ow = __ldg(op + 2 * k + 1);
        const float h = (float)(yo - 1 + k / 3) + oh;
        const float w = (float)(xo - 1 + k % 3) + ow;
        if (h > -1.f && w > -1.f && h < (float)H && w < (float)W) {
          const int hl = (int)floorf(h), wl = (int)floorf(w);
          const int hh_ = hl + 1, wh_ = wl + 1;
          const float lh = h - (float)hl, lw = w - (float)wl;
          const float hh = 1.f - lh, hw = 1.f - lw;
          const int base = t.img * H;
          if (hl >= 0 && wl >= 0) { wts[0] = hh * hw; offs[0] = ((base + hl) * W + wl) * d.x_cs; }
          if (hl >= 0 && wh_ <= W - 1) { wts[1] = hh * lw; offs[1] = ((base + hl) * W + wh_) * d.x_cs; }
          if (hh_ <= H - 1 && wl >= 0) { wts[2] = lh * hw; offs[2] = ((base + hh_) * W + wl) * d.x_cs; }
          if (hh_ <= H - 1 && wh_ <= W - 1) { wts[3] = lh * lw; offs[3] = ((base + hh_) * W + wh_) * d.x_cs; }
        }
      }
      const uint32_t sa = setup_base + (uint32_t)item * 32u;
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(sa), "f"(wts[0]), "f"(wts[1]), "f"(wts[2]), "f"(wts[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sa + 16u), "r"(offs[0]), "r"(offs[1]), "r"(offs[2]), "r"(offs[3]) : "memory");
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
    // ---- units are claimed dynamically (any number of gather warps stays balanced; a warp may run ahead into the next
    //      K step's ring slot): unit u = (K step u / 16, rows 8 * (u % 16) ..), K steps chunk-major / tap-minor
    while (true) {
      uint32_t u = 0;
      if (lane == 0) asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(u) : "r"(ctr_addr) : "memory");
      u = __shfl_sync(0xffffffffu, u, 0);
      if (u >= units_per_tile) break;
      const uint32_t step = u >> 4, part = u & 15u;
      const uint32_t cc = step / 9u, k = step - cc * 9u;
      const uint32_t sg = step_base + step;             // K step counted over all tiles of this CTA -> ring slot and its use count
      const uint32_t use = sg / a_stages, as = sg - use * a_stages;
      mbar_wait(rg.pempty((int)as), (use & 1u) ^ 1u);
      const uint32_t dst = rg.a_base + as * rg.a_bytes;
      const int r = (int)(part * 8u) + (lane >> 2);
      const float* xc = d.x + cc * T32_KC + j * 8;
      {
        const uint32_t sa = setup_base + (uint32_t)(k * BLOCK_M + r) * 32u;
        float wq[4];
        int oq[4];
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(wq[0]), "=f"(wq[1]), "=f"(wq[2]), "=f"(wq[3]) : "r"(sa));
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(oq[0]), "=r"(oq[1]), "=r"(oq[2]), "=r"(oq[3]) : "r"(sa + 16u));
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = 0.f;
        // the reference accumulates w1*v1 + w2*v2 + w3*v3 + w4*v4 left to right (dmcn_im2col_bilinear); same order here
        float4 v0[4], v1[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {           // corners outside the image carry weight 0 (branch-free: finite inputs)
          v0[c] = __ldg(reinterpret_cast<const float4*>(xc + oq[c]));
          v1[c] = __ldg(reinterpret_cast<const float4*>(xc + oq[c]) + 1);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          acc[0] += wq[c] * v0[c].x; acc[1] += wq[c] * v0[c].y; acc[2] += wq[c] * v0[c].z; acc[3] += wq[c] * v0[c].w;
          acc[4] += wq[c] * v1[c].x; acc[5] += wq[c] * v1[c].y; acc[6] += wq[c] * v1[c].z; acc[7] += wq[c] * v1[c].w;
        }
        uint32_t hp[4], lp[4];
        bool over = false;
#pragma unroll
        for (int q = 0; q < 4; ++q) split_pair_f16(acc[2 * q], acc[2 * q + 1], hp[q], lp[q], over);
        if (over) atomicAdd(&g_tc32_overflow, 1u);
        const uint32_t off = (uint32_t)r * 64u + ((((uint32_t)j) ^ ((uint32_t)(r >> 1) & 3u)) << 4);
        const uint32_t pm = dst + off, pl = pm + (uint32_t)e.plane_bytes;
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(pm), "r"(hp[0]), "r"(hp[1]), "r"(hp[2]), "r"(hp[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(pl), "r"(lp[0]), "r"(lp[1]), "r"(lp[2]), "r"(lp[3]) : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(rg.pfull((int)as));                   // 16 warp-units complete a K step's operand planes
    }
    step_base += (uint32_t)steps_per_tile;
    asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");      // the set-up table and the unit counter are rewritten for the next tile
  }
}

// ---------------------------------------------------------------- warps 1 and 2: MMA issuers
// One thread can retire a dependent instruction only every ~5 clocks, so the instruction count of the issue loop IS the
// pipeline rate (measured with VPS_CONV_STATS: a single issuer needed ~1000 clocks per K step for 6 MMAs + 4 barrier
// operations, against 384 clocks of tensor-pipe time at N = 128).  The work is therefore split by accumulator: warp 1 issues
// the main product (2 MMAs per step, group buffers), warp 2 the two correction products (4 MMAs per step, the tile's
// correction buffer); both wait for the same operand / weight barriers and both commit to the slots' empty barriers
// (arrival count 2).  Descriptors are built from 32-bit halves inside the asm block (no 64-bit integer code in the loop).
__device__ __forceinline__ void umma_f16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "setp.ne.b32 p, %6, 0;\n"
      "mov.b64 da, {%1, %2};\n"
      "mov.b64 db, {%3, %4};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// high word of a K-major SWIZZLE_64B descriptor (64-byte rows): stride byte offset, version 1, layout type 4
__device__ __forceinline__ uint32_t desc_hi32(uint32_t sbo) { return (sbo >> 4) | (1u << 14) | (4u << 29); }

// ROLE 0: main product (stats slots [0] group-buffer wait, [1] planes, [2] weights, [4] total); ROLE 1: corrections
// (stats [3] correction-buffer wait)
// PAR (ROLE 1 only): -1 = this warp issues every K step; 0 / 1 = it issues the even / odd steps of a tile and only keeps the
// ring bookkeeping of the others.  The issue loops are bound by the latency of their dependent instructions (ncu: ~130 per
// step for the corrections at ~8 clocks each -- with EVERY tcgen05.mma removed the kernel is only 10 % faster), so the
// per-step work of the slowest role is halved by alternating steps between two warps.
template <int ROLE, bool HALO, bool STATS, int PAR = -1>
__device__ __forceinline__ void mma32(const ConvTcParams& p, const Tc32Extra& e, const Ring32& rg, uint32_t tmem_base) {
  const uint32_t idesc = (1u << 4) | ((uint32_t)(p.block_n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);   // D = f32, A = B = f16
  const int ntaps = p.kh * p.kw, kw = p.kw;
  const uint32_t row_skip = HALO ? (uint32_t)(p.halo_w - kw) * 4u : 0u;          // descriptor units (16 B) to the next halo row
  const uint32_t a_hi = desc_hi32(HALO ? (uint32_t)p.halo_w * 64u : 512u), b_hi = desc_hi32(512u);
  const uint32_t a_plane16 = (uint32_t)e.plane_bytes >> 4, b_plane16 = (uint32_t)e.b_plane_bytes >> 4;
  const uint32_t a_bytes16 = rg.a_bytes >> 4, b_bytes16 = rg.b_bytes >> 4;
  const uint32_t a_base16 = (rg.a_base & 0x3FFFF) >> 4, b_base16 = (rg.b_base & 0x3FFFF) >> 4;
  const int G = e.group, last_cc = p.cin_chunks - 1, a_stages = p.a_stages, b_stages = p.b_stages;
  const int nbuf = ROLE == 0 ? e.nmain : e.ncorr;
  const uint32_t buf0 = tmem_base + (ROLE == 0 ? 0u : (uint32_t)(e.nmain * e.buf_cols)), buf_cols = (uint32_t)e.buf_cols;
  // a split corrections warp accumulates the steps of its parity in its OWN correction buffer (index PAR; the promotion adds
  // both): two warps feeding one accumulator would make the order of its truncating additions depend on their relative timing
  int as = 0, bs = 0, tb = (ROLE == 1 && PAR > 0) ? PAR : 0;
  uint32_t aphase = 0, bphase = 0, tphase = 0;       // tphase: one parity bit per TMEM buffer of this role
  uint32_t nstep = 0;                                // K steps issued so far (all tiles)
  const uint32_t sync_addr = rg.issue_sync();      // steps issued by the main-product warp(s): [even | odd]
  long long w_t = 0, w_a = 0, w_b = 0;
  const long long t_begin = STATS ? clock64() : 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    int in_group = 0;
    uint32_t d_tmem = 0, first = 0;
    uint32_t par = 0;                                // parity of the step inside the tile
    bool tile_waited = false;
    for (int cc = 0; cc <= last_cc; ++cc) {
      const bool two = cc != last_cc || e.nk_last > 1;
      uint32_t a16 = 0;
      int sx = 0;
      bool a_waited = false;
      for (int tap = 0; tap < ntaps; ++tap, par ^= 1u) {
        const bool last_step = cc == last_cc && tap == ntaps - 1;
        // ownership: corrections by the parity of the step inside the tile (step 0 resets the tile's accumulator), the main
        // product by the parity of the CTA-wide step count (= the parity of its group buffer: nmain is even when it is split)
        const uint32_t gpar = nstep & 1u;
        const bool mine = PAR < 0 || (ROLE == 0 ? gpar == (uint32_t)PAR : par == (uint32_t)PAR);
        // the last step of the tile / last tap of the chunk THIS warp issues (the other parity owns the very last one
        // every second time); a split is only configured for tiles of >= 2 steps
        const bool my_last_step = PAR < 0 ? last_step : (last_step ? mine : (mine && cc == last_cc && tap == ntaps - 2 && ntaps >= 2) ||
                                                                             (mine && ntaps == 1 && cc == last_cc - 1));
        ++nstep;
        if (ROLE == 0 ? (in_group == 0 && mine) : (PAR < 0 ? (cc == 0 && tap == 0) : (mine && !tile_waited))) {
          // ROLE 0: a new group of the main product starts on a drained buffer with accumulate = 0
          // ROLE 1: the tile's correction buffer must have been drained by the promotion warps
          const long long t0 = STATS ? clock64() : 0;
          mbar_wait(ROLE == 0 ? rg.gempty(tb) : rg.cempty(tb), ((tphase >> tb) & 1u) ^ 1u);
          if (STATS) w_t += clock64() - t0;
          if (STATS && ROLE == 0) trace_ev(p, 1, nstep - 1u);
          d_tmem = buf0 + (uint32_t)tb * buf_cols;
          first = 0;
          tile_waited = true;
        }
        if (HALO ? (tap == 0) : true) a16 = a_base16 + (uint32_t)as * a_bytes16;
        const bool item_done = !HALO || tap == ntaps - 1;
        // last tap of this chunk issued by this warp: its commit releases the operand planes
        const bool my_item_done = !HALO ? mine : (PAR < 0 ? item_done : (item_done ? mine : (mine && tap == ntaps - 2)));
        if (mine) {
        if (ROLE == 1) {
          // the tensor pipe executes MMAs in issue order: a correction issuer that ran ahead (it never waits for a group
          // buffer) would queue several steps of its 4-MMA batches in front of the main product and stretch the latency of
          // every promoted group -- it issues step s only after the main-product warp has issued step s.  This comes BEFORE the
          // barrier waits: a warp that skips every other use of a ring slot re-visits the slot's barrier two phases later with
          // the same parity, and only the fact that the main warp (which waits on every phase) is already past this step
          // makes that wait unambiguous.
          uint32_t seen;
          const uint32_t main_ctr = sync_addr + (e.split4 ? 4u * gpar : 0u);      // split main product: one counter per parity
          do {
            asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(seen) : "r"(main_ctr) : "memory");
          } while ((int32_t)(seen - nstep) < 0);
        }
        if (HALO ? !a_waited : true) {
          const long long t0 = STATS ? clock64() : 0;
          mbar_wait(rg.pfull(as), aphase);
          if (STATS) w_a += clock64() - t0;
          a_waited = true;
        }
        {
          const long long t0 = STATS ? clock64() : 0;
          mbar_wait(rg.bfull(bs), bphase);
          if (STATS) w_b += clock64() - t0;
          if (STATS) trace_ev(p, ROLE == 0 ? 2 : 4, nstep - 1u);
        }
        tc_fence_after();
        }
        const bool close = ROLE == 0 ? (++in_group == G || last_step) : last_step;
        const uint32_t b16 = b_base16 + (uint32_t)bs * b_bytes16;
        if (mine && elect_one()) {
          if (ROLE == 0) {                 // main: A x B
            if (!(e.dbg & 4)) {
            umma_f16_lohi(d_tmem, a16, a_hi, b16, b_hi, idesc, first);
            if (two) umma_f16_lohi(d_tmem, a16 + 2, a_hi, b16 + 2, b_hi, idesc, 1u);
            }
            asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(sync_addr + (PAR == 1 ? 4u : 0u)), "r"(nstep) : "memory");
          } else {                         // corrections: A2 x B + A x B2 (scaled by 2^-11 when the buffer is added)
            if (!(e.dbg & 2)) {
            umma_f16_lohi(d_tmem, a16 + a_plane16, a_hi, b16, b_hi, idesc, first);
            if (two) umma_f16_lohi(d_tmem, a16 + a_plane16 + 2, a_hi, b16 + 2, b_hi, idesc, 1u);
            }
            if (!(e.dbg & 1)) {
            umma_f16_lohi(d_tmem, a16, a_hi, b16 + b_plane16, b_hi, idesc, 1u);
            if (two) umma_f16_lohi(d_tmem, a16 + 2, a_hi, b16 + b_plane16 + 2, b_hi, idesc, 1u);
            }
          }
          umma_commit(rg.bempty(bs));
          if (my_item_done) umma_commit(rg.pempty(as));
          if (ROLE == 0 ? close : my_last_step) umma_commit(ROLE == 0 ? rg.gfull(tb) : rg.cfull(tb));
        }
        if (mine) first = 1;
        if (STATS && mine) trace_ev(p, ROLE == 0 ? 3 : 5, nstep - 1u);
        if (close) {
          tphase ^= 1u << tb;
          if (!(ROLE == 1 && PAR >= 0) && ++tb == nbuf) tb = 0;
          in_group = 0;
        }
        if (item_done) { if (++as == a_stages) { as = 0; aphase ^= 1; } }
        if (++bs == b_stages) { bs = 0; bphase ^= 1; }
        if (HALO) {                        // next tap: one pixel (64 B = 4 units) to the right, or the start of the next halo row
          a16 += 4u;
          if (++sx == kw) { sx = 0; a16 += row_skip; }
        }
      }
    }
  }
  if (STATS && (threadIdx.x & 31) == 0) {
    long long* o = p.stats + blockIdx.x * 8;
    if (ROLE == 0) { o[0] = w_t; o[1] = w_a; o[2] = w_b; o[4] = clock64() - t_begin; }
    else o[3] = w_t;
  }
}

template <int ROLE, int PAR = -1>
__device__ __forceinline__ void mma32_dispatch(const ConvTcParams& p, const Tc32Extra& e, const Ring32& rg, uint32_t tmem_base) {
  if (p.stats) {
    if (p.halo) mma32<ROLE, true, true, PAR>(p, e, rg, tmem_base); else mma32<ROLE, false, true, PAR>(p, e, rg, tmem_base);
  } else {
    if (p.halo) mma32<ROLE, true, false, PAR>(p, e, rg, tmem_base); else mma32<ROLE, false, false, PAR>(p, e, rg, tmem_base);
  }
}

// ---------------------------------------------------------------- TMA-store epilogue of one 32-channel chunk
// The promotion leaves a lane with ONE pixel and 32 channels.  Stores from that layout cost either 32 partial-line write
// requests per instruction (256-bit stores: 4.0k clocks per 128 x 128 tile in tools/mb/mb_store.cu, and the bias / activation /
// address code in front of them made the whole epilogue 13k clocks -- ncu: the promotion warps are issue-latency bound, ~2000
// dependent instructions per tile) or a shuffle transpose that needs even more instructions.  Instead every promotion warp owns
// a 4 KB SWIZZLE_128B scratch: a lane writes its 32 finished values as eight conflict-free 16-byte stores, and one elected lane
// hands the [32 pixels][32 channels] box to the TMA, which writes full lines, clips pixels / channels outside the output
// tensor and runs asynchronously to the next chunk's arithmetic.  A warp's 32 pixels are rows q*32 .. q*32+31 of the tile =
// a bw x bh pixel box (bw = min(tw, 32)).
__device__ __forceinline__ void tma_store_4d(const void* tmap, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(tmap), "r"(src), "r"(c0),
               "r"(c1), "r"(c2), "r"(c3)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// the calling lane's earlier bulk stores have finished READING shared memory (the scratch may be rewritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// v: the lane's 32 promoted sums for channels n0 .. n0+31 of its pixel `pix` (valid = inside the output); all 32 lanes call
// PLAIN: no bias / residual / activation / scale (the DCN kernel)
template <int ACT, bool PLAIN>
__device__ __forceinline__ void epi_chunk_tma(const ConvTcParams& p, const CUtensorMap* tmY, uint32_t scratch, float (&v)[32], int lane,
                                              int64_t pix, bool valid, int n0, int nlim, int x0, int y0, int img) {
  const int nv = min(32, nlim - n0);
  if (!PLAIN) {
  if (p.bias) {
    const float4* bp = reinterpret_cast<const float4*>(p.bias + n0);   // n0 % 32 == 0, bias 16-byte aligned (host check)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (4 * j + 3 < nv) {
        const float4 b = __ldg(bp + j);
        v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (4 * j + c < nv) v[4 * j + c] += __ldg(p.bias + n0 + 4 * j + c);
      }
    }
  }
  // fp32 residual with 16-byte aligned rows (host check); channels past nlim are never stored (the TMA clips them)
  const float* rq = p.res ? (const float*)p.res + pix * p.res_cs + n0 : nullptr;
  auto add_res = [&]() {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (valid && 4 * j < nv) {
        const float4 f = *reinterpret_cast<const float4*>(rq + 4 * j);
        v[4 * j] += f.x; v[4 * j + 1] += f.y; v[4 * j + 2] += f.z; v[4 * j + 3] += f.w;
      }
    }
  };
  if (rq && !p.res_after_act) add_res();
  const float scale = p.out_scale;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float t = v[j];
    const int act = ACT < 0 ? p.act : ACT;
    if (act == VPS_ACT_RELU) t = fmaxf(t, 0.f);
    else if (act == VPS_ACT_LRELU) t = t > 0.f ? t : t * p.slope;
    else if (act == VPS_ACT_SIGMOID) t = 1.f / (1.f + __expf(-t));
    v[j] = t * scale;
  }
  if (rq && p.res_after_act) add_res();
  }
  // the previous box of this warp must have left the scratch
  if (lane == 0) tma_store_wait_read();
  __syncwarp();
  const uint32_t row = scratch + (uint32_t)lane * 128u;
  const uint32_t sw = (uint32_t)(lane & 7);
#pragma unroll
  for (int j = 0; j < 8; ++j)
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row + ((((uint32_t)j) ^ sw) << 4)), "f"(v[4 * j]), "f"(v[4 * j + 1]),
                 "f"(v[4 * j + 2]), "f"(v[4 * j + 3]) : "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  if (lane == 0) tma_store_4d(tmY, scratch, n0, x0, y0, img);
  // the TMA clips the channel axis in 16-byte units, so its tensor map ends at cout & ~3: the last cout % 4 channels are
  // stored per lane
  const int tail = p.cout & 3;
  if (!PLAIN && tail && nlim == p.cout && valid) {
    const int j0 = (nlim & ~3) - n0;
    float* yp = (float*)p.y + pix * p.y_cs + n0;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j >= j0 && j < j0 + tail) yp[j] = v[j];
  }
}

// ---------------------------------------------------------------- warps 8..15: promotion (TMEM groups -> register sums) + epilogue
// warp -> TMEM lane quarter q = warp % 4 (hardware restriction); the two warps of a quarter take alternate 32-column
// chunks, so a thread owns one output pixel and up to 2 x 32 channels of running sums.
// Fallback epilogue of one chunk for outputs the TMA cannot write (bf16 output, rows that are not 16-byte aligned): per-lane
// scalar accesses, written for small code and few registers -- no layer of the FuseTrack path takes it in the tc32 precision.
template <int ACT>
__device__ __forceinline__ void epi_chunk_scalar(const ConvTcParams& p, const float (&v)[32], int64_t pix, int n0, int nlim) {
  const int nv = min(32, nlim - n0);
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    if (j < nv) {
      float t = v[j];
      if (p.bias) t += __ldg(p.bias + n0 + j);
      float r = 0.f;
      if (p.res) {
        const int64_t ro = pix * p.res_cs + n0 + j;
        r = p.res_dtype == VPS_BF16 ? __bfloat162float(((const __nv_bfloat16*)p.res)[ro]) : ((const float*)p.res)[ro];
      }
      if (!p.res_after_act) t += r;
      const int act = ACT < 0 ? p.act : ACT;
      if (act == VPS_ACT_RELU) t = fmaxf(t, 0.f);
      else if (act == VPS_ACT_LRELU) t = t > 0.f ? t : t * p.slope;
      else if (act == VPS_ACT_SIGMOID) t = 1.f / (1.f + __expf(-t));
      t *= p.out_scale;
      if (p.res_after_act) t += r;
      const int64_t yo = pix * p.y_cs + n0 + j;
      if (p.y_dtype == VPS_BF16) ((__nv_bfloat16*)p.y)[yo] = __float2bfloat16_rn(t);
      else ((float*)p.y)[yo] = t;
    }
  }
}

struct TmY4 {
  CUtensorMap m[MAX_PROB];       // output tensor maps of the launch's problems (the stride phases of a transposed convolution)
};

template <int ACT, bool STATS, bool PLAIN = false>
__device__ __forceinline__ void promote_epilogue(const ConvTcParams& p, const Tc32Extra& e, const Ring32& rg, uint32_t tmem_base,
                                                 int warp, int lane, const TmY4* tmY, uint32_t scratch_base) {
  const int q = warp & 3, half = (warp - 8) >> 2;
  const int row = q * 32 + lane;
  const int ty_in = row / p.tw, tx_in = row - ty_in * p.tw;
  const int row_w = q * 32;                       // the warp's first tile row -> top-left pixel of its bw x bh store box
  const int ty_w = row_w / p.tw, tx_w = row_w - ty_w * p.tw;
  const int tiles_per_img = p.tiles_y * p.tiles_x;
  const int total_steps = p.cin_chunks * p.kh * p.kw;
  const int ngroups = (total_steps + e.group - 1) / e.group;
  const int bn = p.block_n;
  const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
  const int c0a = half * 32, c0b = (half + 2) * 32;          // this warp's two 32-column chunks
  const bool has_a = c0a < bn, has_b = c0b < bn;
  uint32_t scratch = scratch_base + (uint32_t)(warp - 8) * 4096u;
  // Loop-invariant addresses live in registers the compiler cannot re-derive: left alone it rematerialises them from the kernel
  // parameters (shared-memory window base via S2UR, ring sizes via LDCU / UIMAD: a dozen dependent uniform-datapath
  // instructions in front of every barrier operation), and this role is bound by its dependent-instruction latency.
  uint32_t gfull0 = rg.gfull(0), lane_base_r = lane_base, buf_cols_r = (uint32_t)e.buf_cols, nmain_r = (uint32_t)e.nmain;
  asm volatile("" : "+r"(gfull0), "+r"(lane_base_r), "+r"(buf_cols_r), "+r"(nmain_r), "+r"(scratch));
  constexpr uint32_t GEMPTY_OFF = 8u * T32_MAX_MAIN;
  uint32_t gb = 0, cb = 0, pgroup = 0;
  uint32_t gphase = 0, cphase = 0;
  constexpr bool st = STATS;
  long long w_g = 0, t_store = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    float sum[2][32];
    for (int g = 0; g < ngroups; ++g) {
      const long long t0 = st ? clock64() : 0;
      const uint32_t gf = gfull0 + 8u * gb;
      mbar_wait(gf, (gphase >> gb) & 1u);
      if (st) w_g += clock64() - t0;
      if (st && warp == 8) trace_ev(p, 6, pgroup);
      tc_fence_after();
      const uint32_t t_row = lane_base_r + gb * buf_cols_r;
      // one 32-column chunk in flight at a time: with both (64 staging registers next to the 64 running sums) ptxas spills ~35
      // sums around every tcgen05.ld even at 192 registers (re-measured with the TMA epilogue); the buffer is released before
      // the last chunk's adds
      uint32_t r[32];
      if (has_a) {
        tmem_ld32(t_row + (uint32_t)c0a, r);
        tmem_ld_wait();
        if (g == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[0][j] = __uint_as_float(r[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[0][j] = __fadd_rn(sum[0][j], __uint_as_float(r[j]));
        }
      }
      if (has_b) {
        tmem_ld32(t_row + (uint32_t)c0b, r);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(gf + GEMPTY_OFF);   // one arrival per warp (256 per-thread arrivals on one mbarrier serialise)
      if (st && warp == 8) trace_ev(p, 7, pgroup++);
      if (has_b) {
        if (g == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[1][j] = __uint_as_float(r[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[1][j] = __fadd_rn(sum[1][j], __uint_as_float(r[j]));
        }
      }
      gphase ^= 1u << gb;
      if (++gb == nmain_r) gb = 0;
    }
    // ---- the tile's correction products (split corrections issuers: one buffer per issuer, both belong to this tile)
    for (int cpass = 0; cpass < (e.corr_split ? 2 : 1); ++cpass) {
    const uint32_t cf = gfull0 + 8u * (2u * T32_MAX_MAIN) + 8u * cb;       // cfull(cb); cempty(cb) = cf + 16
    mbar_wait(cf, (cphase >> cb) & 1u);
    tc_fence_after();
    {
      const uint32_t t_row = lane_base_r + (nmain_r + cb) * buf_cols_r;
      uint32_t r[32];
      if (has_a) {
        tmem_ld32(t_row + (uint32_t)c0a, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) sum[0][j] = __fmaf_rn(__uint_as_float(r[j]), T32_LO_INV, sum[0][j]);
      }
      if (has_b) {
        tmem_ld32(t_row + (uint32_t)c0b, r);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(cf + 16u);
      if (has_b) {
#pragma unroll
        for (int j = 0; j < 32; ++j) sum[1][j] = __fmaf_rn(__uint_as_float(r[j]), T32_LO_INV, sum[1][j]);
      }
    }
    cphase ^= 1u << cb;
    if (++cb == (uint32_t)e.ncorr) cb = 0;
    }
    const long long t1 = st ? clock64() : 0;
    // ---- bias / activation / residual / store of this tile
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
    const int nbase = n_idx * bn;
    const int nlim = min(p.cout, nbase + bn);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int c0 = (half + 2 * k) * 32;
      if (c0 >= bn || nbase + c0 >= nlim) continue;
      if (PLAIN || p.epi_t == 2) {                  // warp-uniform: TMA store through this warp's scratch (clips partial chunks)
        epi_chunk_tma<ACT, PLAIN>(p, &tmY->m[prob], scratch, sum[k], lane, pix, valid, nbase + c0, nlim, tx * p.tw + tx_w,
                                  ty * p.th + ty_w, img);
      } else if (valid) {
        epi_chunk_scalar<ACT>(p, sum[k], pix, nbase + c0, nlim);
      }
    }
    if (st) t_store += clock64() - t1;
  }
  if ((PLAIN || p.epi_t == 2) && lane == 0) tma_store_wait_all();      // the last boxes are in global memory before the CTA exits
  if (st && warp == 8 && lane == 0) { p.stats[blockIdx.x * 8 + 5] = w_g; p.stats[blockIdx.x * 8 + 6] = t_store; }
}

// ---------------------------------------------------------------- kernel
__global__ void __launch_bounds__(T32_THREADS, 1)
conv_igemm_tc32_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       const __grid_constant__ TmY4 tmY, const ConvTcParams p, const Tc32Extra e) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  Ring32 rg;
  rg.s_base = smem_base; rg.s_bytes = (uint32_t)e.stage_bytes;
  rg.a_base = rg.s_base + T32_STAGE_SLOTS * rg.s_bytes; rg.a_bytes = (uint32_t)T32_PLANES * (uint32_t)e.plane_bytes;
  rg.b_base = rg.a_base + (uint32_t)p.a_stages * rg.a_bytes; rg.b_bytes = (uint32_t)T32_PLANES * (uint32_t)e.b_plane_bytes;
  const uint32_t scratch_base = rg.b_base + (uint32_t)p.b_stages * rg.b_bytes;      // 8 x 4 KB epilogue scratch (epi_t == 2)
  rg.bar_base = scratch_base + (p.epi_t == 2 ? T32_SCRATCH_BYTES : 0u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 2) {
    for (int i = lane; i < T32_NBAR; i += 32) {
      uint32_t count = 1;
      if (i >= MAX_STAGES && i < 3 * MAX_STAGES) count = 32 * (e.split4 ? 3 : (e.corr_split ? 4 : 5));      // sempty, pfull: every converter thread
      if (i >= 5 * MAX_STAGES && i < 6 * MAX_STAGES) count = 2;                    // bempty: the main and ONE correction issuer
      if (i >= 3 * MAX_STAGES && i < 4 * MAX_STAGES) count = !p.halo ? 2 : (e.split4 ? 4 : (e.corr_split ? 3 : 2));      // pempty: halo planes feed all taps
      if ((i >= 6 * MAX_STAGES + T32_MAX_MAIN && i < 6 * MAX_STAGES + 2 * T32_MAX_MAIN) || i >= 6 * MAX_STAGES + 2 * T32_MAX_MAIN + 2)
        count = T32_EPI_WARPS;                                                    // gempty, cempty: one arrival per promotion warp
      mbar_init(rg.bar_base + 8u * i, count);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (p.epi_t == 2) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmY.m[0]) : "memory");
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(rg.issue_sync()), "r"(0u) : "memory");
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(rg.issue_sync() + 4u), "r"(0u) : "memory");
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(rg.issue_sync() + 8u), "r"(0u) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(rg.tmem_slot()), "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(rg.tmem_slot()) : "memory");
  // programmatic dependent launch: the prologue above overlaps the previous kernel's tail (see conv_tc.cu)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // producer / MMA / converter warpgroups give registers away, the two promotion warpgroups take them
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(T32_REGS_LOW));
    const int nissue = e.split4 ? 4 : (e.corr_split ? 3 : 2);      // issuer warps 1 .. nissue, then the converter warps
    if (warp == 0) producer32(p, e, rg, &tmA, &tmB);
    else if (warp == 1) { if (e.split4) mma32_dispatch<0, 0>(p, e, rg, tmem_base); else mma32_dispatch<0>(p, e, rg, tmem_base); }
    else if (warp == 2) { if (e.corr_split) mma32_dispatch<1, 0>(p, e, rg, tmem_base); else mma32_dispatch<1>(p, e, rg, tmem_base); }
    else if (warp == 3 && e.corr_split) mma32_dispatch<1, 1>(p, e, rg, tmem_base);
    else if (warp == 4 && e.split4) mma32_dispatch<0, 1>(p, e, rg, tmem_base);
    else converter32(p, e, rg, (int)threadIdx.x - 32 * (1 + nissue), 32 * (7 - nissue));
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(T32_REGS_HIGH));
    if (p.stats) {     // debugging aid (VPS_CONV_STATS=1): clocks of the generic path only
      promote_epilogue<-1, true>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base);
    } else {
      switch (p.act) {
        case VPS_ACT_RELU: promote_epilogue<VPS_ACT_RELU, false>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base); break;
        case VPS_ACT_LRELU: promote_epilogue<VPS_ACT_LRELU, false>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base); break;
        case VPS_ACT_SIGMOID: promote_epilogue<VPS_ACT_SIGMOID, false>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base); break;
        default: promote_epilogue<VPS_ACT_NONE, false>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base); break;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------- fused DCNv1 kernel (same pipeline, sampling warps feed the ring)
#ifndef VPS_DCN32_LOW        // setmaxnreg redistributes the CTA's OWN allocation (768 threads x 80 registers = 61440): a split
#define VPS_DCN32_LOW 48     // that needs more leaves promotion warps spinning in setmaxnreg.inc forever (measured: deadlock)
#define VPS_DCN32_HIGH 144   // 512 * 48 + 256 * 144 = 61440
#endif
constexpr int DCN32_REGS_LOW = DCN32_THREADS == 768 ? VPS_DCN32_LOW : 80;
constexpr int DCN32_REGS_HIGH = DCN32_THREADS == 768 ? VPS_DCN32_HIGH : 176;     // 512 threads: 256 * 80 + 256 * 176 = 65536
static_assert(DCN32_THREADS != 768 || 512 * DCN32_REGS_LOW + 256 * DCN32_REGS_HIGH <= 768 * 80, "setmaxnreg pool = launch allocation");
__global__ void __launch_bounds__(DCN32_THREADS, 1)
dcn_igemm_tc32_kernel(const __grid_constant__ CUtensorMap tmB, const __grid_constant__ TmY4 tmY, const ConvTcParams p,
                      const Tc32Extra e, const Dcn32Params d) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  Ring32 rg;
  rg.s_base = smem_base; rg.s_bytes = 0;
  rg.a_base = smem_base; rg.a_bytes = (uint32_t)T32_PLANES * (uint32_t)e.plane_bytes;
  rg.b_base = rg.a_base + (uint32_t)p.a_stages * rg.a_bytes; rg.b_bytes = (uint32_t)T32_PLANES * (uint32_t)e.b_plane_bytes;
  const uint32_t setup_base = rg.b_base + (uint32_t)p.b_stages * rg.b_bytes;
  const uint32_t scratch_base = setup_base + DCN32_SETUP_BYTES;
  rg.bar_base = scratch_base + (p.epi_t == 2 ? T32_SCRATCH_BYTES : 0u);
  const uint32_t ctr_addr = rg.issue_sync() + 8u;           // unit counter of the sampling warps
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 2) {
    for (int i = lane; i < T32_NBAR; i += 32) {
      uint32_t count = 1;
      if (i >= 2 * MAX_STAGES && i < 3 * MAX_STAGES) count = DCN32_UNITS_PER_STEP;      // pfull: one arrival per warp-unit
      if ((i >= 3 * MAX_STAGES && i < 4 * MAX_STAGES) || (i >= 5 * MAX_STAGES && i < 6 * MAX_STAGES)) count = 2;
      if ((i >= 6 * MAX_STAGES + T32_MAX_MAIN && i < 6 * MAX_STAGES + 2 * T32_MAX_MAIN) || i >= 6 * MAX_STAGES + 2 * T32_MAX_MAIN + 2)
        count = T32_EPI_WARPS;
      mbar_init(rg.bar_base + 8u * i, count);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(rg.issue_sync()), "r"(0u) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(rg.tmem_slot()), "r"((uint32_t)TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(rg.tmem_slot()) : "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp < 8 || warp >= 16) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(DCN32_REGS_LOW));
    if (warp == 0) producer32(p, e, rg, &tmB, &tmB);
    else if (warp == 1) mma32<0, false, false>(p, e, rg, tmem_base);
    else if (warp == 2) mma32<1, false, false>(p, e, rg, tmem_base);
    else dcn_gather32(p, e, d, rg, setup_base, ctr_addr, warp < 8 ? (int)threadIdx.x - 96 : (int)threadIdx.x - 512 + 160);
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(DCN32_REGS_HIGH));
    promote_epilogue<VPS_ACT_NONE, false, true>(p, e, rg, tmem_base, warp, lane, &tmY, scratch_base);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------- weight packing
// two planes of fp16 words, each [nprob][cout_pad][tap][cin_pad]:  B = fp16(w),  B2 = fp16(2^11 * (w - B))
__global__ void pack_weights_tc32_kernel(const float* __restrict__ src, const float* __restrict__ scale, unsigned short* __restrict__ bm,
                                         unsigned short* __restrict__ bl, int cout, int cin, int kh, int kw, int cout_pad,
                                         int cin_pad, int transposed) {
  const int64_t total = (int64_t)cout_pad * kh * kw * cin_pad;
  bool over = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % cin_pad);
    int64_t t = i / cin_pad;
    const int s = (int)(t % kw); t /= kw;
    const int r = (int)(t % kh); t /= kh;
    const int co = (int)t;
    float v = 0.f;
    if (co < cout && ci < cin) {
      const int64_t si = transposed ? ((((int64_t)ci * cout + co) * kh + r) * kw + s) : ((((int64_t)co * cin + ci) * kh + r) * kw + s);
      v = src[si];
      if (scale) v *= scale[co];
    }
    unsigned short h, l;
    const float m = to_f16_sat(v, h, over);
    bool dummy = false;
    to_f16_sat((v - m) * T32_LO_SCALE, l, dummy);
    bm[i] = h;
    bl[i] = l;
  }
  if (over) atomicAdd(&g_tc32_overflow, 1u);
}

PFN_cuTensorMapEncodeTiled_v12000 get_encode32() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}
int g_num_sms32 = 0;

inline int64_t plane_elems(int cout, int cin, int kh, int kw) {
  const int64_t cout_pad = (cout + 15) / 16 * 16, cin_pad = (cin + T32_KC - 1) / T32_KC * T32_KC;
  return cout_pad * kh * kw * cin_pad;
}

}  // namespace

extern "C" int64_t vps_packed_tc32_bytes(int cout, int cin, int kh, int kw, int nprob) {
  return plane_elems(cout, cin, kh, kw) * 2 * T32_PLANES * nprob;
}

// device address of the saturation counter (library-internal: the correlation's operand split in corr_tc.cu reports into the
// same flag)
extern "C" unsigned int* vps_tc32_overflow_flag() {
  unsigned int* p = nullptr;
  if (cudaGetSymbolAddress((void**)&p, g_tc32_overflow) != cudaSuccess) return nullptr;
  return p;
}

// number of converter / packing threads that met |value| > 65504 (or NaN) since the last reset; synchronises the device
extern "C" int vps_tc32_overflow(int reset) {
  unsigned int v = 0;
  if (cudaMemcpyFromSymbol(&v, g_tc32_overflow, sizeof(v)) != cudaSuccess) return -1;
  if (reset && v) {
    const unsigned int z = 0;
    cudaMemcpyToSymbol(g_tc32_overflow, &z, sizeof(z));
  }
  return (int)v;
}

// problem `prob` of `nprob` (the stride phases of a transposed convolution share one packed buffer; nprob = 1 otherwise)
extern "C" int vps_pack_weights_tc32(const float* w, const float* scale, void* dst, int cout, int cin, int kh, int kw,
                                     int transposed, int prob, int nprob, void* stream) {
  VPS_CHECK_ARG(nprob >= 1 && nprob <= MAX_PROB && prob >= 0 && prob < nprob, "pack_weights_tc32: prob %d of %d", prob, nprob);
  const int cout_pad = (cout + 15) / 16 * 16, cin_pad = (cin + T32_KC - 1) / T32_KC * T32_KC;
  const int64_t n = plane_elems(cout, cin, kh, kw);
  unsigned short* base = (unsigned short*)dst;
  unsigned short* bm = base + (int64_t)prob * n;
  unsigned short* bl = base + n * nprob + (int64_t)prob * n;
  const int blocks = (int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256);
  pack_weights_tc32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, scale, bm, bl, cout, cin, kh, kw, cout_pad, cin_pad, transposed);
  VPS_CUDA_LAST("pack_weights_tc32");
  return VPS_OK;
}

// fp32 activations, fp32 (or bf16) output; args[i].w = the shared buffer of vps_pack_weights_tc32(.., prob i, nprob)
extern "C" int vps_conv2d_tc32_multi(const vps_conv_args* args, int nprob, void* stream) {
  VPS_CHECK_ARG(nprob >= 1 && nprob <= MAX_PROB, "conv2d_tc32: nprob %d", nprob);
  const vps_conv_args* a = &args[0];
  VPS_CHECK_ARG(a->x.dtype == VPS_F32, "conv2d_tc32: x must be fp32");
  VPS_CHECK_ARG(a->x.cs % 4 == 0 && ((uintptr_t)a->x.ptr & 15) == 0, "conv2d_tc32: x not 16B aligned (cs=%d)", a->x.cs);
  VPS_CHECK_ARG(a->sh >= 1 && a->sh <= 2 && a->sw >= 1 && a->sw <= 2, "conv2d_tc32: stride must be 1 or 2");
  VPS_CHECK_ARG(a->cin == a->x.c, "conv2d_tc32: cin %d != x.c %d", a->cin, a->x.c);
  VPS_CHECK_ARG(((uintptr_t)a->w & 127) == 0, "conv2d_tc32: weights not aligned");
  for (int i = 0; i < nprob; ++i) {
    VPS_CHECK_ARG(args[i].w == a->w && args[i].x.ptr == a->x.ptr && args[i].y.ptr == a->y.ptr && args[i].kh == a->kh &&
                      args[i].kw == a->kw && args[i].oh == a->oh && args[i].ow == a->ow && args[i].cout == a->cout &&
                      args[i].bias == a->bias && args[i].act == a->act && args[i].oy_mul == a->oy_mul && args[i].ox_mul == a->ox_mul,
                  "conv2d_tc32_multi: problems must share geometry and the packed weight buffer");
  }
  auto encode = get_encode32();
  if (!encode) { vps::set_error("cuTensorMapEncodeTiled unavailable"); return VPS_E_CUDA; }
  if (!g_num_sms32) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms32, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms32 <= 0) { vps::set_error("no device"); return VPS_E_NODEV; }
  }
  ConvTcParams p = {};
  Tc32Extra e = {};
  p.bk = T32_KC;
  const int cin_pad = (a->cin + T32_KC - 1) / T32_KC * T32_KC;
  const int cout_pad = (a->cout + 15) / 16 * 16;
  p.n_img = a->x.n; p.oh = a->oh; p.ow = a->ow;
  const bool halo = a->sh == 1 && a->sw == 1 && a->kh * a->kw > 1 && a->kh <= 8 && a->kw <= 8;
  p.halo = halo ? 1 : 0;
  if (halo) {
    p.tw = 8; p.th = 16;
  } else {
    int best_tw = 16; int64_t best_area = -1;
    const int cands[5] = {16, 8, 32, 64, 128};
    for (int i = 0; i < 5; ++i) {
      const int tw = cands[i], th = 128 / tw;
      if (tw * a->sw > 256 || th * a->sh > 256) continue;
      const int64_t area = (int64_t)vps::cdiv(a->ow, tw) * tw * vps::cdiv(a->oh, th) * th;
      if (best_area < 0 || area < best_area) { best_area = area; best_tw = tw; }
    }
    p.tw = best_tw; p.th = 128 / best_tw;
  }
  p.halo_w = p.tw + a->kw - 1;
  const int halo_h = p.th + a->kh - 1;
  e.rows = halo ? halo_h * p.halo_w : BLOCK_M;
  p.a_box_bytes = e.rows * 128;
  e.stage_bytes = (e.rows * 128 + 1023) / 1024 * 1024;
  e.plane_bytes = (e.rows * 64 + 1023) / 1024 * 1024;
  p.a_stage_bytes = T32_PLANES * e.plane_bytes;
  p.tiles_x = vps::cdiv(a->ow, p.tw); p.tiles_y = vps::cdiv(a->oh, p.th);
  p.kh = a->kh; p.kw = a->kw; p.sh = a->sh; p.sw = a->sw;
  p.cin_chunks = cin_pad / T32_KC;
  const int rem = a->cin - (p.cin_chunks - 1) * T32_KC;
  e.nk_last = (rem + 15) / 16;
  const int ntaps = a->kh * a->kw;
  p.a_stages = halo ? 2 : 3;
  // epilogue: 2 = TMA store through per-warp scratch boxes (fp32 output with 16-byte aligned pixel rows; a residual must be
  // fp32 with aligned rows; the interleaved output pixels of a transposed-convolution phase are a strided VIEW of y, one
  // tensor map per problem), 0 = per-lane scalar stores (bf16 output, mis-aligned slices)
  {
    static int epi_env = -1;
    if (epi_env < 0) { const char* ev = getenv("VPS_TC32_EPI"); epi_env = ev ? atoi(ev) : 2; }
    const bool y_ok = a->y.dtype == VPS_F32 && (((uintptr_t)a->y.ptr & 15) == 0) && (a->y.cs % 4 == 0);
    const bool r_ok = !a->res.ptr || (a->res.dtype == VPS_F32 && (((uintptr_t)a->res.ptr & 15) == 0) && (a->res.cs % 4 == 0));
    // the TMA clips a box at the end of the channel axis only in 16-byte units (a map ending at cout % 4 != 0 wrote up to 3
    // channels past cout, into neighbouring slices of a concat buffer): the map ends at cout & ~3, epi_chunk_tma stores the rest
    p.epi_t = (y_ok && r_ok && a->y.c == a->cout && a->cout >= 4 && epi_env >= 2) ? 2 : 0;
  }
  const int a_side = T32_STAGE_SLOTS * e.stage_bytes + p.a_stages * p.a_stage_bytes;
  // N tile: divisor of cout_pad (multiple of 16, <= 128) minimising waves * (steps * step clocks + epilogue); a step is
  // 6 MMAs = 3*bn clocks at the MMA floor, ~300 clocks of issue / barrier latency, or its weight bytes at the L2 rate.
  // The TMA-store epilogue writes 32-channel boxes that are clipped only at the END of the tensor's channel axis, so it needs
  // bn % 32 == 0 or a single N tile; when cout_pad > 128 has no such divisor (cout_pad / 16 odd: cout 144, 176, 208, ...)
  // every N tile but the last would write 16 stale channels over its neighbour's, and the scalar epilogue is used instead.
  int block_n = 0, smem_budget = 0;
  for (int pass = 0; pass < 2 && block_n == 0; ++pass) {
    if (pass == 1) p.epi_t = 0;
    smem_budget = 227 * 1024 - 1024 - T32_BAR_BYTES - 64 - (p.epi_t == 2 ? (int)T32_SCRATCH_BYTES : 0);
    const int64_t m_tiles = (int64_t)a->x.n * p.tiles_y * p.tiles_x * nprob;
    double best = -1.0;
    for (int bn = 16; bn <= T32_MAX_N && bn <= cout_pad; bn += 16) {
      if (cout_pad % bn) continue;
      if (a_side + 2 * bn * 64 * T32_PLANES > smem_budget) continue;
      if (p.epi_t == 2 && (bn % 32) && bn != cout_pad) continue;
      const int64_t tiles = m_tiles * (cout_pad / bn);
      const double waves = (double)((tiles + g_num_sms32 - 1) / g_num_sms32);
      const double step = fmax(fmax(300.0, 3.0 * bn), (double)(bn * 64 * T32_PLANES) / 56.0);
      const double t = waves * ((double)(p.cin_chunks * ntaps) * step + 40.0 * bn + 1500.0);
      if (best < 0 || t < best * 0.999) { best = t; block_n = bn; }
    }
  }
  VPS_CHECK_ARG(block_n > 0, "conv2d_tc32: no N tile fits (%d x %d px halo, cout %d)", halo_h, p.halo_w, a->cout);
  p.block_n = block_n; p.n_tiles_n = cout_pad / block_n;
  e.b_plane_bytes = block_n * 64;
  {
    int bst = (smem_budget - a_side) / (T32_PLANES * e.b_plane_bytes);
    p.b_stages = bst > MAX_STAGES ? MAX_STAGES : bst;
    VPS_CHECK_ARG(p.b_stages >= 2, "conv2d_tc32: ring does not fit (%d x %d px halo, bn %d)", halo_h, p.halo_w, block_n);
  }
  static int group_env = -1;
  if (group_env < 0) { const char* ev = getenv("VPS_TC32_GROUP"); group_env = ev ? atoi(ev) : 1; }
  e.group = group_env < 1 ? 1 : group_env;
  { static int dbg_env = -1; if (dbg_env < 0) { const char* ev = getenv("VPS_TC32_DBG"); dbg_env = ev ? atoi(ev) : 0; } e.dbg = dbg_env; }
  { static int sl_env = -1; if (sl_env < 0) { const char* ev = getenv("VPS_TC32_SLEEP"); sl_env = ev ? atoi(ev) : 0; } e.sleep_ns = sl_env; }
  {
    static int split_env = -1;
    // measured neutral (fat layers 0.605 -> 0.609 ms, thin layers +2 %): the corrections issuer is not the pacing role; off
    if (split_env < 0) { const char* ev = getenv("VPS_TC32_SPLIT"); split_env = ev ? atoi(ev) : 2; }
    // four issuer warps (halo layers only: the flat layers need their five converter warps): see mma32
    e.split4 = ((split_env & 2) && halo && e.group == 1 && p.cin_chunks * ntaps >= 4) ? 1 : 0;
    e.corr_split = e.split4;
  }
  e.buf_cols = block_n <= 64 ? 64 : 128;
  // 128-column buffers: long tiles want a third group buffer (slack for the promotion latency), short tiles (1x1 layers
  // with few K steps) a second correction buffer so that the next tile can start while this one is stored
  const bool short_tile = p.cin_chunks * ntaps <= 6;
  e.nmain = block_n <= 64 ? 6 : ((short_tile || e.split4) ? 2 : 3);
  e.ncorr = block_n <= 64 ? 2 : ((short_tile || e.split4) ? 2 : 1);
  p.nprob = nprob;
  p.tiles_per_prob = p.n_img * p.tiles_y * p.tiles_x * p.n_tiles_n;
  p.total_tiles = p.tiles_per_prob * nprob;
  p.y = a->y.ptr; p.y_h = a->y.h; p.y_w = a->y.w; p.y_cs = a->y.cs; p.y_dtype = a->y.dtype;
  const int esz = a->y.dtype == VPS_BF16 ? 2 : 4;
  p.y_vec = (((uintptr_t)a->y.ptr & 15) == 0) && ((a->y.cs * esz) % 16 == 0);
  if (p.y_vec && (((uintptr_t)a->y.ptr & 31) == 0) && ((a->y.cs * esz) % 32 == 0)) p.y_vec = 2;
  p.oy_mul = a->oy_mul; p.ox_mul = a->ox_mul;
  for (int i = 0; i < MAX_PROB; ++i) {
    const vps_conv_args* q = &args[i < nprob ? i : 0];
    p.ph_[i] = q->ph; p.pw_[i] = q->pw; p.oy_off_[i] = q->oy_off; p.ox_off_[i] = q->ox_off;
    VPS_CHECK_ARG((a->oh - 1) * a->oy_mul + q->oy_off < a->y.h && (a->ow - 1) * a->ox_mul + q->ox_off < a->y.w,
                  "conv2d_tc32: output mapping out of range");
  }
  p.res = a->res.ptr; p.res_cs = a->res.cs; p.res_dtype = a->res.dtype; p.res_after_act = a->res_after_act;
  p.res_vec = a->res.ptr && (((uintptr_t)a->res.ptr & 15) == 0) && (a->res.cs % 8 == 0);
  if (p.res_vec && (((uintptr_t)a->res.ptr & 31) == 0) && (a->res.cs % 16 == 0)) p.res_vec = 2;
  VPS_CHECK_ARG(!a->bias || ((uintptr_t)a->bias & 15) == 0, "conv2d_tc32: bias must be 16-byte aligned");
  p.bias = a->bias; p.cout = a->cout; p.act = a->act; p.slope = a->slope; p.out_scale = a->out_scale;
  if (a->res.ptr) VPS_CHECK_ARG(a->res.h == a->y.h && a->res.w == a->y.w, "conv2d_tc32: residual geometry");
  static int stats_env = -1;
  static long long* stats_buf = nullptr;
  if (stats_env < 0) { const char* ev = getenv("VPS_CONV_STATS"); stats_env = ev ? atoi(ev) : 0; }
  p.stats = nullptr;
  if (p.total_tiles == 0) return VPS_OK;

  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[4] = {(cuuint64_t)a->x.c, (cuuint64_t)a->x.w, (cuuint64_t)a->x.h, (cuuint64_t)a->x.n};
    cuuint64_t strides[3] = {(cuuint64_t)a->x.cs * 4, (cuuint64_t)a->x.w * a->x.cs * 4, (cuuint64_t)a->x.h * a->x.w * a->x.cs * 4};
    cuuint32_t box[4] = {(cuuint32_t)T32_KC, (cuuint32_t)(halo ? p.halo_w : p.tw * a->sw), (cuuint32_t)(halo ? halo_h : p.th * a->sh), 1};
    cuuint32_t estr[4] = {1, (cuuint32_t)a->sw, (cuuint32_t)a->sh, 1};
    CUresult r = encode(&tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a->x.ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      vps::set_error("conv2d_tc32: encode A failed (%d) dims %d,%d,%d,%d cs %d", (int)r, a->x.c, a->x.w, a->x.h, a->x.n, a->x.cs);
      return VPS_E_CUDA;
    }
  }
  const int64_t n_plane = (int64_t)cout_pad * ntaps * cin_pad;
  {
    cuuint64_t dims[5] = {(cuuint64_t)cin_pad, (cuuint64_t)cout_pad, (cuuint64_t)ntaps, (cuuint64_t)nprob, T32_PLANES};
    cuuint64_t strides[4] = {(cuuint64_t)ntaps * cin_pad * 2, (cuuint64_t)cin_pad * 2, (cuuint64_t)n_plane * 2,
                             (cuuint64_t)n_plane * nprob * 2};
    cuuint32_t box[5] = {(cuuint32_t)T32_KC, (cuuint32_t)block_n, 1, 1, T32_PLANES};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, (void*)a->w, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { vps::set_error("conv2d_tc32: encode B failed (%d)", (int)r); return VPS_E_CUDA; }
  }
  TmY4 tmY;
  for (int i = 0; i < MAX_PROB; ++i) tmY.m[i] = tmB;      // unused unless epi_t == 2
  if (p.epi_t == 2) {
    // problem i writes output pixel (oy, ox) to y[oy * oy_mul + oy_off_i][ox * ox_mul + ox_off_i]: a [n, oh, ow, cout] view of y
    const int bw = p.tw < 32 ? p.tw : 32, bh = 32 / bw;
    for (int i = 0; i < nprob; ++i) {
      const vps_conv_args* q = &args[i];
      cuuint64_t dims[4] = {(cuuint64_t)(a->cout & ~3), (cuuint64_t)a->ow, (cuuint64_t)a->oh, (cuuint64_t)a->y.n};
      cuuint64_t strides[3] = {(cuuint64_t)a->ox_mul * a->y.cs * 4, (cuuint64_t)a->oy_mul * a->y.w * a->y.cs * 4,
                               (cuuint64_t)a->y.h * a->y.w * a->y.cs * 4};
      cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)bh, 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      void* base = (char*)a->y.ptr + ((int64_t)q->oy_off * a->y.w + q->ox_off) * a->y.cs * 4;
      CUresult r = encode(&tmY.m[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        vps::set_error("conv2d_tc32: encode Y failed (%d) dims %d,%d,%d,%d cs %d", (int)r, a->cout, a->ow, a->oh, a->y.n, a->y.cs);
        return VPS_E_CUDA;
      }
    }
  }
  const int smem = a_side + p.b_stages * T32_PLANES * e.b_plane_bytes + 1024 + T32_BAR_BYTES + (p.epi_t == 2 ? (int)T32_SCRATCH_BYTES : 0);
  static bool smem_set = false;
  if (!smem_set) {
    if (cudaFuncSetAttribute(conv_igemm_tc32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
      vps::set_error("conv2d_tc32: cannot raise dynamic smem: %s", cudaGetErrorString(cudaGetLastError()));
      return VPS_E_CUDA;
    }
    smem_set = true;
  }
  const int grid = p.total_tiles < g_num_sms32 ? p.total_tiles : g_num_sms32;
  static int trace_env = -1;
  static long long* trace_buf = nullptr;
  if (trace_env < 0) { const char* ev = getenv("VPS_CONV_TRACE"); trace_env = ev ? atoi(ev) : 0; }
  p.trace = nullptr;
  if (stats_env) {   // debugging aid: per-role barrier-wait clocks, printed after a device sync (never on in production)
    if (!stats_buf) cudaMalloc(&stats_buf, sizeof(long long) * 8 * 1024);
    cudaMemsetAsync(stats_buf, 0, sizeof(long long) * 8 * grid, (cudaStream_t)stream);
    p.stats = stats_buf;
    if (trace_env) {
      if (!trace_buf) cudaMalloc(&trace_buf, sizeof(long long) * 8 * 256);
      cudaMemsetAsync(trace_buf, 0, sizeof(long long) * 8 * 256, (cudaStream_t)stream);
      p.trace = trace_buf;
    }
  }
  static int pdl_env = -1;
  if (pdl_env < 0) { const char* ev = getenv("VPS_PDL"); pdl_env = ev ? atoi(ev) : 1; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(T32_THREADS); cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_env ? 1 : 0;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, conv_igemm_tc32_kernel, tmA, tmB, tmY, p, e);
  if (le != cudaSuccess) { vps::set_error("conv2d_tc32: launch failed: %s", cudaGetErrorString(le)); return VPS_E_CUDA; }
  VPS_CUDA_LAST("conv_igemm_tc32_kernel");
  if (stats_env) {
    static long long h[8 * 1024];
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaMemcpy(h, stats_buf, sizeof(long long) * 8 * grid, cudaMemcpyDeviceToHost);
    double m[8] = {0};
    for (int i = 0; i < grid; ++i) for (int j = 0; j < 8; ++j) m[j] += (double)h[i * 8 + j] / grid;
    const int tiles_cta = (p.total_tiles + grid - 1) / grid;
    const int steps = ntaps * p.cin_chunks;
    fprintf(stderr, "conv_tc32 stats %dx%d s%d %d->%d @%dx%d halo=%d bn=%d G=%d stages a%d b%d tiles/cta %d steps/tile %d | clk/CTA total %.0f "
            "(%.0f per step) | mma waits: group-buf %.0f planes %.0f weights %.0f corr-buf %.0f | promo: wait gfull %.0f store %.0f\n",
            a->kh, a->kw, a->sh, a->cin, a->cout, a->oh, a->ow, p.halo, block_n, e.group, p.a_stages, p.b_stages, tiles_cta, steps, m[4],
            m[4] / (tiles_cta * steps), m[0], m[1], m[2], m[3], m[5], m[6]);
    if (p.trace) {
      static long long t[8 * 256];
      cudaMemcpy(t, trace_buf, sizeof(t), cudaMemcpyDeviceToHost);
      // steady-state window: steps 40..71 of CTA 0, relative to the main issuer's MMA issue of step 40
      const long long z = t[3 * 256 + 40];
      fprintf(stderr, "trace (CTA 0, clocks relative to main issue of step 40): step | producer-B-issue | main: group-buf ok, weights ok, "
                      "issued | corr: ready, issued | promo: group seen, released\n");
      for (int sidx = 40; sidx < 72 && sidx < steps * tiles_cta; ++sidx)
        fprintf(stderr, "  %3d | %7lld | %7lld %7lld %7lld | %7lld %7lld | %7lld %7lld\n", sidx, t[0 * 256 + sidx] - z, t[1 * 256 + sidx] - z,
                t[2 * 256 + sidx] - z, t[3 * 256 + sidx] - z, t[4 * 256 + sidx] - z, t[5 * 256 + sidx] - z, t[6 * 256 + sidx] - z,
                t[7 * 256 + sidx] - z);
    }
  }
  return VPS_OK;
}

extern "C" int vps_conv2d_tc32(const vps_conv_args* a, void* stream) { return vps_conv2d_tc32_multi(a, 1, stream); }


// Fused DCNv1 3x3 / stride 1 / pad 1 / dilation 1 / 1 deformable group in the tc32 precision (deform_conv.py:15-87 forward,
// deform_conv_cuda.cpp:152-260): x fp32 NHWC (c % 32 == 0), offset fp32 NHWC [.., 18] = (dy, dx) per tap,
// w = vps_pack_weights_tc32 buffer of the [cout, cin, 3, 3] kernel, y fp32 NHWC.  No bias (DeformConv has none).
extern "C" int vps_deform_conv_tc32(const vps_tensor* x, const vps_tensor* offset, const void* w, int cout, const vps_tensor* y,
                                    void* stream) {
  VPS_CHECK_ARG(x->dtype == VPS_F32 && offset->dtype == VPS_F32 && offset->c >= 18, "deform_conv_tc32: dtypes");
  VPS_CHECK_ARG(x->c % T32_KC == 0 && x->cs % 8 == 0 && ((uintptr_t)x->ptr & 31) == 0,
                "deform_conv_tc32: x must have cin %% 32 == 0 and 32-byte aligned pixel rows (256-bit sampling loads)");
  VPS_CHECK_ARG(offset->n == x->n && offset->h == x->h && offset->w == x->w && y->n == x->n && y->h == x->h && y->w == x->w &&
                    y->c == cout, "deform_conv_tc32: shapes");
  VPS_CHECK_ARG((int64_t)x->n * x->h * x->w * x->cs < (1ll << 31), "deform_conv_tc32: tensor too large for 32-bit offsets");
  VPS_CHECK_ARG(((uintptr_t)w & 127) == 0, "deform_conv_tc32: weights not aligned");
  auto encode = get_encode32();
  if (!encode) { vps::set_error("cuTensorMapEncodeTiled unavailable"); return VPS_E_CUDA; }
  if (!g_num_sms32) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms32, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms32 <= 0) { vps::set_error("no device"); return VPS_E_NODEV; }
  }
  const int cout_pad = (cout + 15) / 16 * 16;
  ConvTcParams p = {};
  Tc32Extra e = {};
  p.bk = T32_KC; p.nprob = 1;
  p.n_img = x->n; p.oh = x->h; p.ow = x->w;
  int best_tw = 16; int64_t best_area = -1;
  const int cands[5] = {16, 8, 32, 64, 128};
  for (int i = 0; i < 5; ++i) {
    const int tw = cands[i], th = 128 / tw;
    const int64_t area = (int64_t)vps::cdiv(x->w, tw) * tw * vps::cdiv(x->h, th) * th;
    if (best_area < 0 || area < best_area) { best_area = area; best_tw = tw; }
  }
  p.tw = best_tw; p.th = 128 / best_tw;
  p.tiles_x = vps::cdiv(x->w, p.tw); p.tiles_y = vps::cdiv(x->h, p.th);
  int block_n = cout_pad;
  while (block_n > T32_MAX_N || cout_pad % block_n) block_n -= 16;
  VPS_CHECK_ARG(block_n % 32 == 0 || block_n == cout_pad, "deform_conv_tc32: cout %d has no N tile the TMA epilogue can store", cout);
  p.block_n = block_n; p.n_tiles_n = cout_pad / block_n;
  p.kh = p.kw = 3; p.sh = p.sw = 1; p.halo = 0; p.halo_w = 0;
  p.cin_chunks = x->c / T32_KC;
  e.rows = BLOCK_M; e.dcn = 1;
  e.plane_bytes = BLOCK_M * 64; e.stage_bytes = 0; e.nk_last = 2;
  e.b_plane_bytes = block_n * 64;
  e.buf_cols = block_n <= 64 ? 64 : 128;
  e.nmain = block_n <= 64 ? 6 : 3;
  e.ncorr = block_n <= 64 ? 2 : 1;
  p.a_box_bytes = 0; p.a_stage_bytes = T32_PLANES * e.plane_bytes;
  // Shared memory is kept SMALL on purpose (<= 132 KB -> the 132 KB carve-out, ~120 KB of L1 left): the sampling warps read
  // 4 x 128 B per (tap, pixel, 32-channel chunk) through L1, and the nine taps of a chunk re-read the same ~60 KB footprint of
  // the tile.  With the rings sized like the convolution kernel's (212 KB) only ~28 KB of L1 remained, every tap missed, and the
  // kernel moved ~9.7 GB through L2 per 256->256 layer at 256x512 (1.8-2.1 ms, L2-bandwidth bound whatever the number of
  // sampling warps).
  {
    static int epi_env = -1;
    if (epi_env < 0) { const char* ev = getenv("VPS_TC32_EPI"); epi_env = ev ? atoi(ev) : 2; }
    (void)epi_env;
    VPS_CHECK_ARG(y->dtype == VPS_F32 && (((uintptr_t)y->ptr & 15) == 0) && (y->cs % 4 == 0),
                  "deform_conv_tc32: y must be fp32 with 16-byte aligned pixel rows (cs=%d)", y->cs);
    VPS_CHECK_ARG(cout % 4 == 0, "deform_conv_tc32: cout %d: the TMA epilogue clips channels in 16-byte units", cout);
    p.epi_t = 2;
  }
  static int dcn_a_env = -1, dcn_b_env = -1;
  if (dcn_a_env < 0) { const char* ev = getenv("VPS_DCN32_A_STAGES"); dcn_a_env = ev ? atoi(ev) : 2; }
  if (dcn_b_env < 0) { const char* ev = getenv("VPS_DCN32_B_STAGES"); dcn_b_env = ev ? atoi(ev) : 3; }
  p.a_stages = dcn_a_env < 2 ? 2 : (dcn_a_env > 3 ? 3 : dcn_a_env);
  {
    const int budget = 227 * 1024 - 1024 - T32_BAR_BYTES - 64 - DCN32_SETUP_BYTES - p.a_stages * p.a_stage_bytes -
                       (p.epi_t == 2 ? (int)T32_SCRATCH_BYTES : 0);
    int bst = budget / (T32_PLANES * e.b_plane_bytes);
    p.b_stages = bst > MAX_STAGES ? MAX_STAGES : bst;
    if (p.b_stages > dcn_b_env && dcn_b_env >= 2) p.b_stages = dcn_b_env;
    VPS_CHECK_ARG(p.b_stages >= 2, "deform_conv_tc32: ring does not fit");
  }
  static int group_env = -1;
  if (group_env < 0) { const char* ev = getenv("VPS_TC32_GROUP"); group_env = ev ? atoi(ev) : 1; }
  e.group = group_env < 1 ? 1 : group_env;
  p.tiles_per_prob = p.n_img * p.tiles_y * p.tiles_x * p.n_tiles_n;
  p.total_tiles = p.tiles_per_prob;
  p.y = y->ptr; p.y_h = y->h; p.y_w = y->w; p.y_cs = y->cs; p.y_dtype = y->dtype;
  const int esz = y->dtype == VPS_BF16 ? 2 : 4;
  p.y_vec = (((uintptr_t)y->ptr & 15) == 0) && ((y->cs * esz) % 16 == 0);
  if (p.y_vec && (((uintptr_t)y->ptr & 31) == 0) && ((y->cs * esz) % 32 == 0)) p.y_vec = 2;
  p.oy_mul = p.ox_mul = 1;
  p.res = nullptr; p.bias = nullptr; p.cout = cout; p.act = VPS_ACT_NONE; p.slope = 0.f; p.out_scale = 1.f;
  p.stats = nullptr;
  if (p.total_tiles == 0) return VPS_OK;
  Dcn32Params d;
  d.x = (const float*)x->ptr; d.off = (const float*)offset->ptr; d.x_cs = x->cs; d.off_cs = offset->cs; d.H = x->h; d.W = x->w;
  CUtensorMap tmB;
  {
    const int64_t n_plane = (int64_t)cout_pad * 9 * x->c;
    cuuint64_t dims[5] = {(cuuint64_t)x->c, (cuuint64_t)cout_pad, 9, 1, T32_PLANES};
    cuuint64_t strides[4] = {(cuuint64_t)9 * x->c * 2, (cuuint64_t)x->c * 2, (cuuint64_t)n_plane * 2, (cuuint64_t)n_plane * 2};
    cuuint32_t box[5] = {(cuuint32_t)T32_KC, (cuuint32_t)block_n, 1, 1, T32_PLANES};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, (void*)w, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { vps::set_error("deform_conv_tc32: encode B failed (%d)", (int)r); return VPS_E_CUDA; }
  }
  TmY4 tmY;
  for (int i = 0; i < MAX_PROB; ++i) tmY.m[i] = tmB;
  {
    const int bw = p.tw < 32 ? p.tw : 32, bh = 32 / bw;
    cuuint64_t dims[4] = {(cuuint64_t)y->c, (cuuint64_t)y->w, (cuuint64_t)y->h, (cuuint64_t)y->n};
    cuuint64_t strides[3] = {(cuuint64_t)y->cs * 4, (cuuint64_t)y->w * y->cs * 4, (cuuint64_t)y->h * y->w * y->cs * 4};
    cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)bh, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = encode(&tmY.m[0], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, y->ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { vps::set_error("deform_conv_tc32: encode Y failed (%d)", (int)r); return VPS_E_CUDA; }
  }
  const int smem = p.a_stages * p.a_stage_bytes + p.b_stages * T32_PLANES * e.b_plane_bytes + DCN32_SETUP_BYTES + 1024 + T32_BAR_BYTES +
                   (p.epi_t == 2 ? (int)T32_SCRATCH_BYTES : 0);
  static bool smem_set = false;
  if (!smem_set) {
    if (cudaFuncSetAttribute(dcn_igemm_tc32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
      vps::set_error("deform_conv_tc32: cannot raise dynamic smem: %s", cudaGetErrorString(cudaGetLastError()));
      return VPS_E_CUDA;
    }
    // a hint only: the driver picks the smallest carve-out that holds the launch's dynamic shared memory
    cudaFuncSetAttribute(dcn_igemm_tc32_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, smem <= 132 * 1024 ? 58 : 100);
    (void)cudaGetLastError();
    smem_set = true;
  }
  const int grid = p.total_tiles < g_num_sms32 ? p.total_tiles : g_num_sms32;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(DCN32_THREADS); cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, dcn_igemm_tc32_kernel, tmB, tmY, p, e, d);
  if (le != cudaSuccess) { vps::set_error("deform_conv_tc32: launch failed: %s", cudaGetErrorString(le)); return VPS_E_CUDA; }
  VPS_CUDA_LAST("dcn_igemm_tc32_kernel");
  return VPS_OK;
}
