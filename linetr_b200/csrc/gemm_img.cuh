// Persistent tensor-core GEMM for sm_100a whose operands travel as split-bf16 "tile images".
//
//   Y = act(X W^T + b) (+ R),   X given as an activation image, Y written as fp32 rows and/or
//   as the activation image the next layer consumes.
//
// Activation image (ActImg) of a row-major activation [M, K]: two planes (bf16 hi, bf16 lo with
// x ~= hi + lo), each a sequence of 16 KB tiles [m_tile = row/128][k_block = k/64] holding
// 128 rows x 64 k in the K-major SWIZZLE_128B layout tcgen05 reads.  A tile is therefore ONE
// contiguous cp.async.bulk (TMA) transfer and needs no CUDA-core work on the consumer side.
// Weights use the same trick (TcWeight, tc_weight.cuh).
//
// The main loop is pure TMA + tcgen05:  warp 0 streams A and W tiles through an mbarrier
// ring, warp 1 issues 3 MMAs per k-step (lo*hi + hi*lo + hi*hi, fp32 accumulate in TMEM),
// warps 2-9 drain finished accumulators (tcgen05.ld), apply bias / activation / residual and
// write fp32 rows and/or the split-bf16 image of the result.  TMEM holds two accumulators so
// the epilogue of tile i overlaps the MMAs of tile i+1; CTAs are persistent (one per SM) and
// walk the tile list round-robin.
#pragma once
#include "common.cuh"
#include "linear_f32.cuh"
#include "tc_weight.cuh"
#include "act_img.cuh"
#include "ptx_sm100.cuh"

namespace ltr {

struct GemmImgArgs {
  ActImg A; int a_kb0;       // contract k-blocks [a_kb0 + nb*a_kb_nb, ... + W.K/64) of A for n-block nb
  int a_kb_nb;               // 0 for a plain GEMM; K/64 for a block-diagonal one (each n-block reads its own K slice)
  TcWeight W;
  const float* bias;
  const float* R; int ldr;   // fp32 residual (added after the activation) or nullptr
  ActImg Rimg; int r_kb0;    // OR: residual read from a split-bf16 image (hi + lo), k-block offset
  float* C; int ldc;         // fp32 output or nullptr
  ActImg O; int o_kb0;       // image output (O.hi == nullptr: none); column n -> k-block o_kb0 + n/64
  int M, act;
  // row-normalising epilogue (BN = 256 = N only, one tile spans whole rows):
  //   NORM_LAYER: y = LayerNorm(acc + bias (+ R | Rimg)) * ng + nbeta (+ nadd | NaddImg)      (models/line_attention.py:51-53,73-75)
  //   NORM_L2:    y = (acc + bias) / max(||.||_2, 1e-12)                      (models/line_transformer.py:246)
  int norm; float eps;
  const float* ng; const float* nbeta;
  const float* nadd; int ldadd;   // fp32 rows added AFTER the normalisation or nullptr
  ActImg NaddImg; int nadd_kb0;   // OR: the same addend read from a split-bf16 image
  int m_tiles, n_blks;
  unsigned long long* trace;   // debug: clock64 stamps of CTA 0 (nullptr = off)
};

enum { NORM_NONE = 0, NORM_LAYER = 1, NORM_L2 = 2 };

#define LTR_STAMP(slot) do { if (p.trace && blockIdx.x == 0) p.trace[slot] = clock64(); } while (0)

template <int BN>
struct GemmImgCfg {
  static constexpr int A_TILE = 16384;            // one plane of a 128x64 bf16 tile
  static constexpr int W_TILE = BN * 128;         // one plane of a BN x 64 bf16 tile
  static constexpr int STAGE = 2 * A_TILE + 2 * W_TILE;
  static constexpr int STAGES = BN >= 256 ? 2 : (BN >= 128 ? 3 : 4);
  static constexpr int STG_WARP = 4096;           // per epilogue warp: 32 rows x 32 fp32 (or 2 x [32 x 64 B] bf16)
  static constexpr int OFF_STG = STAGES * STAGE;
  static constexpr int OFF_BAR = OFF_STG + 8 * STG_WARP;
  static constexpr int OFF_XCH = OFF_BAR + 256;                     // row-norm partial sums [2][2][128] fp32 (BN = 256 only)
  static constexpr int XCH = BN == 256 ? 2048 : 0;
  // the dynamic window is declared __align__(1024) (no static shared memory in this kernel, so it starts
  // at the CTA's 1 KB-aligned window base); the in-kernel round-up is then a no-op and the slack below
  // is never consumed - it only keeps the carve-up valid should a toolchain ever place the window at a
  // smaller alignment (BN = 256 has 768 B left under the 227 KB CTA limit)
  static constexpr int SMEM = OFF_XCH + XCH + (BN == 256 ? 768 : 1024);
  static_assert(SMEM <= 232448, "gemm_img: shared memory budget (227 KB per CTA)");
  static constexpr int TMEM_COLS = 2 * BN;        // two accumulators
  static constexpr int THREADS = 320;             // TMA warp, MMA warp, 8 epilogue warps
};


// GELU(x) = x * Phi(x) with the erf form the reference uses (F.gelu default, models/line_attention.py:92).
// erfc(u) = P(t) exp(-u^2), t = 1 / (1 + 0.3275911 u)  (Abramowitz-Stegun 7.1.26, |error| <= 1.5e-7 - the
// size of an fp32 rounding of erf itself) costs 2 SFU ops + ~12 FMAs; erff() is ~35 instructions per value
// and made the 256 -> 1024 FFN epilogue twice as long as its main loop.  Written with erfc on both
// sides of zero so that the negative tail has no 1 - erf cancellation.
__device__ __forceinline__ float gelu_erf(float x) {
  const float u = fabsf(x) * 0.70710678118654752440f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, u, 1.f)));
  float pl = fmaf(1.061405429f, t, -1.453152027f);
  pl = fmaf(pl, t, 1.421413741f);
  pl = fmaf(pl, t, -0.284496736f);
  pl = fmaf(pl, t, 0.254829592f);
  pl *= t;
  const float g = 0.5f * x * pl * ptx::ex2_approx(u * u * -1.4426950408889634f);   // 0.5 x erfc(|x| / sqrt 2)
  return x < 0.f ? g : x - g;
}

// two values at once with packed fp32 arithmetic (mul/fma.f32x2): the same operations in the same order as gelu_erf,
// bit-identical results, ~21 instead of ~34 issue slots per pair (the 256 -> 1024 FFN tiles are epilogue-bound)
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
  const float2 u = __fmul2_rn(make_float2(fabsf(x.x), fabsf(x.y)), make_float2(0.70710678118654752440f, 0.70710678118654752440f));
  const float2 den = __ffma2_rn(make_float2(0.3275911f, 0.3275911f), u, make_float2(1.f, 1.f));
  float2 t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(den.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(den.y));
  float2 pl = __ffma2_rn(make_float2(1.061405429f, 1.061405429f), t, make_float2(-1.453152027f, -1.453152027f));
  pl = __ffma2_rn(pl, t, make_float2(1.421413741f, 1.421413741f));
  pl = __ffma2_rn(pl, t, make_float2(-0.284496736f, -0.284496736f));
  pl = __ffma2_rn(pl, t, make_float2(0.254829592f, 0.254829592f));
  pl = __fmul2_rn(pl, t);
  const float2 arg = __fmul2_rn(__fmul2_rn(u, u), make_float2(-1.4426950408889634f, -1.4426950408889634f));
  const float2 e = make_float2(ptx::ex2_approx(arg.x), ptx::ex2_approx(arg.y));
  const float2 g = __fmul2_rn(__fmul2_rn(__fmul2_rn(make_float2(0.5f, 0.5f), x), pl), e);   // 0.5 x erfc(|x| / sqrt 2)
  return make_float2(x.x < 0.f ? g.x : x.x - g.x, x.y < 0.f ? g.y : x.y - g.y);
}

// ---------------------------------------------------------------- epilogue building blocks
// One epilogue warp owns 32 accumulator rows (row0 .. row0+31, lane = row) and works on 32-column
// chunks `acc[32]` starting at global column `nbase`.  Global traffic goes through the warp's 4 KB
// staging tile so that each load/store instruction touches whole 32-byte sectors of a few rows.

// acc += X[row0 + lane][nbase .. nbase+32) for fp32 rows X (coalesced read of the 32 x 32 tile)
__device__ __forceinline__ void epi_add_rows_f32(const float* __restrict__ X, int ldx, int row0, int nbase, int M, int lane,
                                                 float* stg, float (&acc)[32]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rl = i * 4 + (lane >> 3), c4 = lane & 7;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row0 + rl < M) v = *reinterpret_cast<const float4*>(X + (long long)(row0 + rl) * ldx + nbase + c4 * 4);
    *reinterpret_cast<float4*>(&stg[rl * 32 + ((c4 ^ (rl & 7)) << 2)]) = v;
  }
  __syncwarp();
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) {
    const float4 v = *reinterpret_cast<const float4*>(&stg[lane * 32 + ((c4 ^ (lane & 7)) << 2)]);
    acc[c4 * 4] += v.x; acc[c4 * 4 + 1] += v.y; acc[c4 * 4 + 2] += v.z; acc[c4 * 4 + 3] += v.w;
  }
  __syncwarp();
}

// C[row0 + lane][nbase .. nbase+32) = acc, 256-bit stores: 4 lanes cover one 128-byte row segment
__device__ __forceinline__ void epi_store_rows_f32(float* __restrict__ C, int ldc, int row0, int nbase, int M, int lane,
                                                   float* stg, const float (&acc)[32]) {
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4)
    *reinterpret_cast<float4*>(&stg[lane * 32 + ((c4 ^ (lane & 7)) << 2)]) =
        make_float4(acc[c4 * 4], acc[c4 * 4 + 1], acc[c4 * 4 + 2], acc[c4 * 4 + 3]);
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = i * 8 + (lane >> 2), c8 = lane & 3;
    const float4 v0 = *reinterpret_cast<const float4*>(&stg[rl * 32 + (((2 * c8) ^ (rl & 7)) << 2)]);
    const float4 v1 = *reinterpret_cast<const float4*>(&stg[rl * 32 + (((2 * c8 + 1) ^ (rl & 7)) << 2)]);
    if (row0 + rl < M)
      ptx::st_global_256(C + (long long)(row0 + rl) * ldc + nbase + c8 * 8, *reinterpret_cast<const uint4*>(&v0),
                         *reinterpret_cast<const uint4*>(&v1));
  }
  __syncwarp();
}

// image O, m-tile mt, k-block kb0 + nbase/64: columns nbase .. nbase+32 of rows q*32 + lane <- split-bf16(acc)
__device__ __forceinline__ void epi_store_image(const ActImg& O, int kb0, int mt, int nbase, int q, int row0, int M, int lane,
                                                uint8_t* stgb, const float (&acc)[32]) {
  // staging: plane [32 rows][4 chunks of 16 B], chunk slot swizzled by (row>>1)&3
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    uint4 h, l;
    ptx::split8_bf16(&acc[cc * 8], h, l);
    const int slot = (lane * 4 + (cc ^ ((lane >> 1) & 3))) * 16;
    *reinterpret_cast<uint4*>(stgb + slot) = h;
    *reinterpret_cast<uint4*>(stgb + 2048 + slot) = l;
  }
  __syncwarp();
  const int kb_out = kb0 + (nbase >> 6);
  const size_t toff = ((size_t)mt * O.kblocks + kb_out) * IMG_TILE_ELEMS;
  uint8_t* ohi = reinterpret_cast<uint8_t*>(O.hi + toff);
  uint8_t* olo = reinterpret_cast<uint8_t*>(O.lo + toff);
  const int gch0 = (nbase & 63) >> 3;   // first 16-byte chunk of these 32 columns inside the 64-wide k-block
  // 256-bit stores: the 4 chunks of a row form one aligned 64-byte group of its 128-byte tile
  // line; lane pair (2 x 32 B) per row and plane, 16 rows per instruction
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int rl = i * 16 + (lane >> 1), hp = lane & 1;     // hp: which 32-byte half of the 64-byte group
    const int r_in = q * 32 + rl;
    // physical chunk index inside the group = (gch0 + cc) ^ (r_in & 7) restricted to the group's 2 low bits
    const int base_phys = (gch0 ^ (r_in & 7)) & 4;          // which 64-byte half of the 128-byte line
    uint4 vh[2], vl[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int phys = hp * 2 + e;                           // physical chunk (0..3) inside the group
      const int cc = (phys ^ (r_in & 3));                    // logical chunk stored there (low two bits of the XOR)
      const int slot = (rl * 4 + (cc ^ ((rl >> 1) & 3))) * 16;
      vh[e] = *reinterpret_cast<const uint4*>(stgb + slot);
      vl[e] = *reinterpret_cast<const uint4*>(stgb + 2048 + slot);
    }
    if (row0 + rl < M) {
      const uint32_t off = (r_in >> 3) * 1024u + (r_in & 7u) * 128u + (uint32_t)(base_phys + hp * 2) * 16u;
      ptx::st_global_256(ohi + off, vh[0], vh[1]);
      ptx::st_global_256(olo + off, vl[0], vl[1]);
    }
  }
  __syncwarp();
}

// acc += X[rows q*32 + lane of m-tile mt][columns nbase .. nbase+32) for a split-bf16 image X (k-block kb0 + nbase/64):
// coalesced 16-byte chunk loads -> staging -> own row; bf16 -> fp32 is a 16-bit shift
__device__ __forceinline__ void epi_add_rows_img(const ActImg& X, int kb0, int mt, int nbase, int q, int row0, int M, int lane,
                                                 uint8_t* stgb, float (&acc)[32]) {
  const size_t rtoff = ((size_t)mt * X.kblocks + kb0 + (nbase >> 6)) * IMG_TILE_ELEMS;
  const uint8_t* rhi = reinterpret_cast<const uint8_t*>(X.hi + rtoff);
  const uint8_t* rlo = reinterpret_cast<const uint8_t*>(X.lo + rtoff);
  const int gch0r = (nbase & 63) >> 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = i * 8 + (lane >> 2), cc = lane & 3;
    uint4 vh = make_uint4(0u, 0u, 0u, 0u), vl = vh;
    if (row0 + rl < M) {
      const uint32_t off = ptx::sw128_offset(q * 32 + rl, (gch0r + cc) * 8);
      vh = *reinterpret_cast<const uint4*>(rhi + off);
      vl = *reinterpret_cast<const uint4*>(rlo + off);
    }
    const int slot = (rl * 4 + (cc ^ ((rl >> 1) & 3))) * 16;
    *reinterpret_cast<uint4*>(stgb + slot) = vh;
    *reinterpret_cast<uint4*>(stgb + 2048 + slot) = vl;
  }
  __syncwarp();
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    const int slot = (lane * 4 + (cc ^ ((lane >> 1) & 3))) * 16;
    const uint4 vh = *reinterpret_cast<const uint4*>(stgb + slot);
    const uint4 vl = *reinterpret_cast<const uint4*>(stgb + 2048 + slot);
    const uint32_t wh[4] = {vh.x, vh.y, vh.z, vh.w}, wl[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      acc[cc * 8 + 2 * e] += __uint_as_float(wh[e] << 16) + __uint_as_float(wl[e] << 16);
      acc[cc * 8 + 2 * e + 1] += __uint_as_float(wh[e] & 0xFFFF0000u) + __uint_as_float(wl[e] & 0xFFFF0000u);
    }
  }
  __syncwarp();
}

// barrier over the 8 epilogue warps only (the TMA and MMA warps never join it)
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// Row-normalising epilogue of one 128 x 256 tile (see GemmImgArgs::norm).  A row's 256 columns sit
// in two threads (column halves, different warps); partial sums are exchanged through `xch`.
// The accumulator is re-read from TMEM for every pass (cheap) instead of being held in registers.
__device__ __forceinline__ void epi_norm_tile(const GemmImgArgs& p, uint32_t tmem_acc, int mt, int q, int half, int lane,
                                              uint32_t tl, float* stg, uint8_t* stgb, float* xch) {
  const int row0 = mt * 128 + q * 32, r_in = q * 32 + lane, cbeg = half * 128;
  auto chunk = [&](int c0, float (&v)[32]) {
    ptx::tmem_ld32(tmem_acc + (uint32_t)c0, v);
    if (p.bias) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(p.bias + c0 + j);
        v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
      }
    }
    if (p.R) epi_add_rows_f32(p.R, p.ldr, row0, c0, p.M, lane, stg, v);
    if (p.Rimg.hi) epi_add_rows_img(p.Rimg, p.r_kb0, mt, c0, q, row0, p.M, lane, stgb, v);
  };
  float mean = 0.f, scale;
  if (p.norm == NORM_LAYER) {
    float s = 0.f;
#pragma unroll 1
    for (int c0 = cbeg; c0 < cbeg + 128; c0 += 32) {
      float v[32];
      chunk(c0, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) s += v[j];
    }
    xch[half * 128 + r_in] = s;
    epi_bar();
    mean = (s + xch[(half ^ 1) * 128 + r_in]) * (1.f / 256.f);
    float ss = 0.f;
#pragma unroll 1
    for (int c0 = cbeg; c0 < cbeg + 128; c0 += 32) {
      float v[32];
      chunk(c0, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) { const float d = v[j] - mean; ss = fmaf(d, d, ss); }
    }
    xch[256 + half * 128 + r_in] = ss;
    epi_bar();
    ss += xch[256 + (half ^ 1) * 128 + r_in];
    scale = 1.f / sqrtf(ss * (1.f / 256.f) + p.eps);
  } else {
    float* x = xch + (tl & 1) * 256;   // alternate slots: one barrier per tile is enough
    float ss = 0.f;
#pragma unroll 1
    for (int c0 = cbeg; c0 < cbeg + 128; c0 += 32) {
      float v[32];
      chunk(c0, v);
#pragma unroll
      for (int j = 0; j < 32; ++j) ss = fmaf(v[j], v[j], ss);
    }
    x[half * 128 + r_in] = ss;
    epi_bar();
    ss += x[(half ^ 1) * 128 + r_in];
    scale = 1.f / fmaxf(sqrtf(ss), 1e-12f);
  }
#pragma unroll 1
  for (int c0 = cbeg; c0 < cbeg + 128; c0 += 32) {
    float v[32];
    chunk(c0, v);
    if (p.norm == NORM_LAYER) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 g = *reinterpret_cast<const float4*>(p.ng + c0 + j);
        const float4 b = *reinterpret_cast<const float4*>(p.nbeta + c0 + j);
        v[j] = (v[j] - mean) * scale * g.x + b.x;
        v[j + 1] = (v[j + 1] - mean) * scale * g.y + b.y;
        v[j + 2] = (v[j + 2] - mean) * scale * g.z + b.z;
        v[j + 3] = (v[j + 3] - mean) * scale * g.w + b.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] *= scale;
    }
    if (p.nadd) epi_add_rows_f32(p.nadd, p.ldadd, row0, c0, p.M, lane, stg, v);
    if (p.NaddImg.hi) epi_add_rows_img(p.NaddImg, p.nadd_kb0, mt, c0, q, row0, p.M, lane, stgb, v);
    if (p.C) epi_store_rows_f32(p.C, p.ldc, row0, c0, p.M, lane, stg, v);
    if (p.O.hi) epi_store_image(p.O, p.o_kb0, mt, c0, q, row0, p.M, lane, stgb, v);
  }
}

// Plain epilogue of one 128 x BN tile: this warp's 32 rows x its half of the BN columns, 32 columns at a
// time: bias -> activation -> residual (fp32 rows or split-bf16 image) -> fp32 rows and/or image output.
template <int BN>
__device__ __forceinline__ void epi_plain_tile(const GemmImgArgs& p, uint32_t tmem_acc, int mt, int nb, int q, int half, int lane,
                                               float* stg, uint8_t* stgb) {
  const int row0 = mt * 128 + q * 32;   // first row of this warp
#pragma unroll 1
  for (int c0 = half * (BN / 2); c0 < (half + 1) * (BN / 2); c0 += 32) {
    float acc[32];
    ptx::tmem_ld32(tmem_acc + (uint32_t)c0, acc);
    const int nbase = nb * BN + c0;
    if (p.bias) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const float4 b = *reinterpret_cast<const float4*>(p.bias + nbase + j);
        acc[j] += b.x; acc[j + 1] += b.y; acc[j + 2] += b.z; acc[j + 3] += b.w;
      }
    }
    // the activation is uniform per launch: branch ONCE per chunk (an if-converted erff per
    // element costs ~40 instructions even when ReLU/identity is selected)
    if (p.act == ACT_RELU) {
#pragma unroll
      for (int j = 0; j < 32; ++j) acc[j] = fmaxf(acc[j], 0.f);
    } else if (p.act == ACT_GELU) {
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const float2 g = gelu_erf2(make_float2(acc[j], acc[j + 1]));
        acc[j] = g.x; acc[j + 1] = g.y;
      }
    }
    if (p.R) epi_add_rows_f32(p.R, p.ldr, row0, nbase, p.M, lane, stg, acc);
    if (p.Rimg.hi) epi_add_rows_img(p.Rimg, p.r_kb0, mt, nbase, q, row0, p.M, lane, stgb, acc);
    if (p.C) epi_store_rows_f32(p.C, p.ldc, row0, nbase, p.M, lane, stg, acc);
    if (p.O.hi) epi_store_image(p.O, p.o_kb0, mt, nbase, q, row0, p.M, lane, stgb, acc);
  }
}

template <int BN>
__global__ void __launch_bounds__(320, 1) gemm_img_kernel(GemmImgArgs p) {
  using Cfg = GemmImgCfg<BN>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* full = bars;
  uint64_t* empty = bars + Cfg::STAGES;
  uint64_t* acc_full = bars + 2 * Cfg::STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nk = p.W.K / 64;
  const int n_tiles = p.m_tiles * p.n_blks;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&acc_full[b], 1);
      ptx::mbar_init(&acc_empty[b], 8);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // the previous kernel's outputs (A image, residual) are complete and visible from here on

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    if (lane == 0) {
      const uint8_t* whi = reinterpret_cast<const uint8_t*>(p.W.hi);
      const uint8_t* wlo = reinterpret_cast<const uint8_t*>(p.W.lo);
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int mt = tile / p.n_blks, nb = tile - mt * p.n_blks;
        for (int kb = 0; kb < nk; ++kb, ++it) {
          const int s = it % Cfg::STAGES;
          const uint32_t ph = (it / Cfg::STAGES) & 1;
          ptx::mbar_wait(&empty[s], ph ^ 1);
          if (it < 4) LTR_STAMP(it * 16 + 6);
          uint8_t* st = smem + s * Cfg::STAGE;
          const size_t aoff = ((size_t)mt * p.A.kblocks + p.a_kb0 + nb * p.a_kb_nb + kb) * IMG_TILE_ELEMS;
          const size_t woff = ((size_t)kb * (p.W.N / 8) + (size_t)nb * (BN / 8)) * 1024;
          ptx::mbar_arrive_expect_tx(&full[s], Cfg::STAGE);
          ptx::bulk_g2s(st, p.A.hi + aoff, Cfg::A_TILE, &full[s]);
          ptx::bulk_g2s(st + Cfg::A_TILE, p.A.lo + aoff, Cfg::A_TILE, &full[s]);
          ptx::bulk_g2s(st + 2 * Cfg::A_TILE, whi + woff, Cfg::W_TILE, &full[s]);
          ptx::bulk_g2s(st + 2 * Cfg::A_TILE + Cfg::W_TILE, wlo + woff, Cfg::W_TILE, &full[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, BN);
      uint32_t it = 0, tl = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
        const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
        ptx::mbar_wait(&acc_empty[buf], aph ^ 1);
        ptx::tc_fence_after();
        if (tl < 4) LTR_STAMP(tl * 16 + 0);
        const uint32_t d_tmem = tmem_base + buf * BN;
        for (int kb = 0; kb < nk; ++kb, ++it) {
          const int s = it % Cfg::STAGES;
          const uint32_t ph = (it / Cfg::STAGES) & 1;
          ptx::mbar_wait(&full[s], ph);
          ptx::tc_fence_after();
          if (tl < 4 && kb == 0) LTR_STAMP(tl * 16 + 1);
          const uint32_t a_hi = ptx::smem_u32(smem + s * Cfg::STAGE);
          const uint32_t a_lo = a_hi + Cfg::A_TILE;
          const uint32_t w_hi = a_hi + 2 * Cfg::A_TILE;
          const uint32_t w_lo = w_hi + Cfg::W_TILE;
#pragma unroll
          for (int k16 = 0; k16 < 4; ++k16) {
            const uint32_t ko = k16 * 32;
            const uint64_t dah = ptx::make_sw128_kmajor_desc(a_hi + ko, 1024);
            const uint64_t dal = ptx::make_sw128_kmajor_desc(a_lo + ko, 1024);
            const uint64_t dwh = ptx::make_sw128_kmajor_desc(w_hi + ko, 1024);
            const uint64_t dwl = ptx::make_sw128_kmajor_desc(w_lo + ko, 1024);
            ptx::umma_bf16(d_tmem, dal, dwh, idesc, (kb | k16) != 0);
            ptx::umma_bf16(d_tmem, dah, dwl, idesc, 1);
            ptx::umma_bf16(d_tmem, dah, dwh, idesc, 1);
          }
          ptx::umma_commit(&empty[s]);
        }
        ptx::umma_commit(&acc_full[buf]);
        if (tl < 4) LTR_STAMP(tl * 16 + 2);
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue (8 warps)
    // A thread owns one accumulator row (TMEM lane).  Global traffic goes through a per-warp
    // 4 KB staging tile so that every global load/store instruction of a warp touches whole
    // 32-byte sectors of a few rows instead of 16 bytes of 32 different rows.
    const int q = warp & 3;            // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;  // which half of the BN columns
    float* stg = reinterpret_cast<float*>(smem + Cfg::OFF_STG + (warp - 2) * Cfg::STG_WARP);
    uint8_t* stgb = reinterpret_cast<uint8_t*>(stg);
    uint32_t tl = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
      const int mt = tile / p.n_blks, nb = tile - mt * p.n_blks;
      const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
      ptx::mbar_wait(&acc_full[buf], aph);
      ptx::tc_fence_after();
      if (tl < 4 && warp == 2 && lane == 0) LTR_STAMP(tl * 16 + 3);
      if constexpr (BN == 256) {
        if (p.norm != NORM_NONE) {
          epi_norm_tile(p, tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN, mt, q, half, lane, tl, stg, stgb,
                        reinterpret_cast<float*>(smem + Cfg::OFF_XCH));
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
          continue;
        }
      }
      epi_plain_tile<BN>(p, tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN, mt, nb, q, half, lane, stg, stgb);
      ptx::tc_fence_before();
      __syncwarp();
      if (tl < 4 && warp == 2 && lane == 0) LTR_STAMP(tl * 16 + 5);
      if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ---------------------------------------------------------------- chained GEMMs (one launch, several row-local layers, CTA pairs)
// Layers whose inputs are row-local (every output row depends only on the same row of the previous layer's
// output) can run back to back inside ONE persistent launch: a CTA owns a 128-row m-tile and walks through
// all n-blocks of op 0, then of op 1, ... for that m-tile.  Compared with one launch per layer this removes
// the per-launch fill / drain / wave-quantisation bubbles (mlp1: 256 tiles and mlp2: 128 tiles on 148 SMs
// are 2 resp. 0.86 waves; chained, 128 CTAs do 3 + 3 tiles each) - the signature layer's
//   mlp1 (ReLU) -> mlp2 (+ residual) -> qkv of the NEXT layer (or final_proj + L2 norm)
// chain (models/line_transformer.py:157-166,176-183,245-246) is one launch instead of three.  BN = 256 only.
constexpr int CHAIN_MAX_OPS = 4;
struct GemmChainArgs {
  GemmImgArgs op[CHAIN_MAX_OPS];
  int n_ops, m_tiles;
};

// The chain runs on CTA pairs (tcgen05 cta_group::2).  With 128 x 256 tiles one SM has to pull 96 KB of operands
// (A 32 KB + W 64 KB, split-bf16) per 64-deep k-block against 12 x 128 = 1536 tensor cycles: 62.5 B/cycle/SM, more
// than the ~43 B/cycle/SM the L2 -> SM path delivers (measured: 12.7 TB/s aggregate), so a single-CTA engine
// (gemm_img_kernel) tops out near 0.65 of the tensor pipe.
// A CTA pair (cluster of 2 on one TPC) shares every W tile: each CTA loads only HALF of it (128 of the 256
// n-rows) plus its own 128-row A tile, and one tcgen05.mma.cta_group::2 of the leader CTA multiplies
// M = 256 (128 rows per CTA) x N = 256: 64 KB per SM per k-block = 41.7 B/cycle/SM.
//   barriers: full (local TMA) + peer_full (peer's stage landed, relayed by the peer's otherwise idle MMA warp
//   with a remote arrive), empty / acc_full (tcgen05.commit multicast to both CTAs), acc_empty (leader, 16
//   arrivals: the 8 epilogue warps of each CTA).
// Epilogue and op-to-op dependencies.  The trace of the first version (profiles/r2_chain_trace.md) showed the
// MMA loop at the tensor peak but only 45 % of the launch inside it: at every op boundary the next op waited
// for the WHOLE epilogue of the previous op's last tile (8-12 k cycles through per-warp staging + LDS + STG)
// plus a fence and a TMA round trip.  Now tiles with an image output are drained in k-block order (row norms
// included: their statistics passes read the accumulator from TMEM, the biased values are written back with
// tcgen05.st): all 8 epilogue warps work on the same 64-column k-block, write its hi / lo planes into one of two
// 32 KB staging tiles in the image's own swizzled layout and a dedicated STORE WARP (warp 10) stores them with two
// 16 KB bulk copies (TMA store); epilogue and store warp hand a staging tile back and forth through two mbarriers
// (tile_ready: 8 warp arrivals, tile_free: the bulk copies have read the tile), so no epilogue warp ever waits for a
// global store to complete.  The store warp also publishes every finished output k-block in the shared sequence
// counter `seq_done`; the producer of the NEXT op loads A k-block j as soon as output k-block j of the previous
// op is in memory - the next op's MMAs start while the previous tile is still being drained - and ops with a single
// n-block skip memory altogether (chain2_direct).  Only tiles with fp32-row side inputs keep the per-warp staging
// path (one hand-over per tile, four k-blocks published at once); the encoder no longer produces any.
struct GemmPairCfg {
  static constexpr int BN = 256;
  static constexpr int A_TILE = 16384;
  static constexpr int W_HALF = 16384;            // one plane of this CTA's 128 x 64 half of the W tile
  // Operand ring: FIVE 32 KB slots (hi + lo plane of one tile); k-block `it` takes slot (2 it) % 5 for its half of
  // W and (2 it + 1) % 5 for its A tile - 2.5 k-blocks in flight.  Three whole 64 KB stages left room for only one
  // staging tile, and then the hand-over of that tile (all 8 warps written -> two bulk copies issued -> copies have
  // read the tile -> warps may write again) was 45 % of the epilogue's time (ncu warp-state samples,
  // profiles/r2_chain_trace.md); the 32 KB taken from the ring pay for a second staging tile.
  static constexpr int SLOT = 2 * A_TILE;
  static constexpr int SLOTS = 5;
  static constexpr int STG_TILE = 2 * A_TILE;     // [hi 16 KB | lo 16 KB] of one 128 x 64 output k-block
  static constexpr int STG_WARP = 4096;           // staged path: per-warp 4 KB inside the staging tile
  static constexpr int OFF_STG = SLOTS * SLOT;
  static constexpr int OFF_BAR = OFF_STG + 2 * STG_TILE;
  static constexpr int OFF_XCH = OFF_BAR + 256;
  static constexpr int SMEM = OFF_XCH + 2048 + 768;
  static constexpr int TMEM_COLS = 512;
  static constexpr int THREADS = 352;             // TMA warp, MMA / relay warp, 8 epilogue warps, store warp
};
static_assert(GemmPairCfg::SMEM <= 232448, "gemm pair: shared memory budget");

// spin with a deadline: a protocol bug must end in a trap (launch failure), not in a hung GPU box.
// NB: plain `mbarrier.try_wait.parity.shared::cta` also for the phases that are completed from the peer CTA
// (multicast tcgen05.commit, remote arrives) - as CUTLASS' ClusterBarrier does.  An `.acquire.cluster` poll compiles
// to SYNCS.PHASECHK + CCTL.IVALL, i.e. EVERY poll invalidates the SM's L1: the ncu source view of the first version
// (profiles/r2_chain_trace.md) had 26 % of all stall samples on that CCTL and the epilogue's bias loads missing L1.
// Nothing a waiter reads afterwards travels through L1: accumulators come from TMEM (tcgen05.fence), operands are
// read by the tensor core / TMA through the async proxy.
__device__ __forceinline__ void mbar_wait_dl(uint64_t* bar, uint32_t parity, bool /*completed_by_peer*/) {
  if (ptx::mbar_test_wait(bar, parity)) return;
  const long long t0 = clock64();
  // test_wait (pure polling) rather than try_wait: the waiters here are single elected threads or warps with nothing else
  // to do, and the hardware-suspended form measured ~1 % slower end to end (57.1 k vs 57.7 k pairs/s)
  while (!ptx::mbar_test_wait(bar, parity))
    if (clock64() - t0 > 4000000000LL) __trap();
}

// Tiles with an image output and no fp32-row side inputs leave through the streamed epilogue (row norms included; fp32
// rows C are written straight from registers); anything else takes the per-warp staged path.
__device__ __forceinline__ bool chain2_streamed(const GemmImgArgs& p) { return p.O.hi && !p.R && !p.nadd; }
// The output tiles of a streamed op ARE the A operand tiles of the next op of the chain (same rows, same layout): the
// epilogue warps write every finished k-block ALSO into the ring slot of that A tile and arrive on its `full` barrier (one
// arrival per warp; a TMA fill arrives with count 8, so every use of a slot is one phase whoever filled it), next to
// the staging tile the store warp ships to global memory.  Through memory the next op's first MMAs waited ~4 k cycles
// for the store to complete plus ~2 k for the load (clock64 trace, profiles/r2_chain_trace.md) at every op boundary.
// (A shared -> shared bulk copy by the store warp does the same without the second set of stores, but moved 32 KB in
// ~4 k cycles - it was slower than the round trip through L2.)
// Only for ops with ONE n-block: their four output k-blocks map to ring uses at most 7 beyond the op's last one, so the
// writers wait for a slot at most one mbarrier phase ahead (the parity wait cannot tell phases two apart); the first
// n-block of a wider op would have to be handed over while the op's later n-blocks still cycle the ring.
__device__ __forceinline__ bool chain2_direct(const GemmImgArgs& p) { return chain2_streamed(p) && p.n_blks == 1; }

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(352, 1) gemm_chain2_kernel(const __grid_constant__ GemmChainArgs c) {
  using Cfg = GemmPairCfg;
  constexpr int BN = Cfg::BN;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* full = bars;                          // [5] local: this CTA's tile of the slot has landed
  uint64_t* peer_full = full + Cfg::SLOTS;        // [5] used in the leader: the peer's tile of the slot has landed
  uint64_t* empty = peer_full + Cfg::SLOTS;       // [5] local, multicast commit: the MMAs reading the slot are complete
  uint64_t* acc_full = empty + Cfg::SLOTS;        // [2] local, multicast commit
  uint64_t* acc_empty = acc_full + 2;             // [2] used in the leader, 16 arrivals
  uint64_t* tile_ready = acc_empty + 2;           // [2] local: the 8 epilogue warps filled staging tile b / finished a staged tile
  uint64_t* tile_free = tile_ready + 2;           // [2] local: the store warp's bulk copies have read staging tile b
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tile_free + 2);
  volatile uint32_t* seq_done = tmem_slot + 1;    // output k-blocks (64 columns of one m-tile) completed by this CTA's epilogue

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int n_ctiles = (c.m_tiles + 1) >> 1;      // cluster tiles: pairs of 128-row m-tiles
  const int cl0 = blockIdx.x >> 1, cl_step = gridDim.x >> 1;
  pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < Cfg::SLOTS; ++s) {
      ptx::mbar_init(&full[s], 8);   // a TMA fill arrives with count 8; a direct hand-over = one arrival per epilogue warp
      ptx::mbar_init(&peer_full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&acc_full[b], 1);
      ptx::mbar_init(&acc_empty[b], 16);
      ptx::mbar_init(&tile_ready[b], 8);
      ptx::mbar_init(&tile_free[b], 1);
    }
    *seq_done = 0;
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();          // both CTAs' barriers are initialised before any remote arrive / multicast commit
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // operand slot of ring use u (see GemmPairCfg): W half of k-block it = use 2 it, A tile = use 2 it + 1
  auto slot_of = [](uint32_t u) { return (int)(u % Cfg::SLOTS); };
  auto phase_of = [](uint32_t u) { return (u / Cfg::SLOTS) & 1u; };

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer (both CTAs: own A tile, own half of W)
    if (lane == 0) {
      // this CTA's 128 x 64 half (hi + lo plane) of W k-block kb, n-block nb of op p -> the slot of ring use u
      auto load_w = [&](const GemmImgArgs& p, int nb, int kb, uint32_t u) {
        const int sl = slot_of(u);
        mbar_wait_dl(&empty[sl], phase_of(u) ^ 1, true);
        uint8_t* st = smem + sl * Cfg::SLOT;
        const size_t woff = ((size_t)kb * (p.W.N / 8) + (size_t)nb * (BN / 8) + (size_t)rank * 16) * 1024;
        ptx::mbar_expect_tx(&full[sl], Cfg::SLOT);
        ptx::mbar_arrive_cnt(&full[sl], 8);
        ptx::bulk_g2s(st, reinterpret_cast<const uint8_t*>(p.W.hi) + woff, Cfg::W_HALF, &full[sl]);
        ptx::bulk_g2s(st + Cfg::W_HALF, reinterpret_cast<const uint8_t*>(p.W.lo) + woff, Cfg::W_HALF, &full[sl]);
      };
      // The weights do not depend on the kernel in front of this one: the first two k-blocks' W tiles are on their way
      // before griddepcontrol.wait returns.
      int pre = 0;
      if (cl0 < n_ctiles) {
        const GemmImgArgs& p0 = c.op[0];
        pre = min(2, p0.W.K / 64);
        for (int kb = 0; kb < pre; ++kb) load_w(p0, 0, kb, 2u * kb);
      }
      pdl_wait();   // A images, residuals: the previous kernel's outputs are complete and visible from here on
      LTR_DBG_STAMP(110);
      uint32_t it = 0, seq_prev = 0, seq_base = 0;   // seq_prev: sequence number of the previous op's first output k-block
      for (int ct = cl0; ct < n_ctiles; ct += cl_step) {
        const int mt = 2 * ct + (int)rank;
        for (int o = 0; o < c.n_ops; ++o) {
          const GemmImgArgs& p = c.op[o];
          const int nk = p.W.K / 64;
          for (int nb = 0; nb < p.n_blks; ++nb)
            for (int kb = 0; kb < nk; ++kb, ++it) {
              if ((int)it >= pre) load_w(p, nb, kb, 2u * it);
              // A k-block kb of this op = output k-block kb of the previous op (same m-tile, same CTA).  For the first
              // n-block the store warp copies it from the staging tile straight into this ring slot (chain2_direct) -
              // nothing to do here; later n-blocks re-read it from global memory, after the store has been published
              const bool direct = o > 0 && chain2_direct(c.op[o - 1]);
              if (direct && nb == 0) continue;
              if (o > 0 && (nb == 0 || direct)) {
                // wait until the epilogue has published it (bulk store completed / generic stores fenced)
                const uint32_t need = seq_prev + (uint32_t)kb + 1;
                if (*seq_done < need) {
                  const long long t0 = clock64();
                  while (*seq_done < need)
                    if (clock64() - t0 > 4000000000LL) __trap();
                }
                __threadfence_block();
                ptx::fence_proxy_async_all();
                if (kb == 0 && o < 8) LTR_DBG_STAMP(100 + o);
              }
              const uint32_t u = 2u * it + 1u;
              const int sl = slot_of(u);
              mbar_wait_dl(&empty[sl], phase_of(u) ^ 1, true);
              uint8_t* st = smem + sl * Cfg::SLOT;
              const size_t aoff = ((size_t)mt * p.A.kblocks + p.a_kb0 + kb) * IMG_TILE_ELEMS;
              ptx::mbar_expect_tx(&full[sl], Cfg::SLOT);
              ptx::mbar_arrive_cnt(&full[sl], 8);
              ptx::bulk_g2s(st, p.A.hi + aoff, Cfg::A_TILE, &full[sl]);
              ptx::bulk_g2s(st + Cfg::A_TILE, p.A.lo + aoff, Cfg::A_TILE, &full[sl]);
            }
          seq_prev = seq_base;
          seq_base += 4u * (uint32_t)p.n_blks;
        }
      }
    }
  } else if (warp == 1) {
    pdl_wait();
    if (lane == 0 && !leader) {
      // ---------------------------------------------------------------- peer: relay "my tile of the slot landed" to the leader
      uint32_t u = 0;
      for (int ct = cl0; ct < n_ctiles; ct += cl_step)
        for (int o = 0; o < c.n_ops; ++o) {
          const int n_use = 2 * c.op[o].n_blks * (c.op[o].W.K / 64);
          for (int i = 0; i < n_use; ++i, ++u) {
            const int sl = slot_of(u);
            mbar_wait_dl(&full[sl], phase_of(u), false);
            ptx::mbar_arrive_cluster(ptx::mapa_shared(&peer_full[sl], 0));
          }
        }
    } else if (lane == 0) {
      // ---------------------------------------------------------------- leader: MMA issuer for the pair
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(256, BN);
      uint32_t it = 0, tl = 0;
      for (int ct = cl0; ct < n_ctiles; ct += cl_step)
        for (int o = 0; o < c.n_ops; ++o) {
          const int nk = c.op[o].W.K / 64, n_blks = c.op[o].n_blks;
          for (int nb = 0; nb < n_blks; ++nb, ++tl) {
            const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
            mbar_wait_dl(&acc_empty[buf], aph ^ 1, true);
            ptx::tc_fence_after();
            if (tl < 10) LTR_DBG_STAMP(40 + tl * 4);
            const uint32_t d_tmem = tmem_base + buf * BN;
            for (int kb = 0; kb < nk; ++kb, ++it) {
              const uint32_t uw = 2u * it, ua = uw + 1u;
              const int sw = slot_of(uw), sa = slot_of(ua);
              mbar_wait_dl(&full[sw], phase_of(uw), false);
              mbar_wait_dl(&peer_full[sw], phase_of(uw), true);
              mbar_wait_dl(&full[sa], phase_of(ua), false);
              mbar_wait_dl(&peer_full[sa], phase_of(ua), true);
              ptx::tc_fence_after();
              if (tl < 10 && kb == 0) LTR_DBG_STAMP(41 + tl * 4);
              const uint32_t a_hi = ptx::smem_u32(smem + sa * Cfg::SLOT);
              const uint32_t a_lo = a_hi + Cfg::A_TILE;
              const uint32_t w_hi = ptx::smem_u32(smem + sw * Cfg::SLOT);
              const uint32_t w_lo = w_hi + Cfg::W_HALF;
#pragma unroll
              for (int k16 = 0; k16 < 4; ++k16) {
                const uint32_t ko = k16 * 32;
                const uint64_t dah = ptx::make_sw128_kmajor_desc(a_hi + ko, 1024);
                const uint64_t dal = ptx::make_sw128_kmajor_desc(a_lo + ko, 1024);
                const uint64_t dwh = ptx::make_sw128_kmajor_desc(w_hi + ko, 1024);
                const uint64_t dwl = ptx::make_sw128_kmajor_desc(w_lo + ko, 1024);
                ptx::umma2_bf16(d_tmem, dal, dwh, idesc, (kb | k16) != 0);
                ptx::umma2_bf16(d_tmem, dah, dwl, idesc, 1);
                ptx::umma2_bf16(d_tmem, dah, dwh, idesc, 1);
              }
              ptx::umma2_commit(&empty[sw], 3);
              ptx::umma2_commit(&empty[sa], 3);
            }
            ptx::umma2_commit(&acc_full[buf], 3);
            if (tl < 10) LTR_DBG_STAMP(42 + tl * 4);
          }
        }
    }
  } else if (warp == 10) {
    pdl_wait();
    // ---------------------------------------------------------------- store warp: staging tiles -> global (TMA store), publish
    if (lane == 0) {
      uint32_t hs = 0, unpub = 0;                   // hs: hand-overs so far; unpub: k-blocks stored but not yet published
      for (int ct = cl0; ct < n_ctiles; ct += cl_step) {
        const int mt = 2 * ct + (int)rank;
        // With an odd tile count the rank-1 CTA of the last cluster computes a tile past the end (mt == m_tiles): it
        // runs the whole barrier protocol (the leader's MMAs cover both CTAs' rows) but its output goes nowhere.  The
        // last op's image may be the caller's descriptor tile image, which is only 128-row padded: a store there would
        // land in the lo plane (hi) and past the end of the buffer (lo).
        const bool real_tile = mt < c.m_tiles;
        for (int o = 0; o < c.n_ops; ++o) {
          const GemmImgArgs& p = c.op[o];
          const bool streamed = chain2_streamed(p);
          for (int nb = 0; nb < p.n_blks; ++nb) {
            if (streamed) {
              for (int kbl = 0; kbl < 4; ++kbl, ++hs) {
                const uint32_t b = hs & 1, ph = (hs >> 1) & 1;
                uint8_t* tile = smem + Cfg::OFF_STG + b * Cfg::STG_TILE;
                mbar_wait_dl(&tile_ready[b], ph, false);
                const size_t toff = ((size_t)mt * p.O.kblocks + p.o_kb0 + nb * 4 + kbl) * IMG_TILE_ELEMS;
                if (real_tile) {
                  ptx::bulk_s2g(p.O.hi + toff, tile, 16384);
                  ptx::bulk_s2g(p.O.lo + toff, tile + 16384, 16384);
                }
                ptx::bulk_commit();                   // an empty group for a phantom tile keeps the wait counts below
                ++unpub;
                ptx::bulk_wait_read_all();            // the copies have read staging tile b: hand it back (the epilogue
                ptx::mbar_arrive(&tile_free[b]);      // is filling the other tile meanwhile)
                // publish what is in memory.  Waiting for THIS k-block's store here would make the store round trip
                // (~4 k cycles until the write is complete, trace) the period of the whole epilogue: let one store stay
                // in flight, except for the tile's last k-block (the next op needs it before this CTA produces anything
                // else).  Nobody inside this launch reads what the LAST op writes: its stores only have to be done
                // reading the staging tile (above) - the grid's completion makes them visible to the next kernel - so the
                // CTA does not sit out a store round trip at the end of every launch.
                if (o + 1 < c.n_ops || ct + cl_step < n_ctiles) {
                  if (kbl == 3) ptx::bulk_wait_all();
                  else ptx::bulk_wait_but_one();
                  const uint32_t n = kbl == 3 ? unpub : unpub - 1;
                  if (n) {
                    __threadfence_block();
                    *seq_done = *seq_done + n;
                    unpub -= n;
                  }
                }
                if (hs < 24) LTR_DBG_STAMP(16 + hs);   // trace: hand-over hs processed (published up to here)
              }
            } else {
              const uint32_t b = hs & 1, ph = (hs >> 1) & 1;
              mbar_wait_dl(&tile_ready[b], ph, false);   // all epilogue warps finished (and fenced) a staged tile
              ++hs;
              __threadfence_block();
              *seq_done = *seq_done + 4;
              ptx::mbar_arrive(&tile_free[b]);
            }
          }
        }
      }
    }
  } else {
    pdl_wait();
    // ---------------------------------------------------------------- epilogue (8 warps per CTA, own 128 rows)
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    // streamed path: staging tile hs & 1 = [hi 16 KB | lo 16 KB] of one output k-block; staged path: per-warp 4 KB in it
    float* xch = reinterpret_cast<float*>(smem + Cfg::OFF_XCH);
    const int r_in = q * 32 + lane;
    uint32_t tl = 0, hs = 0;                        // hs: hand-overs of the staging memory to the store warp so far
    // Per-column vectors (bias, LayerNorm gain / shift) of a streamed tile: lane j keeps column j of each of this warp's
    // four 32-column chunks and the chunk code broadcasts with shuffles.  A broadcast global load per chunk put an L2
    // round trip (every bias line is touched once per CTA and tile, so it never hits L1) in front of each chunk's
    // arithmetic: ~1 k cycles per chunk in the clock64 trace against ~350 of issue time (profiles/r2_chain_trace.md).
    // The bias is fetched one tile ahead.
    auto col_vec = [&](const float* v, int nb, float (&b)[4]) {
#pragma unroll
      for (int k = 0; k < 4; ++k) b[k] = v ? v[nb * BN + k * 64 + half * 32 + lane] : 0.f;
    };
    auto sel4 = [](const float (&a)[4], int k) { return k == 0 ? a[0] : k == 1 ? a[1] : k == 2 ? a[2] : a[3]; };
    float bcur[4] = {0.f, 0.f, 0.f, 0.f}, bnxt[4] = {0.f, 0.f, 0.f, 0.f};
    if (cl0 < n_ctiles) col_vec(c.op[0].bias, 0, bcur);
    uint32_t it_cnt = 0;                            // ring k-blocks of all ops so far (the producer's `it` at the end of the op)
    for (int ct = cl0; ct < n_ctiles; ct += cl_step) {
      const int mt = 2 * ct + (int)rank;
      for (int o = 0; o < c.n_ops; ++o) {
        const GemmImgArgs& p = c.op[o];
        const bool streamed = chain2_streamed(p);
        it_cnt += (uint32_t)(p.n_blks * (p.W.K / 64));
        // direct hand-over (chain2_direct): output k-block j of this op = A k-block j of the next op's first n-block,
        // ring use 2 (it_cnt + j) + 1
        const int nk_next = (o + 1 < c.n_ops && chain2_direct(p)) ? c.op[o + 1].W.K / 64 : 0;
        for (int nb = 0; nb < p.n_blks; ++nb, ++tl) {
          const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
          {   // next tile of this CTA (this op's next n-block, the next op, the next cluster tile)
            int no = o, nnb = nb + 1;
            if (nnb == p.n_blks) { nnb = 0; no = o + 1 < c.n_ops ? o + 1 : (ct + cl_step < n_ctiles ? 0 : -1); }
            if (no >= 0) col_vec(c.op[no].bias, nnb, bnxt);
          }
          // Everything the chunk loops need from the op descriptor, in registers: the descriptor sits in the kernel
          // parameter bank at a dynamic index, and every asm volatile with a memory clobber (tcgen05.ld, mbarrier,
          // fences) made the compiler re-read its fields - indexed LDC + compare + branch chains were a third of the
          // warp-state samples inside the chunk arithmetic (ncu source view, profiles/r2_chain_trace.md).
          const int norm = p.norm, act = p.act;
          const bool has_bias = p.bias != nullptr;
          const __nv_bfloat16* res_hi = p.Rimg.hi;
          const __nv_bfloat16* res_lo = p.Rimg.lo;
          const size_t res_t0 = ((size_t)mt * p.Rimg.kblocks + p.r_kb0 + nb * 4) * IMG_TILE_ELEMS;
          const __nv_bfloat16* add_hi = p.NaddImg.hi;
          const __nv_bfloat16* add_lo = p.NaddImg.lo;
          const size_t add_t0 = ((size_t)mt * p.NaddImg.kblocks + p.nadd_kb0 + nb * 4) * IMG_TILE_ELEMS;
          float* const crow = (p.C && mt * 128 + r_in < p.M) ? p.C + (long long)(mt * 128 + r_in) * p.ldc + nb * BN : nullptr;
          const float eps = p.eps;
          float gk[4] = {1.f, 1.f, 1.f, 1.f}, bek[4] = {0.f, 0.f, 0.f, 0.f};
          if (streamed && norm == NORM_LAYER) { col_vec(p.ng, 0, gk); col_vec(p.nbeta, 0, bek); }
          // Side input of a streamed tile from a split-bf16 image (residual, post-norm addend): this thread's own row,
          // 4 x 16 B per plane and chunk.  Chunk 0 is requested before the accumulator wait, chunk k + 1 right after
          // chunk k was consumed - an L2 round trip per chunk otherwise (mlp2: 14.5 k cycles per tile against 9 k).
          uint4 rh[4], rl[4];
          auto img_load = [&](const __nv_bfloat16* xh, const __nv_bfloat16* xl, size_t toff) {
            const uint8_t* xhi = reinterpret_cast<const uint8_t*>(xh + toff);
            const uint8_t* xlo = reinterpret_cast<const uint8_t*>(xl + toff);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              const uint32_t off = ptx::sw128_offset(r_in, half * 32 + cc * 8);
              rh[cc] = *reinterpret_cast<const uint4*>(xhi + off);
              rl[cc] = *reinterpret_cast<const uint4*>(xlo + off);
            }
          };
          auto img_add = [&](float (&acc)[32]) {
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              const uint32_t wh[4] = {rh[cc].x, rh[cc].y, rh[cc].z, rh[cc].w}, wl[4] = {rl[cc].x, rl[cc].y, rl[cc].z, rl[cc].w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                acc[cc * 8 + 2 * e] += __uint_as_float(wh[e] << 16) + __uint_as_float(wl[e] << 16);
                acc[cc * 8 + 2 * e + 1] += __uint_as_float(wh[e] & 0xFFFF0000u) + __uint_as_float(wl[e] & 0xFFFF0000u);
              }
            }
          };
          auto add_bias = [&](float (&acc)[32], int kbl) {
            const float bk = sel4(bcur, kbl);
#pragma unroll
            for (int j = 0; j < 32; j += 2) {   // packed fp32 pair add (add.f32x2): bit-identical, half the issue slots
              const float2 v = __fadd2_rn(make_float2(acc[j], acc[j + 1]),
                                          make_float2(__shfl_sync(0xffffffffu, bk, j), __shfl_sync(0xffffffffu, bk, j + 1)));
              acc[j] = v.x; acc[j + 1] = v.y;
            }
          };
          if (streamed && res_hi) img_load(res_hi, res_lo, res_t0);
          mbar_wait_dl(&acc_full[buf], aph, true);
          ptx::tc_fence_after();
          const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN;
          if (tl < 10 && warp == 2 && lane == 0) LTR_DBG_STAMP(80 + tl);
          if (tl == 2 && lane == 0) LTR_DBG_STAMP(112 + warp - 2);   // trace: per-warp start of the third tile
          if (streamed) {
            float mean = 0.f, scale = 1.f;
            if (norm != NORM_NONE) {
              // ---- row statistics (N == 256: the tile holds whole rows; the two threads of a row exchange partial sums).
              //      v = acc + bias (+ residual) goes BACK into the accumulator columns (tcgen05.st), so the later passes
              //      are plain TMEM reads: no second trip to the bias / residual.
              float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
              for (int kbl = 0; kbl < 4; ++kbl) {
                const int c0 = kbl * 64 + half * 32;
                float acc[32];
                ptx::tmem_ld32(tacc + (uint32_t)c0, acc);
                if (has_bias) add_bias(acc, kbl);
                if (res_hi) {
                  img_add(acc);
                  if (kbl < 3) img_load(res_hi, res_lo, res_t0 + (size_t)(kbl + 1) * IMG_TILE_ELEMS);
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) { s1 += acc[j]; s2 = fmaf(acc[j], acc[j], s2); }
                ptx::tmem_st32(tacc + (uint32_t)c0, acc);
              }
              if (add_hi) img_load(add_hi, add_lo, add_t0);   // lands under the exchanges below
              if (norm == NORM_LAYER) {
                xch[half * 128 + r_in] = s1;
                epi_bar();
                mean = (s1 + xch[(half ^ 1) * 128 + r_in]) * (1.f / 256.f);
                float ss = 0.f;
#pragma unroll 1
                for (int kbl = 0; kbl < 4; ++kbl) {
                  float acc[32];
                  ptx::tmem_ld32(tacc + (uint32_t)(kbl * 64 + half * 32), acc);
#pragma unroll
                  for (int j = 0; j < 32; ++j) { const float d = acc[j] - mean; ss = fmaf(d, d, ss); }
                }
                xch[256 + half * 128 + r_in] = ss;
                epi_bar();
                ss += xch[256 + (half ^ 1) * 128 + r_in];
                scale = 1.f / sqrtf(ss * (1.f / 256.f) + eps);
              } else {
                float* x = xch + (tl & 1) * 256;   // alternate slots: one barrier per tile is enough
                x[half * 128 + r_in] = s2;
                epi_bar();
                s2 += x[(half ^ 1) * 128 + r_in];
                scale = 1.f / fmaxf(sqrtf(s2), 1e-12f);
              }
            }
#pragma unroll 1
            for (int kbl = 0; kbl < 4; ++kbl) {
              const int c0 = kbl * 64 + half * 32;
              float acc[32];
              const bool fine = tl == 0 && warp == 2 && lane == 0;   // fine-grained trace of the first tile (slots 0..15)
              if (fine) LTR_DBG_STAMP(kbl * 4);
              ptx::tmem_ld32(tacc + (uint32_t)c0, acc);
              if (fine) LTR_DBG_STAMP(kbl * 4 + 1);
              if (kbl == 3) {   // this warp has read everything it needs from the accumulator
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                  if (leader) ptx::mbar_arrive(&acc_empty[buf]);
                  else ptx::mbar_arrive_cluster(ptx::mapa_shared(&acc_empty[buf], 0));
                }
              }
              if (norm == NORM_NONE) {
                if (has_bias) add_bias(acc, kbl);
                if (act == ACT_RELU) {
#pragma unroll
                  for (int j = 0; j < 32; ++j) acc[j] = fmaxf(acc[j], 0.f);
                } else if (act == ACT_GELU) {
#pragma unroll
                  for (int j = 0; j < 32; j += 2) {
                    const float2 g = gelu_erf2(make_float2(acc[j], acc[j + 1]));
                    acc[j] = g.x; acc[j + 1] = g.y;
                  }
                }
                if (res_hi) {
                  img_add(acc);
                  if (kbl < 3) img_load(res_hi, res_lo, res_t0 + (size_t)(kbl + 1) * IMG_TILE_ELEMS);
                }
              } else {
                if (norm == NORM_LAYER) {
                  const float gg = sel4(gk, kbl), bb = sel4(bek, kbl);
#pragma unroll
                  for (int j = 0; j < 32; ++j)
                    acc[j] = (acc[j] - mean) * scale * __shfl_sync(0xffffffffu, gg, j) + __shfl_sync(0xffffffffu, bb, j);
                } else {
#pragma unroll
                  for (int j = 0; j < 32; ++j) acc[j] *= scale;
                }
                if (add_hi) {
                  img_add(acc);
                  if (kbl < 3) img_load(add_hi, add_lo, add_t0 + (size_t)(kbl + 1) * IMG_TILE_ELEMS);
                }
              }
              if (crow) {   // fp32 rows: this thread's 128 contiguous bytes, four 256-bit stores
#pragma unroll
                for (int j = 0; j < 32; j += 8)
                  ptx::st_global_256(crow + c0 + j, make_uint4(__float_as_uint(acc[j]), __float_as_uint(acc[j + 1]), __float_as_uint(acc[j + 2]), __float_as_uint(acc[j + 3])),
                                     make_uint4(__float_as_uint(acc[j + 4]), __float_as_uint(acc[j + 5]), __float_as_uint(acc[j + 6]), __float_as_uint(acc[j + 7])));
              }
              uint4 h[4], l[4];
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) ptx::split8_bf16(&acc[cc * 8], h[cc], l[cc]);
              if (fine) LTR_DBG_STAMP(kbl * 4 + 2);
              const uint32_t sb = hs & 1;
              uint8_t* tile = smem + Cfg::OFF_STG + sb * Cfg::STG_TILE;
              mbar_wait_dl(&tile_free[sb], ((hs >> 1) & 1) ^ 1, false);   // its previous contents have been read by the store warp's copies
              ++hs;
              if (fine) LTR_DBG_STAMP(kbl * 4 + 3);
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) {
                const uint32_t off = ptx::sw128_offset(r_in, (c0 & 63) + cc * 8);
                *reinterpret_cast<uint4*>(tile + off) = h[cc];
                *reinterpret_cast<uint4*>(tile + 16384 + off) = l[cc];
              }
              if (kbl < nk_next) {   // the same 64 B per plane also into the next op's A slot (n_blks == 1: nb == 0)
                const uint32_t uc = 2u * (it_cnt + (uint32_t)kbl) + 1u;
                const int slc = slot_of(uc);
                uint8_t* aslot = smem + slc * Cfg::SLOT;
                mbar_wait_dl(&empty[slc], phase_of(uc) ^ 1, true);   // the MMAs that read the slot's previous tile are complete
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                  const uint32_t off = ptx::sw128_offset(r_in, (c0 & 63) + cc * 8);
                  *reinterpret_cast<uint4*>(aslot + off) = h[cc];
                  *reinterpret_cast<uint4*>(aslot + Cfg::A_TILE + off) = l[cc];
                }
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                  ptx::mbar_arrive(&tile_ready[sb]);
                  ptx::mbar_arrive(&full[slc]);
                }
              } else {
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&tile_ready[sb]);
              }
              if (tl == 2 && kbl == 0 && lane == 0) LTR_DBG_STAMP(90 + warp - 2);   // trace: per-warp first hand-over of the third tile
            }
          } else {
            const uint32_t sb = hs & 1;
            float* stg = reinterpret_cast<float*>(smem + Cfg::OFF_STG + sb * Cfg::STG_TILE + (warp - 2) * Cfg::STG_WARP);
            uint8_t* stgb = reinterpret_cast<uint8_t*>(stg);
            mbar_wait_dl(&tile_free[sb], ((hs >> 1) & 1) ^ 1, false);   // the per-warp staging areas alias staging tile sb
            ++hs;
            if (p.norm != NORM_NONE)
              epi_norm_tile(p, tacc, mt, q, half, lane, tl, stg, stgb, xch);
            else
              epi_plain_tile<BN>(p, tacc, mt, nb, q, half, lane, stg, stgb);
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (leader) ptx::mbar_arrive(&acc_empty[buf]);
              else ptx::mbar_arrive_cluster(ptx::mapa_shared(&acc_empty[buf], 0));
            }
            // generic-proxy global stores of this tile -> visible to the bulk copies of the next op's producer
            __threadfence();
            ptx::fence_proxy_async_all();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tile_ready[sb]);   // the store warp publishes the tile's four k-blocks
          }
          if (tl < 10 && warp == 2 && lane == 0) LTR_DBG_STAMP(43 + tl * 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) bcur[k] = bnxt[k];
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();          // nobody leaves (or frees TMEM) while the peer may still signal / multiply
  if (tid == 0) LTR_DBG_STAMP(111);
  if (warp == 1) ptx::tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
}

inline int device_sm_count() {
  static std::atomic<int> sms[64];   // zero-initialised; benign duplicate queries, no torn state
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return 148;
  int v = sms[dev].load(std::memory_order_relaxed);
  if (!v) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (v <= 0) v = 148;
    sms[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

template <int BN>
static int launch_gemm_img_bn(GemmImgArgs a, cudaStream_t s) {
  using Cfg = GemmImgCfg<BN>;
  LTR_CUDA_TRY(ensure_dynamic_smem(gemm_img_kernel<BN>, Cfg::SMEM));
  a.m_tiles = cdiv(a.M, 128);
  a.n_blks = a.W.N / BN;
  const int tiles = a.m_tiles * a.n_blks;
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  LaunchScope ls(KC_LINEAR, s);
  LTR_CUDA_TRY(launch_pdl(gemm_img_kernel<BN>, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM, s, a));
  return 0;
}

// bn_hint: 0 = choose (256 when N % 256 == 0 and that still gives >= 1 tile per SM, else 128)
inline int launch_gemm_img(const GemmImgArgs& a, cudaStream_t s, int bn_hint = 0) {
  if (a.M <= 0) return 0;
  if (a.W.K % 64 || a.W.N % 64 || (a.C && a.ldc % 8) || (a.R && a.ldr % 4))
    return set_error(-1, "gemm_img: K%64, N%64, ldc%8, ldr%4 required");
  {   // operand / output k-block ranges must lie inside their images (a wrong d_inner would otherwise alias tiles silently)
    const int nblk = a.a_kb_nb ? a.W.N / 64 : 1;   // block-diagonal: 64-wide n-blocks, each with its own K slice
    if (a.a_kb0 < 0 || a.a_kb0 + (nblk - 1) * a.a_kb_nb + a.W.K / 64 > a.A.kblocks)
      return set_error(-1, "gemm_img: A k-block range exceeds the activation image");
    if (a.O.hi && (a.o_kb0 < 0 || a.o_kb0 + a.W.N / 64 > a.O.kblocks))
      return set_error(-1, "gemm_img: output columns exceed the output image");
    if (a.Rimg.hi && (a.r_kb0 < 0 || a.r_kb0 + a.W.N / 64 > a.Rimg.kblocks))
      return set_error(-1, "gemm_img: residual columns exceed the residual image");
  }
  if (a.norm != NORM_NONE) {
    if (a.W.N != 256 || a.act != ACT_NONE || (a.nadd && a.ldadd % 4) || (a.norm == NORM_LAYER && (!a.ng || !a.nbeta)) ||
        (a.R && a.Rimg.hi) || (a.nadd && a.NaddImg.hi) ||
        (a.NaddImg.hi && (a.nadd_kb0 < 0 || a.nadd_kb0 + 4 > a.NaddImg.kblocks)))
      return set_error(-1, "gemm_img: the row-norm epilogue needs N == 256, no activation, fp32 residual");
    return launch_gemm_img_bn<256>(a, s);
  }
  if (bn_hint == 64 || a.W.N % 128) return launch_gemm_img_bn<64>(a, s);
  int bn = bn_hint;
  if (!bn) {
    bn = 128;
    if (a.W.N % 256 == 0 && (long long)cdiv(a.M, 128) * (a.W.N / 256) >= device_sm_count()) bn = 256;
  }
  if (bn == 256 && a.W.N % 256 == 0) return launch_gemm_img_bn<256>(a, s);
  return launch_gemm_img_bn<128>(a, s);
}

// Chain of row-local layers in one launch of gemm_chain2_kernel (see "chained GEMMs" above).  Every op: N % 256 == 0,
// plain A (no block-diagonal slices); op i+1 must read what op i writes for the same rows only.  The images the chain
// reads (A, residual, addend) must be padded to 256 rows (ltr_api.cu carve does).  O may be padded to 128 rows only
// (the caller's descriptor tile image): the store warp drops the output of the phantom tile an odd tile count gives the
// last cluster.
inline int launch_gemm_chain(const GemmImgArgs* ops, int n_ops, cudaStream_t s) {
  if (n_ops < 1 || n_ops > CHAIN_MAX_OPS) return set_error(-1, "gemm_chain: 1..4 ops");
  if (ops[0].M <= 0) return 0;
  GemmChainArgs c{};
  c.n_ops = n_ops;
  c.m_tiles = cdiv(ops[0].M, 128);
  for (int i = 0; i < n_ops; ++i) {
    GemmImgArgs a = ops[i];
    if (a.M != ops[0].M || a.W.K % 64 || a.W.N % 256 || a.a_kb_nb || (a.C && a.ldc % 8) || (a.R && a.ldr % 4))
      return set_error(-1, "gemm_chain: ops need equal M, K%64, N%256, no block-diagonal A");
    if (a.a_kb0 < 0 || a.a_kb0 + a.W.K / 64 > a.A.kblocks || (a.O.hi && (a.o_kb0 < 0 || a.o_kb0 + a.W.N / 64 > a.O.kblocks)) ||
        (a.Rimg.hi && (a.r_kb0 < 0 || a.r_kb0 + a.W.N / 64 > a.Rimg.kblocks)))
      return set_error(-1, "gemm_chain: k-block range exceeds an image");
    if (a.norm != NORM_NONE && (a.W.N != 256 || a.act != ACT_NONE || (a.norm == NORM_LAYER && (!a.ng || !a.nbeta))))
      return set_error(-1, "gemm_chain: the row-norm epilogue needs N == 256 and no activation");
    if ((a.R && a.Rimg.hi) || (a.nadd && a.NaddImg.hi) || ((a.nadd || a.NaddImg.hi) && a.norm == NORM_NONE) ||
        (a.NaddImg.hi && (a.nadd_kb0 < 0 || a.nadd_kb0 + a.W.N / 64 > a.NaddImg.kblocks)))
      return set_error(-1, "gemm_chain: residual / addend given twice, addend without a row norm, or its k-blocks exceed the image");
    // op i > 0 reads, k-block for k-block, what op i-1 wrote for the same rows (the kernel's dependency rule)
    if (i > 0 && (a.A.hi != ops[i - 1].O.hi || a.a_kb0 != ops[i - 1].o_kb0 || a.W.K > ops[i - 1].W.N))
      return set_error(-1, "gemm_chain: op i must consume the image op i-1 writes (same k-blocks)");
    a.m_tiles = c.m_tiles;
    a.n_blks = a.W.N / 256;
    c.op[i] = a;
  }
  using Cfg = GemmPairCfg;
  LTR_CUDA_TRY(ensure_dynamic_smem(gemm_chain2_kernel, Cfg::SMEM));
  const int clusters = std::min((c.m_tiles + 1) / 2, device_sm_count() / 2);
  LaunchScope ls(KC_LINEAR, s);
  const bool traced = dbg_chain_sel() >= 0 && dbg_chain_cnt()++ == dbg_chain_sel();
  static const int k_on = 1, k_off = 0;
  if (traced) cudaMemcpyToSymbolAsync(g_dbg_on, &k_on, sizeof(int), 0, cudaMemcpyHostToDevice, s);
  LTR_CUDA_TRY(launch_pdl(gemm_chain2_kernel, dim3(2 * clusters), dim3(Cfg::THREADS), Cfg::SMEM, s, c));   // __cluster_dims__(2,1,1)
  if (traced) cudaMemcpyToSymbolAsync(g_dbg_on, &k_off, sizeof(int), 0, cudaMemcpyHostToDevice, s);
  return 0;
}

// ---------------------------------------------------------------- image <-> fp32 helpers
// fp32 rows [M, K] (ld) -> image k-blocks [kb0, kb0 + K/64); one thread per 8 consecutive k.
__global__ void __launch_bounds__(256) to_image_kernel(const float* __restrict__ x, int ld, int M, int K, ActImg o, int kb0) {
  const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
  const int k8 = K / 8;
  if (idx >= (long long)M * k8) return;
  const int row = (int)(idx / k8), k = (int)(idx % k8) * 8;
  const float4 a = *reinterpret_cast<const float4*>(x + (long long)row * ld + k);
  const float4 b = *reinterpret_cast<const float4*>(x + (long long)row * ld + k + 4);
  const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint4 h, l;
  ptx::split8_bf16(v, h, l);
  const size_t toff = ((size_t)(row >> 7) * o.kblocks + kb0 + (k >> 6)) * IMG_TILE_ELEMS;
  const uint32_t off = ptx::sw128_offset(row & 127, k & 63);
  *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(o.hi + toff) + off) = h;
  *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(o.lo + toff) + off) = l;
}

// image k-blocks [kb0, kb0 + K/64) -> fp32 rows (hi + lo); test helper.
__global__ void __launch_bounds__(256) from_image_kernel(ActImg a, int kb0, float* __restrict__ y, int ld, int M, int K) {
  const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
  if (idx >= (long long)M * K) return;
  const int row = (int)(idx / K), k = (int)(idx % K);
  const size_t toff = ((size_t)(row >> 7) * a.kblocks + kb0 + (k >> 6)) * IMG_TILE_ELEMS;
  const uint32_t off = ptx::sw128_offset(row & 127, k & 63) / 2;
  y[(long long)row * ld + k] = __bfloat162float(a.hi[toff + off]) + __bfloat162float(a.lo[toff + off]);
}

}  // namespace ltr
