// Tensor-core descriptor matcher (K3): all-pairs distance D = 2 - 2 <a_i, b_j> on tcgen05 with the
// row-argmin fused into the epilogue, for BOTH directions (side 0 rows vs side 1 and side 1 rows vs
// side 0 - the second one is the column argmin the mutual check needs), a tail kernel that applies
// threshold + mutual check + per-pair counts and lists the decisions the tensor-core arithmetic cannot
// make safely, and an exact fp32 kernel that re-takes those over the whole GPU.
//
// Reference: get_dist_matrix (models/line_process.py:198-201: einsum('bdn,bdm->bnm'), (2 - 2 s).clip(0)),
// nn_matcher / nn_matcher_distmat (models/nn_matcher.py:3-43: argmin axis 1, strict '<' threshold,
// argmin axis 0, mutual check), and - distance mode 1 - the training-side matcher
// evaluations/matcher.py:51-102 (||a||^2 + ||b||^2 - 2 ab).
//
// Precision contract.  The contraction is a 3-term split-bf16 product (hi*hi + lo*hi + hi*lo, fp32
// accumulate in TMEM): ~1e-5 absolute on a distance.  Match indices must be bit-exact, so every row
// whose best and second-best distance are closer than MATCH_EPS, or whose best distance lies within
// MATCH_EPS of the threshold, is recomputed by match_exact_kernel with fp32 FMAs in ascending k order
// (the arithmetic of the round-1 FFMA matcher the golden vectors were pinned with) before any decision
// is taken.  Exact ties therefore resolve to the lowest index exactly as np.argmin does.
//
// Operands are "descriptor tile images": the split-bf16 activation-image format of gemm_img.cuh
// (planes hi / lo, 16 KB tiles [row/128][k/64] of 128 rows x 64 k, K-major SWIZZLE_128B), 4 k-blocks
// per 128-row tile.  Either the encoder's final GEMM writes them (pairs whose first line is 128-aligned
// in the batch - every uniform batch with L % 128 == 0) or desc_tiles_kernel builds pair-aligned tiles
// from fp32 descriptors (rows [n, 256] or channel-first [256, n]).
#pragma once
#include "act_img.cuh"
#include "common.cuh"
#include "ptx_sm100.cuh"

namespace ltr {

constexpr float MATCH_EPS = 1e-4f;
constexpr int MT_D = 256;                         // descriptor dimension the tensor-core matcher is built for
constexpr int MT_KB = MT_D / 64;                  // k-blocks per tile row
constexpr int MT_TILE = 16384;                    // one plane of a 128 x 64 bf16 tile
constexpr int MT_A_BYTES = MT_KB * 2 * MT_TILE;   // resident A: 4 k-blocks x (hi + lo) = 128 KB
constexpr int MT_STAGE = 2 * MT_TILE;             // B ring stage: one k-block, hi + lo
constexpr int MT_STAGES = 3;
constexpr int MT_OFF_B = MT_A_BYTES;
constexpr int MT_OFF_BAR = MT_OFF_B + MT_STAGES * MT_STAGE;
constexpr int MT_OFF_XCH = MT_OFF_BAR + 256;      // half-merge exchange: 3 x 128 x 4 B
constexpr int MT_SMEM = MT_OFF_XCH + 1536 + 1024; // + alignment slack (<= 227 KB)
constexpr int MT_THREADS = 320;                   // TMA warp, MMA warp, 8 epilogue warps
static_assert(MT_SMEM <= 232448, "match_tc: shared memory budget");

// One side of a batch of pairs.
struct MatchSide {
  ActImg img;            // descriptor tile image (kblocks = 4)
  const int* cu;         // [n_pairs + 1] line offsets or nullptr (uniform n)
  int n;                 // lines per pair when cu == nullptr
  int tile_mode;         // 0: pair p starts at tile p * tmax (pair-aligned scratch tiles)
                         // 1: pair p starts at tile (tile_row0 + first line of p) / 128 (encoder image, aligned pairs)
  int tile_row0;         // mode 1: row of this side's first line inside the image
  int tmax;              // row tiles per pair (grid sizing; tile stride in mode 0)
  const float* sq;       // mode-1 distance only: squared norms, indexed like the lines (cu / p * n)
  uint2* slot;           // out: per line {bits(best distance), best index | ambiguous << 31}
};

// Work list of the exact re-check: an item is one line whose tensor-core argmin cannot be trusted, a tile up to
// XT_ITEMS items of one pair and side.  match_tail_kernel appends, match_exact_kernel takes.
constexpr int XT_ITEMS = 32;
struct ExactTile {
  int pair, side, n, pad;
  int line[XT_ITEMS];    // lines inside the pair
};
// counters (zeroed by match_tc_kernel, or by a memset when it does not run)
constexpr int XQ_TILES = 0;      // tiles on the list
constexpr int XQ_HEAD = 1;       // next tile to take
constexpr int XQ_PAIRS = 2;      // pairs with at least one tile
constexpr int XQ_FINISHED = 3;   // pairs whose open decisions are made (multi-GPU publication)
constexpr int XQ_HDR = 4;        // then tiles per pair [n_pairs], finished tiles per pair [n_pairs]
struct ExactQueue {
  int* ctr;
  ExactTile* tiles;      // capacity: 256 / XT_ITEMS + 1 tiles per tail block
  uint2* res[2];         // per line of each side: {bits(exact best distance), exact best index}, items only
};

struct MatchTcArgs {
  MatchSide s[2];
  int dist_mode;         // 0: 2 - 2 s (unit descriptors, nn_matcher.py:37-38)   1: |a|^2 + |b|^2 - 2 s (evaluations/matcher.py:66-70)
  float* dist;           // optional dense output of side 0 vs side 1, pair p at p * dist_stride, row-major [n0_p, n1_p]
  long long dist_stride;
  int* counts;           // zeroed here (the tail and exact kernels accumulate into it)
  int* xq_ctr;           // exact work-list counters (XQ_HDR + 2 n_pairs), zeroed here
  int n_pairs;
};

__device__ __forceinline__ void side_range(const MatchSide& s, int pair, int& b, int& e) { image_range(s.cu, s.n, pair, b, e); }
__device__ __forceinline__ int side_tile0(const MatchSide& s, int pair, int b) {
  return s.tile_mode ? (s.tile_row0 + b) >> 7 : pair * s.tmax;
}

__device__ __forceinline__ void mt_epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// grid = (tmax0 + tmax1, n_pairs): CTA x < tmax0 handles row block x of side 0 against all of side 1,
// the others row block x - tmax0 of side 1 against all of side 0.
__global__ void __launch_bounds__(MT_THREADS, 1) match_tc_kernel(MatchTcArgs p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + MT_OFF_BAR);
  uint64_t* full = bars;                   // [STAGES] B stage landed
  uint64_t* empty = bars + MT_STAGES;      // [STAGES] B stage consumed
  uint64_t* a_full = bars + 2 * MT_STAGES; // [1] resident A landed
  uint64_t* acc_full = a_full + 1;         // [2]
  uint64_t* acc_empty = acc_full + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* xch = reinterpret_cast<float*>(smem + MT_OFF_XCH);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int pair = blockIdx.y;
  const int side = (int)blockIdx.x >= p.s[0].tmax ? 1 : 0;
  const int rb = side ? (int)blockIdx.x - p.s[0].tmax : (int)blockIdx.x;
  const MatchSide& SA = p.s[side];
  const MatchSide& SB = p.s[side ^ 1];
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < MT_STAGES; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    ptx::mbar_init(a_full, 1);
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(&acc_full[b], 1);
      ptx::mbar_init(&acc_empty[b], 8);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 256);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // descriptors / tile images of the producing kernel are complete from here on

  int ba, ea, bb, eb;
  side_range(SA, pair, ba, ea);
  side_range(SB, pair, bb, eb);
  const int na = ea - ba, nb = eb - bb;
  if (p.counts && blockIdx.x == 0 && tid == 0) p.counts[pair] = 0;
  if (p.xq_ctr && blockIdx.x == 0 && tid == 0) {
    p.xq_ctr[XQ_HDR + pair] = 0;
    p.xq_ctr[XQ_HDR + p.n_pairs + pair] = 0;
    if (pair == 0)
      for (int i = 0; i < XQ_HDR; ++i) p.xq_ctr[i] = 0;
  }
  const bool active = rb * 128 < na && nb > 0;   // uniform per CTA
  const int n_ct = active ? (nb + 127) >> 7 : 0;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    if (lane == 0 && active) {
      const size_t ta = (size_t)(side_tile0(SA, pair, ba) + rb) * MT_KB;
      ptx::mbar_arrive_expect_tx(a_full, MT_A_BYTES);
#pragma unroll
      for (int kb = 0; kb < MT_KB; ++kb) {
        ptx::bulk_g2s(smem + kb * 2 * MT_TILE, SA.img.hi + (ta + kb) * IMG_TILE_ELEMS, MT_TILE, a_full);
        ptx::bulk_g2s(smem + kb * 2 * MT_TILE + MT_TILE, SA.img.lo + (ta + kb) * IMG_TILE_ELEMS, MT_TILE, a_full);
      }
      const size_t tb0 = (size_t)side_tile0(SB, pair, bb) * MT_KB;
      uint32_t it = 0;
      for (int ct = 0; ct < n_ct; ++ct)
        for (int kb = 0; kb < MT_KB; ++kb, ++it) {
          const int s = it % MT_STAGES;
          const uint32_t ph = (it / MT_STAGES) & 1;
          ptx::mbar_wait(&empty[s], ph ^ 1);
          uint8_t* st = smem + MT_OFF_B + s * MT_STAGE;
          const size_t toff = (tb0 + (size_t)ct * MT_KB + kb) * IMG_TILE_ELEMS;
          ptx::mbar_arrive_expect_tx(&full[s], MT_STAGE);
          ptx::bulk_g2s(st, SB.img.hi + toff, MT_TILE, &full[s]);
          ptx::bulk_g2s(st + MT_TILE, SB.img.lo + toff, MT_TILE, &full[s]);
        }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    if (lane == 0 && active) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16_f32(128, 128);
      ptx::mbar_wait(a_full, 0);
      ptx::tc_fence_after();
      uint32_t it = 0;
      for (int ct = 0; ct < n_ct; ++ct) {
        const uint32_t buf = ct & 1, aph = (ct >> 1) & 1;
        ptx::mbar_wait(&acc_empty[buf], aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * 128;
        for (int kb = 0; kb < MT_KB; ++kb, ++it) {
          const int s = it % MT_STAGES;
          const uint32_t ph = (it / MT_STAGES) & 1;
          ptx::mbar_wait(&full[s], ph);
          ptx::tc_fence_after();
          const uint32_t a_hi = ptx::smem_u32(smem + kb * 2 * MT_TILE), a_lo = a_hi + MT_TILE;
          const uint32_t b_hi = ptx::smem_u32(smem + MT_OFF_B + s * MT_STAGE), b_lo = b_hi + MT_TILE;
#pragma unroll
          for (int k16 = 0; k16 < 4; ++k16) {
            const uint32_t ko = k16 * 32;
            const uint64_t dah = ptx::make_sw128_kmajor_desc(a_hi + ko, 1024);
            const uint64_t dal = ptx::make_sw128_kmajor_desc(a_lo + ko, 1024);
            const uint64_t dbh = ptx::make_sw128_kmajor_desc(b_hi + ko, 1024);
            const uint64_t dbl = ptx::make_sw128_kmajor_desc(b_lo + ko, 1024);
            ptx::umma_bf16(d_tmem, dal, dbh, idesc, (kb | k16) != 0);
            ptx::umma_bf16(d_tmem, dah, dbl, idesc, 1);
            ptx::umma_bf16(d_tmem, dah, dbh, idesc, 1);
          }
          ptx::umma_commit(&empty[s]);
        }
        ptx::umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue (8 warps)
    // thread = accumulator row (TMEM lane) x one half of the tile's 128 columns; running best /
    // second-best over all column tiles stay in registers.
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int r_in = q * 32 + lane;
    const int row = rb * 128 + r_in;             // line of side A inside the pair
    const bool valid_row = row < na;
    float best = INFINITY, second = INFINITY;
    int bidx = 0x7fffffff;
    const float sqa = (p.dist_mode == 1 && valid_row) ? SA.sq[ba + row] : 0.f;
    float* drow = (p.dist && side == 0 && valid_row) ? p.dist + (long long)pair * p.dist_stride + (long long)row * nb : nullptr;
    const bool dvec = drow && (nb % 8 == 0) && (p.dist_stride % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.dist) & 31) == 0);
    for (int ct = 0; ct < n_ct; ++ct) {
      const uint32_t buf = ct & 1, aph = (ct >> 1) & 1;
      ptx::mbar_wait(&acc_full[buf], aph);
      ptx::tc_fence_after();
#pragma unroll 1
      for (int c0 = half * 64; c0 < half * 64 + 64; c0 += 32) {
        float acc[32];
        ptx::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * 128 + (uint32_t)c0, acc);
        const int j0 = ct * 128 + c0;            // first column (line of side B) of this chunk
        if (j0 >= nb) continue;                  // whole chunk is padding
        if (p.dist_mode == 1) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 sb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j0 + j + 3 < nb) {
              sb.x = SB.sq[bb + j0 + j]; sb.y = SB.sq[bb + j0 + j + 1]; sb.z = SB.sq[bb + j0 + j + 2]; sb.w = SB.sq[bb + j0 + j + 3];
            } else {
              if (j0 + j < nb) sb.x = SB.sq[bb + j0 + j];
              if (j0 + j + 1 < nb) sb.y = SB.sq[bb + j0 + j + 1];
              if (j0 + j + 2 < nb) sb.z = SB.sq[bb + j0 + j + 2];
            }
            acc[j] = fmaxf((sqa + sb.x) - 2.f * acc[j], 0.f);
            acc[j + 1] = fmaxf((sqa + sb.y) - 2.f * acc[j + 1], 0.f);
            acc[j + 2] = fmaxf((sqa + sb.z) - 2.f * acc[j + 2], 0.f);
            acc[j + 3] = fmaxf((sqa + sb.w) - 2.f * acc[j + 3], 0.f);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[j] = fmaxf(fmaf(-2.f, acc[j], 2.f), 0.f);
        }
        if (j0 + 32 <= nb) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float v = acc[j];
            if (v < best) { second = best; best = v; bidx = j0 + j; }
            else if (v < second) second = v;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float v = (j0 + j < nb) ? acc[j] : INFINITY;
            if (v < best) { second = best; best = v; bidx = j0 + j; }
            else if (v < second) second = v;
          }
        }
        if (drow) {
          if (dvec && j0 + 32 <= nb) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              const uint4 a = make_uint4(__float_as_uint(acc[j]), __float_as_uint(acc[j + 1]), __float_as_uint(acc[j + 2]), __float_as_uint(acc[j + 3]));
              const uint4 b = make_uint4(__float_as_uint(acc[j + 4]), __float_as_uint(acc[j + 5]), __float_as_uint(acc[j + 6]), __float_as_uint(acc[j + 7]));
              ptx::st_global_256(drow + j0 + j, a, b);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j0 + j < nb) drow[j0 + j] = acc[j];
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
    }
    // merge the two column halves of every row (lexicographic (value, index): first minimum wins)
    if (half == 1) {
      xch[r_in] = best;
      xch[128 + r_in] = second;
      reinterpret_cast<int*>(xch)[256 + r_in] = bidx;
    }
    mt_epi_bar();
    if (half == 0 && valid_row) {
      const float ob = xch[r_in], os = xch[128 + r_in];
      const int oi = reinterpret_cast<int*>(xch)[256 + r_in];
      if (ob < best || (ob == best && oi < bidx)) { second = fminf(best, os); best = ob; bidx = oi; }
      else second = fminf(second, ob);
      const bool amb = !(second - best >= MATCH_EPS);   // also true for NaN
      SA.slot[ba + row] = make_uint2(__float_as_uint(best), (uint32_t)bidx | (amb ? 0x80000000u : 0u));
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, 256);
}

// ---------------------------------------------------------------- fp32 descriptors -> pair-aligned tile images
struct DescTilesArgs {
  const float* d[2];     // fp32 descriptors of side 0 / 1
  int layout;            // 0 rows [n, 256] per line; 1 channel-first [256, n_p] per pair (pair p at 256 * first line)
  const int* cu[2]; int n[2];
  ActImg img[2]; int tmax[2];
  float* sq[2];          // optional squared norms per line (distance mode 1) or nullptr
};

// grid = (max(tmax0, tmax1) * 4, n_pairs, 2): block = 32 lines of one tile; 256 threads.
__global__ void __launch_bounds__(256) desc_tiles_kernel(DescTilesArgs p) {
  __shared__ float part[8][33];
  pdl_launch_dependents();
  pdl_wait();
  const int side = blockIdx.z, pair = blockIdx.y;
  const int tile = blockIdx.x >> 2, sub = blockIdx.x & 3;
  if (tile >= p.tmax[side]) return;
  int b, e;
  image_range(p.cu[side], p.n[side], pair, b, e);
  const int n = e - b;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* __restrict__ src = p.d[side];
  const ActImg& img = p.img[side];
  const size_t t0 = ((size_t)pair * p.tmax[side] + tile) * MT_KB;
  uint8_t* hi = reinterpret_cast<uint8_t*>(img.hi);
  uint8_t* lo = reinterpret_cast<uint8_t*>(img.lo);
  if (p.layout == 0) {
    // warp -> 4 consecutive lines, lane -> 8 consecutive k
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r_in = sub * 32 + warp * 4 + i, r = tile * 128 + r_in;
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (r < n) {
        const float4 a = *reinterpret_cast<const float4*>(src + (size_t)(b + r) * MT_D + lane * 8);
        const float4 c = *reinterpret_cast<const float4*>(src + (size_t)(b + r) * MT_D + lane * 8 + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
      }
      uint4 h, l;
      ptx::split8_bf16(v, h, l);
      const size_t off = (t0 + (lane >> 3)) * (size_t)MT_TILE + ptx::sw128_offset(r_in, (lane & 7) * 8);
      *reinterpret_cast<uint4*>(hi + off) = h;
      *reinterpret_cast<uint4*>(lo + off) = l;
      if (p.sq[side]) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) s = fmaf(v[j], v[j], s);
        s = warp_sum(s);
        if (lane == 0 && r < n) p.sq[side][b + r] = s;
      }
    }
  } else {
    // lane -> line, warp -> groups of 8 consecutive k (4 groups per warp): loads coalesced along lines
    const int r_in = sub * 32 + lane, r = tile * 128 + r_in;
    const float* __restrict__ base = src + (size_t)b * MT_D;   // [256, n] of this pair
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int k0 = (g * 8 + warp) * 8;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (r < n) ? base[(size_t)(k0 + j) * n + r] : 0.f;
      uint4 h, l;
      ptx::split8_bf16(v, h, l);
      const size_t off = (t0 + (k0 >> 6)) * (size_t)MT_TILE + ptx::sw128_offset(r_in, k0 & 63);
      *reinterpret_cast<uint4*>(hi + off) = h;
      *reinterpret_cast<uint4*>(lo + off) = l;
#pragma unroll
      for (int j = 0; j < 8; ++j) s = fmaf(v[j], v[j], s);
    }
    if (p.sq[side]) {
      part[warp][lane] = s;
      __syncthreads();
      if (warp == 0 && r < n) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += part[w][lane];
        p.sq[side][b + r] = t;
      }
    }
  }
}

constexpr int GATHER_SLOTS = 8;   // = LTR_GATHER_SLOTS
__device__ __forceinline__ void multimem_st_u32(int* mc_addr, int v) {
  asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(mc_addr), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---------------------------------------------------------------- tail: threshold, mutual check, counts, exact work list
struct MatchTailArgs {
  const int* cu[2]; int n[2];
  const uint2* slot[2];
  float thr; int mutual;
  int* matches0; float* scores0; int* nn1; int* counts;
  int max0;                        // max lines of side 0 per pair (row part of the grid)
  ExactQueue xq;
};

// grid = (ceil((max0 + max1) / 256), n_pairs), 256 threads, one line per thread: items below max0 decide side-0
// lines (matches0 / scores0 / counts), the others publish nn1 (argmin over axis 0).  Lines whose tensor-core
// argmin cannot be trusted (ambiguous slot, or a side-0 score next to the threshold) are appended to the exact
// work list in tiles of up to XT_ITEMS lines of one pair and side; match_exact_kernel takes them.  A side-0 row
// whose only doubt is an ambiguous partner column keeps its own tensor-core result and is left undecided: it
// needs that column's exact argmin, and the column is on the list.
__global__ void __launch_bounds__(256) match_tail_kernel(MatchTailArgs p) {
  __shared__ int list[2][256];
  __shared__ int n_list[2], n_keep, tile0[2];
  pdl_launch_dependents();
  pdl_wait();
  const int pair = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
  int b0, e0, b1, e1;
  image_range(p.cu[0], p.n[0], pair, b0, e0);
  image_range(p.cu[1], p.n[1], pair, b1, e1);
  const int n0 = e0 - b0, n1 = e1 - b1;
  if (tid == 0) { n_list[0] = 0; n_list[1] = 0; n_keep = 0; }
  __syncthreads();
  const int w = blockIdx.x * 256 + tid;
  bool keep = false;
  if (w < p.max0) {
    const int i = w;
    if (i < n0) {
      if (n1 == 0) {
        p.matches0[b0 + i] = -1;
        p.scores0[b0 + i] = INFINITY;
      } else {
        const uint2 s = p.slot[0][b0 + i];
        const float v = __uint_as_float(s.x);
        const int idx = (int)(s.y & 0x7fffffffu);
        if ((s.y >> 31) || !(fabsf(v - p.thr) >= MATCH_EPS)) {
          list[0][atomicAdd(&n_list[0], 1)] = i;
        } else {
          keep = v < p.thr;   // strict '<' (nn_matcher.py:18)
          bool defer = false;
          if (keep && p.mutual) {
            const uint2 t = p.slot[1][b1 + idx];
            defer = (t.y >> 31) != 0;
            keep = !defer && (int)(t.y & 0x7fffffffu) == i;
          }
          if (!defer) { p.matches0[b0 + i] = keep ? idx : -1; p.scores0[b0 + i] = v; }
        }
      }
    }
  } else if (p.mutual) {
    const int j = w - p.max0;
    if (j < n1) {
      if (n0 == 0) p.nn1[b1 + j] = -1;
      else {
        const uint2 t = p.slot[1][b1 + j];
        if (t.y >> 31) list[1][atomicAdd(&n_list[1], 1)] = j;
        else p.nn1[b1 + j] = (int)(t.y & 0x7fffffffu);
      }
    }
  }
  const unsigned kb = __ballot_sync(0xffffffffu, keep);
  if (lane == 0 && kb) atomicAdd(&n_keep, __popc(kb));
  __syncthreads();
  if (tid == 0) {
    if (n_keep) atomicAdd(&p.counts[pair], n_keep);
    const int t0 = (n_list[0] + XT_ITEMS - 1) / XT_ITEMS, t1 = (n_list[1] + XT_ITEMS - 1) / XT_ITEMS;
    if (t0 + t1) {
      const int first = atomicAdd(&p.xq.ctr[XQ_TILES], t0 + t1);
      tile0[0] = first;
      tile0[1] = first + t0;
      if (atomicAdd(&p.xq.ctr[XQ_HDR + pair], t0 + t1) == 0) atomicAdd(&p.xq.ctr[XQ_PAIRS], 1);
    }
  }
  __syncthreads();
#pragma unroll
  for (int sd = 0; sd < 2; ++sd) {
    const int n = n_list[sd];
    if (tid < n) {
      ExactTile& t = p.xq.tiles[tile0[sd] + tid / XT_ITEMS];
      t.line[tid % XT_ITEMS] = list[sd][tid];
      if (tid % XT_ITEMS == 0) { t.pair = pair; t.side = sd; t.n = min(XT_ITEMS, n - tid); }
    }
  }
}

// ---------------------------------------------------------------- exact re-check of the work list
struct MatchExactArgs {
  const float* d[2]; int layout;   // the fp32 descriptors the tiles were made from
  const int* cu[2]; int n[2];
  const float* sq[2];              // distance mode 1
  int dist_mode;
  const uint2* slot[2];
  float thr; int mutual;
  int* matches0; float* scores0; int* nn1; int* counts;
  ExactQueue xq;
  // multi-GPU publication of `counts` (LtrPeerGather): symmetric buffer = counts[SLOTS][world][n_pairs] | flags[SLOTS][world]
  int* mc_base; int* const* peer_bases;
  int rank, world, gslot, epoch, n_pairs;
};

constexpr int XK_THREADS = 256;
constexpr int XK_COLS = 128;          // lines of the other side per streamed chunk
constexpr int XK_KC = 32;             // channels per streamed chunk
constexpr int XK_AS = MT_D + 4;       // row stride (floats) of the staged items: conflict-free float4 reads
constexpr int XK_BS = XK_KC + 4;      // row stride of the streamed chunk
constexpr int XK_SMEM = (XT_ITEMS * XK_AS + XK_COLS * XK_BS + 4 * XT_ITEMS * 2 + 2 * XT_ITEMS) * 4;
constexpr int XK_CTAS_PER_SM = 2;

__device__ __forceinline__ void lex_min(float& v, int& i, float ov, int oi) {
  if (ov < v || (ov == v && oi < i)) { v = ov; i = oi; }
}

// chunk (lines c0 .. c0 + 127 of the other side, channels k0 .. k0 + 31) -> 4 float4 per thread
__device__ __forceinline__ void xk_load_chunk(const MatchExactArgs& p, const float* __restrict__ B, int bb, int nb, int c0, int k0,
                                              float4 (&r)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int f = threadIdx.x + XK_THREADS * u;
    r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.layout == 0) {   // 8 lanes read one line's 128 contiguous bytes
      const int c = f >> 3, q = f & 7;
      if (c0 + c < nb) r[u] = __ldg(reinterpret_cast<const float4*>(B + (size_t)(bb + c0 + c) * MT_D + k0 + 4 * q));
    } else {               // lanes read consecutive lines of one channel
      const int c = f & (XK_COLS - 1), q = f >> 7;
      if (c0 + c < nb) {
        const float* y = B + (size_t)bb * MT_D + (size_t)(k0 + 4 * q) * nb + c0 + c;
        r[u] = make_float4(__ldg(y), __ldg(y + nb), __ldg(y + 2 * (size_t)nb), __ldg(y + 3 * (size_t)nb));
      }
    }
  }
}

__device__ __forceinline__ void xk_store_chunk(const MatchExactArgs& p, float* Bs, const float4 (&r)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int f = threadIdx.x + XK_THREADS * u;
    const int c = p.layout == 0 ? f >> 3 : f & (XK_COLS - 1);
    const int q = p.layout == 0 ? f & 7 : f >> 7;
    *reinterpret_cast<float4*>(Bs + c * XK_BS + 4 * q) = r[u];
  }
}

// The decisions of one pair that the tail left open, once every tile of the pair is done: side-0 rows with an
// exact argmin or an ambiguous partner column (matches0 / scores0 / counts) and ambiguous side-1 columns (nn1).
__device__ __forceinline__ void exact_finish_pair(const MatchExactArgs& p, int pair) {
  int b0, e0, b1, e1;
  image_range(p.cu[0], p.n[0], pair, b0, e0);
  image_range(p.cu[1], p.n[1], pair, b1, e1);
  const int n0 = e0 - b0, n1 = e1 - b1;
  int kept = 0;
  for (int i = threadIdx.x; i < n0; i += XK_THREADS) {
    const uint2 s = p.slot[0][b0 + i];
    float v = __uint_as_float(s.x);
    int idx = (int)(s.y & 0x7fffffffu);
    const bool hard = (s.y >> 31) || !(fabsf(v - p.thr) >= MATCH_EPS);
    if (hard) {
      const uint2 x = __ldcg(p.xq.res[0] + b0 + i);
      v = __uint_as_float(x.x);
      idx = (int)x.y;
    }
    bool keep = v < p.thr;   // strict '<' (nn_matcher.py:18)
    if (keep && p.mutual) {
      const uint2 t = p.slot[1][b1 + idx];
      if (!hard && !(t.y >> 31)) continue;   // decided by the tail
      const int back = (t.y >> 31) ? (int)__ldcg(p.xq.res[1] + b1 + idx).y : (int)(t.y & 0x7fffffffu);
      keep = back == i;
    } else if (!hard) {
      continue;
    }
    p.matches0[b0 + i] = keep ? idx : -1;
    p.scores0[b0 + i] = v;
    kept += keep;
  }
  if (p.mutual)
    for (int j = threadIdx.x; j < n1; j += XK_THREADS)
      if (p.slot[1][b1 + j].y >> 31) p.nn1[b1 + j] = (int)__ldcg(p.xq.res[1] + b1 + j).y;
  kept = __reduce_add_sync(0xffffffffu, kept);
  if ((threadIdx.x & 31) == 0 && kept) atomicAdd(&p.counts[pair], kept);
}

// The rank's counts to every rank over NVLink (whole block).
__device__ __forceinline__ void publish_counts(const MatchExactArgs& p) {
  __threadfence();
  const long long cnt_off = ((long long)p.gslot * p.world + p.rank) * p.n_pairs;
  const long long flag_off = (long long)GATHER_SLOTS * p.world * p.n_pairs + (long long)p.gslot * p.world + p.rank;
  for (int i = threadIdx.x; i < p.n_pairs; i += XK_THREADS) {
    const int v = __ldcg(p.counts + i);
    if (p.mc_base) multimem_st_u32(p.mc_base + cnt_off + i, v);
    else
      for (int r = 0; r < p.world; ++r) p.peer_bases[r][cnt_off + i] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    if (p.mc_base) multimem_st_u32(p.mc_base + flag_off, p.epoch);
    else
      for (int r = 0; r < p.world; ++r) *reinterpret_cast<volatile int*>(p.peer_bases[r] + flag_off) = p.epoch;
    __threadfence_system();
  }
}

// Persistent CTAs take tiles of the work list from an atomic queue.  A tile's items (up to 32 lines of side A)
// stay in shared memory; the other side's descriptors stream through shared memory in chunks of 128 lines x
// 32 channels.  Each thread owns 4 items x 4 lines of a chunk, every distance the ascending-k fmaf chain from 0
// (the arithmetic of the round-1 FFMA matcher), so distances, minima and first-minimum indices are bit-identical
// to a sequential fp32 evaluation.  The CTA that finishes a pair's last tile makes that pair's open decisions;
// with several GPUs, the CTA that finishes the last such pair (or CTA 0 if the list is empty) publishes the counts.
__global__ void __launch_bounds__(XK_THREADS, XK_CTAS_PER_SM) match_exact_kernel(MatchExactArgs p) {
  extern __shared__ __align__(16) float xk_smem[];
  float* As = xk_smem;                              // [XT_ITEMS][XK_AS]
  float* Bs = As + XT_ITEMS * XK_AS;                // [XK_COLS][XK_BS]
  float* red_v = Bs + XK_COLS * XK_BS;              // [4][XT_ITEMS] per column-group quarter
  int* red_i = reinterpret_cast<int*>(red_v + 4 * XT_ITEMS);
  float* s_sq = reinterpret_cast<float*>(red_i + 4 * XT_ITEMS);
  int* s_line = reinterpret_cast<int*>(s_sq + XT_ITEMS);
  __shared__ int s_tile, s_last, s_pub;
  pdl_launch_dependents();
  pdl_wait();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = p.xq.ctr[XQ_TILES];
  const int li = (lane >> 3) + 16 * (warp & 1);     // items li + 4 e, e = 0..3
  const int cq = warp >> 1;
  const int cg = cq * 8 + (lane & 7);               // lines c0 + cg + 32 e of each chunk
  for (;;) {
    if (tid == 0) s_tile = atomicAdd(&p.xq.ctr[XQ_HEAD], 1);
    __syncthreads();
    const int t = s_tile;
    if (t >= n_tiles) break;
    const ExactTile& T = p.xq.tiles[t];
    const int pair = T.pair, sa = T.side, sb = sa ^ 1, n = T.n;
    int ba, ea, bb, eb;
    image_range(p.cu[sa], p.n[sa], pair, ba, ea);
    image_range(p.cu[sb], p.n[sb], pair, bb, eb);
    const int na = ea - ba, nb = eb - bb;
    const float* __restrict__ A = p.d[sa];
    const float* __restrict__ B = p.d[sb];
    if (tid < XT_ITEMS) {
      const int r = tid < n ? T.line[tid] : 0;
      s_line[tid] = r;
      s_sq[tid] = (p.dist_mode == 1 && tid < n) ? p.sq[sa][ba + r] : 0.f;
    }
    __syncthreads();
    // stage the items (rows past n are zero)
    if (p.layout == 0) {
      for (int f = tid; f < XT_ITEMS * MT_D / 4; f += XK_THREADS) {
        const int it = f >> 6, q = f & 63;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (it < n) v = __ldg(reinterpret_cast<const float4*>(A + (size_t)(ba + s_line[it]) * MT_D) + q);
        *reinterpret_cast<float4*>(As + it * XK_AS + 4 * q) = v;
      }
    } else {
      for (int f = tid; f < XT_ITEMS * MT_D; f += XK_THREADS) {
        const int it = f >> 8, k = f & (MT_D - 1);
        As[it * XK_AS + k] = it < n ? __ldg(A + (size_t)ba * MT_D + (size_t)k * na + s_line[it]) : 0.f;
      }
    }
    float best[4], sqa[4];
    int bidx[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) { best[e] = INFINITY; bidx[e] = 0x7fffffff; }
    const bool live = 16 * (warp & 1) < n;          // warp-uniform: this warp's items exist
    float4 pre[4];
    xk_load_chunk(p, B, bb, nb, 0, 0, pre);
    for (int c0 = 0; c0 < nb; c0 += XK_COLS) {
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 1
      for (int k0 = 0; k0 < MT_D; k0 += XK_KC) {
        __syncthreads();                              // the previous chunk is consumed
        xk_store_chunk(p, Bs, pre);
        __syncthreads();
        const int nk = k0 + XK_KC == MT_D ? 0 : k0 + XK_KC, nc = nk ? c0 : c0 + XK_COLS;
        if (nc < nb) xk_load_chunk(p, B, bb, nb, nc, nk, pre);
        if (live) {
#pragma unroll
          for (int kq = 0; kq < XK_KC / 4; ++kq) {
            float4 a[4], b[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) a[e] = *reinterpret_cast<const float4*>(As + (li + 4 * e) * XK_AS + k0 + 4 * kq);
#pragma unroll
            for (int e = 0; e < 4; ++e) b[e] = *reinterpret_cast<const float4*>(Bs + (cg + 32 * e) * XK_BS + 4 * kq);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float c = acc[i][j];
                c = fmaf(a[i].x, b[j].x, c);
                c = fmaf(a[i].y, b[j].y, c);
                c = fmaf(a[i].z, b[j].z, c);
                c = fmaf(a[i].w, b[j].w, c);
                acc[i][j] = c;
              }
          }
        }
      }
      if (p.dist_mode == 1) {
#pragma unroll
        for (int i = 0; i < 4; ++i) sqa[i] = s_sq[li + 4 * i];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {                  // ascending lines: strict '<' keeps the first minimum
        const int c = c0 + cg + 32 * j;
        if (c < nb) {
          const float sqb = p.dist_mode == 1 ? p.sq[sb][bb + c] : 0.f;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float v = p.dist_mode == 1 ? fmaxf((sqa[i] + sqb) - 2.f * acc[i][j], 0.f) : fmaxf(2.f - 2.f * acc[i][j], 0.f);
            if (v < best[i]) { best[i] = v; bidx[i] = c; }
          }
        }
      }
    }
    // first minimum over the 32 column groups: 8 lanes of a warp, then the 4 warp pairs
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int o = 1; o < 8; o <<= 1)
        lex_min(best[i], bidx[i], __shfl_xor_sync(0xffffffffu, best[i], o), __shfl_xor_sync(0xffffffffu, bidx[i], o));
      if ((lane & 7) == 0) { red_v[cq * XT_ITEMS + li + 4 * i] = best[i]; red_i[cq * XT_ITEMS + li + 4 * i] = bidx[i]; }
    }
    __syncthreads();
    if (tid < n) {
      float v = red_v[tid];
      int ix = red_i[tid];
#pragma unroll
      for (int g = 1; g < 4; ++g) lex_min(v, ix, red_v[g * XT_ITEMS + tid], red_i[g * XT_ITEMS + tid]);
      p.xq.res[sa][ba + s_line[tid]] = make_uint2(__float_as_uint(v), (uint32_t)ix);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&p.xq.ctr[XQ_HDR + p.n_pairs + pair], 1) == p.xq.ctr[XQ_HDR + pair] - 1;
    __syncthreads();
    if (s_last) {
      __threadfence();
      exact_finish_pair(p, pair);
      if (p.world > 1) {
        __threadfence();
        __syncthreads();
        if (tid == 0) s_pub = atomicAdd(&p.xq.ctr[XQ_FINISHED], 1) == p.xq.ctr[XQ_PAIRS] - 1;
        __syncthreads();
        if (s_pub) publish_counts(p);
      }
    }
  }
  if (p.world > 1 && n_tiles == 0 && blockIdx.x == 0) publish_counts(p);
}

// one block: wait until every rank's flag of the slot reached `epoch`, then copy the gathered counts out
__global__ void __launch_bounds__(256) gather_wait_kernel(const int* base, int world, int n_pairs, int slot, int epoch, int* out) {
  pdl_launch_dependents();
  pdl_wait();
  const int* flags = base + (long long)GATHER_SLOTS * world * n_pairs + (long long)slot * world;
  if ((int)threadIdx.x < world) {
    const long long t0 = clock64();
    while (ld_acquire_sys(flags + threadIdx.x) < epoch)
      if (clock64() - t0 > 20000000000LL) __trap();   // ~10 s: a rank died - fail loudly instead of hanging
  }
  __syncthreads();
  const int* src = base + (long long)slot * world * n_pairs;
  for (int i = threadIdx.x; i < world * n_pairs; i += 256) out[i] = __ldcv(src + i);
}

}  // namespace ltr
