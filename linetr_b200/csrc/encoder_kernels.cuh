// CUDA-core kernels of the line-descriptor forward that are not GEMMs: the narrow head of the line
// positional encoder and the final L2 normalisation of the channel-first output.
#pragma once
#include "act_img.cuh"
#include "common.cuh"

namespace ltr {

// ------------------------------------------------------------------------------------
// Narrow head of the line positional encoder: 5 -> 32 -> 64 -> 128, eval-BatchNorm folded,
// ReLU after each layer.  Reference: MLP() models/line_transformer.py:9-20 as used by
// LinePositionalEncoder (:46-50, inputs: mid x, mid y, response, cos2t, sin2t), after
// normalize_keylines (:22-38).  One warp owns SM_ROWS rows at a time; weights live in shared memory.
struct SmallMlpWeights {
  const float* w1;  // [32][5]
  const float* b1;  // [32]
  const float* w2;  // [64][32]
  const float* b2;
  const float* w3;  // [128][64]
  const float* b3;
};

constexpr int SM_ROWS = 4;
constexpr int SM_WARPS = 8;
constexpr int SM_K2 = 32 + 4, SM_K3 = 64 + 4;  // padded leading dims (bank-conflict-free float4)

struct SmallMlpSmem {
  float w1[32 * 5];
  float b1[32], b2[64], b3[128];
  __align__(16) float w2[64 * SM_K2];
  __align__(16) float w3[128 * SM_K3];
  __align__(16) float h1[SM_WARPS][SM_ROWS][32];
  __align__(16) float h2[SM_WARPS][SM_ROWS][64];
};

// row = line, inputs sublines[row][2][2] (in0), resp[row] (in1), angle[row][2] (in2)
__global__ void __launch_bounds__(SM_WARPS * 32)
small_mlp_kernel(SmallMlpWeights w, const float* __restrict__ in0, const float* __restrict__ in1,
                 const float* __restrict__ in2, ActImg out, int rows, float cx, float cy,
                 float scale) {
  constexpr int IN = 5;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  auto& S = *reinterpret_cast<SmallMlpSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_launch_dependents();
  for (int i = tid; i < 32 * IN; i += blockDim.x) S.w1[i] = w.w1[i];
  for (int i = tid; i < 32; i += blockDim.x) S.b1[i] = w.b1[i];
  for (int i = tid; i < 64; i += blockDim.x) S.b2[i] = w.b2[i];
  for (int i = tid; i < 128; i += blockDim.x) S.b3[i] = w.b3[i];
  for (int i = tid; i < 64 * 32; i += blockDim.x) S.w2[(i >> 5) * SM_K2 + (i & 31)] = w.w2[i];
  for (int i = tid; i < 128 * 64; i += blockDim.x) S.w3[(i >> 6) * SM_K3 + (i & 63)] = w.w3[i];
  __syncthreads();
  pdl_wait();

  const int groups = (rows + SM_ROWS - 1) / SM_ROWS;
  for (int g = blockIdx.x * SM_WARPS + warp; g < groups; g += gridDim.x * SM_WARPS) {
    const int r0 = g * SM_ROWS;
    // layer 1: lane = output channel
    float x[SM_ROWS][IN];
#pragma unroll
    for (int r = 0; r < SM_ROWS; ++r) {
      int row = min(r0 + r, rows - 1);
      // normalise both end points first, then take the mid point (reference order)
      float ax = (in0[4 * row + 0] - cx) / scale, ay = (in0[4 * row + 1] - cy) / scale;
      float bx = (in0[4 * row + 2] - cx) / scale, by = (in0[4 * row + 3] - cy) / scale;
      x[r][0] = (ax + bx) / 2.f;
      x[r][1] = (ay + by) / 2.f;
      x[r][2] = in1[row];
      x[r][3] = in2[2 * row];
      x[r][4] = in2[2 * row + 1];
    }
#pragma unroll
    for (int r = 0; r < SM_ROWS; ++r) {
      float a = S.b1[lane];
#pragma unroll
      for (int i = 0; i < IN; ++i) a = fmaf(S.w1[lane * IN + i], x[r][i], a);
      S.h1[warp][r][lane] = fmaxf(a, 0.f);
    }
    __syncwarp();
    // layer 2: lane owns channels lane, lane+32
    {
      float acc[2][SM_ROWS];
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int r = 0; r < SM_ROWS; ++r) acc[j][r] = S.b2[lane + 32 * j];
#pragma unroll
      for (int k4 = 0; k4 < 8; ++k4) {
        float4 h[SM_ROWS];
#pragma unroll
        for (int r = 0; r < SM_ROWS; ++r) h[r] = *reinterpret_cast<const float4*>(&S.h1[warp][r][k4 * 4]);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          float4 ww = *reinterpret_cast<const float4*>(&S.w2[(lane + 32 * j) * SM_K2 + k4 * 4]);
#pragma unroll
          for (int r = 0; r < SM_ROWS; ++r) {
            acc[j][r] = fmaf(ww.x, h[r].x, acc[j][r]);
            acc[j][r] = fmaf(ww.y, h[r].y, acc[j][r]);
            acc[j][r] = fmaf(ww.z, h[r].z, acc[j][r]);
            acc[j][r] = fmaf(ww.w, h[r].w, acc[j][r]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int r = 0; r < SM_ROWS; ++r) S.h2[warp][r][lane + 32 * j] = fmaxf(acc[j][r], 0.f);
    }
    __syncwarp();
    // layer 3: lane owns channels lane + 32 j, j < 4
    {
      float acc[4][SM_ROWS];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int r = 0; r < SM_ROWS; ++r) acc[j][r] = S.b3[lane + 32 * j];
#pragma unroll 4
      for (int k4 = 0; k4 < 16; ++k4) {
        float4 h[SM_ROWS];
#pragma unroll
        for (int r = 0; r < SM_ROWS; ++r) h[r] = *reinterpret_cast<const float4*>(&S.h2[warp][r][k4 * 4]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 ww = *reinterpret_cast<const float4*>(&S.w3[(lane + 32 * j) * SM_K3 + k4 * 4]);
#pragma unroll
          for (int r = 0; r < SM_ROWS; ++r) {
            acc[j][r] = fmaf(ww.x, h[r].x, acc[j][r]);
            acc[j][r] = fmaf(ww.y, h[r].y, acc[j][r]);
            acc[j][r] = fmaf(ww.z, h[r].z, acc[j][r]);
            acc[j][r] = fmaf(ww.w, h[r].w, acc[j][r]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < SM_ROWS; ++r) {
        int row = r0 + r;
        if (row < rows) {
#pragma unroll
          for (int j = 0; j < 4; ++j) img_store1(out, row, lane + 32 * j, fmaxf(acc[j][r], 0.f));
        }
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------
// F.normalize(p=2, dim=channel, eps=1e-12) of the final projection
// (models/line_transformer.py:245-246) and the write of both output layouts:
// rows [n_lines, 256] and channel-first per image [256, L_i] (the reference's line_desc).
__global__ void __launch_bounds__(256)
final_norm_kernel(const float* __restrict__ y, float* __restrict__ out_rows, float* __restrict__ out_cf,
                  const int* __restrict__ cu, int lpi) {
  __shared__ float tile[32][257];
  pdl_launch_dependents();
  pdl_wait();
  int lb, le;
  image_range(cu, lpi, blockIdx.y, lb, le);
  const int L = le - lb, l0 = blockIdx.x * 32;
  if (l0 >= L) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int r = warp; r < 32; r += 8) {
    int li = l0 + r;
    if (li < L) {
      const float* p = y + (long long)(lb + li) * 256;
      float4 a = *reinterpret_cast<const float4*>(p + lane * 4);
      float4 b = *reinterpret_cast<const float4*>(p + 128 + lane * 4);
      float ss = a.x * a.x + a.y * a.y + a.z * a.z + a.w * a.w + b.x * b.x + b.y * b.y + b.z * b.z + b.w * b.w;
      ss = warp_sum(ss);
      float inv = 1.f / fmaxf(sqrtf(ss), 1e-12f);
      a.x *= inv; a.y *= inv; a.z *= inv; a.w *= inv;
      b.x *= inv; b.y *= inv; b.z *= inv; b.w *= inv;
      if (out_rows) {
        float* o = out_rows + (long long)(lb + li) * 256;
        *reinterpret_cast<float4*>(o + lane * 4) = a;
        *reinterpret_cast<float4*>(o + 128 + lane * 4) = b;
      }
      tile[r][lane * 4 + 0] = a.x; tile[r][lane * 4 + 1] = a.y; tile[r][lane * 4 + 2] = a.z; tile[r][lane * 4 + 3] = a.w;
      tile[r][128 + lane * 4 + 0] = b.x; tile[r][128 + lane * 4 + 1] = b.y;
      tile[r][128 + lane * 4 + 2] = b.z; tile[r][128 + lane * 4 + 3] = b.w;
    }
  }
  if (!out_cf) return;
  __syncthreads();
  float* base = out_cf + (long long)lb * 256;
  if (l0 + lane < L) {
    for (int c = warp; c < 256; c += 8) base[(long long)c * L + l0 + lane] = tile[lane][c];
  }
}

}  // namespace ltr
