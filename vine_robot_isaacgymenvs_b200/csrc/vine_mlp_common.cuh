// vine_mlp_common.cuh — what the actor-critic MLP kernels share: the packed parameter block (bf16 weights in the UMMA
// row-blocked layout + f32 biases; written by vine_mlp_pack and vine_ppo_adam) and the per-row TMEM epilogues.
// Network: cfg/train/Vine5LinkMovingBasePPO.yaml:10-30 -- MLP [256,128,64] ELU, heads mu[2] + value[1] (padded to 16).
#pragma once
#include "../../include/vine_b200.h"
#include "vine_umma.cuh"

namespace vine_mlp {
using namespace vine_umma;

constexpr int H1 = 256, H2 = 128, H3 = 64, NH = 16, K1 = 32;
constexpr int TILE = 128, THREADS = 256;
// packed parameter block: identical to vine_mlp.cu (vine_mlp_pack / vine_mlp_forward share it)
constexpr int OFF_W1 = 0;
constexpr int OFF_W2 = OFF_W1 + H1 * K1 * 2;
constexpr int OFF_W3 = OFF_W2 + H2 * H1 * 2;
constexpr int OFF_W4 = OFF_W3 + H3 * H2 * 2;
constexpr int OFF_B = OFF_W4 + NH * H3 * 2;  // f32: b1[256] b2[128] b3[64] bh[16]
constexpr int PACKED_BYTES = OFF_B + (H1 + H2 + H3 + NH) * 4;
static_assert(PACKED_BYTES == VINE_MLP_PACKED_BYTES, "header constant out of date");
// shared-memory map common to the kernels: [packed block][x][h1][h2][h3]
constexpr int OFF_X = 102400;                      // x   [128 x 32]  bf16
constexpr int OFF_A1 = OFF_X + TILE * K1 * 2;      // h1 [128 x 256]
constexpr int OFF_A2 = OFF_A1 + TILE * H1 * 2;     // h2 [128 x 128]
constexpr int OFF_A3 = OFF_A2 + TILE * H2 * 2;     // h3 [128 x 64]
constexpr int OFF_END = OFF_A3 + TILE * H3 * 2;
static_assert(PACKED_BYTES <= OFF_X, "packed block overlaps the activation tiles");

// exp / reciprocal straight on the SFU (flush-to-zero variants: no denormal fix-up code around MUFU)
__device__ __forceinline__ float fast_exp(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float elu(float x) { return x > 0.f ? x : fast_exp(x) - 1.f; }

// 32 accumulator columns (already in registers) -> bias + ELU -> bf16 -> tile columns [c_out, c_out+32) of row `row`
template <int KL>
__device__ __forceinline__ void fwd_chunk(const uint32_t (&r)[32], int c_out, const float* bias, uint8_t* tile, int row) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + c_out + g * 8);
    const float4 b1 = *reinterpret_cast<const float4*>(bias + c_out + g * 8 + 4);
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      w[i] = pack_bf16(elu(__uint_as_float(r[g * 8 + 2 * i]) + bb[2 * i]), elu(__uint_as_float(r[g * 8 + 2 * i + 1]) + bb[2 * i + 1]));
    *reinterpret_cast<uint4*>(tile + tile_offset(row, c_out + g * 8, KL)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// accumulator columns [taddr, taddr+ncols) -> tile columns [c_out, c_out+ncols); ncols = 32 or 64 (both TMEM loads in flight)
// 8 accumulator columns -> bias + ELU -> bf16 -> one 16-byte chunk of the tile
template <int KL>
__device__ __forceinline__ void fwd_group8(const uint32_t* r, int c, const float* bias, uint8_t* tile, int row) {
  const float4 b0 = *reinterpret_cast<const float4*>(bias + c), b1 = *reinterpret_cast<const float4*>(bias + c + 4);
  *reinterpret_cast<uint4*>(tile + tile_offset(row, c, KL)) =
      make_uint4(pack_bf16(elu(__uint_as_float(r[0]) + b0.x), elu(__uint_as_float(r[1]) + b0.y)),
                 pack_bf16(elu(__uint_as_float(r[2]) + b0.z), elu(__uint_as_float(r[3]) + b0.w)),
                 pack_bf16(elu(__uint_as_float(r[4]) + b1.x), elu(__uint_as_float(r[5]) + b1.y)),
                 pack_bf16(elu(__uint_as_float(r[6]) + b1.z), elu(__uint_as_float(r[7]) + b1.w)));
}
template <int KL>
__device__ __forceinline__ void bwd_group8(const uint32_t* r, int c, uint8_t* tile, int row) {
  uint4* p = reinterpret_cast<uint4*>(tile + tile_offset(row, c, KL));
  const uint4 hv = *p;
  const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 h = unpack_bf16(hw[i]);
    w[i] = pack_bf16(__uint_as_float(r[2 * i]) * (h.x > 0.f ? 1.f : h.x + 1.f), __uint_as_float(r[2 * i + 1]) * (h.y > 0.f ? 1.f : h.y + 1.f));
  }
  *p = make_uint4(w[0], w[1], w[2], w[3]);
}

template <int KL>
__device__ __forceinline__ void fwd_epilogue(uint32_t taddr, int ncols, int c_out, const float* bias, uint8_t* tile, int row) {
  if (ncols == 16) {
    uint32_t r[16];
    tmem_ld16(taddr, r);
    fwd_group8<KL>(r, c_out, bias, tile, row);
    fwd_group8<KL>(r + 8, c_out + 8, bias, tile, row);
    return;
  }
  uint32_t r0[32], r1[32];
  tmem_ld32_async(taddr, r0);
  if (ncols > 32) {
    tmem_ld32_async(taddr + 32, r1);
    tmem_wait(r1);
  }
  tmem_wait(r0);
  fwd_chunk<KL>(r0, c_out, bias, tile, row);
  if (ncols > 32) fwd_chunk<KL>(r1, c_out + 32, bias, tile, row);
}

// dz = dh * ELU'(h) with ELU'(h) = h > 0 ? 1 : h + 1, written over h in place
template <int KL>
__device__ __forceinline__ void bwd_chunk(const uint32_t (&r)[32], int c_out, uint8_t* tile, int row) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint4* p = reinterpret_cast<uint4*>(tile + tile_offset(row, c_out + g * 8, KL));
    const uint4 hv = *p;
    const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 h = unpack_bf16(hw[i]);
      const float d0 = __uint_as_float(r[g * 8 + 2 * i]) * (h.x > 0.f ? 1.f : h.x + 1.f);
      const float d1 = __uint_as_float(r[g * 8 + 2 * i + 1]) * (h.y > 0.f ? 1.f : h.y + 1.f);
      w[i] = pack_bf16(d0, d1);
    }
    *p = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
template <int KL>
__device__ __forceinline__ void bwd_epilogue(uint32_t taddr, int ncols, int c_out, uint8_t* tile, int row) {
  if (ncols == 16) {
    uint32_t r[16];
    tmem_ld16(taddr, r);
    bwd_group8<KL>(r, c_out, tile, row);
    bwd_group8<KL>(r + 8, c_out + 8, tile, row);
    return;
  }
  uint32_t r0[32], r1[32];
  tmem_ld32_async(taddr, r0);
  if (ncols > 32) {
    tmem_ld32_async(taddr + 32, r1);
    tmem_wait(r1);
  }
  tmem_wait(r0);
  bwd_chunk<KL>(r0, c_out, tile, row);
  if (ncols > 32) bwd_chunk<KL>(r1, c_out + 32, tile, row);
}

// Reductions over the 128 rows of a row-blocked [128 x NC] bf16 tile by the 8 warps of the CTA: a warp owns whole
// 8-column groups (NC/64 of them); its lanes are 8 rows of a core matrix (128 contiguous bytes: conflict-free 16-byte
// loads) x 4 row-group phases, so one butterfly over the warp finishes the sum and lane 0 is the only writer of the
// result -- no shared-memory float atomics (those are CAS loops).
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// out[c] += sum over rows of tile[row][c]   (out: shared, f32, owned by this CTA)
template <int NC>
__device__ __forceinline__ void column_sums(const uint8_t* tile, float* out, int tid) {
  const int warp = tid >> 5, lane = tid & 31, r8 = lane & 7, ph = lane >> 3;
#pragma unroll
  for (int j = 0; j < NC / 64; ++j) {
    const int cg = warp * (NC / 64) + j;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int rg = ph; rg < TILE / 8; rg += 4) {
      const uint4 v = *reinterpret_cast<const uint4*>(tile + tile_offset(rg * 8 + r8, cg * 8, NC));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f = unpack_bf16(w[k]);
        acc[2 * k] += f.x, acc[2 * k + 1] += f.y;
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float t = warp_sum_f(acc[k]);
      if (lane == 0) out[cg * 8 + k] += t;
    }
  }
}

__device__ __forceinline__ float bf16_at(const uint8_t* tile, int row, int col, int KL) {
  return __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(tile + tile_offset(row, col, KL)));
}

// normalised observation row -> bf16 x tile (this thread: 16 of the 32 padded columns of its row); optionally copies
// the raw observation out (rollout buffer) and plants the constant 1 in column 31 (bias gradient through dW1).
// RAW (normalize_input off): x = obs as it is, mean / inv_std are not read and there is no clamp.  A template parameter, so
// the normalising instantiation is the same code whether or not the raw one exists.
template <int CPT = 16, bool RAW = false>   // columns per thread: 16 (two threads per row) or 8 (four threads per row)
__device__ __forceinline__ void build_x_tile(uint8_t* x_t, int row, int part, bool valid, const float* __restrict__ obs_row,
                                             const float* __restrict__ mean, const float* __restrict__ inv_std, int O,
                                             bool ones_column, float* __restrict__ obs_copy_row) {
  const int k0 = part * CPT;
  float x[CPT];
#pragma unroll
  for (int i = 0; i < CPT; ++i) {
    const int k = k0 + i;
    float v = 0.f;
    if (valid && k < O) {
      const float raw = obs_row[k];
      if (obs_copy_row) obs_copy_row[k] = raw;
      v = RAW ? raw : fminf(fmaxf((raw - mean[k]) * inv_std[k], -5.f), 5.f);
    }
    if (ones_column && valid && k == K1 - 1) v = 1.f;
    x[i] = v;
  }
#pragma unroll
  for (int g = 0; g < CPT / 8; ++g)
    *reinterpret_cast<uint4*>(x_t + tile_offset(row, k0 + g * 8, K1)) =
        make_uint4(pack_bf16(x[g * 8], x[g * 8 + 1]), pack_bf16(x[g * 8 + 2], x[g * 8 + 3]),
                   pack_bf16(x[g * 8 + 4], x[g * 8 + 5]), pack_bf16(x[g * 8 + 6], x[g * 8 + 7]));
}

}  // namespace vine_mlp
