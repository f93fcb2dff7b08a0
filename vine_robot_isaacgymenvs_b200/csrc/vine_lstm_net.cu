// vine_lstm_net.cu — the recurrent half of the reference's actor-critic on hand-written sm_100a kernels:
//   u = [MLP(x) (64) | x (32, padded)]  ->  LSTM 256 (gates = u W_ih^T + h W_hh^T + b, torch order i,f,g,o)  ->  LayerNorm
//   ->  mu (2), value (1)                                   (cfg/train/Vine5LinkMovingBasePPO.yaml:10-40, rl_games A2CBuilder)
//
// Data lives in HBM as 128-row tiles in the UMMA row-blocked layout (vine_umma.cuh), so every GEMM operand is one bulk-TMA
// copy and the same bytes serve forward (K-major) and backward/weight-gradient (MN-major) GEMMs:
//   U  [tile]        [128 x 128] bf16: cols 0..63 MLP output, 64..95 normalised observation (col 95 == 1), 96..127 zero
//   HM [tile][half]  [128 x 128] bf16: recurrent input of the step = not_done * h_prev (hidden units 128*half ..)
//   HH [tile][half]  [128 x 128] bf16: h of the step (input of LayerNorm and, masked, of the next step)
//   ACT[tile][piece] [128 x 64]  bf16: activated gates of 16 hidden units: [i(16) f(16) g(16) o(16)]   (saved for backward)
//   C  [n, 256] f32 row-major cell state
// Packed LSTM parameters (vine_lstm_pack): W_ih as 16 pieces [64 x 128] (piece p row g*16+k = gate g of hidden unit 16p+k,
// columns = U's columns), W_hh as [2 halves][16 pieces][64 x 128], then f32: bias (same row order), LayerNorm gamma/beta,
// head weights [3][256] (mu0, mu1, v) and head biases.
//
// vine_lstm_step  : one LSTM time step for every 128-sequence tile; CTA = (tile, half of the hidden units): resident A tile,
//                   weight pieces streamed through a bulk-TMA ring, tcgen05.mma into ping-pong TMEM accumulators, cell
//                   epilogue per row overlapped with the next piece (warp-specialised).
// vine_lstm_head  : LayerNorm + heads per row (one warp per row) + Gaussian sampling / neglogp (rollout).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "vine_device.cuh"
#include "vine_p2p.cuh"
#include "vine_mlp_common.cuh"
#include "vine_launch.cuh"

namespace {
using namespace vine_mlp;

constexpr int HID = 256, GATES = 4 * HID, UK = 128;            // U tile width
constexpr int PIECE_ROWS = 64, NPIECE = GATES / PIECE_ROWS;    // 16 pieces of 16 hidden units
constexpr int TILE_BYTES = TILE * UK * 2;                      // 32 KB: one [128 x 128] bf16 tile
constexpr int PIECE_BYTES = PIECE_ROWS * UK * 2;               // 16 KB: one [64 x 128] weight piece
constexpr int ACT_BYTES = TILE * PIECE_ROWS * 2;               // 16 KB: one [128 x 64] gate tile
constexpr int LP_WIH = 0;
constexpr int LP_WHH = LP_WIH + NPIECE * PIECE_BYTES;          // [half][piece]
constexpr int LP_BIAS = LP_WHH + 2 * NPIECE * PIECE_BYTES;     // f32 [1024] (piece row order)
constexpr int LP_LNG = LP_BIAS + GATES * 4;
constexpr int LP_LNB = LP_LNG + HID * 4;
constexpr int LP_WH = LP_LNB + HID * 4;                        // f32 [3][256]
constexpr int LP_BH = LP_WH + 3 * HID * 4;                     // f32 [4]
constexpr int LP_BYTES = LP_BH + 16;
static_assert(LP_BYTES == VINE_LSTM_PACKED_BYTES, "header constant out of date");

// packed gate row (piece, r) <-> torch gate row
__host__ __device__ inline int torch_gate_row(int packed_row) {
  const int p = packed_row / PIECE_ROWS, r = packed_row % PIECE_ROWS;
  return (r / 16) * HID + 16 * p + (r % 16);
}

__global__ void vine_lstm_pack_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b_ih,
                                      const float* __restrict__ b_hh, const float* __restrict__ ln_g, const float* __restrict__ ln_b,
                                      const float* __restrict__ w_mu, const float* __restrict__ b_mu, const float* __restrict__ w_v,
                                      const float* __restrict__ b_v, int O, uint8_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int in_w = H3 + O;   // torch W_ih is [1024, 64 + O]: MLP output first, then the observation (concat_input)
  if (i < GATES * UK) {      // W_ih pieces
    const int R = i / UK, c = i % UK, tr = torch_gate_row(R);
    float v = 0.f;
    if (c < H3) v = w_ih[tr * in_w + c];
    else if (c - H3 < O) v = w_ih[tr * in_w + c];
    *reinterpret_cast<__nv_bfloat16*>(out + LP_WIH + (R / PIECE_ROWS) * PIECE_BYTES + tile_offset(R % PIECE_ROWS, c, UK)) =
        __float2bfloat16_rn(v);
  }
  if (i < GATES * HID) {     // W_hh [half][piece]
    const int R = i / HID, c = i % HID, tr = torch_gate_row(R);
    *reinterpret_cast<__nv_bfloat16*>(out + LP_WHH + ((c / UK) * NPIECE + R / PIECE_ROWS) * PIECE_BYTES +
                                      tile_offset(R % PIECE_ROWS, c % UK, UK)) = __float2bfloat16_rn(w_hh[tr * HID + c]);
  }
  if (i < GATES) {
    const int tr = torch_gate_row(i);
    reinterpret_cast<float*>(out + LP_BIAS)[i] = b_ih[tr] + b_hh[tr];
  }
  if (i < HID) {
    reinterpret_cast<float*>(out + LP_LNG)[i] = ln_g[i];
    reinterpret_cast<float*>(out + LP_LNB)[i] = ln_b[i];
    reinterpret_cast<float*>(out + LP_WH)[i] = w_mu[i];
    reinterpret_cast<float*>(out + LP_WH)[HID + i] = w_mu[HID + i];
    reinterpret_cast<float*>(out + LP_WH)[2 * HID + i] = w_v[i];
  }
  if (i < 4) reinterpret_cast<float*>(out + LP_BH)[i] = i < 2 ? b_mu[i] : (i == 2 ? b_v[0] : 0.f);
}

// ---------------------------------------------------------------------------------------------------------------
// One MUFU each (tanh.approx.f32, max relative error 2^-11: below the bf16 rounding of every stored gate / hidden value;
// exp + reciprocal cost two per function, and the cell epilogue evaluates five per hidden unit).
__device__ __forceinline__ float tanh_(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_(float x) { return fmaf(tanh_(0.5f * x), 0.5f, 0.5f); }

// CTA = (tile of 128 sequences, half of the hidden units).  A = [U | HM] (96 KB) stays resident; the CTA's 8 weight pieces
// (16 hidden units x 4 gates each, 48 KB: W_ih piece + the two W_hh half pieces) stream through a 2-stage ring of bulk copies;
// the gate accumulators ping-pong between two TMEM buffers, so the tensor core works on piece p+1 and the copy engine on
// piece p+2 while the 8 epilogue warps run the cell update of piece p.  Warp 8 (one lane) is producer + MMA issuer.
constexpr int SO_U = 0, SO_HM = TILE_BYTES, SO_RING = 3 * TILE_BYTES, RING_STAGE = 3 * PIECE_BYTES, SO_BIAS = SO_RING + 2 * RING_STAGE;
constexpr int SO_BAR = SO_BIAS + 2048;
constexpr int STEP_SMEM = SO_BAR + 128;
constexpr int STEP_THREADS = THREADS + 32;

__global__ void __launch_bounds__(STEP_THREADS, 1) vine_lstm_step_kernel(const VineLstmStep a) {
  vine_launch::grid_dependency_sync();
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int tile = blockIdx.x;
  const int PIECES_PER_CTA = NPIECE / (int)gridDim.y;                // gridDim.y = 2 (8 pieces) or 4 (4 pieces: small batches)
  const uint32_t bar0 = smem_u32(smem + SO_BAR);
  const uint32_t bar_a = bar0, bar_hm = bar0 + 72u;                  // U + bias landed | HM landed
  auto full = [&](int st) { return bar0 + 8u + 8u * st; };           // ring stage filled
  auto done = [&](int st) { return bar0 + 24u + 8u * st; };          // ring stage consumed by the tensor core
  auto acc_full = [&](int b) { return bar0 + 40u + 8u * b; };        // accumulator buffer complete
  auto acc_empty = [&](int b) { return bar0 + 56u + 8u * b; };       // accumulator buffer drained by the epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SO_BAR + 96);
  const uint8_t* P = reinterpret_cast<const uint8_t*>(a.params);
  const int piece0 = (int)blockIdx.y * PIECES_PER_CTA, hf = piece0 / (NPIECE / 2);
  if (tid == 0) {
    mbar_init(bar_a, 1);
    mbar_init(bar_hm, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(full(i), 1); mbar_init(done(i), 1); mbar_init(acc_full(i), 1); mbar_init(acc_empty(i), 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 8) {
    if ((tid & 31) == 0) {
      auto load_b = [&](int p, int st) {
        const uint32_t dst = smem_u32(smem + SO_RING + st * RING_STAGE);
        mbar_expect_tx(full(st), RING_STAGE);
        bulk_g2s(dst, P + LP_WIH + (size_t)(piece0 + p) * PIECE_BYTES, PIECE_BYTES, full(st));
        bulk_g2s(dst + PIECE_BYTES, P + LP_WHH + (size_t)(piece0 + p) * PIECE_BYTES, PIECE_BYTES, full(st));
        bulk_g2s(dst + 2 * PIECE_BYTES, P + LP_WHH + (size_t)(NPIECE + piece0 + p) * PIECE_BYTES, PIECE_BYTES, full(st));
      };
      // K-chunked operand barriers: the first MMAs (U columns) start after U + the first weight piece, not after all 192 KB
      mbar_expect_tx(bar_a, TILE_BYTES + PIECES_PER_CTA * 256);
      bulk_g2s(smem_u32(smem + SO_U), reinterpret_cast<const uint8_t*>(a.u) + (size_t)tile * TILE_BYTES, TILE_BYTES, bar_a);
      bulk_g2s(smem_u32(smem + SO_BIAS), P + LP_BIAS + (size_t)piece0 * PIECE_ROWS * 4, PIECES_PER_CTA * 256, bar_a);
      load_b(0, 0);
      mbar_expect_tx(bar_hm, 2 * TILE_BYTES);
      bulk_g2s(smem_u32(smem + SO_HM), reinterpret_cast<const uint8_t*>(a.hm) + (size_t)tile * 2 * TILE_BYTES, 2 * TILE_BYTES, bar_hm);
      load_b(1, 1);
      mbar_wait(bar_a, 0);
      const uint32_t idesc = instr_desc(PIECE_ROWS, false, false);
      const Operand aU = k_major(smem_u32(smem + SO_U), UK), aH0 = k_major(smem_u32(smem + SO_HM), UK),
                    aH1 = k_major(smem_u32(smem + SO_HM + TILE_BYTES), UK);
      for (int p = 0; p < PIECES_PER_CTA; ++p) {
        const int st = p & 1;
        const uint32_t ph = (uint32_t)((p >> 1) & 1);
        mbar_wait(full(st), ph);
        if (p >= 2) mbar_wait(acc_empty(st), ph ^ 1u);     // completion #(p/2 - 1) of this buffer's drain
        fence_after_sync();
        const uint32_t base = smem_u32(smem + SO_RING + st * RING_STAGE), acc = tmem + 64u * st;
        mma_sequence(acc, aU, k_major(base, UK), idesc, 96 / 16, false);
        if (p == 0) {
          mbar_wait(bar_hm, 0);
          fence_after_sync();
        }
        mma_sequence(acc, aH0, k_major(base + PIECE_BYTES, UK), idesc, UK / 16, true);
        mma_sequence(acc, aH1, k_major(base + 2 * PIECE_BYTES, UK), idesc, UK / 16, true);
        mma_commit(acc_full(st));
        mma_commit(done(st));
        if (p + 2 < PIECES_PER_CTA) {
          mbar_wait(done(st), ph);
          load_b(p + 2, st);
        }
      }
    }
  } else {
    // ---- epilogue warps: thread = (sequence row, 8 of the piece's 16 hidden units) ----
    const int row = tid & 127, sub = tid >> 7;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int64_t s = (int64_t)tile * TILE + row;
    const bool valid = s < a.n;
    const float m = (valid && a.not_done) ? a.not_done[s] : 1.f;
    const float mn = (valid && a.not_done_next) ? a.not_done_next[s] : 1.f;
    mbar_wait(bar_a, 0);   // bias slice
    uint8_t* hh_t = reinterpret_cast<uint8_t*>(a.hh) + ((size_t)tile * 2 + hf) * TILE_BYTES;
    uint8_t* hm_t = a.hm_next ? reinterpret_cast<uint8_t*>(a.hm_next) + ((size_t)tile * 2 + hf) * TILE_BYTES : nullptr;
    // cell state of the next piece is fetched while the current one is processed (the load latency is otherwise exposed)
    float4 cq0 = make_float4(0.f, 0.f, 0.f, 0.f), cq1 = cq0;
    if (valid) {
      cq0 = *reinterpret_cast<const float4*>(a.c_prev + s * HID + 16 * piece0 + 8 * sub);
      cq1 = *reinterpret_cast<const float4*>(a.c_prev + s * HID + 16 * piece0 + 8 * sub + 4);
    }
#pragma unroll 1
    for (int p = 0; p < PIECES_PER_CTA; ++p) {
      const int b = p & 1;
      const float4 c0 = cq0, c1 = cq1;
      if (valid && p + 1 < PIECES_PER_CTA) {
        cq0 = *reinterpret_cast<const float4*>(a.c_prev + s * HID + 16 * (piece0 + p + 1) + 8 * sub);
        cq1 = *reinterpret_cast<const float4*>(a.c_prev + s * HID + 16 * (piece0 + p + 1) + 8 * sub + 4);
      }
      mbar_wait(acc_full(b), (uint32_t)((p >> 1) & 1));
      fence_after_sync();
      uint32_t gi[8], gf[8], gg[8], go[8];
      const uint32_t t0 = lane_base + 64u * b + 8u * sub;
      tmem_ld8_async(t0, gi);
      tmem_ld8_async(t0 + 16, gf);
      tmem_ld8_async(t0 + 32, gg);
      tmem_ld8_async(t0 + 48, go);
      tmem_wait8(gi, gf, gg, go);
      fence_before_sync();
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(acc_empty(b));   // this warp's lanes hold their accumulator values in registers
      if (!valid) continue;
      const int piece = piece0 + p, unit0 = 16 * piece + 8 * sub;
      const float* sb = reinterpret_cast<const float*>(smem + SO_BIAS) + p * PIECE_ROWS + 8 * sub;
      const float cp[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
      float cn[8], hn[8], ai[8], af[8], ag[8], ao[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        ai[k] = sigmoid_(__uint_as_float(gi[k]) + sb[k]);
        af[k] = sigmoid_(__uint_as_float(gf[k]) + sb[16 + k]);
        ag[k] = tanh_(__uint_as_float(gg[k]) + sb[32 + k]);
        ao[k] = sigmoid_(__uint_as_float(go[k]) + sb[48 + k]);
        cn[k] = fmaf(af[k], cp[k] * m, ai[k] * ag[k]);
        hn[k] = ao[k] * tanh_(cn[k]);
      }
      float* co = a.c + s * HID + unit0;
      *reinterpret_cast<float4*>(co) = make_float4(cn[0], cn[1], cn[2], cn[3]);
      *reinterpret_cast<float4*>(co + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
      const int off = tile_offset(row, unit0 % UK, UK);
      *reinterpret_cast<uint4*>(hh_t + off) =
          make_uint4(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]), pack_bf16(hn[4], hn[5]), pack_bf16(hn[6], hn[7]));
      if (hm_t)
        *reinterpret_cast<uint4*>(hm_t + off) = make_uint4(pack_bf16(hn[0] * mn, hn[1] * mn), pack_bf16(hn[2] * mn, hn[3] * mn),
                                                           pack_bf16(hn[4] * mn, hn[5] * mn), pack_bf16(hn[6] * mn, hn[7] * mn));
      if (a.act) {
        uint8_t* at = reinterpret_cast<uint8_t*>(a.act) + ((size_t)tile * NPIECE + piece) * ACT_BYTES;
        auto st8 = [&](int col, const float (&v)[8]) {
          *reinterpret_cast<uint4*>(at + tile_offset(row, col, PIECE_ROWS)) =
              make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
        };
        st8(8 * sub, ai);
        st8(16 + 8 * sub, af);
        st8(32 + 8 * sub, ag);
        st8(48 + 8 * sub, ao);
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem) : "memory");
}

// h tile rows -> masked copy (rollout: the done flag of the env step arrives after the LSTM step has run)
__global__ void vine_lstm_mask_kernel(const uint8_t* __restrict__ hh, const float* __restrict__ not_done, int64_t n, uint8_t* __restrict__ hm) {
  vine_launch::grid_dependency_sync();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte chunk (8 hidden units of one row)
  const int64_t chunks = ((n + TILE - 1) / TILE) * 2 * (TILE_BYTES / 16);
  if (i >= chunks) return;
  const int64_t tile = i / (2 * (TILE_BYTES / 16));
  const int within = (int)(i % (TILE_BYTES / 16));
  const int row = (within / 128) * 8 + (within % 8);   // chunk -> row of the row-blocked [128 x 128] tile
  const int64_t s = tile * TILE + row;
  const float m = (s < n) ? not_done[s] : 0.f;
  const uint4 v = reinterpret_cast<const uint4*>(hh)[i];
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 f = unpack_bf16(w[k]);
    o[k] = pack_bf16(f.x * m, f.y * m);
  }
  reinterpret_cast<uint4*>(hm)[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

// ---------------------------------------------------------------------------------------------------------------
// LayerNorm + heads, one warp per row; lane l owns hidden units [8l, 8l+8)
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(256) vine_lstm_head_kernel(const VineLstmHead a) {
  vine_launch::grid_dependency_sync();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const uint8_t* P = reinterpret_cast<const uint8_t*>(a.params);
  const float* lng = reinterpret_cast<const float*>(P + LP_LNG) + 8 * lane;
  const float* lnb = reinterpret_cast<const float*>(P + LP_LNB) + 8 * lane;
  const float* wh = reinterpret_cast<const float*>(P + LP_WH) + 8 * lane;
  const float* bh = reinterpret_cast<const float*>(P + LP_BH);
  float g[8], b[8], w0[8], w1[8], w2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) g[k] = lng[k], b[k] = lnb[k], w0[k] = wh[k], w1[k] = wh[HID + k], w2[k] = wh[2 * HID + k];
  const bool sample = a.actions != nullptr;
  const uint32_t ctr = (sample && a.rng_counter) ? *a.rng_counter : 0u;
  const float ls0 = sample ? a.logstd[0] : 0.f, ls1 = sample ? a.logstd[1] : 0.f;
  const float vmean = a.value_stats[0], vstd = a.value_stats[1];
  for (int64_t s = warp0; s < a.n; s += nwarps) {
    const int64_t tile = s / TILE;
    const int row = (int)(s % TILE), unit = 8 * lane;
    const uint4 hv = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(a.hh) + ((size_t)tile * 2 + unit / UK) * TILE_BYTES +
                                                     tile_offset(row, unit % UK, UK));
    const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
    float h[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = unpack_bf16(hw[k]);
      h[2 * k] = f.x, h[2 * k + 1] = f.y;
    }
    // same summation order as vine_lstm_head_train_kernel: the first training pass reproduces the rollout's mu bit for bit
    const float sm = ((h[0] + h[1]) + (h[2] + h[3])) + ((h[4] + h[5]) + (h[6] + h[7]));
    const float mean = wsum(sm) * (1.f / HID);
    float t[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) h[k] -= mean, t[k] = h[k] * h[k];
    const float sq = ((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]));
    const float rstd = rsqrtf(wsum(sq) * (1.f / HID) + 1e-5f);     // torch.nn.LayerNorm: biased variance, eps 1e-5
    float d0 = 0.f, d1 = 0.f, d2 = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float y = fmaf(h[k] * rstd, g[k], b[k]);
      d0 = fmaf(y, w0[k], d0), d1 = fmaf(y, w1[k], d1), d2 = fmaf(y, w2[k], d2);
    }
    const float mu0 = wsum(d0) + bh[0], mu1 = wsum(d1) + bh[1], v = wsum(d2) + bh[2];
    if (lane == 0) {
      const float value = fminf(fmaxf(v, -5.f), 5.f) * vstd + vmean;
      if (a.mu) *reinterpret_cast<float2*>(a.mu + 2 * s) = make_float2(mu0, mu1);
      if (a.value) a.value[s] = value;
      if (sample) {
        float z[4];
        normal4(philox4x32((uint32_t)a.seed, (uint32_t)(a.seed >> 32), (uint32_t)(a.global_env_offset + s), 16u, ctr, 0u), z);
        const float act0 = fmaf(__expf(ls0), z[0], mu0), act1 = fmaf(__expf(ls1), z[1], mu1);
        *reinterpret_cast<float2*>(a.actions + 2 * s) = make_float2(act0, act1);
        if (a.neglogp) a.neglogp[s] = 0.5f * (z[0] * z[0] + z[1] * z[1]) + 1.8378770664093453f + ls0 + ls1;
        if (a.env_actions)
          *reinterpret_cast<float2*>(a.env_actions + 2 * s) =
              make_float2(fminf(fmaxf(act0, -1.f), 1.f), fminf(fmaxf(act1, -1.f), 1.f));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Training: LayerNorm + heads forward, the PPO losses (same formulas as vine_ppo_minibatch_kernel), and their backward
// down to dh (one warp per row).  Parameter gradients accumulate in registers over the warp's rows, are combined per
// block in shared memory and written as one partial per block (`grads` [blocks][HG_FLOATS]; vine_lstm_reduce sums them).
constexpr int HG_LNG = 0, HG_LNB = HID, HG_WH = 2 * HID, HG_BH = 5 * HID, HG_LS = 5 * HID + 4, HG_STATS = 5 * HID + 6;
constexpr int HG_FLOATS = 5 * HID + 16;
static_assert(HG_FLOATS == VINE_LSTM_HEAD_GRAD_FLOATS, "header constant out of date");

// Latency, not arithmetic, bounds this kernel (≈350 warp-instructions per row in four dependent butterfly rounds): every
// warp keeps HT_ROWS rows in flight, the parameters live in shared memory (conflict-free float4 columns) instead of 40
// registers, and only A_j[k] = sum_rows d_j yh[k] (j = mu0, mu1, v) is accumulated per lane — the gradients of the
// LayerNorm gain/bias and of the head weights are linear in those sums and are assembled once per block at the end.
constexpr int HT_ROWS = 2;

__global__ void __launch_bounds__(256, 2) vine_lstm_head_train_kernel(const VineLstmHeadTrain a) {
  vine_launch::grid_dependency_sync();
  __shared__ float red[HG_FLOATS];
  __shared__ float4 prm[5][2][32];   // g, b, w0, w1, w2: [array][half of the lane's 8 units][lane]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const uint8_t* P = reinterpret_cast<const uint8_t*>(a.params);
  for (int i = threadIdx.x; i < 5 * 64; i += blockDim.x) {
    const int arr = i / 64, r = i % 64, l = r >> 1, half = r & 1;
    const float* src = arr == 0 ? reinterpret_cast<const float*>(P + LP_LNG)
                     : arr == 1 ? reinterpret_cast<const float*>(P + LP_LNB)
                                : reinterpret_cast<const float*>(P + LP_WH) + (arr - 2) * HID;
    prm[arr][half][l] = *reinterpret_cast<const float4*>(src + 8 * l + 4 * half);
  }
  for (int i = threadIdx.x; i < HG_FLOATS; i += blockDim.x) red[i] = 0.f;
  const float* bh = reinterpret_cast<const float*>(P + LP_BH);
  const float bh0_ = bh[0], bh1_ = bh[1], bh2_ = bh[2];
  float A[3][8];
#pragma unroll
  for (int j = 0; j < 3; ++j)
#pragma unroll
    for (int k = 0; k < 8; ++k) A[j][k] = 0.f;
  float sc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // dbh[3], dlogstd[2], a_loss, c_loss, kl, b_loss (same in every lane)
  const float ls0 = a.logstd[0], ls1 = a.logstd[1], lso0 = a.logstd_old[0], lso1 = a.logstd_old[1];
  const float sig0 = __expf(ls0), sig1 = __expf(ls1), sigo0 = __expf(lso0), sigo1 = __expf(lso1);
  // sigma is a parameter, not a per-row quantity: every division of the row math below is by one of these constants, so the
  // eight IEEE divisions per row (~17 dependent instructions each, in all 32 lanes) become multiplications
  const float inv_sig0 = 1.f / sig0, inv_sig1 = 1.f / sig1;
  // rl_games policy_kl(p0 = current policy, p1 = the policy the rows were last evaluated with), as in vine_ppo_minibatch_kernel
  const float klc0 = __logf(sigo0 / sig0 + 1e-5f) - 0.5f, klc1 = __logf(sigo1 / sig1 + 1e-5f) - 0.5f;
  const float klq0 = 1.f / (2.f * (sigo0 * sigo0 + 1e-5f)), klq1 = 1.f / (2.f * (sigo1 * sigo1 + 1e-5f));
  const float lo = 1.f - a.e_clip, hi = 1.f + a.e_clip;
  const bool clip_value = !a.value_loss_unclipped;   // rl_games clip_value
  __syncthreads();
  auto load8 = [&](int arr, float* v) {
    const float4 x = prm[arr][0][lane], y = prm[arr][1][lane];
    v[0] = x.x, v[1] = x.y, v[2] = x.z, v[3] = x.w, v[4] = y.x, v[5] = y.y, v[6] = y.z, v[7] = y.w;
  };
  for (int64_t s0 = warp0; s0 < a.n; s0 += HT_ROWS * nwarps) {
    int64_t srow[HT_ROWS];
    bool ok[HT_ROWS];
    size_t off[HT_ROWS];
    uint4 hv[HT_ROWS];
    float4 q0[HT_ROWS], q1[HT_ROWS];
#pragma unroll
    for (int r = 0; r < HT_ROWS; ++r) {   // every load of the rows in flight is issued before anything waits on one
      const int64_t s = s0 + r * nwarps;
      ok[r] = s < a.n;
      srow[r] = ok[r] ? s : s0;
      const int64_t tile = srow[r] / TILE;
      const int row = (int)(srow[r] % TILE), unit = 8 * lane;
      off[r] = ((size_t)tile * 2 + unit / UK) * TILE_BYTES + tile_offset(row, unit % UK, UK);
      hv[r] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(a.hh) + off[r]));
      const float4* q = reinterpret_cast<const float4*>(a.scalars + 8 * srow[r]);
      q0[r] = __ldg(q), q1[r] = __ldg(q + 1);
    }
    float yh[HT_ROWS][8], rstd[HT_ROWS], mean[HT_ROWS], sq[HT_ROWS];
#pragma unroll
    for (int r = 0; r < HT_ROWS; ++r) {
      const uint32_t hw[4] = {hv[r].x, hv[r].y, hv[r].z, hv[r].w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f = unpack_bf16(hw[k]);
        yh[r][2 * k] = f.x, yh[r][2 * k + 1] = f.y;
      }
      mean[r] = ((yh[r][0] + yh[r][1]) + (yh[r][2] + yh[r][3])) + ((yh[r][4] + yh[r][5]) + (yh[r][6] + yh[r][7]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r) mean[r] += __shfl_xor_sync(0xffffffffu, mean[r], o);
#pragma unroll
    for (int r = 0; r < HT_ROWS; ++r) {
      mean[r] *= (1.f / HID);
      float t[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) yh[r][k] -= mean[r], t[k] = yh[r][k] * yh[r][k];
      sq[r] = ((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r) sq[r] += __shfl_xor_sync(0xffffffffu, sq[r], o);
    float d[HT_ROWS][3];
    {
      float g[8], b[8], w0[8], w1[8], w2[8];
      load8(0, g), load8(1, b), load8(2, w0), load8(3, w1), load8(4, w2);
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r) {
        rstd[r] = rsqrtf(sq[r] * (1.f / HID) + 1e-5f);   // torch.nn.LayerNorm: biased variance, eps 1e-5
        d[r][0] = d[r][1] = d[r][2] = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          yh[r][k] *= rstd[r];
          const float y = fmaf(yh[r][k], g[k], b[k]);
          d[r][0] = fmaf(y, w0[k], d[r][0]), d[r][1] = fmaf(y, w1[k], d[r][1]), d[r][2] = fmaf(y, w2[k], d[r][2]);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r)
#pragma unroll
        for (int j = 0; j < 3; ++j) d[r][j] += __shfl_xor_sync(0xffffffffu, d[r][j], o);
    // ---- PPO losses and their gradient with respect to (mu0, mu1, v); every lane computes the same numbers ----
    float gr[HT_ROWS][3];
#pragma unroll
    for (int r = 0; r < HT_ROWS; ++r) {
      const float mu0 = d[r][0] + bh0_, mu1 = d[r][1] + bh1_, v = d[r][2] + bh2_;
      const float act0 = q0[r].x, act1 = q0[r].y, muo0 = q0[r].z, muo1 = q0[r].w, nlpo = q1[r].x, vo = q1[r].y, ret = q1[r].z, adv = q1[r].w;
      const float e0 = (act0 - mu0) * inv_sig0, e1 = (act1 - mu1) * inv_sig1;
      const float nlp = 0.5f * (e0 * e0 + e1 * e1) + 1.8378770664093453f + ls0 + ls1;
      const float ratio = __expf(nlpo - nlp);
      const float t1 = -adv * ratio, t2 = -adv * fminf(fmaxf(ratio, lo), hi);
      const bool inside = ratio >= lo && ratio <= hi;
      const float g_nlp = ((inside || t1 > t2) ? -adv : 0.f) * (-ratio);
      float dmu0 = g_nlp * (-e0 * inv_sig0), dmu1 = g_nlp * (-e1 * inv_sig1);
      const float dls0 = g_nlp * (1.f - e0 * e0) - a.entropy_coef, dls1 = g_nlp * (1.f - e1 * e1) - a.entropy_coef;
      const float dvo = v - vo, vclip = vo + fminf(fmaxf(dvo, -a.e_clip), a.e_clip);
      const float r1 = v - ret, r2 = vclip - ret, c1 = r1 * r1, c2 = r2 * r2;
      const float pass2 = (fabsf(dvo) <= a.e_clip) ? 1.f : 0.f;
      const float dvc = !clip_value ? 2.f * r1 : c1 > c2 ? 2.f * r1 : (c2 > c1 ? 2.f * r2 * pass2 : r1 + r2 * pass2);
      float dv = 0.5f * a.critic_coef * dvc;
      const float bh0 = fmaxf(mu0 - 1.1f, 0.f), bl0 = fminf(mu0 + 1.1f, 0.f), bh1 = fmaxf(mu1 - 1.1f, 0.f), bl1 = fminf(mu1 + 1.1f, 0.f);
      dmu0 += a.bounds_loss_coef * 2.f * (bh0 + bl0);
      dmu1 += a.bounds_loss_coef * 2.f * (bh1 + bl1);
      const float m0 = mu0 - muo0, m1 = mu1 - muo1;
      const float kl = klc0 + (sig0 * sig0 + m0 * m0) * klq0 + klc1 + (sig1 * sig1 + m1 * m1) * klq1;
      const float w = ok[r] ? a.inv_B : 0.f;   // a row past the end contributes nothing
      dmu0 *= w, dmu1 *= w, dv *= w;
      gr[r][0] = dmu0, gr[r][1] = dmu1, gr[r][2] = dv;
      sc[0] += dmu0, sc[1] += dmu1, sc[2] += dv;
      sc[3] += dls0 * w, sc[4] += dls1 * w;
      sc[5] += fmaxf(t1, t2) * w, sc[6] += (clip_value ? fmaxf(c1, c2) : c1) * w, sc[7] += kl * w;
      sc[8] += (bh0 * bh0 + bl0 * bl0 + bh1 * bh1 + bl1 * bl1) * w;
      if (lane == 0 && ok[r]) {
        const int64_t s = srow[r];
        if (a.mu_writeback) {   // dataset.update_mu_sigma: row s = [step l][chunk c][env e] of the minibatch -> row (c L + l, e0 + e) of [T, N, 8]
          const int64_t per_step = a.wb_chunks * a.wb_env_count;
          const int64_t l = s / per_step, rem = s - l * per_step, c = rem / a.wb_env_count, e = rem - c * a.wb_env_count;
          float* dst = a.mu_writeback + ((c * a.wb_seq_len + l) * a.wb_num_envs + a.wb_env_begin + e) * 8 + 2;
          *reinterpret_cast<float2*>(dst) = make_float2(mu0, mu1);
        }
        if (a.debug_out) {
          float* dd = a.debug_out + 4 * s;
          dd[0] = mu0, dd[1] = mu1, dd[2] = v, dd[3] = nlp;
        }
      }
    }
    // ---- backward: heads -> LayerNorm -> dh ----
    float dyh[HT_ROWS][8], s1[HT_ROWS], s2[HT_ROWS];
    {
      float g[8], w0[8], w1[8], w2[8];
      load8(0, g), load8(2, w0), load8(3, w1), load8(4, w2);
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r) {
        s1[r] = s2[r] = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float dy = fmaf(gr[r][0], w0[k], fmaf(gr[r][1], w1[k], gr[r][2] * w2[k]));
          A[0][k] = fmaf(gr[r][0], yh[r][k], A[0][k]);
          A[1][k] = fmaf(gr[r][1], yh[r][k], A[1][k]);
          A[2][k] = fmaf(gr[r][2], yh[r][k], A[2][k]);
          dyh[r][k] = dy * g[k];
          s1[r] += dyh[r][k], s2[r] = fmaf(dyh[r][k], yh[r][k], s2[r]);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
      for (int r = 0; r < HT_ROWS; ++r) {
        s1[r] += __shfl_xor_sync(0xffffffffu, s1[r], o);
        s2[r] += __shfl_xor_sync(0xffffffffu, s2[r], o);
      }
#pragma unroll
    for (int r = 0; r < HT_ROWS; ++r) {
      const float mean1 = s1[r] * (1.f / HID), mean2 = s2[r] * (1.f / HID);
      uint32_t o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        o[k] = pack_bf16(rstd[r] * (dyh[r][2 * k] - mean1 - yh[r][2 * k] * mean2),
                         rstd[r] * (dyh[r][2 * k + 1] - mean1 - yh[r][2 * k + 1] * mean2));
      if (ok[r]) *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(a.dh) + off[r]) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
  // ---- the parameter gradients from the sums: with y = yh g + b and dy = sum_j d_j w_j,
  //        d(gain)[k] = sum_j w_j[k] A_j[k]     d(bias)[k] = sum_j w_j[k] S_j     d(w_j)[k] = g[k] A_j[k] + b[k] S_j
  //      (S_j = sum_rows d_j = sc[0..2]); the 8 warps of the block take turns on the block's partial in shared memory ----
  {
    float g[8], b[8], w0[8], w1[8], w2[8];
    load8(0, g), load8(1, b), load8(2, w0), load8(3, w1), load8(4, w2);
    for (int w = 0; w < 8; ++w) {
      if (warp == w) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          red[HG_LNG + 8 * lane + k] += fmaf(w0[k], A[0][k], fmaf(w1[k], A[1][k], w2[k] * A[2][k]));
          red[HG_LNB + 8 * lane + k] += fmaf(w0[k], sc[0], fmaf(w1[k], sc[1], w2[k] * sc[2]));
          red[HG_WH + 8 * lane + k] += fmaf(g[k], A[0][k], b[k] * sc[0]);
          red[HG_WH + HID + 8 * lane + k] += fmaf(g[k], A[1][k], b[k] * sc[1]);
          red[HG_WH + 2 * HID + 8 * lane + k] += fmaf(g[k], A[2][k], b[k] * sc[2]);
        }
        if (lane == 0) {
          red[HG_BH] += sc[0], red[HG_BH + 1] += sc[1], red[HG_BH + 2] += sc[2];
          red[HG_LS] += sc[3], red[HG_LS + 1] += sc[4];
          red[HG_STATS] += sc[5], red[HG_STATS + 1] += sc[6], red[HG_STATS + 2] += sc[7], red[HG_STATS + 3] += sc[8];
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < HG_FLOATS; i += blockDim.x) a.grads[(size_t)blockIdx.x * HG_FLOATS + i] = red[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Backward of the cell (pointwise) on the tile layouts.
//   dh = dh_out + dh_rec ;  dc = dc_next + dh o (1 - tanh^2 c) ;  dG = (dc g i(1-i), dc c_in f(1-f), dc i (1-g^2), dh tanh(c) o(1-o))
//   dc_prev = dc f nd          (c_in = nd c_prev; dh_rec arrives already masked from vine_lstm_bwd_gemm)
// Thread mapping: block = (tile, piece of 16 hidden units), 512 threads; the four threads of a sequence row are neighbouring
// lanes (4 hidden units each) and a warp covers 8 consecutive rows, so a warp's loads fall into 8 (row-major f32 cell
// arrays) or 2 (row-blocked bf16 tiles) 128-byte lines instead of 32.
constexpr int CB_THREADS = 4 * TILE;

__global__ void __launch_bounds__(CB_THREADS) vine_lstm_cell_bwd_tiles_kernel(const VineLstmCellBwd a) {
  vine_launch::grid_dependency_sync();
  const int tile = blockIdx.x, piece = blockIdx.y, row = threadIdx.x >> 2, q = threadIdx.x & 3;
  const int64_t s = (int64_t)tile * TILE + row;
  if (s >= a.n) return;
  const int col = 4 * q, unit0 = 16 * piece + col;
  const uint8_t* at = reinterpret_cast<const uint8_t*>(a.act) + ((size_t)tile * NPIECE + piece) * ACT_BYTES;
  uint8_t* dg = reinterpret_cast<uint8_t*>(a.dg) + ((size_t)tile * NPIECE + piece) * ACT_BYTES;
  auto ld4 = [&](const uint8_t* p, float (&o)[4]) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 f0 = unpack_bf16(v.x), f1 = unpack_bf16(v.y);
    o[0] = f0.x, o[1] = f0.y, o[2] = f1.x, o[3] = f1.y;
  };
  auto ldf4 = [&](const float* p, float (&o)[4]) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = v.x, o[1] = v.y, o[2] = v.z, o[3] = v.w;
  };
  float gi[4], gf[4], gg[4], go[4], dh[4], cp[4], cc[4], dc[4] = {0.f, 0.f, 0.f, 0.f};
  ld4(at + tile_offset(row, col, PIECE_ROWS), gi);
  ld4(at + tile_offset(row, 16 + col, PIECE_ROWS), gf);
  ld4(at + tile_offset(row, 32 + col, PIECE_ROWS), gg);
  ld4(at + tile_offset(row, 48 + col, PIECE_ROWS), go);
  const size_t hoff = ((size_t)tile * 2 + unit0 / UK) * TILE_BYTES + tile_offset(row, unit0 % UK, UK);
  ld4(reinterpret_cast<const uint8_t*>(a.dh) + hoff, dh);
  if (a.dh_rec) {
    float dr[4];
    ld4(reinterpret_cast<const uint8_t*>(a.dh_rec) + hoff, dr);
#pragma unroll
    for (int k = 0; k < 4; ++k) dh[k] += dr[k];
  }
  const float m = a.not_done ? __ldg(a.not_done + s) : 1.f;
  ldf4(a.c_prev + s * HID + unit0, cp);
  ldf4(a.c + s * HID + unit0, cc);
  if (a.dc_next) ldf4(a.dc_next + s * HID + unit0, dc);
  float di[4], df[4], dgg[4], dob[4], dcp[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float t = tanh_(cc[k]);
    const float d = fmaf(dh[k] * go[k], 1.f - t * t, dc[k]);
    di[k] = d * gg[k] * gi[k] * (1.f - gi[k]);
    df[k] = d * cp[k] * m * gf[k] * (1.f - gf[k]);
    dgg[k] = d * gi[k] * (1.f - gg[k] * gg[k]);
    dob[k] = dh[k] * t * go[k] * (1.f - go[k]);
    dcp[k] = d * gf[k] * m;
  }
  auto st4 = [&](uint8_t* p, const float (&v)[4]) { *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3])); };
  st4(dg + tile_offset(row, col, PIECE_ROWS), di);
  st4(dg + tile_offset(row, 16 + col, PIECE_ROWS), df);
  st4(dg + tile_offset(row, 32 + col, PIECE_ROWS), dgg);
  st4(dg + tile_offset(row, 48 + col, PIECE_ROWS), dob);
  *reinterpret_cast<float4*>(a.dc_prev + s * HID + unit0) = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
}

// ---------------------------------------------------------------------------------------------------------------
// Backward data GEMM of one time step for a 128-sequence tile:  d[U(:, 0:64) | HM] = dG [128 x 1024] W  (reduction over the
// 1024 gate rows, streamed as 16 pieces of 64 through a 3-stage ring of bulk copies; W pieces are read as MN-major
// operands, i.e. the forward weights serve unchanged).  Outputs: dh3 (f32 [n, 64], the gradient of the MLP output) and the
// recurrent gradient for the previous step, masked with this step's not_done, as bf16 tiles.
constexpr int BG_STAGES = 3, BG_STAGE_BYTES = 4 * PIECE_BYTES;
constexpr int BG_BAR = BG_STAGES * BG_STAGE_BYTES;
constexpr int BG_SMEM = BG_BAR + 128;
constexpr uint32_t BG_TM_DU = 0, BG_TM_DH = 64;

__global__ void __launch_bounds__(THREADS, 1) vine_lstm_bwd_gemm_kernel(const VineLstmBwdGemm a) {
  vine_launch::grid_dependency_sync();
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & 127, half = tid >> 7;
  const int tile = blockIdx.x, part = blockIdx.y;          // part 0: d U(:, 0:64) and d HM half 0;  part 1: d HM half 1
  const uint32_t bar0 = smem_u32(smem + BG_BAR);          // full[3] | done[3] | final
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + BG_BAR + 64);
  const uint8_t* P = reinterpret_cast<const uint8_t*>(a.params);
  const uint8_t* DG = reinterpret_cast<const uint8_t*>(a.dg) + (size_t)tile * NPIECE * ACT_BYTES;
  auto full = [&](int st) { return bar0 + 8u * st; };
  auto done = [&](int st) { return bar0 + 24u + 8u * st; };
  const uint32_t fin = bar0 + 48u;
  auto load = [&](int p, int st) {
    const uint32_t dst = smem_u32(smem + st * BG_STAGE_BYTES);
    mbar_expect_tx(full(st), part == 0 ? 3 * PIECE_BYTES : 2 * PIECE_BYTES);
    bulk_g2s(dst, DG + (size_t)p * ACT_BYTES, ACT_BYTES, full(st));
    if (part == 0) {
      bulk_g2s(dst + PIECE_BYTES, P + LP_WIH + (size_t)p * PIECE_BYTES, PIECE_BYTES, full(st));
      bulk_g2s(dst + 2 * PIECE_BYTES, P + LP_WHH + (size_t)p * PIECE_BYTES, PIECE_BYTES, full(st));
    } else {
      bulk_g2s(dst + 3 * PIECE_BYTES, P + LP_WHH + (size_t)(NPIECE + p) * PIECE_BYTES, PIECE_BYTES, full(st));
    }
  };
  if (tid == 0) {
    for (int i = 0; i < 7; ++i) mbar_init(bar0 + 8u * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int p = 0; p < BG_STAGES; ++p) load(p, p);
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  if (tid == 0) {
    for (int p = 0; p < NPIECE; ++p) {
      const int st = p % BG_STAGES;
      const uint32_t ph = (uint32_t)((p / BG_STAGES) & 1);
      mbar_wait(full(st), ph);
      fence_after_sync();
      const uint32_t base = smem_u32(smem + st * BG_STAGE_BYTES);
      const Operand A = k_major(base, PIECE_ROWS);
      if (part == 0) {
        mma_sequence(tmem + BG_TM_DU, A, mn_major(base + PIECE_BYTES, UK), instr_desc(64, false, true), PIECE_ROWS / 16, p > 0);
        mma_sequence(tmem + BG_TM_DH, A, mn_major(base + 2 * PIECE_BYTES, UK), instr_desc(128, false, true), PIECE_ROWS / 16, p > 0);
      } else {
        mma_sequence(tmem + BG_TM_DH, A, mn_major(base + 3 * PIECE_BYTES, UK), instr_desc(128, false, true), PIECE_ROWS / 16, p > 0);
      }
      mma_commit(done(st));
      if (p + BG_STAGES < NPIECE) {
        mbar_wait(done(st), ph);
        load(p + BG_STAGES, st);
      }
    }
    mma_commit(fin);
  }
  mbar_wait(fin, 0);
  fence_after_sync();
  const int64_t s = (int64_t)tile * TILE + row;
  const float m = (s < a.n && a.not_done) ? a.not_done[s] : 1.f;
  if (part == 0) {
    uint32_t r[32];
    tmem_ld32(lane_base + BG_TM_DU + half * 32, r);
    if (s < a.n) {
      float4* dst = reinterpret_cast<float4*>(a.dh3 + s * H3 + half * 32);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
    }
  }
#pragma unroll 1
  for (int c0 = half * 64; c0 < half * 64 + 64; c0 += 32) {   // this thread: hidden units 128*part + c0 .. +31 of its row
    uint32_t r[32];
    tmem_ld32(lane_base + BG_TM_DH + c0, r);
    if (a.dh_rec && s < a.n) {
      uint8_t* dst = reinterpret_cast<uint8_t*>(a.dh_rec) + ((size_t)tile * 2 + part) * TILE_BYTES;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        *reinterpret_cast<uint4*>(dst + tile_offset(row, c0 + 8 * q, UK)) =
            make_uint4(pack_bf16(__uint_as_float(r[8 * q]) * m, __uint_as_float(r[8 * q + 1]) * m),
                       pack_bf16(__uint_as_float(r[8 * q + 2]) * m, __uint_as_float(r[8 * q + 3]) * m),
                       pack_bf16(__uint_as_float(r[8 * q + 4]) * m, __uint_as_float(r[8 * q + 5]) * m),
                       pack_bf16(__uint_as_float(r[8 * q + 6]) * m, __uint_as_float(r[8 * q + 7]) * m));
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// Weight gradients of the LSTM:  dW^T[f][R] = sum over all (step, sequence) rows of  in[row][f] * dG[row][R]
// with in = U (f = U column; column 95 == 1 carries the bias gradient) or HM half (f = hidden unit).  Both operands are the
// activation tiles read as MN-major operands (reduction over the tile's 128 rows).  CTA = (output block, K split):
// output block = (input part: U | HM0 | HM1) x (quarter of the gate rows = 4 pieces = 256 columns) -> [128 x 256] f32 in
// TMEM; the K range (row tiles) streams through a 2-stage ring of bulk copies.  Partials go to a workspace
// [split][12][128][256] that vine_lstm_reduce sums.
constexpr int WG_STAGES = 2, WG_STAGE_BYTES = TILE_BYTES + 4 * ACT_BYTES;   // 96 KB
constexpr int WG_BAR = WG_STAGES * WG_STAGE_BYTES;
constexpr int WG_SMEM = WG_BAR + 128;
constexpr int WG_BLOCKS = 12, WG_BLOCK_FLOATS = TILE * 256;

__global__ void __launch_bounds__(THREADS, 1) vine_lstm_wgrad_kernel(const VineLstmWgrad a) {
  vine_launch::grid_dependency_sync();
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & 127, half = tid >> 7;
  const int blk = blockIdx.x, sp = blockIdx.y, part = blk >> 2, nq = blk & 3;
  const int64_t per = (a.ntiles + gridDim.y - 1) / gridDim.y;
  const int64_t k0 = (int64_t)sp * per, k1 = (k0 + per < a.ntiles) ? k0 + per : a.ntiles;
  const uint32_t bar0 = smem_u32(smem + WG_BAR);          // full[2] | done[2] | final
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + WG_BAR + 64);
  auto full = [&](int st) { return bar0 + 8u * st; };
  auto done = [&](int st) { return bar0 + 16u + 8u * st; };
  const uint32_t fin = bar0 + 32u;
  auto load = [&](int64_t k, int st) {
    const uint32_t dst = smem_u32(smem + st * WG_STAGE_BYTES);
    const uint8_t* A = part == 0 ? reinterpret_cast<const uint8_t*>(a.u) + (size_t)k * TILE_BYTES
                                 : reinterpret_cast<const uint8_t*>(a.hm) + ((size_t)k * 2 + (part - 1)) * TILE_BYTES;
    mbar_expect_tx(full(st), WG_STAGE_BYTES);
    bulk_g2s(dst, A, TILE_BYTES, full(st));
    bulk_g2s(dst + TILE_BYTES, reinterpret_cast<const uint8_t*>(a.dg) + ((size_t)k * NPIECE + 4 * nq) * ACT_BYTES, 4 * ACT_BYTES, full(st));
  };
  if (tid == 0) {
    for (int i = 0; i < 5; ++i) mbar_init(bar0 + 8u * i, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int i = 0; i < WG_STAGES; ++i)
      if (k0 + i < k1) load(k0 + i, i);
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  if (tid == 0) {
    for (int64_t k = k0; k < k1; ++k) {
      const int it = (int)(k - k0), st = it % WG_STAGES;
      const uint32_t ph = (uint32_t)((it / WG_STAGES) & 1);
      mbar_wait(full(st), ph);
      fence_after_sync();
      const uint32_t base = smem_u32(smem + st * WG_STAGE_BYTES);
      const Operand A = mn_major(base, UK);
#pragma unroll 1
      for (int j = 0; j < 4; ++j)
        mma_sequence(tmem + 64 * j, A, mn_major(base + TILE_BYTES + j * ACT_BYTES, PIECE_ROWS), instr_desc(64, true, true), TILE / 16, it > 0);
      mma_commit(done(st));
      if (k + WG_STAGES < k1) {
        mbar_wait(done(st), ph);
        load(k + WG_STAGES, st);
      }
    }
    mma_commit(fin);
  }
  mbar_wait(fin, 0);
  fence_after_sync();
  float* out = a.workspace + ((size_t)sp * WG_BLOCKS + blk) * WG_BLOCK_FLOATS + (size_t)row * 256 + half * 128;
#pragma unroll 1
  for (int c0 = 0; c0 < 128; c0 += 32) {
    uint32_t r[32];
    if (k1 > k0) tmem_ld32(lane_base + half * 128 + c0, r);
    else {
#pragma unroll
      for (int i = 0; i < 32; ++i) r[i] = 0u;
    }
    float4* dst = reinterpret_cast<float4*>(out + c0);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// Flat f32 parameter vector of the recurrent half (torch layouts, this order):
//   W_ih[1024, 64+O]  W_hh[1024, 256]  b_ih[1024]  b_hh[1024]  ln_gamma[256]  ln_beta[256]  W_mu[2,256]  b_mu[2]  W_v[1,256]
//   b_v[1]  logstd[2]
__host__ __device__ inline int lstm_num_params(int O) { return GATES * (H3 + O) + GATES * HID + 2 * GATES + 2 * HID + 2 * HID + 2 + HID + 1 + 2; }
__host__ __device__ inline int packed_gate_row(int torch_row) {
  const int g_ = torch_row / HID, unit = torch_row % HID;
  return (unit / 16) * PIECE_ROWS + g_ * 16 + (unit % 16);
}

struct LstmSeg { int wih, whh, bih, bhh, lng, lnb, wmu, bmu, wv, bv, ls, end; };
__host__ __device__ inline LstmSeg lstm_segments(int O) {
  LstmSeg s;
  s.wih = 0; s.whh = s.wih + GATES * (H3 + O); s.bih = s.whh + GATES * HID; s.bhh = s.bih + GATES; s.lng = s.bhh + GATES;
  s.lnb = s.lng + HID; s.wmu = s.lnb + HID; s.bmu = s.wmu + 2 * HID; s.wv = s.bmu + 2; s.bv = s.wv + HID; s.ls = s.bv + 1; s.end = s.ls + 2;
  return s;
}

// sum of the head kernel's per-block partials: block = 4 slots, thread = every 128th partial
__global__ void __launch_bounds__(128) vine_lstm_head_sum_kernel(const float* __restrict__ hg, int parts, float* __restrict__ out) {
  vine_launch::grid_dependency_sync();
  __shared__ float red[4][4];
  const int slot0 = blockIdx.x * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = threadIdx.x; k < parts; k += 128) {
    const float4 v = *reinterpret_cast<const float4*>(hg + (size_t)k * HG_FLOATS + slot0);
    acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
  }
  acc.x = wsum(acc.x), acc.y = wsum(acc.y), acc.z = wsum(acc.z), acc.w = wsum(acc.w);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][0] = acc.x, red[threadIdx.x >> 5][1] = acc.y, red[threadIdx.x >> 5][2] = acc.z, red[threadIdx.x >> 5][3] = acc.w;
  __syncthreads();
  if (threadIdx.x < 4) out[slot0 + threadIdx.x] = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
}

// flat gradient vector from the weight-gradient partials: one thread per workspace slot (coalesced reads over the K splits),
// scattered write to the slot's parameter; the parameters fed by the head kernel come from the summed head buffer.
__global__ void __launch_bounds__(256) vine_lstm_reduce_kernel(const float* __restrict__ ws, int splits, const float* __restrict__ hsum, int O,
                                                               float* __restrict__ flat, const VineP2PChannel* ch) {
  vine_launch::grid_dependency_sync();
  if (ch) flat = p2p_local_buffer(ch);   // multi-GPU: straight into this rank's peer-visible buffer (vine_p2p.cuh)
  const LstmSeg sg = lstm_segments(O);
  const int PL = sg.end;
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  constexpr int SLOTS = WG_BLOCKS * WG_BLOCK_FLOATS;
  if (w < SLOTS) {
    const int blk = w / WG_BLOCK_FLOATS, f = (w % WG_BLOCK_FLOATS) / 256, R = (blk & 3) * 256 + (w & 255), part = blk >> 2;
    const int tr = torch_gate_row(R);
    int p = -1, p2 = -1;
    if (part == 0) {
      if (f < H3 + O) p = sg.wih + tr * (H3 + O) + f;
      else if (f == UK - 33) { p = sg.bih + tr; p2 = sg.bhh + tr; }     // U column 95 == 1: d(b_ih) == d(b_hh)
    } else {
      p = sg.whh + tr * HID + (part - 1) * UK + f;
    }
    if (p >= 0) {
      float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;   // fixed order: split k goes to accumulator k % 4
      int k = 0;
      for (; k + 3 < splits; k += 4) {   // four independent loads in flight per thread
        const float v0 = __ldg(ws + (size_t)k * SLOTS + w), v1 = __ldg(ws + (size_t)(k + 1) * SLOTS + w),
                    v2 = __ldg(ws + (size_t)(k + 2) * SLOTS + w), v3 = __ldg(ws + (size_t)(k + 3) * SLOTS + w);
        acc0 += v0, acc1 += v1, acc2 += v2, acc3 += v3;
      }
      if (k < splits) acc0 += __ldg(ws + (size_t)k * SLOTS + w);
      if (k + 1 < splits) acc1 += __ldg(ws + (size_t)(k + 1) * SLOTS + w);
      if (k + 2 < splits) acc2 += __ldg(ws + (size_t)(k + 2) * SLOTS + w);
      const float total = (acc0 + acc1) + (acc2 + acc3);
      flat[p] = total;
      if (p2 >= 0) flat[p2] = total;
    }
  } else {
    const int q = w - SLOTS;   // LayerNorm, heads, logstd, statistics
    if (q < HID) flat[sg.lng + q] = hsum[HG_LNG + q];
    else if (q < 2 * HID) flat[sg.lnb + q - HID] = hsum[HG_LNB + q - HID];
    else if (q < 4 * HID) flat[sg.wmu + q - 2 * HID] = hsum[HG_WH + q - 2 * HID];
    else if (q < 5 * HID) flat[sg.wv + q - 4 * HID] = hsum[HG_WH + 2 * HID + q - 4 * HID];
    else if (q < 5 * HID + 2) flat[sg.bmu + q - 5 * HID] = hsum[HG_BH + q - 5 * HID];
    else if (q == 5 * HID + 2) flat[sg.bv] = hsum[HG_BH + 2];
    else if (q < 5 * HID + 5) flat[sg.ls + q - 5 * HID - 3] = hsum[HG_LS + q - 5 * HID - 3];
    else if (q < 5 * HID + 9) flat[PL + q - 5 * HID - 5] = hsum[HG_STATS + q - 5 * HID - 5];
  }
  if (ch) p2p_producer_done(const_cast<VineP2PChannel*>(ch));
}

__global__ void vine_lstm_adam_kernel(const float* __restrict__ flat, float scale, float* __restrict__ params, float* __restrict__ m,
                                      float* __restrict__ v, uint8_t* __restrict__ packed, float* __restrict__ state, int O, float beta1,
                                      float beta2, float eps, const float* __restrict__ clip, VineP2PChannel* ch) {
  vine_launch::grid_dependency_sync();
  const int PL = lstm_num_params(O);
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  // multi-GPU: wait for every rank's gradient buffer, then read the sum over the ranks instead of `flat` (vine_p2p.cuh)
  __shared__ __align__(16) float s_g[256];
  const unsigned seq = ch ? p2p_exchange_begin(ch, false) : 0u;   // vine_lstm_reduce has published this rank's flag
  const int base = blockIdx.x * blockDim.x;
  if (ch) p2p_sum_block(ch, seq, base, min((int)blockDim.x, PL + 4 - base), s_g);
  if (p == PL) {   // loss statistics + the KL that drives the adaptive learning rate (state layout: vine_ppo_adam)
    float st4[4];
    if (ch && PL - base + 4 <= (int)blockDim.x) {   // already in this block's sums
      for (int j = 0; j < 4; ++j) st4[j] = s_g[PL - base + j];
    } else if (ch) {
      p2p_sum4(ch, seq, PL, st4);
    } else {
      st4[0] = flat[PL]; st4[1] = flat[PL + 1]; st4[2] = flat[PL + 2]; st4[3] = flat[PL + 3];
    }
    for (int j = 0; j < 4; ++j) state[4 + j] += st4[j] * scale;
    state[8] += 1.f;
    state[2] = st4[2] * scale;
    state[3] = 1.f;
  }
  const LstmSeg sg = lstm_segments(O);
  // b_hh[tr] is updated by the thread of b_ih[tr] (below), so that one thread writes the packed sum b_ih + b_hh
  if (p < PL && !(p >= sg.bhh && p < sg.lng)) {
  const float lr = state[0], step = state[1];
  const float bc1 = 1.f - powf(beta1, step), bc2 = 1.f - powf(beta2, step);
  auto adam = [&](float g, float& mq, float& vq, float& wq) {
    mq = beta1 * mq + (1.f - beta1) * g;
    vq = beta2 * vq + (1.f - beta2) * g * g;
    wq = wq - (lr / bc1) * mq / (sqrtf(vq) / sqrtf(bc2) + eps);
  };
  const bool bias = p >= sg.bih && p < sg.bhh;
  const int q = p + GATES;   // bias: b_hh of the same gate row
  const float cf = clip ? *clip : 1.f;   // vine_grad_clip's coefficient (exactly 1 below the threshold; g * 1 == g)
  float g = (ch ? s_g[threadIdx.x] : flat[p]) * scale;
  if (clip) g *= cf;
  float mp = m[p], vp = v[p], w = params[p], g2 = 0.f, mq = 0.f, vq = 0.f, w_hh = 0.f;
  if (bias) {   // the partner's operands are loaded with the thread's own: these blocks run last, one memory round trip
    g2 = (ch ? p2p_sum(ch, seq, q) : flat[q]) * scale;
    if (clip) g2 *= cf;
    mq = m[q], vq = v[q], w_hh = params[q];
  }
  adam(g, mp, vp, w);
  m[p] = mp;
  v[p] = vp;
  params[p] = w;
  if (p < sg.whh) {
    const int tr = p / (H3 + O), c = p % (H3 + O), R = packed_gate_row(tr);
    *reinterpret_cast<__nv_bfloat16*>(packed + LP_WIH + (R / PIECE_ROWS) * PIECE_BYTES + tile_offset(R % PIECE_ROWS, c, UK)) = __float2bfloat16_rn(w);
  } else if (p < sg.bih) {
    const int q = p - sg.whh, tr = q / HID, c = q % HID, R = packed_gate_row(tr);
    *reinterpret_cast<__nv_bfloat16*>(packed + LP_WHH + ((c / UK) * NPIECE + R / PIECE_ROWS) * PIECE_BYTES + tile_offset(R % PIECE_ROWS, c % UK, UK)) =
        __float2bfloat16_rn(w);
  } else if (bias) {
    // the kernels use b_ih + b_hh: this thread also updates b_hh[tr] and stores the sum as vine_lstm_pack computes it, so the
    // packed bias is fl(b_ih + b_hh) of the new parameters and the same bits on every run and every rank (the partner's
    // gradient is summed over the ranks in the same order as p2p_sum_block)
    adam(g2, mq, vq, w_hh);
    m[q] = mq;
    v[q] = vq;
    params[q] = w_hh;
    reinterpret_cast<float*>(packed + LP_BIAS)[packed_gate_row(p - sg.bih)] = w + w_hh;
  }
  if (p >= sg.lng) {
    float* f32 = nullptr;
    if (p < sg.lnb) f32 = reinterpret_cast<float*>(packed + LP_LNG) + (p - sg.lng);
    else if (p < sg.wmu) f32 = reinterpret_cast<float*>(packed + LP_LNB) + (p - sg.lnb);
    else if (p < sg.bmu) f32 = reinterpret_cast<float*>(packed + LP_WH) + (p - sg.wmu);
    else if (p < sg.wv) f32 = reinterpret_cast<float*>(packed + LP_BH) + (p - sg.bmu);
    else if (p < sg.bv) f32 = reinterpret_cast<float*>(packed + LP_WH) + 2 * HID + (p - sg.wv);
    else if (p < sg.ls) f32 = reinterpret_cast<float*>(packed + LP_BH) + 2;
    if (f32) *f32 = w;
  }
  }
  if (ch) p2p_exchange_end(ch);
}

// ---------------------------------------------------------------------------------------------------------------
// Minibatch assembly for the recurrent update in ONE launch: rows ordered [step in chunk][chunk, env] gathered from the
// [T, N] rollout buffers (observations, loss scalars, not_done), the initial cell state and the masked initial hidden-state
// tiles of every sequence (saved at the chunk starts of the rollout).
__global__ void __launch_bounds__(256) vine_lstm_gather_kernel(const VineLstmGather a) {
  vine_launch::grid_dependency_sync();
  const int64_t S = (int64_t)a.chunks * a.env_count;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // one piece of (obs | scalars | not_done) per thread: obs in float2 pieces when the width is even (8-byte aligned rows),
  // scalars as two float4, not_done as one float; the host checked that rows * pieces fits 32 bits
  const bool even = (a.num_obs & 1) == 0;
  const unsigned OP = even ? a.num_obs / 2 : a.num_obs, W = OP + 3;
  const unsigned rows = (unsigned)(a.seq_len * S);
  if (i < (int64_t)rows * W) {
    const unsigned iu = (unsigned)i, r = iu / W, c = iu - r * W, Su = (unsigned)S, t = r / Su, sq = r - t * Su;
    const unsigned ck = sq / (unsigned)a.env_count, e = (unsigned)a.env_begin + (sq - ck * (unsigned)a.env_count);
    const int64_t src = ((int64_t)ck * a.seq_len + t) * a.num_envs + e;
    if (c < OP) {
      if (even) reinterpret_cast<float2*>(a.mb_obs + (int64_t)r * a.num_obs)[c] = __ldg(reinterpret_cast<const float2*>(a.obs + src * a.num_obs) + c);
      else a.mb_obs[(int64_t)r * a.num_obs + c] = __ldg(a.obs + src * a.num_obs + c);
    } else if (c < OP + 2) {
      reinterpret_cast<float4*>(a.mb_scalars + (int64_t)r * 8)[c - OP] = __ldg(reinterpret_cast<const float4*>(a.scalars + src * 8) + (c - OP));
    } else {
      a.mb_not_done[r] = __ldg(a.not_done + src);
    }
  }
  // initial state: thread -> one 16-byte chunk (8 hidden units) of one sequence
  const int64_t nchunks = S * (HID / 8);
  if (i < nchunks) {
    const int64_t sq = i / (HID / 8);
    const int ug = (int)(i % (HID / 8)), unit0 = 8 * ug;
    const int ck = (int)(sq / a.env_count), el = (int)(sq % a.env_count), e = a.env_begin + el;
    const float m = a.not_done[((int64_t)ck * a.seq_len) * a.num_envs + e];
    // cell state rows
    const float4* cs = reinterpret_cast<const float4*>(a.c_saved + ((int64_t)ck * a.num_envs + e) * HID + unit0);
    float4* cd = reinterpret_cast<float4*>(a.c0 + sq * HID + unit0);
    cd[0] = cs[0], cd[1] = cs[1];
    // hidden state: saved tiles [chunk][N/128][2] -> masked tiles [S/128][2]
    const int64_t st = (int64_t)ck * (a.num_envs / TILE) + e / TILE, dt = sq / TILE;
    const int half = unit0 / UK, off_s = tile_offset(e % TILE, unit0 % UK, UK), off_d = tile_offset((int)(sq % TILE), unit0 % UK, UK);
    const uint4 v = *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(a.hh_saved) + (st * 2 + half) * TILE_BYTES + off_s);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 f = unpack_bf16(w[k]);
      o[k] = pack_bf16(f.x * m, f.y * m);
    }
    *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(a.hm0) + (dt * 2 + half) * TILE_BYTES + off_d) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

}  // namespace

extern "C" {

int vine_lstm_pack(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, const float* ln_gamma,
                   const float* ln_beta, const float* w_mu, const float* b_mu, const float* w_v, const float* b_v, int num_obs,
                   void* packed, void* stream) {
  if (!w_ih || !w_hh || !b_ih || !b_hh || !ln_gamma || !ln_beta || !w_mu || !b_mu || !w_v || !b_v || !packed || num_obs < 1 ||
      num_obs >= K1)
    return VINE_ERR_INVALID_ARG;
  const int total = GATES * HID;
  vine_lstm_pack_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w_ih, w_hh, b_ih, b_hh, ln_gamma, ln_beta, w_mu, b_mu,
                                                                             w_v, b_v, num_obs, (uint8_t*)packed);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_step(const VineLstmStep* a, void* stream) {
  if (!a || !a->params || !a->u || !a->hm || !a->c_prev || !a->c || !a->hh || a->n <= 0) return VINE_ERR_INVALID_ARG;
  if ((((uintptr_t)a->params) | ((uintptr_t)a->u) | ((uintptr_t)a->hm) | ((uintptr_t)a->hh) | ((uintptr_t)a->c_prev) |
       ((uintptr_t)a->c)) & 15u)
    return VINE_ERR_INVALID_ARG;
  static int configured = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (configured != dev) {
    if (cudaFuncSetAttribute(vine_lstm_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, STEP_SMEM) != cudaSuccess)
      return VINE_ERR_CUDA;
    configured = dev;
  }
  const unsigned tiles = (unsigned)((a->n + TILE - 1) / TILE);
  const dim3 grid(tiles, tiles * 2 <= 74 ? 4 : 2);   // small batches (rollout): 4 CTAs per tile to fill more SMs
  vine_launch::launch(vine_lstm_step_kernel, grid, STEP_THREADS, STEP_SMEM, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_mask(const void* hh, const float* not_done, int64_t n, void* hm, void* stream) {
  if (!hh || !not_done || !hm || n <= 0) return VINE_ERR_INVALID_ARG;
  const int64_t chunks = ((n + TILE - 1) / TILE) * 2 * (TILE_BYTES / 16);
  vine_launch::launch(vine_lstm_mask_kernel, (unsigned)((chunks + 255) / 256), 256, 0, (cudaStream_t)stream, (const uint8_t*)hh, not_done, n, (uint8_t*)hm);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_cell_bwd_tiles(const VineLstmCellBwd* a, void* stream) {
  if (!a || !a->act || !a->c_prev || !a->c || !a->dh || !a->dg || !a->dc_prev || a->n <= 0) return VINE_ERR_INVALID_ARG;
  const dim3 grid((unsigned)((a->n + TILE - 1) / TILE), NPIECE);
  vine_launch::launch(vine_lstm_cell_bwd_tiles_kernel, grid, CB_THREADS, 0, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_bwd_gemm(const VineLstmBwdGemm* a, void* stream) {
  if (!a || !a->params || !a->dg || !a->dh3 || a->n <= 0) return VINE_ERR_INVALID_ARG;
  static int configured = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (configured != dev) {
    if (cudaFuncSetAttribute(vine_lstm_bwd_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BG_SMEM) != cudaSuccess)
      return VINE_ERR_CUDA;
    configured = dev;
  }
  vine_launch::launch(vine_lstm_bwd_gemm_kernel, dim3((unsigned)((a->n + TILE - 1) / TILE), 2), THREADS, BG_SMEM, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_abi_struct_size(int which) {
  switch (which) {
    case 0: return (int)sizeof(VinePolicyAct);
    case 1: return (int)sizeof(VineRolloutPost);
    case 2: return (int)sizeof(VinePpoPrologue);
    case 3: return (int)sizeof(VinePpoMinibatch);
    case 4: return (int)sizeof(VineLstmStep);
    case 5: return (int)sizeof(VineLstmHead);
    case 6: return (int)sizeof(VineLstmHeadTrain);
    case 7: return (int)sizeof(VineLstmCellBwd);
    case 8: return (int)sizeof(VineLstmBwdGemm);
    case 9: return (int)sizeof(VineLstmWgrad);
    case 10: return (int)sizeof(VineLstmGather);
    default: return VINE_ERR_INVALID_ARG;
  }
}

int vine_lstm_gather(const VineLstmGather* a, void* stream) {
  if (!a || !a->obs || !a->scalars || !a->not_done || !a->c_saved || !a->hh_saved || !a->mb_obs || !a->mb_scalars || !a->mb_not_done ||
      !a->c0 || !a->hm0 || a->seq_len < 1 || a->chunks < 1 || a->env_count < 1 || a->env_begin < 0 ||
      a->env_begin + a->env_count > a->num_envs || a->num_envs % TILE || a->env_count % TILE || a->env_begin % TILE || a->num_obs < 1)
    return VINE_ERR_INVALID_ARG;
  const int64_t S = (int64_t)a->chunks * a->env_count, rows = (int64_t)a->seq_len * S;
  const int64_t pieces = ((a->num_obs & 1) ? a->num_obs : a->num_obs / 2) + 3;
  if (rows * pieces >= (int64_t)1 << 31) return VINE_ERR_INVALID_ARG;
  int64_t work = rows * pieces;
  if (S * (HID / 8) > work) work = S * (HID / 8);
  vine_launch::launch(vine_lstm_gather_kernel, (unsigned)((work + 255) / 256), 256, 0, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_num_params(int num_obs) { return (num_obs < 1 || num_obs >= K1) ? VINE_ERR_INVALID_ARG : lstm_num_params(num_obs); }

int vine_lstm_wgrad(const VineLstmWgrad* a, void* stream) {
  if (!a || !a->u || !a->hm || !a->dg || !a->workspace || a->ntiles <= 0 || a->splits < 1 || a->splits > a->ntiles)
    return VINE_ERR_INVALID_ARG;
  static int configured = -1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (configured != dev) {
    if (cudaFuncSetAttribute(vine_lstm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM) != cudaSuccess)
      return VINE_ERR_CUDA;
    configured = dev;
  }
  vine_launch::launch(vine_lstm_wgrad_kernel, dim3(WG_BLOCKS, (unsigned)a->splits), THREADS, WG_SMEM, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_reduce(const float* workspace, int splits, float* head_grads, int head_parts, int num_obs, float* flat, void* p2p_channel,
                     void* stream) {
  if (!workspace || !head_grads || (!flat && !p2p_channel) || splits < 1 || head_parts < 1 || head_parts > VINE_LSTM_HEAD_GRAD_PARTS || num_obs < 1 ||
      num_obs >= K1)
    return VINE_ERR_INVALID_ARG;
  const int n = lstm_num_params(num_obs) + 4;
  // the per-block partials of the head kernel are summed in parallel into the extra row [VINE_LSTM_HEAD_GRAD_PARTS]
  float* hsum = head_grads + (size_t)VINE_LSTM_HEAD_GRAD_PARTS * HG_FLOATS;
  vine_launch::launch(vine_lstm_head_sum_kernel, HG_FLOATS / 4, 128, 0, (cudaStream_t)stream, (const float*)head_grads, head_parts, hsum);
  const int threads = WG_BLOCKS * WG_BLOCK_FLOATS + 5 * HID + 9;
  (void)n;
  vine_launch::launch(vine_lstm_reduce_kernel, (threads + 255) / 256, 256, 0, (cudaStream_t)stream, workspace, splits, (const float*)hsum, num_obs, flat,
                      (const VineP2PChannel*)p2p_channel);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_adam_clipped(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed, float* state,
                           int num_obs, float beta1, float beta2, float eps, const float* clip_coef, void* p2p_channel, void* stream) {
  if ((!flat && !p2p_channel) || !params || !exp_avg || !exp_avg_sq || !packed || !state || num_obs < 1 || num_obs >= K1) return VINE_ERR_INVALID_ARG;
  const int n = lstm_num_params(num_obs) + 1;
  vine_launch::launch(vine_lstm_adam_kernel, (n + 255) / 256, 256, 0, (cudaStream_t)stream, flat, grad_scale, params, exp_avg, exp_avg_sq, (uint8_t*)packed,
                      state, num_obs, beta1, beta2, eps, clip_coef, (VineP2PChannel*)p2p_channel);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_lstm_adam(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed, float* state,
                   int num_obs, float beta1, float beta2, float eps, void* p2p_channel, void* stream) {
  return vine_lstm_adam_clipped(flat, grad_scale, params, exp_avg, exp_avg_sq, packed, state, num_obs, beta1, beta2, eps, nullptr,
                                p2p_channel, stream);
}

int vine_lstm_head_train(const VineLstmHeadTrain* a, void* stream) {
  if (!a || !a->params || !a->hh || !a->scalars || !a->logstd || !a->logstd_old || !a->dh || !a->grads || a->n <= 0)
    return VINE_ERR_INVALID_ARG;
  int64_t blocks = (a->n + 7) / 8;
  if (blocks > 296) blocks = 296;   // 2 resident blocks per SM (128 registers per thread), one wave; <= VINE_LSTM_HEAD_GRAD_PARTS
  vine_launch::launch(vine_lstm_head_train_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? (int)blocks : VINE_ERR_CUDA;   // number of gradient partials written
}

int vine_lstm_head(const VineLstmHead* a, void* stream) {
  if (!a || !a->params || !a->hh || !a->value_stats || a->n <= 0) return VINE_ERR_INVALID_ARG;
  if (a->actions && !a->logstd) return VINE_ERR_INVALID_ARG;
  int64_t blocks = (a->n + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  vine_launch::launch(vine_lstm_head_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

}  // extern "C"
