// vine_ppo.cu — the PPO minibatch update of the actor-critic MLP as ONE fused tcgen05/TMEM kernel (sm_100a),
// plus the gradient reduction and the Adam step that re-packs the weights for the tensor cores.
//
// What it replaces (rl-games 1.5.2 A2CAgent.calc_gradients + torch autograd + torch.optim.Adam for the network of
// cfg/train/Vine5LinkMovingBasePPO.yaml:10-30; in-repo analogue isaacgymenvs/learning/common_agent.py:319-435,482-517):
//   forward  x -> ELU(W1 x+b1) -> ELU(W2 .+b2) -> ELU(W3 .+b3) -> (mu, v)
//   loss     clipped-ratio actor loss + clipped value loss * critic_coef/2 + bound loss - entropy (YP:61-81)
//   backward d(loss)/d(every parameter)
// One CTA owns a tile of 128 samples.  Weights (bf16, UMMA layout, 100 KB) and ALL activations of the tile
// (x, h1, h2, h3: 120 KB) stay resident in shared memory; every GEMM of the tile is a tcgen05.mma sequence:
//   forward      h_l   = h_{l-1} W_l^T        A = activations (K-major),  B = W_l (K-major)
//   backward     dh_l-1 = dz_l W_l            A = dz_l (K-major),         B = W_l (MN-major: same bytes, no W^T copy)
//   weight grad  dW_l += dz_l^T h_{l-1}       A = dz_l (MN-major),        B = h_{l-1} (MN-major): reduction over the
//                                             128 samples of the tile, accumulated in TMEM across the CTA's tiles
// dz_l overwrites h_l in place (ELU' is a function of the output), so nothing is ever written to HBM except the
// per-CTA gradient partials at the end.  TMEM: 128 columns of working accumulator + 384 columns of persistent
// weight-gradient accumulators (dW2 256, dW1 2x32, dW3^T 64) = all 512.  HBM traffic per sample: 72 B of observations
// + 32 B of rollout scalars in, nothing out.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#include "vine_mlp_common.cuh"
#include "vine_p2p.cuh"
#include "vine_launch.cuh"

namespace {
using namespace vine_mlp;

// shared-memory map
// (x column 31 == 1 carries db1 through dW1; dz_l overwrites h_l in place)
constexpr int OFF_DZH = OFF_END;                   // d(mu0,mu1,v) [128 x 16] bf16
constexpr int OFF_ACC = OFF_DZH + TILE * NH * 2;   // f32 accumulators over the CTA's tiles: db2[128] db3[64] dWh[3][64] dbh[3]
constexpr int ACC_B2 = 0, ACC_B3 = H2, ACC_WH = H2 + H3, ACC_BH = H2 + H3 + 3 * H3, ACC_FLOATS = 512;
constexpr int OFF_RED = OFF_ACC + ACC_FLOATS * 4;  // block-reduction scratch
constexpr int OFF_BAR = OFF_RED + 256;
constexpr int SMEM_BYTES = OFF_BAR + 64;
static_assert(SMEM_BYTES <= 232448, "shared-memory budget");
// TMEM columns
constexpr uint32_t TM_DATA = 0, TM_DW2 = 128, TM_DW1 = 384, TM_DW3T = 448;
// per-CTA gradient partial (floats)
constexpr int WS_W2 = 0;                  // [128 out][256 in]
constexpr int WS_W1 = WS_W2 + H2 * H1;    // [256 out][32 in], column 31 = db1
constexpr int WS_W3T = WS_W1 + H1 * K1;   // [128 in][64 out]
constexpr int WS_WH = WS_W3T + H2 * H3;   // [3][64]: mu0, mu1, v
constexpr int WS_BH = WS_WH + 3 * H3;     // [3] (+1 pad)
constexpr int WS_B2 = WS_BH + 4;
constexpr int WS_B3 = WS_B2 + H2;
constexpr int WS_STATS = WS_B3 + H3;      // a_loss, c_loss, kl, b_loss, dlogstd0, dlogstd1, -, -
constexpr int WS_FLOATS = 49664;
static_assert(WS_STATS + 8 <= WS_FLOATS && WS_FLOATS == VINE_PPO_WS_FLOATS, "workspace layout");
// device-resident optimiser state (floats): see include/vine_b200.h
constexpr int ST_LR = 0, ST_STEP = 1, ST_KL = 2, ST_PENDING = 3, ST_SUMS = 4 /* a,c,kl,b */, ST_COUNT = 8;
constexpr int ST_EPOCH = 11, ST_EKL_SUM = 12, ST_EKL_N = 13;   // iteration, KL sum / count of the current mini-epoch

struct MbArgs {
  const uint8_t* packed;
  const float *obs, *act, *nlp_old, *val_old, *ret, *adv, *obs_mean, *obs_inv_std, *logstd, *logstd_old;
  float* mu_old;   // in: the policy mean these rows were last evaluated with; out: this pass's mean (rl_games dataset.update_mu_sigma)
  float *ws, *state, *debug;
  const float* dh3_ext;   // recurrent network: d(loss)/d(h3) comes from the LSTM backward instead of the MLP heads
  int T, N, e0, E, O;
  float e_clip, critic_coef, entropy_coef, bounds_coef, inv_B, kl_threshold, lr_min, lr_max, lr0;
  int adaptive, linear, standard, epoch_begin, mini_epoch_begin, max_epochs, clip_value;
};

// One run of the learning-rate rule (rl_games scheduler.update) on the state block; `kl` is the rank-mean KL it acts on.
__device__ __forceinline__ void lr_schedule_rule(const MbArgs& a, float kl) {
  float lr = a.state[ST_LR];
  if (a.adaptive) {   // AdaptiveScheduler
    if (kl > 2.f * a.kl_threshold) lr = fmaxf(lr / 1.5f, a.lr_min);
    if (kl < 0.5f * a.kl_threshold) lr = fminf(lr * 1.5f, a.lr_max);
  } else if (a.linear) {   // LinearScheduler(use_epochs=True): in f64, one rounding to f32
    const double left = fmax((double)a.max_epochs - (double)a.state[ST_EPOCH], 0.0);
    lr = (float)((double)a.lr_min + ((double)a.lr0 - (double)a.lr_min) * (left / (double)a.max_epochs));
  }
  a.state[ST_LR] = lr;
}


// Q = epilogue threads per row (2 or 4): thread (row, part) owns the columns [part * N/Q, (part+1) * N/Q) of every N-wide
// accumulator; with Q = 4 the SM has 4 warps per sub-partition to hide the TMEM/shared-memory latencies of the epilogues.
// RAW_OBS: normalize_input off (VinePpoMinibatch.raw_obs), the observations enter as they are.
template <int Q, bool RAW_OBS>
__global__ void __launch_bounds__(128 * Q, 1) vine_ppo_minibatch_kernel(const MbArgs a) {
  vine_launch::grid_dependency_sync();
  extern __shared__ __align__(1024) uint8_t smem[];
  constexpr int C128 = 128 / Q, C64 = 64 / Q;
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & 127, part = tid >> 7;
  const uint32_t bar_w = smem_u32(smem + OFF_BAR), bar_mma = bar_w + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 16);
  const float* biases = reinterpret_cast<const float*>(smem + OFF_B);
  float* acc_s = reinterpret_cast<float*>(smem + OFF_ACC);
  for (int i = tid; i < ACC_FLOATS; i += 128 * Q) acc_s[i] = 0.f;

  if (tid == 0) {
    mbar_init(bar_w, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(bar_w, PACKED_BYTES);
    bulk_g2s(smem_u32(smem), a.packed, PACKED_BYTES, bar_w);   // ONE bulk TMA copy: all weights and biases
    if (blockIdx.x == 0) {
      // the learning-rate schedule acts between optimiser steps: `legacy` applies the KL of the previous minibatch now;
      // `standard` adds it to the mini-epoch's sum and applies the mean when a new mini-epoch opens.  Then count this
      // iteration (if it opens one) and this step.  The Adam kernel that follows in the stream reads both.
      if (a.state[ST_PENDING] != 0.f) {
        if (a.standard) {
          a.state[ST_EKL_SUM] += a.state[ST_KL];
          a.state[ST_EKL_N] += 1.f;
        } else {
          lr_schedule_rule(a, a.state[ST_KL]);
        }
        a.state[ST_PENDING] = 0.f;
      }
      if (a.standard && a.mini_epoch_begin && a.state[ST_EKL_N] > 0.f) {
        lr_schedule_rule(a, a.state[ST_EKL_SUM] / a.state[ST_EKL_N]);
        a.state[ST_EKL_SUM] = 0.f;
        a.state[ST_EKL_N] = 0.f;
      }
      if (a.epoch_begin) a.state[ST_EPOCH] += 1.f;
      a.state[ST_STEP] += 1.f;
    }
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);   // this warp's 32 TMEM lanes
  mbar_wait(bar_w, 0);

  uint8_t *x_t = smem + OFF_X, *a1_t = smem + OFF_A1, *a2_t = smem + OFF_A2, *a3_t = smem + OFF_A3, *dzh_t = smem + OFF_DZH;
  const uint32_t sW1 = smem_u32(smem + OFF_W1), sW2 = smem_u32(smem + OFF_W2), sW3 = smem_u32(smem + OFF_W3),
                 sW4 = smem_u32(smem + OFF_W4);
  const uint32_t sX = smem_u32(x_t), sA1 = smem_u32(a1_t), sA2 = smem_u32(a2_t), sA3 = smem_u32(a3_t), sDZH = smem_u32(dzh_t);
  uint32_t phase = 0;

  // One step of the tile's dependency chain: make this thread's smem writes visible to the tensor core, join the
  // CTA, let ONE thread issue the MMAs, optionally do CUDA-core work while they run, then wait for their completion.
  auto mma_step = [&](auto&& issue, auto&& overlap) {
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      issue();
      mma_commit(bar_mma);
    }
    overlap();
    mbar_wait(bar_mma, phase);
    phase ^= 1;
    fence_after_sync();
  };
  auto nothing = [] {};

  // persistent per-thread accumulators
  float st[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // a_loss, c_loss, kl, b_loss, dlogstd0, dlogstd1 (part 0 threads)

  const int64_t B = (int64_t)a.T * a.E;
  const int64_t ntiles = (B + TILE - 1) / TILE;
  const float ls0 = a.logstd[0], ls1 = a.logstd[1], lso0 = a.logstd_old[0], lso1 = a.logstd_old[1];
  const float sig0 = __expf(ls0), sig1 = __expf(ls1), sigo0 = __expf(lso0), sigo1 = __expf(lso1);
  // sigma is a parameter: the row math divides only by these constants, so its eight IEEE divisions become multiplications
  const float inv_sig0 = 1.f / sig0, inv_sig1 = 1.f / sig1;
  // rl_games torch_ext.policy_kl(p0 = current policy, p1 = the policy the rows were last evaluated with):
  //   log(sigma1 / sigma0 + 1e-5) + (sigma0^2 + (mu1 - mu0)^2) / (2 (sigma1^2 + 1e-5)) - 1/2, summed over the actions
  const float klc0 = __logf(sigo0 / sig0 + 1e-5f) - 0.5f, klc1 = __logf(sigo1 / sig1 + 1e-5f) - 0.5f;
  const float klq0 = 1.f / (2.f * (sigo0 * sigo0 + 1e-5f)), klq1 = 1.f / (2.f * (sigo1 * sigo1 + 1e-5f));
  bool first = true;

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, first = false) {
    const int64_t s = tile * TILE + row;
    const bool valid = s < B;
    const int64_t grow = valid ? (s / a.E) * (int64_t)a.N + a.e0 + (s % a.E) : 0;   // row in the [T, N] rollout buffers
    // rollout scalars of this sample (part 0 threads own the loss of their row)
    float act0 = 0.f, act1 = 0.f, muo0 = 0.f, muo1 = 0.f, nlpo = 0.f, vo = 0.f, ret = 0.f, adv = 0.f;
    if (part == 0 && valid && !a.dh3_ext) {
      const float2 av = *reinterpret_cast<const float2*>(a.act + 2 * grow);
      const float2 mv = *reinterpret_cast<const float2*>(a.mu_old + 2 * grow);
      act0 = av.x, act1 = av.y, muo0 = mv.x, muo1 = mv.y;
      nlpo = a.nlp_old[grow], vo = a.val_old[grow], ret = a.ret[grow], adv = a.adv[grow];
    }
    // ---- x tile: normalised observation, bf16, zero padded to K1; column 31 is the constant 1 (bias gradient) ----
    build_x_tile<K1 / Q, RAW_OBS>(x_t, row, part, valid, a.obs + grow * a.O, a.obs_mean, a.obs_inv_std, a.O, true, nullptr);
    // =============================== forward ===============================
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {   // layer 1 in two halves of 128 output features (working accumulator = 128 columns)
      mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sX, K1), k_major(sW1, K1, h * 128), instr_desc(128, false, false), K1 / 16, false); },
               nothing);
      fwd_epilogue<H1>(lane_base + TM_DATA + part * C128, C128, h * 128 + part * C128, biases, a1_t, row);
    }
    mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sA1, H1), k_major(sW2, H1), instr_desc(H2, false, false), H1 / 16, false); }, nothing);
    fwd_epilogue<H2>(lane_base + TM_DATA + part * C128, C128, part * C128, biases + H1, a2_t, row);
    mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sA2, H2), k_major(sW3, H2), instr_desc(H3, false, false), H2 / 16, false); }, nothing);
    fwd_epilogue<H3>(lane_base + TM_DATA + part * C64, C64, part * C64, biases + H1 + H2, a3_t, row);
    if (!a.dh3_ext) {
    mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sA3, H3), k_major(sW4, H3), instr_desc(NH, false, false), H3 / 16, false); }, nothing);
    // =============================== loss ===============================
    if (part == 0) {
      uint32_t r[16];
      tmem_ld16(lane_base + TM_DATA, r);
      const float* bh = biases + H1 + H2 + H3;
      const float mu0 = __uint_as_float(r[0]) + bh[0], mu1 = __uint_as_float(r[1]) + bh[1], v = __uint_as_float(r[2]) + bh[2];
      float dmu0 = 0.f, dmu1 = 0.f, dv = 0.f;
      if (valid) {
        const float d0 = (act0 - mu0) * inv_sig0, d1 = (act1 - mu1) * inv_sig1;
        const float nlp = 0.5f * (d0 * d0 + d1 * d1) + 1.8378770664093453f + ls0 + ls1;
        const float ratio = __expf(nlpo - nlp);
        const float lo = 1.f - a.e_clip, hi = 1.f + a.e_clip;
        const float t1 = -adv * ratio, t2 = -adv * fminf(fmaxf(ratio, lo), hi);
        const bool inside = ratio >= lo && ratio <= hi;
        const float g_nlp = ((inside || t1 > t2) ? -adv : 0.f) * (-ratio);
        dmu0 = g_nlp * (-d0 * inv_sig0);
        dmu1 = g_nlp * (-d1 * inv_sig1);
        float dls0 = g_nlp * (1.f - d0 * d0) - a.entropy_coef, dls1 = g_nlp * (1.f - d1 * d1) - a.entropy_coef;
        // clipped value loss (clip_value: True) or (ret - v)^2 (clip_value: False), both on normalised values
        const float dvo = v - vo, vclip = vo + fminf(fmaxf(dvo, -a.e_clip), a.e_clip);
        const float e1 = v - ret, e2 = vclip - ret, c1 = e1 * e1, c2 = e2 * e2;
        const float pass2 = (fabsf(dvo) <= a.e_clip) ? 1.f : 0.f;
        const float dvc = !a.clip_value ? 2.f * e1 : c1 > c2 ? 2.f * e1 : (c2 > c1 ? 2.f * e2 * pass2 : e1 + e2 * pass2);
        dv = 0.5f * a.critic_coef * dvc;
        // bound loss on mu (soft bound 1.1)
        const float bh0 = fmaxf(mu0 - 1.1f, 0.f), bl0 = fminf(mu0 + 1.1f, 0.f), bh1 = fmaxf(mu1 - 1.1f, 0.f), bl1 = fminf(mu1 + 1.1f, 0.f);
        dmu0 += a.bounds_coef * 2.f * (bh0 + bl0);
        dmu1 += a.bounds_coef * 2.f * (bh1 + bl1);
        const float m0 = mu0 - muo0, m1 = mu1 - muo1;
        const float kl = klc0 + (sig0 * sig0 + m0 * m0) * klq0 + klc1 + (sig1 * sig1 + m1 * m1) * klq1;
        // the next mini-epoch measures its KL against THIS pass (a2c_common train_epoch: dataset.update_mu_sigma(cmu, csigma))
        *reinterpret_cast<float2*>(a.mu_old + 2 * grow) = make_float2(mu0, mu1);
        st[0] += fmaxf(t1, t2) * a.inv_B;
        st[1] += (a.clip_value ? fmaxf(c1, c2) : c1) * a.inv_B;
        st[2] += kl * a.inv_B;
        st[3] += (bh0 * bh0 + bl0 * bl0 + bh1 * bh1 + bl1 * bl1) * a.inv_B;
        st[4] += dls0 * a.inv_B;
        st[5] += dls1 * a.inv_B;
        dmu0 *= a.inv_B, dmu1 *= a.inv_B, dv *= a.inv_B;
        if (a.debug) {
          float* d = a.debug + 4 * s;
          d[0] = mu0, d[1] = mu1, d[2] = v, d[3] = nlp;
        }
      }
      *reinterpret_cast<uint4*>(dzh_t + tile_offset(row, 0, NH)) = make_uint4(pack_bf16(dmu0, dmu1), pack_bf16(dv, 0.f), 0u, 0u);
      *reinterpret_cast<uint4*>(dzh_t + tile_offset(row, 8, NH)) = make_uint4(0u, 0u, 0u, 0u);
    }
    // =============================== backward ===============================
    // heads: dh3 = dzh Wh (reduction over the 16 padded head rows); meanwhile dWh = dzh^T h3 and dbh on CUDA cores
    mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sDZH, NH), mn_major(sW4, H3), instr_desc(H3, false, true), NH / 16, false); },
             [&] {   // warp w < 8 owns columns [8w, 8w+8) of h3; lanes = 8 rows x 4 row-group phases (see column_sums)
               if (warp < 8) {
               const int lane = tid & 31, r8 = lane & 7, ph = lane >> 3;
               float acc[3][8];
#pragma unroll
               for (int j = 0; j < 3; ++j)
#pragma unroll
                 for (int k = 0; k < 8; ++k) acc[j][k] = 0.f;
               float bsum[3] = {0.f, 0.f, 0.f};
#pragma unroll
               for (int rg = ph; rg < TILE / 8; rg += 4) {
                 const int r_ = rg * 8 + r8;
                 const uint4 hv = *reinterpret_cast<const uint4*>(a3_t + tile_offset(r_, warp * 8, H3));
                 const uint2 dv = *reinterpret_cast<const uint2*>(dzh_t + tile_offset(r_, 0, NH));
                 const float2 d01 = unpack_bf16(dv.x), d2_ = unpack_bf16(dv.y);
                 const float d[3] = {d01.x, d01.y, d2_.x};
                 const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
                 for (int k = 0; k < 4; ++k) {
                   const float2 h = unpack_bf16(hw[k]);
#pragma unroll
                   for (int j = 0; j < 3; ++j) {
                     acc[j][2 * k] = fmaf(d[j], h.x, acc[j][2 * k]);
                     acc[j][2 * k + 1] = fmaf(d[j], h.y, acc[j][2 * k + 1]);
                   }
                 }
#pragma unroll
                 for (int j = 0; j < 3; ++j) bsum[j] += d[j];
               }
#pragma unroll
               for (int j = 0; j < 3; ++j) {
#pragma unroll
                 for (int k = 0; k < 8; ++k) {
                   const float t = warp_sum_f(acc[j][k]);
                   if (lane == 0) acc_s[ACC_WH + j * H3 + warp * 8 + k] += t;
                 }
                 if (warp == 0) {   // every warp sees all 128 rows of dzh; one of them records the bias gradient
                   const float t = warp_sum_f(bsum[j]);
                   if (lane == 0) acc_s[ACC_BH + j] += t;
                 }
               }
               }
               __syncthreads();   // h3 is overwritten in place next
             });
    bwd_epilogue<H3>(lane_base + TM_DATA + part * C64, C64, part * C64, a3_t, row);   // dz3 over h3
    } else {
      // dz3 = dh3 (from the LSTM backward, f32 [T, N, 64], rows like obs) * ELU'(h3), written over h3 in place
      __syncthreads();   // every thread is past its h3 stores / the layer-3 accumulator reads
      uint32_t r[C64];
      if (valid) {
        const float4* src = reinterpret_cast<const float4*>(a.dh3_ext + grow * H3 + part * C64);
#pragma unroll
        for (int i = 0; i < C64 / 4; ++i) {
          const float4 v = src[i];
          r[4 * i] = __float_as_uint(v.x), r[4 * i + 1] = __float_as_uint(v.y), r[4 * i + 2] = __float_as_uint(v.z), r[4 * i + 3] = __float_as_uint(v.w);
        }
      } else {
#pragma unroll
        for (int i = 0; i < C64; ++i) r[i] = 0u;
      }
#pragma unroll
      for (int g = 0; g < C64 / 8; ++g) bwd_group8<H3>(r + 8 * g, part * C64 + 8 * g, a3_t, row);
    }
    // layer 3: dW3^T += h2^T dz3 (persistent), dh2 = dz3 W3; meanwhile db3 = column sums of dz3
    mma_step(
        [&] {
          mma_sequence(tmem + TM_DW3T, mn_major(sA2, H2), mn_major(sA3, H3), instr_desc(H3, true, true), TILE / 16, !first);
          mma_sequence(tmem + TM_DATA, k_major(sA3, H3), mn_major(sW3, H2), instr_desc(H2, false, true), H3 / 16, false);
        },
        [&] { if (warp < 8) column_sums<H3>(a3_t, acc_s + ACC_B3, tid); });
    bwd_epilogue<H2>(lane_base + TM_DATA + part * C128, C128, part * C128, a2_t, row);   // dz2 over h2
    // layer 2: dW2 += dz2^T h1 (persistent), dh1[:, 0:128] = dz2 W2[:, 0:128]; meanwhile db2
    mma_step(
        [&] {
          mma_sequence(tmem + TM_DW2, mn_major(sA2, H2), mn_major(sA1, H1), instr_desc(H1, true, true), TILE / 16, !first);
          mma_sequence(tmem + TM_DATA, k_major(sA2, H2), mn_major(sW2, H1, 0), instr_desc(128, false, true), H2 / 16, false);
        },
        [&] { if (warp < 8) column_sums<H2>(a2_t, acc_s + ACC_B2, tid); });
    bwd_epilogue<H1>(lane_base + TM_DATA + part * C128, C128, part * C128, a1_t, row);           // dz1[:, 0:128] over h1
    mma_step([&] { mma_sequence(tmem + TM_DATA, k_major(sA2, H2), mn_major(sW2, H1, 128), instr_desc(128, false, true), H2 / 16, false); },
             nothing);
    bwd_epilogue<H1>(lane_base + TM_DATA + part * C128, C128, 128 + part * C128, a1_t, row);     // dz1[:, 128:256]
    // layer 1: dW1 += dz1^T x (two halves of 128 output features; x column 31 == 1 gives db1)
    mma_step(
        [&] {
          mma_sequence(tmem + TM_DW1, mn_major(sA1, H1, 0), mn_major(sX, K1), instr_desc(K1, true, true), TILE / 16, !first);
          mma_sequence(tmem + TM_DW1 + K1, mn_major(sA1, H1, 128), mn_major(sX, K1), instr_desc(K1, true, true), TILE / 16, !first);
        },
        nothing);
  }

  // ---- per-CTA gradient partial: TMEM accumulators + register accumulators -> workspace ----
  float* ws = a.ws + (size_t)blockIdx.x * WS_FLOATS;
  {
    uint32_t r[32];
#pragma unroll 1
    for (int c0 = 0; c0 < 256 / Q; c0 += 32) {   // dW2: lane = output feature, 256 columns, this thread's share
      tmem_ld32(lane_base + TM_DW2 + part * (256 / Q) + c0, r);
      float4* dst = reinterpret_cast<float4*>(ws + WS_W2 + row * H1 + part * (256 / Q) + c0);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
    }
    if (part < 2) {   // dW1: accumulator h holds output features h*128 + lane, 32 columns
      tmem_ld32(lane_base + TM_DW1 + part * K1, r);
      float4* dst = reinterpret_cast<float4*>(ws + WS_W1 + (part * 128 + row) * K1);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
    } else {          // (warp-uniform: whole warps share `part`)
    }
    if (Q == 2 || part >= 2) {   // dW3^T: lane = input feature, 64 columns: two threads x 32
      const int hsel = Q == 2 ? part : part - 2;
      tmem_ld32(lane_base + TM_DW3T + hsel * 32, r);
      float4* dst = reinterpret_cast<float4*>(ws + WS_W3T + row * H3 + hsel * 32);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
    }
  }
  __syncthreads();   // the last tile's shared-memory atomics
  if (tid < H2) ws[WS_B2 + tid] = acc_s[ACC_B2 + tid];
  else if (tid < H2 + H3) ws[WS_B3 + tid - H2] = acc_s[ACC_B3 + tid - H2];
  if (tid < 3 * H3) ws[WS_WH + tid] = acc_s[ACC_WH + tid];
  else if (tid < 3 * H3 + 3) ws[WS_BH + tid - 3 * H3] = acc_s[ACC_BH + tid - 3 * H3];
  // loss statistics + d(logstd): reduce over the 128 sample-owning threads
  float* red = reinterpret_cast<float*>(smem + OFF_RED);
  if (part == 0) {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      float v = st[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((tid & 31) == 0) red[warp * 8 + j] = v;
    }
  }
  fence_before_sync();
  __syncthreads();
  if (tid < 6) ws[WS_STATS + tid] = red[tid] + red[8 + tid] + red[16 + tid] + red[24 + tid];
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// flat parameter vector (torch layouts): W1[256,O] b1[256] W2[128,256] b2[128] W3[64,128] b3[64] Wmu[2,64] bmu[2]
// Wv[1,64] bv[1] logstd[2].  For parameter p: where its gradient sits in a CTA partial, and where its tensor-core
// copy sits in the packed block (bf16 weight / f32 bias; -1 = none).
__host__ __device__ inline int num_params(int O) { return H1 * O + H1 + H2 * H1 + H2 + H3 * H2 + H3 + 2 * H3 + 2 + H3 + 1 + 2; }

__device__ inline void param_map(int p, int O, int& ws_off, int& pk_off, bool& pk_is_f32) {
  pk_is_f32 = false;
  int q = p;
  if (q < H1 * O) { const int o = q / O, i = q % O; ws_off = WS_W1 + o * K1 + i; pk_off = OFF_W1 + tile_offset(o, i, K1); return; }
  q -= H1 * O;
  if (q < H1) { ws_off = WS_W1 + q * K1 + (K1 - 1); pk_off = OFF_B + 4 * q; pk_is_f32 = true; return; }
  q -= H1;
  if (q < H2 * H1) { const int o = q / H1, i = q % H1; ws_off = WS_W2 + o * H1 + i; pk_off = OFF_W2 + tile_offset(o, i, H1); return; }
  q -= H2 * H1;
  if (q < H2) { ws_off = WS_B2 + q; pk_off = OFF_B + 4 * (H1 + q); pk_is_f32 = true; return; }
  q -= H2;
  if (q < H3 * H2) { const int o = q / H2, i = q % H2; ws_off = WS_W3T + i * H3 + o; pk_off = OFF_W3 + tile_offset(o, i, H2); return; }
  q -= H3 * H2;
  if (q < H3) { ws_off = WS_B3 + q; pk_off = OFF_B + 4 * (H1 + H2 + q); pk_is_f32 = true; return; }
  q -= H3;
  if (q < 2 * H3) { ws_off = WS_WH + q; pk_off = OFF_W4 + tile_offset(q / H3, q % H3, H3); return; }
  q -= 2 * H3;
  if (q < 2) { ws_off = WS_BH + q; pk_off = OFF_B + 4 * (H1 + H2 + H3 + q); pk_is_f32 = true; return; }
  q -= 2;
  if (q < H3) { ws_off = WS_WH + 2 * H3 + q; pk_off = OFF_W4 + tile_offset(2, q, H3); return; }
  q -= H3;
  if (q < 1) { ws_off = WS_BH + 2; pk_off = OFF_B + 4 * (H1 + H2 + H3 + 2); pk_is_f32 = true; return; }
  q -= 1;
  ws_off = WS_STATS + 4 + q;
  pk_off = -1;
}

// inverse of param_map: which parameter (or statistic, as P + j) a workspace slot carries; -1 = padding
__device__ inline int ws_to_param(int w, int O) {
  const int P = num_params(O);
  const int bW1 = 0, bb1 = H1 * O, bW2 = bb1 + H1, bb2 = bW2 + H2 * H1, bW3 = bb2 + H2, bb3 = bW3 + H3 * H2, bWmu = bb3 + H3,
            bbmu = bWmu + 2 * H3, bWv = bbmu + 2, bbv = bWv + H3;
  if (w < WS_W1) return bW2 + w;
  if (w < WS_W3T) { const int r = w - WS_W1, o = r / K1, i = r % K1; return i < O ? bW1 + o * O + i : (i == K1 - 1 ? bb1 + o : -1); }
  if (w < WS_WH) { const int r = w - WS_W3T, i = r / H3, o = r % H3; return bW3 + o * H2 + i; }
  if (w < WS_BH) { const int r = w - WS_WH; return r < 2 * H3 ? bWmu + r : bWv + (r - 2 * H3); }
  if (w < WS_B2) { const int r = w - WS_BH; return r < 2 ? bbmu + r : (r == 2 ? bbv : -1); }
  if (w < WS_B3) return bb2 + (w - WS_B2);
  if (w < WS_STATS) return bb3 + (w - WS_B3);
  const int r = w - WS_STATS;
  return r < 4 ? P + r : (r < 6 ? P - 2 + (r - 4) : -1);
}

// flat[p] = sum over CTA partials (parameter order); flat[P + j] = loss statistics j (a_loss, c_loss, kl, b_loss).
// One workspace slot per (x) thread so the partial reads are coalesced, RED_SPLIT threads share a slot's partials.
constexpr int RED_SLOTS = 64, RED_SPLIT = 4;
__global__ void __launch_bounds__(RED_SLOTS* RED_SPLIT) vine_ppo_reduce_kernel(const float* __restrict__ ws, int n_partials, int O,
                                                                               float* __restrict__ flat, const float* __restrict__ logstd,
                                                                               float* __restrict__ logstd_old_out, const VineP2PChannel* ch) {
  vine_launch::grid_dependency_sync();
  if (ch) { flat = p2p_local_buffer(ch); p2p_producer_begin(const_cast<VineP2PChannel*>(ch)); }   // multi-GPU: the sum goes straight into this rank's peer-visible buffer (vine_p2p.cuh)
  // sigma half of dataset.update_mu_sigma: the log-std this minibatch was evaluated with becomes its rows' "old" one. Done
  // here because this launch sits between the last reader (the minibatch kernel) and the writer (Adam) of the parameter.
  if (logstd_old_out && blockIdx.x == 0 && threadIdx.x < 2) logstd_old_out[threadIdx.x] = logstd[threadIdx.x];
  __shared__ float part[RED_SPLIT][RED_SLOTS];
  const int lane = threadIdx.x % RED_SLOTS, grp = threadIdx.x / RED_SLOTS;
  const int w = blockIdx.x * RED_SLOTS + lane;
  float acc0 = 0.f, acc1 = 0.f;
  if (w < WS_STATS + 8) {
    int k = grp;
    for (; k + RED_SPLIT < n_partials; k += 2 * RED_SPLIT) {
      acc0 += ws[(size_t)k * WS_FLOATS + w];
      acc1 += ws[(size_t)(k + RED_SPLIT) * WS_FLOATS + w];
    }
    if (k < n_partials) acc0 += ws[(size_t)k * WS_FLOATS + w];
  }
  part[grp][lane] = acc0 + acc1;
  __syncthreads();
  if (grp == 0 && w < WS_STATS + 8) {
    const int p = ws_to_param(w, O);
    if (p >= 0) flat[p] = part[0][lane] + part[1][lane] + part[2][lane] + part[3][lane];
  }
  if (ch) p2p_producer_done(const_cast<VineP2PChannel*>(ch));
}

// Gradient-norm clipping (torch.nn.utils.clip_grad_norm_ over the whole model) for one or two flat gradient vectors:
// total = sqrt(sum of (flat[i] * scale)^2 over i < count of each vector), coef = min(max_norm / (total + 1e-6), 1) with a NaN
// kept (torch's clamp(max=1)), both written to the state block; the Adam kernels multiply the coefficient in.  The sum of
// squares has a fixed order -- per block a fixed tree, then the last block to finish (self-resetting ticket in the workspace)
// sums the block partials in a fixed tree -- so every rank that holds the same summed gradient computes the same bits.
// No block waits for another block of the grid.  Multi-GPU (peer memory), this kernel is the consumer of each channel: it
// writes the rank-order sum of all `len` floats (gradient + loss statistics) into the local `flat`, which Adam then reads
// without a channel.
constexpr int CLIP_THREADS = 256, CLIP_CHUNK = 4 * CLIP_THREADS, CLIP_MAX_BLOCKS = VINE_GRAD_CLIP_WS_FLOATS - 1;
constexpr int ST_CLIP_COEF = 9, ST_GRAD_NORM = 10;
struct ClipArgs {
  float* flat[2];
  VineP2PChannel* ch[2];
  int count[2], len[2], chunks0, chunks;   // chunks0 = chunks of vector 0; blocks stride over all chunks of both
  float scale, max_norm;
  float *state, *ws;                      // ws[0]: ticket (u32 bits), ws[1 + b]: partial of block b
};

// deterministic sum over the block (every thread gets the result; CLIP_THREADS / 32 warps added in warp order)
__device__ __forceinline__ float clip_block_sum(float v, float* red) {
  v = warp_sum_f(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < CLIP_THREADS / 32; ++w) s += red[w];
  __syncthreads();   // red is reused
  return s;
}

__global__ void __launch_bounds__(CLIP_THREADS) vine_grad_clip_kernel(const ClipArgs a) {
  vine_launch::grid_dependency_sync();
  __shared__ __align__(16) float s_g[CLIP_CHUNK];
  __shared__ float red[CLIP_THREADS / 32];
  __shared__ int s_last;
  // vine_ppo_reduce / vine_lstm_reduce have published this rank's flags
  const unsigned seq0 = a.ch[0] ? p2p_exchange_begin(a.ch[0], false) : 0u, seq1 = a.ch[1] ? p2p_exchange_begin(a.ch[1], false) : 0u;
  float acc = 0.f;
  for (int c = blockIdx.x; c < a.chunks; c += gridDim.x) {   // (selects instead of a[v]: no local-memory copy of the arguments)
    const bool second = c >= a.chunks0;
    const int base = (second ? c - a.chunks0 : c) * CLIP_CHUNK, n = min(CLIP_CHUNK, (second ? a.len[1] : a.len[0]) - base);
    const int count = second ? a.count[1] : a.count[0];
    float* flat = second ? a.flat[1] : a.flat[0];
    VineP2PChannel* ch = second ? a.ch[1] : a.ch[0];
    if (ch) p2p_sum_block(ch, second ? seq1 : seq0, base, n, s_g);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = threadIdx.x + k * CLIP_THREADS;
      if (i < n) {
        float x;
        if (ch) flat[base + i] = x = s_g[i];
        else x = flat[base + i];
        const float g = x * a.scale;
        if (base + i < count) acc = fmaf(g, g, acc);
      }
    }
    if (ch) __syncthreads();   // s_g is refilled by the next chunk
  }
  if (a.ch[0]) p2p_exchange_end(a.ch[0]);
  if (a.ch[1]) p2p_exchange_end(a.ch[1]);
  const float part = clip_block_sum(acc, red);
  unsigned* ticket = reinterpret_cast<unsigned*>(a.ws);
  if (threadIdx.x == 0) {
    a.ws[1 + blockIdx.x] = part;
    __threadfence();
    s_last = atomicAdd(ticket, 1u) + 1u == gridDim.x;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  float t = 0.f;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += CLIP_THREADS) t += __ldcg(a.ws + 1 + b);
  const float sumsq = clip_block_sum(t, red);
  if (threadIdx.x == 0) {
    const float total = sqrtf(sumsq);
    const float coef = a.max_norm / (total + 1e-6f);
    a.state[ST_CLIP_COEF] = coef > 1.f ? 1.f : coef;   // NaN stays NaN, as with torch.clamp(max=1.0)
    a.state[ST_GRAD_NORM] = total;
    *ticket = 0u;                                      // ready for the next call (and the next replay of a graph)
  }
}

// torch.optim.Adam (no weight decay, no amsgrad) on the flat parameter vector + re-pack for the tensor cores
__global__ void vine_ppo_adam_kernel(const float* __restrict__ flat, float scale, float* __restrict__ params, float* __restrict__ m,
                                     float* __restrict__ v, uint8_t* __restrict__ packed, float* __restrict__ state, int O,
                                     float beta1, float beta2, float eps, int bookkeeping, const float* __restrict__ clip,
                                     VineP2PChannel* ch) {
  vine_launch::grid_dependency_sync();
  const int P = num_params(O);
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  // multi-GPU: wait for every rank's gradient buffer, then read the sum over the ranks instead of `flat` (vine_p2p.cuh)
  __shared__ __align__(16) float s_g[128];
  const unsigned seq = ch ? p2p_exchange_begin(ch, false) : 0u;   // vine_ppo_reduce has published this rank's flag
  const int base = blockIdx.x * blockDim.x;
  if (ch) p2p_sum_block(ch, seq, base, min((int)blockDim.x, P + 4 - base), s_g);
  if (p == P && bookkeeping) {   // bookkeeping by exactly one thread
    float st4[4];
    if (ch && P - base + 4 <= (int)blockDim.x) {   // the statistics sit right behind the last parameters: already in this block's sums
      for (int j = 0; j < 4; ++j) st4[j] = s_g[P - base + j];
    } else if (ch) {
      p2p_sum4(ch, seq, P, st4);
    } else {
      st4[0] = flat[P]; st4[1] = flat[P + 1]; st4[2] = flat[P + 2]; st4[3] = flat[P + 3];
    }
    for (int j = 0; j < 4; ++j) state[ST_SUMS + j] += st4[j] * scale;
    state[ST_COUNT] += 1.f;
    state[ST_KL] = st4[2] * scale;
    state[ST_PENDING] = 1.f;
  }
  if (p < P) {
    const float lr = state[ST_LR], step = state[ST_STEP];
    float g = (ch ? s_g[threadIdx.x] : flat[p]) * scale;
    if (clip) g *= *clip;   // vine_grad_clip's coefficient: exactly 1 when the norm is below max_norm, and g * 1 == g
    const float mn = beta1 * m[p] + (1.f - beta1) * g;
    const float vn = beta2 * v[p] + (1.f - beta2) * g * g;
    m[p] = mn;
    v[p] = vn;
    const float bc1 = 1.f - powf(beta1, step), bc2 = 1.f - powf(beta2, step);
    const float w = params[p] - (lr / bc1) * mn / (sqrtf(vn) / sqrtf(bc2) + eps);
    params[p] = w;
    int ws_off, pk_off;
    bool f32;
    param_map(p, O, ws_off, pk_off, f32);
    if (pk_off >= 0) {
      if (f32) *reinterpret_cast<float*>(packed + pk_off) = w;
      else *reinterpret_cast<__nv_bfloat16*>(packed + pk_off) = __float2bfloat16_rn(w);
    }
  }
  if (ch) p2p_exchange_end(ch);
}

}  // namespace

extern "C" {

int vine_ppo_num_params(int num_obs) { return (num_obs < 1 || num_obs >= K1) ? VINE_ERR_INVALID_ARG : num_params(num_obs); }

int vine_ppo_max_ctas(void) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return VINE_ERR_CUDA;
  return sms;
}

int vine_ppo_minibatch(const VinePpoMinibatch* b, void* stream) {
  if (!b || !b->packed || !b->obs || (!b->raw_obs && (!b->obs_mean || !b->obs_inv_std)) || !b->logstd || !b->logstd_old ||
      !b->workspace || !b->state)
    return VINE_ERR_INVALID_ARG;
  if (!b->dh3_ext && (!b->actions || !b->mu_old || !b->neglogp_old || !b->values_old || !b->returns || !b->advantages))
    return VINE_ERR_INVALID_ARG;
  if (b->horizon < 1 || b->num_envs < 1 || b->env_count < 1 || b->env_begin < 0 || b->env_begin + b->env_count > b->num_envs ||
      b->num_obs < 1 || b->num_obs >= K1 || (((uintptr_t)b->packed) & 15u) || (((uintptr_t)b->workspace) & 15u))
    return VINE_ERR_INVALID_ARG;
  if (b->lr_linear && (b->adaptive_lr || b->max_epochs < 1)) return VINE_ERR_INVALID_ARG;
  static int configured = -1, q4 = 1;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (configured != dev) {
    if (cudaFuncSetAttribute(vine_ppo_minibatch_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(vine_ppo_minibatch_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(vine_ppo_minibatch_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(vine_ppo_minibatch_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES) != cudaSuccess)
      return VINE_ERR_CUDA;
    configured = dev;
  }
  q4 = b->reserved != 2;   // VinePpoMinibatch.reserved: 2 = two epilogue threads per row (A/B switch), anything else four
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t B = (int64_t)b->horizon * b->env_count;
  const int64_t ntiles = (B + TILE - 1) / TILE;
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  if (b->workspace_ctas < grid) return VINE_ERR_INVALID_ARG;
  MbArgs a;
  a.packed = (const uint8_t*)b->packed;
  a.obs = b->obs, a.act = b->actions, a.mu_old = b->mu_old, a.nlp_old = b->neglogp_old, a.val_old = b->values_old;
  a.ret = b->returns, a.adv = b->advantages, a.obs_mean = b->obs_mean, a.obs_inv_std = b->obs_inv_std;
  a.logstd = b->logstd, a.logstd_old = b->logstd_old, a.ws = b->workspace, a.state = b->state, a.debug = b->debug_out;
  a.dh3_ext = b->dh3_ext;
  a.T = b->horizon, a.N = b->num_envs, a.e0 = b->env_begin, a.E = b->env_count, a.O = b->num_obs;
  a.e_clip = b->e_clip, a.critic_coef = b->critic_coef, a.entropy_coef = b->entropy_coef, a.bounds_coef = b->bounds_loss_coef;
  a.inv_B = 1.0f / (float)B, a.kl_threshold = b->kl_threshold, a.lr_min = b->lr_min, a.lr_max = b->lr_max, a.adaptive = b->adaptive_lr;
  a.lr0 = b->lr0, a.linear = b->lr_linear, a.standard = b->schedule_standard, a.epoch_begin = b->epoch_begin;
  a.mini_epoch_begin = b->mini_epoch_begin, a.max_epochs = b->max_epochs, a.clip_value = !b->value_loss_unclipped;
  const cudaStream_t st = (cudaStream_t)stream;
  if (b->raw_obs) {
    if (q4) vine_launch::launch(vine_ppo_minibatch_kernel<4, true>, grid, 512, SMEM_BYTES, st, a);
    else vine_launch::launch(vine_ppo_minibatch_kernel<2, true>, grid, 256, SMEM_BYTES, st, a);
  } else {
    if (q4) vine_launch::launch(vine_ppo_minibatch_kernel<4, false>, grid, 512, SMEM_BYTES, st, a);
    else vine_launch::launch(vine_ppo_minibatch_kernel<2, false>, grid, 256, SMEM_BYTES, st, a);
  }
  if (cudaGetLastError() != cudaSuccess) return VINE_ERR_CUDA;
  return grid;   // number of gradient partials written (>= 1)
}

int vine_ppo_reduce(const float* workspace, int n_partials, int num_obs, float* flat, const float* logstd, float* logstd_old_out,
                    void* p2p_channel, void* stream) {
  if (!workspace || (!flat && !p2p_channel) || n_partials < 1 || num_obs < 1 || num_obs >= K1 || (logstd_old_out && !logstd))
    return VINE_ERR_INVALID_ARG;
  const int slots = WS_STATS + 8;
  vine_launch::launch(vine_ppo_reduce_kernel, (slots + RED_SLOTS - 1) / RED_SLOTS, RED_SLOTS * RED_SPLIT, 0, (cudaStream_t)stream,
                      workspace, n_partials, num_obs, flat, logstd, logstd_old_out, (const VineP2PChannel*)p2p_channel);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_ppo_adam_clipped(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed,
                          float* state, int num_obs, float beta1, float beta2, float eps, int bookkeeping, const float* clip_coef,
                          void* p2p_channel, void* stream) {
  if ((!flat && !p2p_channel) || !params || !exp_avg || !exp_avg_sq || !packed || !state || num_obs < 1 || num_obs >= K1)
    return VINE_ERR_INVALID_ARG;
  const int n = num_params(num_obs) + 1;
  vine_launch::launch(vine_ppo_adam_kernel, (n + 127) / 128, 128, 0, (cudaStream_t)stream, flat, grad_scale, params, exp_avg, exp_avg_sq,
                      (uint8_t*)packed, state, num_obs, beta1, beta2, eps, bookkeeping, clip_coef, (VineP2PChannel*)p2p_channel);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_ppo_adam(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed,
                  float* state, int num_obs, float beta1, float beta2, float eps, int bookkeeping, void* p2p_channel, void* stream) {
  return vine_ppo_adam_clipped(flat, grad_scale, params, exp_avg, exp_avg_sq, packed, state, num_obs, beta1, beta2, eps, bookkeeping,
                               nullptr, p2p_channel, stream);
}

int vine_grad_clip(float* flat, int count, int length, float* flat2, int count2, int length2, float grad_scale, float max_norm,
                   float* state, float* workspace, void* p2p_channel, void* p2p_channel2, void* stream) {
  if (!flat || !state || !workspace || count < 1 || count > length || !isfinite(max_norm)) return VINE_ERR_INVALID_ARG;
  if (flat2 ? (count2 < 1 || count2 > length2) : (count2 != 0 || length2 != 0 || p2p_channel2)) return VINE_ERR_INVALID_ARG;
  const int64_t chunks0 = ((int64_t)length + CLIP_CHUNK - 1) / CLIP_CHUNK;
  const int64_t chunks = chunks0 + (flat2 ? ((int64_t)length2 + CLIP_CHUNK - 1) / CLIP_CHUNK : 0);
  ClipArgs a;
  a.flat[0] = flat, a.flat[1] = flat2;
  a.ch[0] = (VineP2PChannel*)p2p_channel, a.ch[1] = (VineP2PChannel*)p2p_channel2;
  a.count[0] = count, a.count[1] = count2, a.len[0] = length, a.len[1] = length2;
  a.chunks0 = (int)chunks0, a.chunks = (int)chunks;
  a.scale = grad_scale, a.max_norm = max_norm, a.state = state, a.ws = workspace;
  const int grid = (int)(chunks < CLIP_MAX_BLOCKS ? chunks : CLIP_MAX_BLOCKS);
  vine_launch::launch(vine_grad_clip_kernel, grid, CLIP_THREADS, 0, (cudaStream_t)stream, a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}


// ------------------------------------------------------------------------------------------
// peer-memory regions and channels of the gradient all-reduce (vine_p2p.cuh)
// ------------------------------------------------------------------------------------------
}  // extern "C"

// In-place sum over the ranks of a SHORT f64 vector (the running-statistics moments of vine_ppo_moments: 2 O + 4 doubles) in one
// single-block launch: producer and consumer of the exchange in one kernel (one block, so nothing has to be co-resident).
// The doubles travel as their two 32-bit halves in a channel of 2 n floats; sums in rank order: bit-identical on all ranks.
__global__ void __launch_bounds__(256) vine_p2p_allreduce_f64_kernel(VineP2PChannel* ch, double* __restrict__ buf, int n) {
  float* mine = p2p_local_buffer(ch);
  for (int i = threadIdx.x; i < n; i += blockDim.x) reinterpret_cast<double*>(mine)[i] = buf[i];
  __syncthreads();                                   // all of this block's stores precede thread r's system fence + flag store
  const unsigned seq = p2p_exchange_begin(ch);
  const int W = ch->world;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double acc = 0.0;
    for (int r = 0; r < W; ++r) acc += __ldcv(reinterpret_cast<const double*>(p2p_buffer(ch, r, seq)) + i);
    buf[i] = acc;
  }
  p2p_exchange_end(ch);
}

extern "C" {

int vine_p2p_allreduce_f64(void* channel, double* buf, int n, void* stream) {
  if (!channel || !buf || n < 1) return VINE_ERR_INVALID_ARG;
  vine_p2p_allreduce_f64_kernel<<<1, 256, 0, (cudaStream_t)stream>>>((VineP2PChannel*)channel, buf, n);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

static int64_t p2p_padded(int64_t count) { return (count + 3) & ~(int64_t)3; }   // buffers are read with 128-bit loads
static size_t p2p_region_bytes(int64_t count) { return (size_t)VINE_P2P_FLAG_BYTES + 2u * (size_t)p2p_padded(count) * sizeof(float); }

int vine_p2p_alloc(int64_t count, void** region, void* ipc_handle_out) {
  if (count < 1 || !region || !ipc_handle_out) return VINE_ERR_INVALID_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == VINE_P2P_HANDLE_BYTES, "handle size");
  void* p = nullptr;
  if (cudaMalloc(&p, p2p_region_bytes(count)) != cudaSuccess) return VINE_ERR_CUDA;
  if (cudaMemset(p, 0, p2p_region_bytes(count)) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) { cudaFree(p); return VINE_ERR_CUDA; }
  cudaIpcMemHandle_t h;
  if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaFree(p); return VINE_ERR_CUDA; }
  memcpy(ipc_handle_out, &h, sizeof(h));
  *region = p;
  return VINE_OK;
}

int vine_p2p_open(const void* ipc_handle, void** region) {
  if (!ipc_handle || !region) return VINE_ERR_INVALID_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof(h));
  return cudaIpcOpenMemHandle(region, h, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_p2p_close(void* region) { return cudaIpcCloseMemHandle(region) == cudaSuccess ? VINE_OK : VINE_ERR_CUDA; }
int vine_p2p_free(void* region) { return cudaFree(region) == cudaSuccess ? VINE_OK : VINE_ERR_CUDA; }

int vine_p2p_channel_create(void* const* regions, int world, int rank, int64_t count, void** channel) {
  if (!regions || !channel || world < 1 || world > VINE_P2P_MAX_RANKS || rank < 0 || rank >= world || count < 1) return VINE_ERR_INVALID_ARG;
  VineP2PChannel h;
  memset(&h, 0, sizeof(h));
  for (int r = 0; r < world; ++r) {
    if (!regions[r]) return VINE_ERR_INVALID_ARG;
    h.peer_base[r] = (unsigned long long)(uintptr_t)regions[r];
  }
  h.world = world; h.rank = rank; h.count = p2p_padded(count);
  void* d = nullptr;
  if (cudaMalloc(&d, sizeof(h)) != cudaSuccess) return VINE_ERR_CUDA;
  if (cudaMemcpy(d, &h, sizeof(h), cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return VINE_ERR_CUDA; }
  *channel = d;
  return VINE_OK;
}

// exchanges completed and the timeout flag of a channel (synchronises the device: for tests and error reporting)
int vine_p2p_channel_status(const void* channel, uint32_t* seq, uint32_t* error) {
  if (!channel) return VINE_ERR_INVALID_ARG;
  VineP2PChannel h;
  if (cudaMemcpy(&h, channel, sizeof(h), cudaMemcpyDeviceToHost) != cudaSuccess) return VINE_ERR_CUDA;
  if (seq) *seq = h.seq;
  if (error) *error = h.error;
  return VINE_OK;
}

// mean ns per exchange, as seen by block 0 of the consumer: [0] entry -> own flag stored at every peer, [1 + r] entry -> rank
// r's flag seen here (r == own rank: the local store); resets the accumulators.  Synchronises the device.
int vine_p2p_channel_timing(void* channel, double* out, int n_out) {
  if (!channel || !out || n_out < 1 + VINE_P2P_MAX_RANKS) return VINE_ERR_INVALID_ARG;
  VineP2PChannel h;
  if (cudaMemcpy(&h, channel, sizeof(h), cudaMemcpyDeviceToHost) != cudaSuccess) return VINE_ERR_CUDA;
  const double n = h.t_n ? (double)h.t_n : 1.0;
  out[0] = (double)h.t_signal / n;
  for (int r = 0; r < VINE_P2P_MAX_RANKS; ++r) out[1 + r] = (double)h.t_wait[r] / n;
  if (n_out >= 3 + VINE_P2P_MAX_RANKS) { out[1 + VINE_P2P_MAX_RANKS] = (double)h.t_kernel / n; out[2 + VINE_P2P_MAX_RANKS] = (double)h.t_loads / n; }
  if (n_out >= 6 + VINE_P2P_MAX_RANKS) {
    out[3 + VINE_P2P_MAX_RANKS] = (double)h.t_mb / n; out[4 + VINE_P2P_MAX_RANKS] = (double)h.t_prod / n; out[5 + VINE_P2P_MAX_RANKS] = (double)h.t_gap / n;
  }
  h.t_signal = 0; h.t_n = 0; h.t_kernel = 0; h.t_loads = 0; h.t_mb = 0; h.t_prod = 0; h.t_gap = 0; h.t_prev_end = 0;
  for (int r = 0; r < VINE_P2P_MAX_RANKS; ++r) h.t_wait[r] = 0;
  // only the accumulators are written back (seq / ticket belong to the kernels)
  const size_t off = offsetof(VineP2PChannel, t_signal);   // t_signal .. the end: all timing fields
  if (cudaMemcpy((char*)channel + off, (char*)&h + off, sizeof(h) - off, cudaMemcpyHostToDevice) != cudaSuccess) return VINE_ERR_CUDA;
  return VINE_OK;
}

int vine_p2p_channel_destroy(void* channel) { return cudaFree(channel) == cudaSuccess ? VINE_OK : VINE_ERR_CUDA; }

}  // extern "C"
