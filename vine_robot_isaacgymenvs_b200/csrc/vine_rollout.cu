// vine_rollout.cu — the PPO rollout and update-prologue kernels around the fused env step (sm_100a).
//
//   vine_policy_act      one launch per control step: observation normalisation -> actor-critic MLP on tcgen05/TMEM ->
//                        Gaussian action sampling (Philox keyed by the GLOBAL env id) -> neglogp, and every rollout-buffer
//                        write of that step (obs, action, mu, neglogp, value) + the clamped action the env consumes.
//                        (rl_games A2CAgent.get_action_values / play_steps; in-repo analogue learning/common_agent.py:257-314)
//   vine_rollout_post    after the env step: reward shaper + value bootstrap on time-outs (YP:56-59), dones, episode
//                        statistics (device-side, no host sync).
//   vine_ppo_moments / vine_ppo_finalize
//                        running mean/std of observations and values (rl_games RunningMeanStd), advantage normalisation,
//                        normalised value targets: sufficient statistics in f64 (all-reducible), then one finalize pass.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "vine_device.cuh"
#include "vine_mlp_common.cuh"
#include "vine_launch.cuh"

namespace {
using namespace vine_mlp;

constexpr int OFF_BAR = OFF_END;
constexpr int ACT_SMEM_BYTES = OFF_BAR + 64;
constexpr uint32_t VINE_SITE_POLICY = 16;   // Philox "site" of the policy's action noise (env sites: vine_params.h:20)

__global__ void __launch_bounds__(THREADS, 1) vine_policy_act_kernel(const VinePolicyAct a) {
  vine_launch::grid_dependency_sync();
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, row = tid & 127, half = tid >> 7;
  const uint32_t bar_w = smem_u32(smem + OFF_BAR), bar_mma = bar_w + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 16);
  const float* biases = reinterpret_cast<const float*>(smem + OFF_B);

  if (tid == 0) {
    mbar_init(bar_w, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(bar_w, PACKED_BYTES);
    bulk_g2s(smem_u32(smem), a.packed, PACKED_BYTES, bar_w);
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  mbar_wait(bar_w, 0);

  uint8_t *x_t = smem + OFF_X, *a1_t = smem + OFF_A1, *a2_t = smem + OFF_A2, *a3_t = smem + OFF_A3;
  const uint32_t sW1 = smem_u32(smem + OFF_W1), sW2 = smem_u32(smem + OFF_W2), sW3 = smem_u32(smem + OFF_W3),
                 sW4 = smem_u32(smem + OFF_W4);
  const uint32_t sX = smem_u32(x_t), sA1 = smem_u32(a1_t), sA2 = smem_u32(a2_t), sA3 = smem_u32(a3_t);
  uint32_t phase = 0;
  auto mma_step = [&](auto&& issue) {
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    if (tid == 0) {
      fence_after_sync();
      issue();
      mma_commit(bar_mma);
    }
    mbar_wait(bar_mma, phase);
    phase ^= 1;
    fence_after_sync();
  };
  const bool sample = a.actions != nullptr;
  const uint32_t ctr = (sample && a.rng_counter) ? *a.rng_counter : 0u;
  float ls0 = 0.f, ls1 = 0.f;
  if (sample) ls0 = a.logstd[0], ls1 = a.logstd[1];
  const float vmean = a.value_stats[0], vstd = a.value_stats[1];
  const int O = a.num_obs;
  const int64_t ntiles = (a.n + TILE - 1) / TILE;

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t e = tile * TILE + row;
    const bool valid = e < a.n;
    build_x_tile(x_t, row, half, valid, a.obs + e * O, a.obs_mean, a.obs_inv_std, O, a.u_out != nullptr,
                 (valid && a.obs_copy) ? a.obs_copy + e * O : nullptr);
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      mma_step([&] { mma_sequence(tmem, k_major(sX, K1), k_major(sW1, K1, h * 128), instr_desc(128, false, false), K1 / 16, false); });
      fwd_epilogue<H1>(lane_base + half * 64, 64, h * 128 + half * 64, biases, a1_t, row);
    }
    mma_step([&] { mma_sequence(tmem, k_major(sA1, H1), k_major(sW2, H1), instr_desc(H2, false, false), H1 / 16, false); });
    fwd_epilogue<H2>(lane_base + half * 64, 64, half * 64, biases + H1, a2_t, row);
    mma_step([&] { mma_sequence(tmem, k_major(sA2, H2), k_major(sW3, H2), instr_desc(H3, false, false), H2 / 16, false); });
    fwd_epilogue<H3>(lane_base + half * 32, 32, half * 32, biases + H1 + H2, a3_t, row);
    if (a.u_out) {
      // recurrent network: emit the LSTM input tile U = [h3 (64) | x (32) | 0 (32)] (row-blocked [128 x 128] bf16) and stop;
      // LayerNorm and the heads follow the LSTM (vine_lstm_step / vine_lstm_head)
      __syncthreads();   // both column halves of h3 are in shared memory
      uint8_t* ut = reinterpret_cast<uint8_t*>(a.u_out) + (size_t)tile * (TILE * 128 * 2);
#pragma unroll
      for (int q = half * 8; q < half * 8 + 8; ++q) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (q < 8) v = *reinterpret_cast<const uint4*>(a3_t + tile_offset(row, 8 * q, H3));
        else if (q < 12) v = *reinterpret_cast<const uint4*>(x_t + tile_offset(row, 8 * (q - 8), K1));
        *reinterpret_cast<uint4*>(ut + tile_offset(row, 8 * q, 128)) = v;
      }
      __syncthreads();   // x / h3 tiles are rewritten by the next tile
      continue;
    }
    mma_step([&] { mma_sequence(tmem, k_major(sA3, H3), k_major(sW4, H3), instr_desc(NH, false, false), H3 / 16, false); });
    if (half == 0) {
      uint32_t r[16];
      tmem_ld16(lane_base, r);
      if (valid) {
        const float* bh = biases + H1 + H2 + H3;
        const float mu0 = __uint_as_float(r[0]) + bh[0], mu1 = __uint_as_float(r[1]) + bh[1], v = __uint_as_float(r[2]) + bh[2];
        const float value = fminf(fmaxf(v, -5.f), 5.f) * vstd + vmean;   // RunningMeanStd(unnorm=True)
        if (a.mu) *reinterpret_cast<float2*>(a.mu + 2 * e) = make_float2(mu0, mu1);
        if (a.value) a.value[e] = value;
        if (sample) {
          const uint32_t gid = (uint32_t)(a.global_env_offset + e);
          float z[4];
          normal4(philox4x32((uint32_t)a.seed, (uint32_t)(a.seed >> 32), gid, VINE_SITE_POLICY, ctr, 0u), z);
          const float act0 = fmaf(__expf(ls0), z[0], mu0), act1 = fmaf(__expf(ls1), z[1], mu1);
          *reinterpret_cast<float2*>(a.actions + 2 * e) = make_float2(act0, act1);
          if (a.neglogp) a.neglogp[e] = 0.5f * (z[0] * z[0] + z[1] * z[1]) + 1.8378770664093453f + ls0 + ls1;
          if (a.env_actions)   // rl_games preprocess_actions: clamp to [-1, 1] for the env, keep the raw action for the loss
            *reinterpret_cast<float2*>(a.env_actions + 2 * e) =
                make_float2(fminf(fmaxf(act0, -1.f), 1.f), fminf(fmaxf(act1, -1.f), 1.f));
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(256) vine_rollout_post_kernel(const VineRolloutPost a) {
  vine_launch::grid_dependency_sync();
  __shared__ double red[8][4];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  if (i < a.n) {
    const float rew = a.rewards[i];
    const float d = a.resets[i] != 0 ? 1.f : 0.f;
    // rl_games DefaultRewardsShaper: (r + shift) * scale, clamped like torch.clamp (comparisons keep a NaN, fminf would not)
    float shaped = (a.reward_shift != 0.f ? rew + a.reward_shift : rew) * a.reward_scale;
    if (a.reward_clamp) {
      if (shaped < a.reward_min) shaped = a.reward_min;
      if (shaped > a.reward_max) shaped = a.reward_max;
    }
    if (a.value_bootstrap && a.timeouts[i]) shaped += a.gamma * a.values[i];   // Vine5LinkMovingBasePPO.yaml:56
    a.shaped_rewards[i] = shaped;
    a.dones_next[i] = d;
    if (a.not_done_next) a.not_done_next[i] = 1.f - d;
    const float er = a.ep_return[i] + rew, el = a.ep_length[i] + 1.f;
    if (d != 0.f) {   // episode statistics; success == the 1000-point "Position Success" term fired (V5:1507)
      s0 = 1.0, s1 = rew > a.success_reward_threshold ? 1.0 : 0.0, s2 = er, s3 = el;
    }
    a.ep_return[i] = d != 0.f ? 0.f : er;
    a.ep_length[i] = d != 0.f ? 0.f : el;
  }
  s0 = warp_sum(s0), s1 = warp_sum(s1), s2 = warp_sum(s2), s3 = warp_sum(s3);
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) red[warp][0] = s0, red[warp][1] = s1, red[warp][2] = s2, red[warp][3] = s3;
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
    if (t != 0.0) atomicAdd(a.ep_stats + threadIdx.x, t);
  }
  if (i == 0 && a.rng_counter) *a.rng_counter += 1u;   // every act launch of this step has read it (stream order)
}

// ---------------------------------------------------------------------------------------------------------------
// moments layout (f64): [0,O) sum obs, [O,2O) sum obs^2, then sum v, sum v^2 (values and returns pooled), sum adv, sum adv^2
__global__ void __launch_bounds__(256) vine_ppo_moments_kernel(const VinePpoPrologue a) {
  __shared__ double red[8][2 * 32];
  const int tid = threadIdx.x, f = tid & 31, lane8 = tid >> 5, O = a.num_obs;
  double s = 0.0, q = 0.0;
  if (f < O)
    for (int64_t i = (int64_t)blockIdx.x * 8 + lane8; i < a.count; i += (int64_t)gridDim.x * 8) {
      const double x = a.obs[i * O + f];
      s += x, q += x * x;
    }
  red[lane8][f] = s, red[lane8][32 + f] = q;
  __syncthreads();
  if (tid < 64) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w][tid];
    const int ff = tid & 31;
    if (ff < O) atomicAdd(a.moments + (tid < 32 ? ff : O + ff), t);
  }
  __syncthreads();
  double m[4] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < a.count; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = a.values[i], r = a.returns[i], ad = (double)(a.returns[i] - a.values[i]);
    m[0] += v + r, m[1] += v * v + r * r, m[2] += ad, m[3] += ad * ad;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    m[j] = warp_sum(m[j]);
    if ((tid & 31) == 0) red[tid >> 5][j] = m[j];
  }
  __syncthreads();
  if (tid < 4) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w][tid];
    atomicAdd(a.moments + 2 * O + tid, t);
  }
}

// rl_games RunningMeanStd.update (parallel-variance merge) from pooled sufficient statistics
__device__ inline void rms_merge(double sum, double sumsq, double n, double* mean, double* var, double count_old, double* count_new) {
  const double bmean = sum / n;
  const double bvar = fmax(sumsq - n * bmean * bmean, 0.0) / fmax(n - 1.0, 1.0);
  const double delta = bmean - *mean, tot = count_old + n;
  const double m_a = *var * count_old, m_b = bvar * n;
  *var = (m_a + m_b + delta * delta * count_old * n / tot) / tot;
  *mean = *mean + delta * n / tot;
  *count_new = tot;
}

__global__ void vine_ppo_finalize_kernel(const VinePpoPrologue a) {
  const int tid = threadIdx.x, O = a.num_obs;
  const double n = (double)a.count * a.world;   // moments were summed over ranks
  if (tid < O) {
    double mean = a.obs_mean[tid], var = a.obs_var[tid], cnt;
    rms_merge(a.moments[tid], a.moments[O + tid], n, &mean, &var, *a.obs_count, &cnt);
    a.obs_mean[tid] = mean, a.obs_var[tid] = var;
    a.obs_mean_f[tid] = (float)mean;
    a.obs_inv_std_f[tid] = rsqrtf((float)var + 1e-5f);
  }
  __syncthreads();   // every thread has read the old obs count
  if (tid == 0) {
    *a.obs_count += n;
    double mean = *a.val_mean, var = *a.val_var, cnt;
    rms_merge(a.moments[2 * O], a.moments[2 * O + 1], 2.0 * n, &mean, &var, *a.val_count, &cnt);
    *a.val_mean = mean, *a.val_var = var, *a.val_count = cnt;
    a.value_stats[0] = (float)mean;
    a.value_stats[1] = sqrtf((float)var + 1e-5f);
    const double am = a.moments[2 * O + 2] / n;
    const double astd = sqrt(fmax((a.moments[2 * O + 3] - n * am * am) / (n - 1.0), 0.0));
    a.adv_stats[0] = a.normalize_advantage ? (float)am : 0.f;
    a.adv_stats[1] = a.normalize_advantage ? 1.f / ((float)astd + 1e-8f) : 1.f;
  }
  __syncthreads();
  if (tid < 2 * O + 4) a.moments[tid] = 0.0;   // ready for the next iteration
}

__global__ void __launch_bounds__(256) vine_ppo_normalize_kernel(const VinePpoPrologue a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.count) return;
  const float vm = a.value_stats[0], vinv = 1.f / a.value_stats[1];
  const float v = a.values[i], r = a.returns[i];
  a.values_n[i] = fminf(fmaxf((v - vm) * vinv, -5.f), 5.f);
  a.returns_n[i] = fminf(fmaxf((r - vm) * vinv, -5.f), 5.f);
  a.advantages_n[i] = ((r - v) - a.adv_stats[0]) * a.adv_stats[1];
}

}  // namespace

extern "C" {

int vine_policy_act(const VinePolicyAct* a, void* stream) {
  if (!a || !a->packed || !a->obs || !a->obs_mean || !a->obs_inv_std || !a->value_stats || a->n <= 0 || a->num_obs < 1 ||
      a->num_obs > K1 || (((uintptr_t)a->packed) & 15u))
    return VINE_ERR_INVALID_ARG;
  if (a->actions && !a->logstd) return VINE_ERR_INVALID_ARG;
  if (!a->actions && !a->mu && !a->value && !a->u_out) return VINE_ERR_INVALID_ARG;
  if (a->u_out && (a->num_obs >= K1 || (((uintptr_t)a->u_out) & 15u))) return VINE_ERR_INVALID_ARG;
  static int configured = -1;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return VINE_ERR_CUDA;
  if (configured != dev) {
    if (cudaFuncSetAttribute(vine_policy_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ACT_SMEM_BYTES) != cudaSuccess)
      return VINE_ERR_CUDA;
    configured = dev;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t ntiles = (a->n + TILE - 1) / TILE;
  const int grid = (int)(ntiles < sms ? ntiles : sms);
  vine_launch::launch(vine_policy_act_kernel, grid, THREADS, ACT_SMEM_BYTES, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_mlp_forward(const void* packed, const float* obs, const float* obs_mean, const float* obs_inv_std, int64_t n,
                     int num_obs, const float* value_stats, float* mu, float* value, void* stream) {
  if (!mu || !value) return VINE_ERR_INVALID_ARG;
  VinePolicyAct a = {};
  a.packed = packed, a.obs = obs, a.obs_mean = obs_mean, a.obs_inv_std = obs_inv_std, a.value_stats = value_stats;
  a.mu = mu, a.value = value, a.n = n, a.num_obs = num_obs;
  return vine_policy_act(&a, stream);
}

int vine_rollout_post(const VineRolloutPost* a, void* stream) {
  if (!a || !a->rewards || !a->resets || !a->timeouts || !a->values || !a->shaped_rewards || !a->dones_next || !a->ep_return ||
      !a->ep_length || !a->ep_stats || a->n <= 0)
    return VINE_ERR_INVALID_ARG;
  vine_launch::launch(vine_rollout_post_kernel, (unsigned)((a->n + 255) / 256), 256, 0, (cudaStream_t)stream, *a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

static int prologue_ok(const VinePpoPrologue* a) {
  return a && a->obs && a->values && a->returns && a->moments && a->obs_mean && a->obs_var && a->obs_count && a->val_mean &&
         a->val_var && a->val_count && a->obs_mean_f && a->obs_inv_std_f && a->value_stats && a->adv_stats && a->values_n &&
         a->returns_n && a->advantages_n && a->count > 1 && a->num_obs >= 1 && a->num_obs <= 32 && a->world >= 1;
}

int vine_ppo_moments(const VinePpoPrologue* a, void* stream) {
  if (!prologue_ok(a)) return VINE_ERR_INVALID_ARG;
  // one block per SM at most: the row loop is latency-bound (a warp reads one 72-byte observation row per load), so it wants
  // as many blocks as there are SMs, and no more (every block ends in ~40 f64 atomics on the same addresses)
  int64_t blocks = (a->count + 255) / 256;
  if (blocks > 148) blocks = 148;
  vine_ppo_moments_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(*a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_ppo_finalize(const VinePpoPrologue* a, void* stream) {
  if (!prologue_ok(a)) return VINE_ERR_INVALID_ARG;
  vine_ppo_finalize_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(*a);
  vine_ppo_normalize_kernel<<<(unsigned)((a->count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*a);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

}  // extern "C"
