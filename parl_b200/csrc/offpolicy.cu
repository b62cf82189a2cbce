// Off-policy continuous control (DDPG / TD3 / SAC): fused exploration into the HBM replay ring, and uniform replay
// sampling with the row count and draw index read from device memory.
//
// rl_explore_mlp replaces, per env step, the reference's agent.sample -> env.step -> rpm.append round trip
// (benchmark/torch/{td3,sac,ddpg}/train.py).  The reference actors (17->256->256->6 TD3, 17->256->256->{6,6} SAC,
// 17->400->300->6 DDPG: 290-531 KB of fp32) do not fit one CTA's shared memory, so the output rows of every layer are
// split over the C CTAs of a thread-block cluster.  Each CTA keeps ITS slice of every layer resident in shared memory
// (transposed, [in][rows]) for all K steps; all C CTAs of a cluster work on the same tile of 32 envs, each computes
// its rows of a layer for the 32 envs and stores them into the activation buffer of every CTA of the cluster through
// distributed shared memory, then one cluster barrier per layer.  The env step itself is cheap and deterministic, so
// every CTA advances its own copy of the observations; rank 0 alone writes the replay rows and the episode statistics.
//
// Register tile: thread = 4 output rows x 4 envs, weights and activations both read as float4 (16 FMA per 2 LDS.128).
#include <string.h>

#include <cooperative_groups.h>

#include "common.cuh"
#include "env_common.cuh"

namespace cg = cooperative_groups;

namespace rl {

constexpr int kExThreads = 128;
constexpr int kExTN = 32;           // envs per cluster (one warp of env threads: episode bookkeeping is warp-wide)
constexpr int kExXS = 36;           // row stride of the observation tile: float4-aligned, and a column read (one env's
                                    // observation, consecutive threads walk k) touches 8 banks instead of 1
constexpr int kExMaxLayers = 4;
constexpr int kExMaxSeg = 8;
constexpr int kExMaxWidth = 512;    // widest layer
constexpr int kExMaxCluster = 8;    // portable cluster size limit
constexpr size_t kExSmemLimit = 220 * 1024;

struct ExSeg {
  const float* w;   // [rows, in] row-major (torch nn.Linear.weight)
  const float* b;   // [rows] or NULL
  int layer, row0, rows;
};

struct ExploreArgs {
  int L, C, n_seg;
  int dims[kExMaxLayers + 1];
  int inp[kExMaxLayers];      // padded input width of layer l (multiple of 4)
  int R[kExMaxLayers];        // output rows of layer l owned by each CTA (multiple of 4)
  int w_off[kExMaxLayers];    // float offsets of the CTA's slice: weights [inp][R], then bias [R]
  int w_floats;               // 0 when the actor is not evaluated (mode 0)
  int H;                      // rows of each hidden activation buffer
  int O;                      // rows of the head's output buffer
  ExSeg seg[kExMaxSeg];
  int head, mode, K, B, AD, D, max_steps;
  float sigma;
  float* obs_cur;             // [B, D]
  EpisodeStats st;
  uint32_t k0, k1, step0, env_offset, done_thr;
  float* rm_obs;              // [cap, D]
  float* rm_act;              // [cap, AD]
  float* rm_rew;              // [cap]
  int* rm_term;               // [cap]
  float* rm_next;             // [cap, D]
  int cap, pos;
};

__device__ __forceinline__ uint32_t ex_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}

__device__ __forceinline__ void ex_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

// rows [rank*R, rank*R + R) of layer l for the 32 envs: out[j][n] = act(b[j] + sum_k W[j][k] in[k][n]),
// stored into the buffer `out_local` of EVERY CTA of the cluster (DSMEM).  act: 0 relu, 2 none.
__device__ __forceinline__ void ex_layer(const float* __restrict__ wt, const float* __restrict__ bias,
                                         const float* __restrict__ in, int in_stride, float* out_local, int inp, int R,
                                         int row_base, int act, int C) {
  cg::cluster_group cluster = cg::this_cluster();
  const int nblk = (R >> 2) * (kExTN / 4);
  for (int blk = threadIdx.x; blk < nblk; blk += kExThreads) {
    const int jq = blk >> 3, nq = blk & 7;
    float acc[4][4];
    const float4 bv = *reinterpret_cast<const float4*>(bias + jq * 4);
    const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = bb[i];
#pragma unroll 4
    for (int k = 0; k < inp; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(in + k * in_stride + nq * 4);
      const float4 w = *reinterpret_cast<const float4*>(wt + k * R + jq * 4);
      const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(wv[i], a.x, acc[i][0]), acc[i][1] = fmaf(wv[i], a.y, acc[i][1]);
        acc[i][2] = fmaf(wv[i], a.z, acc[i][2]), acc[i][3] = fmaf(wv[i], a.w, acc[i][3]);
      }
    }
    float4 o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (act == 0) {
        o[i] = make_float4(fmaxf(acc[i][0], 0.f), fmaxf(acc[i][1], 0.f), fmaxf(acc[i][2], 0.f), fmaxf(acc[i][3], 0.f));
      } else {
        o[i] = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      }
    }
    const int j0 = row_base + jq * 4;
    for (int c = 0; c < C; ++c) {
      float* dst = cluster.map_shared_rank(out_local, c);
#pragma unroll
      for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(dst + (j0 + i) * kExTN + nq * 4) = o[i];
    }
  }
}

__global__ void __launch_bounds__(kExThreads) explore_mlp_kernel(const ExploreArgs p) {
  extern __shared__ __align__(16) float smem_f[];
  float* s_w = smem_f;
  float* s_x = s_w + p.w_floats;                  // observations [Dp][kExXS]
  const int Dp = (p.D + 3) & ~3;
  float* s_h0 = s_x + Dp * kExXS;                 // activation ping [H][32]
  float* s_h1 = s_h0 + p.H * kExTN;               // activation pong
  float* s_o = s_h1 + p.H * kExTN;                // head outputs [O][32]: a buffer of its own, so that a peer that
                                                  // starts the next step never overwrites what warp 0 still reads
  const int rank = (int)ex_cluster_rank();
  const int tile = blockIdx.x / p.C;
  const int n0 = tile * kExTN;
  const int tid = threadIdx.x;
  const int D = p.D, B = p.B, AD = p.AD;

  // this CTA's weight slice: transposed [inp][R] + bias [R], zero beyond the layer's rows / inputs
  if (p.w_floats > 0) {
    for (int i = tid; i < p.w_floats; i += kExThreads) s_w[i] = 0.f;
    __syncthreads();
    for (int s = 0; s < p.n_seg; ++s) {
      const ExSeg& g = p.seg[s];
      const int l = g.layer, in = p.dims[l], R = p.R[l];
      const int lo = max(g.row0, rank * R), hi = min(g.row0 + g.rows, rank * R + R);
      if (lo >= hi) continue;
      float* wt = s_w + p.w_off[l];
      for (int i = tid; i < (hi - lo) * in; i += kExThreads) {
        const int r = lo + i / in, k = i % in;
        wt[k * R + (r - rank * R)] = g.w[(size_t)(r - g.row0) * in + k];
      }
      if (g.b)
        for (int r = lo + tid; r < hi; r += kExThreads) wt[p.inp[l] * R + (r - rank * R)] = g.b[r - g.row0];
    }
  }
  for (int i = tid; i < Dp * kExTN; i += kExThreads) {
    const int n = i / Dp, k = i - n * Dp;
    s_x[k * kExXS + n] = (k < D && n0 + n < B) ? p.obs_cur[(size_t)(n0 + n) * D + k] : 0.f;
  }
  ex_cluster_sync();                               // every CTA's buffers exist before a peer stores into them

  for (int t = 0; t < p.K; ++t) {
    const uint32_t step = p.step0 + (uint32_t)t;
    if (rank == 0) {
      for (int i = tid; i < kExTN * D; i += kExThreads) {
        const int n = i / D, k = i - n * D;
        if (n0 + n < B) {
          const size_t row = ((size_t)p.pos + (size_t)t * B + n0 + n) % (size_t)p.cap;
          p.rm_obs[row * D + k] = s_x[k * kExXS + n];
        }
      }
    }
    if (p.mode != 0) {
      for (int l = 0; l < p.L; ++l) {
        const float* in = l == 0 ? s_x : ((l - 1) % 2 == 0 ? s_h0 : s_h1);
        float* out = l + 1 == p.L ? s_o : (l % 2 == 0 ? s_h0 : s_h1);
        ex_layer(s_w + p.w_off[l], s_w + p.w_off[l] + p.inp[l] * p.R[l], in, l == 0 ? kExXS : kExTN, out, p.inp[l],
                 p.R[l], rank * p.R[l], l + 1 < p.L ? 0 : 2, p.C);
        ex_cluster_sync();
      }
    }
    // one thread per env (warp 0): action, env step, replay row, episode bookkeeping
    if (rank == 0 && tid < kExTN) {
      const int b = n0 + tid;
      const bool valid = b < B;
      float reward = 0.f;
      bool done = false;
      if (valid) {
        const uint32_t env = p.env_offset + (uint32_t)b;
        const size_t row = ((size_t)p.pos + (size_t)t * B + b) % (size_t)p.cap;
        float* ao = p.rm_act + row * AD;
        for (int blk = 0; blk * 4 < AD; ++blk) {
          float z[4];
          if (p.mode == 0) {
            const uint4 x = philox4x32_10(env, step, (uint32_t)blk, STREAM_ACTION, p.k0, p.k1);
            z[0] = u01_24(x.x), z[1] = u01_24(x.y), z[2] = u01_24(x.z), z[3] = u01_24(x.w);
          } else {
            gauss_block(env, step, (uint32_t)blk, STREAM_GAUSS, p.k0, p.k1, z);
          }
#pragma unroll
          for (int k = 0; k < 4 && blk * 4 + k < AD; ++k) {
            const int d = blk * 4 + k;
            float a;
            if (p.mode == 0) {
              a = __fsub_rn(__fmul_rn(2.f, z[k]), 1.f);
            } else if (p.mode == 1) {
              const float mu = tanhf(s_o[d * kExTN + tid]);
              a = fminf(fmaxf(fmaf(p.sigma, z[k], mu), -1.f), 1.f);
            } else {
              const float mean = s_o[d * kExTN + tid];
              const float ls = fminf(fmaxf(s_o[(AD + d) * kExTN + tid], -20.f), 2.f);
              a = tanhf(fmaf(expf(ls), z[k], mean));
            }
            ao[d] = a;
          }
        }
        const uint4 x = philox4x32_10(env, step, 0u, STREAM_REWDONE, p.k0, p.k1);
        reward = (float)(x.x & 1u);
        done = x.y < p.done_thr;
        const bool time_limit = p.max_steps > 0 && p.st.ep_len[b] + 1 >= p.max_steps;
        p.rm_rew[row] = reward;
        p.rm_term[row] = (done && !time_limit) ? 1 : 0;
        done = done || time_limit;
      }
      episode_update(p.st, b, valid, reward, done);
    }
    __syncthreads();                               // s_x (and the head's outputs) read before they are replaced
    // next observation of every env (each CTA keeps its own copy), one Box-Muller block per task
    const int nblk = (D + 3) >> 2;
    for (int task = tid; task < kExTN * nblk; task += kExThreads) {
      const int blk = task / kExTN, n = task - blk * kExTN;
      const int b = n0 + n;
      if (b >= B) continue;
      float z[4];
      gauss_block(p.env_offset + (uint32_t)b, step + 1u, (uint32_t)blk, STREAM_OBS, p.k0, p.k1, z);
      const size_t row = ((size_t)p.pos + (size_t)t * B + b) % (size_t)p.cap;
#pragma unroll
      for (int k = 0; k < 4 && blk * 4 + k < D; ++k) {
        const int d = blk * 4 + k;
        s_x[d * kExXS + n] = z[k];
        if (rank == 0) p.rm_next[row * D + d] = z[k];
      }
    }
    __syncthreads();
  }
  if (rank == 0) {
    for (int i = tid; i < kExTN * D; i += kExThreads) {
      const int n = i / D, k = i - n * D;
      if (n0 + n < B) p.obs_cur[(size_t)(n0 + n) * D + k] = s_x[k * kExXS + n];
    }
  }
  ex_cluster_sync();                               // no CTA leaves while a peer may still store into it
}

// shared-memory bytes of the explore kernel with cluster size C (0: does not fit the shape limits)
static size_t explore_layout(ExploreArgs& a, int C, bool with_weights) {
  a.C = C;
  int off = 0, H = 4;
  for (int l = 0; l < a.L; ++l) {
    a.inp[l] = (a.dims[l] + 3) & ~3;
    const int per = (a.dims[l + 1] + C - 1) / C;
    a.R[l] = (per + 3) & ~3;
    a.w_off[l] = off;
    off += (a.inp[l] + 1) * a.R[l];
    if (l + 1 < a.L) H = max(H, C * a.R[l]);
  }
  // without the actor (mode 0) only the observation tile is used
  a.w_floats = with_weights ? off : 0;
  a.H = with_weights ? H : 0;
  a.O = with_weights ? C * a.R[a.L - 1] : 0;
  const int Dp = (a.dims[0] + 3) & ~3;
  return ((size_t)a.w_floats + (size_t)Dp * kExXS + (2 * (size_t)a.H + a.O) * kExTN) * sizeof(float);
}

// ---------------------------------------------------------------------------------------------------------------
// Uniform replay sampling: row i of draw d = (x * size) >> 32 with x = word 0 of philox(i, d, 0, STREAM_REPLAY);
// one warp per sampled row gathers obs / action / next_obs and widens reward / terminal to float32.
struct ReplaySampleArgs {
  const float* obs;
  const float* act;
  const float* rew;
  const int* term;
  const float* next;
  int D, AD, n, cap;
  const int* size_dev;
  const int* draw_dev;
  uint32_t k0, k1;
  float* obs_out;
  float* act_out;
  float* rew_out;
  float* term_out;
  float* next_out;
  int* idx_out;
};

__global__ void __launch_bounds__(256) replay_sample_uniform_kernel(const ReplaySampleArgs p) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= p.n) return;
  const uint32_t size = (uint32_t)min(max(*p.size_dev, 1), p.cap);     // never past the ring's last row
  const uint32_t d = (uint32_t)*p.draw_dev;
  const uint4 x = philox4x32_10((uint32_t)i, d, 0u, STREAM_REPLAY, p.k0, p.k1);
  const size_t row = (size_t)(((uint64_t)x.x * (uint64_t)size) >> 32);
  for (int k = lane; k < p.D; k += 32) {
    p.obs_out[(size_t)i * p.D + k] = p.obs[row * p.D + k];
    p.next_out[(size_t)i * p.D + k] = p.next[row * p.D + k];
  }
  for (int k = lane; k < p.AD; k += 32) p.act_out[(size_t)i * p.AD + k] = p.act[row * p.AD + k];
  if (lane == 0) {
    p.rew_out[i] = p.rew[row];
    p.term_out[i] = p.term[row] != 0 ? 1.f : 0.f;
    if (p.idx_out) p.idx_out[i] = (int)row;
  }
}

}  // namespace rl

extern "C" int rl_explore_mlp(int n_layers, const int* dims, int n_seg, const int* seg_layer, const int* seg_rows,
                              const float* const* seg_w, const float* const* seg_b, int head, int mode, int K, int B,
                              int action_dim, float expl_noise, float* obs_cur, float* ep_ret, int32_t* ep_len,
                              float* totals, float* ring_ret, int32_t* ring_len, uint32_t* ring_head, int ring_cap,
                              uint64_t seed, uint32_t step0, uint32_t env_offset, float p_done, int max_episode_steps,
                              float* rm_obs, float* rm_action, float* rm_reward, int32_t* rm_terminal,
                              float* rm_next_obs, int rm_max_size, int rm_pos, rl_stream_t stream) {
  using namespace rl;
  RL_CHECK_ARG(dims && seg_layer && seg_rows && seg_w && obs_cur && ep_ret && ep_len && totals && rm_obs && rm_action &&
                   rm_reward && rm_terminal && rm_next_obs,
               "explore_mlp: null pointer");
  RL_CHECK_ARG(n_layers >= 2 && n_layers <= kExMaxLayers, "explore_mlp: %d layers (1..%d hidden layers + head)", n_layers,
               kExMaxLayers - 1);
  RL_CHECK_ARG(n_seg >= n_layers && n_seg <= kExMaxSeg, "explore_mlp: %d parameter segments (need %d..%d)", n_seg,
               n_layers, kExMaxSeg);
  RL_CHECK_ARG(head == 0 || head == 1, "explore_mlp: head %d not in {0 tanh, 1 mean|log-std}", head);
  RL_CHECK_ARG(mode >= 0 && mode <= 2, "explore_mlp: mode %d not in {0 warm-up, 1 deterministic + noise, 2 SAC}", mode);
  RL_CHECK_ARG(mode != 1 || head == 0, "explore_mlp: mode 1 needs the tanh head");
  RL_CHECK_ARG(mode != 2 || head == 1, "explore_mlp: mode 2 needs the mean|log-std head");
  RL_CHECK_ARG(K >= 1 && B >= 1 && action_dim >= 1, "explore_mlp: K=%d B=%d action_dim=%d", K, B, action_dim);
  RL_CHECK_ARG(rm_max_size >= 1 && rm_pos >= 0 && rm_pos < rm_max_size, "explore_mlp: replay pos %d / size %d", rm_pos,
               rm_max_size);
  RL_CHECK_ARG((long long)K * B <= rm_max_size,
               "explore_mlp: K*B = %lld transitions exceed the replay capacity %d (a launch would overwrite its own rows)",
               (long long)K * B, rm_max_size);
  ExploreArgs a;
  memset(&a, 0, sizeof(a));
  a.L = n_layers, a.n_seg = n_seg;
  for (int l = 0; l <= n_layers; ++l) {
    RL_CHECK_ARG(dims[l] >= 1 && dims[l] <= kExMaxWidth, "explore_mlp: width %d of layer %d outside 1..%d", dims[l], l,
                 kExMaxWidth);
    a.dims[l] = dims[l];
  }
  RL_CHECK_ARG(dims[n_layers] == (head == 0 ? action_dim : 2 * action_dim),
               "explore_mlp: actor has %d outputs, head %d with action_dim %d needs %d", dims[n_layers], head,
               action_dim, head == 0 ? action_dim : 2 * action_dim);
  int rows_seen[kExMaxLayers] = {0, 0, 0, 0};
  for (int s = 0; s < n_seg; ++s) {
    const int l = seg_layer[s];
    RL_CHECK_ARG(l >= 0 && l < n_layers && seg_rows[s] >= 1 && seg_w[s], "explore_mlp: bad segment %d", s);
    a.seg[s].w = seg_w[s], a.seg[s].b = seg_b ? seg_b[s] : nullptr;
    a.seg[s].layer = l, a.seg[s].row0 = rows_seen[l], a.seg[s].rows = seg_rows[s];
    rows_seen[l] += seg_rows[s];
  }
  for (int l = 0; l < n_layers; ++l)
    RL_CHECK_ARG(rows_seen[l] == dims[l + 1], "explore_mlp: segments of layer %d cover %d of %d rows", l, rows_seen[l],
                 dims[l + 1]);
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = (B + kExTN - 1) / kExTN;
  // cluster size: the smallest that holds the actor, doubled while the grid leaves SMs idle
  int C = 1;
  size_t smem = 0;
  if (mode == 0) {
    smem = explore_layout(a, 1, false);
  } else {
    while (C <= kExMaxCluster && explore_layout(a, C, true) > kExSmemLimit) C *= 2;
    RL_CHECK_ARG(C <= kExMaxCluster, "explore_mlp: actor too large for a %d-CTA cluster (%zu B of shared memory)",
                 kExMaxCluster, explore_layout(a, kExMaxCluster, true));
    while (C < kExMaxCluster && tiles * C < nsm) C *= 2;
    smem = explore_layout(a, C, true);
  }
  a.head = head, a.mode = mode, a.K = K, a.B = B, a.AD = action_dim, a.D = dims[0], a.max_steps = max_episode_steps;
  a.sigma = expl_noise, a.obs_cur = obs_cur;
  a.st = make_episode_stats(ep_ret, ep_len, totals, ring_ret, ring_len, ring_head, ring_cap);
  a.k0 = (uint32_t)seed, a.k1 = (uint32_t)(seed >> 32), a.step0 = step0, a.env_offset = env_offset;
  a.done_thr = prob_threshold(p_done);
  a.rm_obs = rm_obs, a.rm_act = rm_action, a.rm_rew = rm_reward, a.rm_term = rm_terminal, a.rm_next = rm_next_obs;
  a.cap = rm_max_size, a.pos = rm_pos;
  RL_SMEM_OPTIN(explore_mlp_kernel);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(tiles * a.C), 1, 1);
  cfg.blockDim = dim3(kExThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)a.C, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr, cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, explore_mlp_kernel, a) != cudaSuccess) {
    set_error("explore_mlp: launch failed (cluster %d, %zu B shared memory): %s", a.C, smem,
              cudaGetErrorString(cudaGetLastError()));
    return RL_ERR_CUDA;
  }
  return RL_OK;
}

extern "C" int rl_replay_sample_uniform(const float* obs, const float* action, const float* reward,
                                        const int32_t* terminal, const float* next_obs, int obs_dim, int act_dim,
                                        const int32_t* size_dev, const int32_t* draw_dev, int capacity, int n,
                                        uint64_t seed,
                                        float* obs_out, float* action_out, float* reward_out, float* terminal_out,
                                        float* next_obs_out, int32_t* idx_out, rl_stream_t stream) {
  using namespace rl;
  RL_CHECK_ARG(obs && action && reward && terminal && next_obs && size_dev && draw_dev && obs_out && action_out &&
                   reward_out && terminal_out && next_obs_out,
               "replay_sample_uniform: null pointer");
  RL_CHECK_ARG(n >= 1 && obs_dim >= 1 && act_dim >= 1 && capacity >= 1,
               "replay_sample_uniform: n=%d obs_dim=%d act_dim=%d capacity=%d", n, obs_dim, act_dim, capacity);
  ReplaySampleArgs a;
  a.obs = obs, a.act = action, a.rew = reward, a.term = terminal, a.next = next_obs;
  a.D = obs_dim, a.AD = act_dim, a.n = n, a.cap = capacity, a.size_dev = size_dev, a.draw_dev = draw_dev;
  a.k0 = (uint32_t)seed, a.k1 = (uint32_t)(seed >> 32);
  a.obs_out = obs_out, a.act_out = action_out, a.rew_out = reward_out, a.term_out = terminal_out;
  a.next_out = next_obs_out, a.idx_out = idx_out;
  replay_sample_uniform_kernel<<<(n + 7) / 8, 256, 0, (cudaStream_t)stream>>>(a);
  RL_CHECK_LAUNCH("rl_replay_sample_uniform");
  return RL_OK;
}
