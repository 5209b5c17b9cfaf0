// Rollout collection fused into one kernel (BASELINE configs[4]; SURVEY section 3.6 / a15): what rllab's
// BatchSampler does around the reference env, one Python call and twelve FFI calls per policy step
// (rllab/envs/trpo_cassie.py:13-55 -> rollout() -> GaussianMLPPolicy.get_action -> NormalizedEnv.step
// -> Cassie2dEnv.step), here T policy steps per launch for every env:
//   obs -> tanh MLP (26|17 -> 32 -> 32 -> adim) -> a = mean + exp(log_std) * eps -> NormalizedEnv affine
//   map + clip -> n_substeps x Step* -> obs / reward / done -> auto-reset at done or max_path_length.
// The policy is 2.0 k MAC per policy step against ~0.5 MFLOP for the ten simulator steps it drives
// (0.4 %), so it runs as per-thread FP32 FMAs with the weights broadcast from shared memory; a
// tensor-core tile for a [N x 32] x [32 x 32] product would be launch- and fill-latency bound
// (DESIGN.md section 9).  eps comes from Philox4x32-10 keyed by (seed, global env id, policy step), so
// results do not depend on the launch partition or the GPU count.
#pragma once
#include "env_kernels.cuh"
#include "rollout_philox.cuh"
#include "rollout_args.h"
#include <cstdlib>
#include <cstring>

namespace cassie {

constexpr int kHidden = 32;  // hidden_sizes=(32, 32), trpo_cassie.py:24

// ---- tensor-core variant of the policy forward (A/B of VERDICT r1 item 8; CASSIE_MLP=tc, fp32 builds, thread engine)
// One warp = 32 envs = the M dimension: H[32 x 32] = X[32 x K] W[K x 32] as mma.sync m16n8k8 TF32 tiles, every product
// split 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo) so that the result keeps fp32 accuracy (the parity bar against the
// PyTorch fp32 reference is 1e-5; plain TF32 gives 1e-3).  Activations stay feature-major in shared memory
// ([feature][env], the layout the scalar path stages the observation in), two buffers in ping-pong.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hi) : "f"(x));
  const float r = x - __uint_as_float(hi);
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lo) : "f"(r));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// out[j][env] = act(sum_i xs[i][env] w[i * ldw + j] + bias[j]) for the warp's 32 envs; NT = n-tiles of 8 outputs
template <int NT, bool TANH>
__device__ __forceinline__ void warp_dense_tc(const float* xs, int ldx, int K, const float* w, int ldw, int N, const float* bias,
                                              float* out, int ldo) {
  const int lane = (int)(threadIdx.x & 31u), g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; mt++) {
    float acc[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
      const int j0 = 8 * nt + 2 * t;
      const float b0 = j0 < N ? bias[j0] : 0.0f, b1 = j0 + 1 < N ? bias[j0 + 1] : 0.0f;
      acc[nt][0] = b0; acc[nt][1] = b1; acc[nt][2] = b0; acc[nt][3] = b1;
    }
    for (int kt = 0; 8 * kt < K; kt++) {
      const int i0 = 8 * kt + t, i1 = i0 + 4, r0 = 16 * mt + g;
      const float a0 = i0 < K ? xs[i0 * ldx + r0] : 0.0f, a1 = i0 < K ? xs[i0 * ldx + r0 + 8] : 0.0f;
      const float a2 = i1 < K ? xs[i1 * ldx + r0] : 0.0f, a3 = i1 < K ? xs[i1 * ldx + r0 + 8] : 0.0f;
      uint32_t ah[4], al[4];
      split_tf32(a0, ah[0], al[0]); split_tf32(a1, ah[1], al[1]); split_tf32(a2, ah[2], al[2]); split_tf32(a3, ah[3], al[3]);
#pragma unroll
      for (int nt = 0; nt < NT; nt++) {
        const int j = 8 * nt + g;
        const float w0 = (i0 < K && j < N) ? w[i0 * ldw + j] : 0.0f, w1 = (i1 < K && j < N) ? w[i1 * ldw + j] : 0.0f;
        uint32_t bh[2], bl[2];
        split_tf32(w0, bh[0], bl[0]); split_tf32(w1, bh[1], bl[1]);
        mma_tf32(acc[nt], al, bh);
        mma_tf32(acc[nt], ah, bl);
        mma_tf32(acc[nt], ah, bh);
      }
    }
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
      const int j0 = 8 * nt + 2 * t, r0 = 16 * mt + g;
      float c0 = acc[nt][0], c1 = acc[nt][1], c2 = acc[nt][2], c3 = acc[nt][3];
      if (TANH) { c0 = tanhf(c0); c1 = tanhf(c1); c2 = tanhf(c2); c3 = tanhf(c3); }
      if (j0 < N) { out[j0 * ldo + r0] = c0; out[j0 * ldo + r0 + 8] = c2; }
      if (j0 + 1 < N) { out[(j0 + 1) * ldo + r0] = c1; out[(j0 + 1) * ldo + r0 + 8] = c3; }
    }
  }
  __syncwarp();
}

template <typename T>
struct RolloutDev {
  int task, flags, n_sub, T_steps, max_path_length, normalize, mlp_tc;
  uint64_t seed;
  uint32_t env0;       // global id of this batch's env 0
  const T* params;     // flat [W1(in x 32) | b1 | W2(32 x 32) | b2 | W3(32 x adim) | b3 | log_std(adim)]  (Lasagne order)
  T* obs;              // [T][n][odim]
  T* act;              // [T][n][adim]  raw policy actions (what rllab stores in paths)
  T* mean;             // [T][n][adim]  agent_infos["mean"]
  T* rew;              // [T][n]
  uint8_t* done;       // [T][n]  1 = env terminated, 2 = max_path_length reached
  T act_lo[7], act_hi[7];
  T reset_state[26];
};

template <typename T, int MODE>
__global__ void __launch_bounds__(kBlock, CASSIE_MIN_BLOCKS) k_rollout(const __grid_constant__ ModelPair<T> mp, const BatchView<T> v,
                                                     const __grid_constant__ RolloutDev<T> a) {
  constexpr int adim = action_dim(MODE);
  const int odim = a.task == kTaskStand ? 17 : 26;
  extern __shared__ unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  const int n_params = odim * kHidden + kHidden + kHidden * kHidden + kHidden + kHidden * adim + adim + adim;
  for (int i = threadIdx.x; i < n_params; i += kBlock) sp[i] = a.params[i];
  T* sobs = sp + n_params;  // [26][kBlock] per-thread observation staging (+ [32][kBlock] hidden buffer, tensor-core variant)
  T* shid = sobs + 26 * kBlock;
  __syncthreads();
  const T* W1 = sp; const T* b1 = W1 + odim * kHidden; const T* W2 = b1 + kHidden; const T* b2 = W2 + kHidden * kHidden;
  const T* W3 = b2 + kHidden; const T* b3 = W3 + kHidden * adim; const T* lstd = b3 + adim;

  const int e = blockIdx.x * kBlock + threadIdx.x;
  if (e >= v.n) return;
  T q[kNV], qd[kNV], w[kNV], u[kNU];
  load_env(v, e, q, qd, w);
  alignas(16) Rows<T> rows;
  OpState<T> op;
  load_op(v, e, op);
  StepStats st = {0, 0, 0u};
  OscStats qs = {0, 0};
  double t = v.clock[e];
  unsigned qps = v.qp_set[e];
  int ep_len = v.ep_len[e];
  uint32_t pstep = (uint32_t)v.policy_step[e];
  const size_t n = (size_t)v.n;
  int n_diverged = 0;

  for (int k = 0; k < a.T_steps; k++) {
    // ---- observation of the current state (what the previous step / reset returned)
    T o18[18], ref9[9];
    op_state_array(op, q, qd, o18);
    const bool fresh = ep_len == 0;   // the observation env.reset() returned: reference slots are zero (cassie2d.py:78-95)
    write_obs(v, a.task, e, o18, t, a.obs + (size_t)k * n * odim, ref9, fresh);
    {
      T o[17];
      pos_invariant_obs(o18, o);
#pragma unroll
      for (int i = 0; i < 17; i++) sobs[i * kBlock + threadIdx.x] = o[i];
      if (a.task != kTaskStand) {
#pragma unroll
        for (int i = 0; i < 9; i++) sobs[(17 + i) * kBlock + threadIdx.x] = fresh ? T(0) : ref9[i];
      }
    }
    // ---- GaussianMLPPolicy forward: tanh hidden layers, linear mean head (trpo_cassie.py:21-27)
    T mu[adim], act[7];
    bool mlp_done = false;
    if constexpr (sizeof(T) == 4) {
      if (a.mlp_tc) {
        // whole warps only (the host enables this variant when n % 32 == 0): 32 envs x 32 hidden units per warp
        const int wb = (int)(threadIdx.x & ~31u);
        float* xs = reinterpret_cast<float*>(sobs) + wb;
        float* hs = reinterpret_cast<float*>(shid) + wb;
        __syncwarp();
        warp_dense_tc<4, true>(xs, kBlock, odim, (const float*)W1, kHidden, kHidden, (const float*)b1, hs, kBlock);
        warp_dense_tc<4, true>(hs, kBlock, kHidden, (const float*)W2, kHidden, kHidden, (const float*)b2, xs, kBlock);
        warp_dense_tc<1, false>(xs, kBlock, kHidden, (const float*)W3, adim, adim, (const float*)b3, hs, kBlock);
#pragma unroll
        for (int c = 0; c < adim; c++) mu[c] = (T)hs[c * kBlock + (threadIdx.x & 31u)];
        __syncwarp();
        mlp_done = true;
      }
    }
    if (!mlp_done) {
    T h1[kHidden], h2[kHidden];
#pragma unroll
    for (int j = 0; j < kHidden; j++) h1[j] = b1[j];
    for (int i = 0; i < odim; i++) {
      const T x = sobs[i * kBlock + threadIdx.x];
#pragma unroll
      for (int j = 0; j < kHidden; j++) h1[j] += x * W1[i * kHidden + j];
    }
#pragma unroll
    for (int j = 0; j < kHidden; j++) { h1[j] = tanh(h1[j]); h2[j] = b2[j]; }
#pragma unroll
    for (int i = 0; i < kHidden; i++) {
#pragma unroll
      for (int j = 0; j < kHidden; j++) h2[j] += h1[i] * W2[i * kHidden + j];
    }
#pragma unroll
    for (int j = 0; j < kHidden; j++) h2[j] = tanh(h2[j]);
#pragma unroll
    for (int c = 0; c < adim; c++) {
      T s = b3[c];
#pragma unroll
      for (int i = 0; i < kHidden; i++) s += h2[i] * W3[i * adim + c];
      mu[c] = s;
    }
    }
    // ---- a = mean + exp(log_std) * eps ; NormalizedEnv: lb + (a + 1) / 2 (ub - lb), clipped (trpo_cassie.py:13)
    T eps[8];
    normal8(a.seed, a.env0 + (uint32_t)e, pstep, eps);
#pragma unroll
    for (int c = 0; c < adim; c++) {
      const T raw = mu[c] + exp(lstd[c]) * eps[c];
      a.act[((size_t)k * n + e) * adim + c] = raw;
      a.mean[((size_t)k * n + e) * adim + c] = mu[c];
      T x = raw;
      if (a.normalize) x = a.act_lo[c] + (raw + T(1)) * T(0.5) * (a.act_hi[c] - a.act_lo[c]);
      act[c] = x < a.act_lo[c] ? a.act_lo[c] : (x > a.act_hi[c] ? a.act_hi[c] : x);
    }
    // ---- Cassie2dEnv.step(action, n)
    for (int s = 0; s < a.n_sub; s++) {
      controller_step<MODE>(mp.phys, mp.phys_d, ctrl_model<MODE>(mp), mp.ctrl_d, q, qd, w, act, rows, u, s == a.n_sub - 1 ? &op : nullptr, &st, &qs, &qps);
      t += 0.0005;
    }
    T r;
    int done;
    const bool diverged = state_diverged(q, qd);   // mj_checkPos/Vel/Acc [EXT]: report done, reset, flag in stats
    op_state_array(op, q, qd, o18);
    if (a.task == kTaskStand) {
      T o[17];
      pos_invariant_obs(o18, o);
      stand_reward(o18, o, act, adim, r, done);
    } else {
      const int idx9[9] = {0, 1, 2, 3, 4, 6, 8, 9, 11};
      const int row = v.traj ? traj_index(t, v.traj_tmax, v.traj_rows) : 0;
#pragma unroll
      for (int i = 0; i < 9; i++) ref9[i] = v.traj ? (T)v.traj[(size_t)row * 13 + idx9[i]] : T(0);
      const T jsum = (a.flags & 4) ? q[3] + q[4] + q[6] + q[8] + q[9] + q[11] : v.jsum0[e];
      imitate_reward(o18, ref9, jsum, r, done);
    }
    if (diverged) { r = T(0); done = 1; qs.status = kStatusDiverged; n_diverged++; }
    ep_len++;
    pstep++;
    int flag = done ? 1 : (ep_len >= a.max_path_length ? 2 : 0);
    a.rew[(size_t)k * n + e] = r;
    a.done[(size_t)k * n + e] = (uint8_t)flag;
    if (flag) {  // rollout(): the path ends, the sampler calls env.reset()
      state26_to_q(a.reset_state, q, qd);
      t = 0.0;
      ep_len = 0;
      v.jsum0[e] = q[3] + q[4] + q[6] + q[8] + q[9] + q[11];
      if ((a.flags & 2) || diverged) {
        Kin<T> kc;
        forward_kinematics(mp.ctrl, q, qd, kc);
        op_state_from_kin(mp.ctrl, kc, q, op);
      }
      if (diverged) {
#pragma unroll
        for (int i = 0; i < kNV; i++) w[i] = T(0);
        qps = 0u;
      }
    }
  }
  v.clock[e] = t;
  v.qp_set[e] = qps;
  v.ep_len[e] = ep_len;
  v.policy_step[e] = (int32_t)pstep;
  store_env(v, e, q, qd, w);
  store_op(v, e, op);
  if (n_diverged) qs.status = kStatusDiverged;   // sticky for the launch: the env diverged and was reset at least once
  store_stats(v.stats, v.n, e, st, qs);
}


// Discounted returns of the collected paths, R_t = r_t + gamma * R_{t+1} within a path (rllab
// special.discount_cumsum applied per path in BatchPolopt.process_samples [EXT]; discount = 0.99,
// trpo_cassie.py:38).  One thread per env scans its column of the [T][n] buffers backwards; a path
// boundary (done != 0) restarts the sum.  tail[n] (optional) = value to bootstrap the last,
// unfinished path of each env with (0 when null).
template <typename T>
__global__ void __launch_bounds__(128) k_discounted_returns(const T* __restrict__ rew, const uint8_t* __restrict__ done,
                                                            const T* __restrict__ tail, T gamma, int T_steps, int n, T* __restrict__ ret) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  T acc = tail ? tail[e] : T(0);
  for (int k = T_steps - 1; k >= 0; k--) {
    const size_t i = (size_t)k * n + e;
    acc = rew[i] + (done[i] ? T(0) : gamma * acc);
    ret[i] = acc;
  }
}
template <typename T>
cudaError_t launch_discounted_returns(const void* rew, const uint8_t* done, const void* tail, double gamma, int T_steps, int n,
                                      void* ret, cudaStream_t s) {
  k_discounted_returns<T><<<grid_for(n, 128), 128, 0, s>>>((const T*)rew, done, (const T*)tail, (T)gamma, T_steps, n, (T*)ret);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// LinearFeatureBaseline + advantages (rllab [EXT], used by trpo_cassie.py:29-41): features of a sample =
// [clip(o, -10, 10), clip(o)^2, al, al^2, al^3, 1] with al = (step index within its path) / 100.
// k_path_index recovers the in-path step index from the done flags; k_baseline_moments accumulates the
// normal equations F'F (D x D) and F'y (D) over all T x n samples (the D x D solve itself is host-side
// glue on 38 x 38 numbers); k_advantages evaluates the baseline and runs the backward GAE scan
//   delta_t = r_t + gamma V_{t+1} - V_t,  A_t = delta_t + gamma lambda A_{t+1}   (V = 0 past a path end).
// The capacities are template parameters: the planar observations below, the 3-D one in rollout_args.h.
constexpr int kMaxFeat = 2 * 26 + 4, kMomentsPerThread = 8;

template <typename T>
__device__ __forceinline__ void baseline_features(const T* __restrict__ o, int odim, int step_in_path, T* f) {
  for (int i = 0; i < odim; i++) {
    T x = o[i];
    x = x < T(-10) ? T(-10) : (x > T(10) ? T(10) : x);
    f[i] = x;
    f[odim + i] = x * x;
  }
  const T al = (T)step_in_path / T(100);
  f[2 * odim] = al; f[2 * odim + 1] = al * al; f[2 * odim + 2] = al * al * al; f[2 * odim + 3] = T(1);
}

// in-path step index of every sample; start[n] (in/out, optional) carries the index across collect() calls
template <typename T>
__global__ void __launch_bounds__(128) k_path_index(const uint8_t* __restrict__ done, int T_steps, int n, const int32_t* start,
                                                    int32_t* __restrict__ idx) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int k = start ? start[e] : 0;
  for (int t = 0; t < T_steps; t++) {
    idx[(size_t)t * n + e] = k;
    k = done[(size_t)t * n + e] ? 0 : k + 1;
  }
}

// one CTA per chunk of samples: features staged in shared memory, thread p owns entries p, p + 256, ... of
// the packed upper triangle (+ the F'y column); double accumulation, one atomicAdd per entry per CTA.
// MAXF = feature capacity (D <= MAXF), EPT = entries per thread (D (D + 1) / 2 + D <= 256 EPT).
template <typename T, int MAXF, int EPT>
__global__ void __launch_bounds__(256) k_baseline_moments(const T* __restrict__ obs, const T* __restrict__ ret,
                                                          const int32_t* __restrict__ idx, int odim, long n_samples,
                                                          int chunk, double* __restrict__ out) {
  const int D = 2 * odim + 4, n_ent = D * (D + 1) / 2 + D;
  __shared__ T sf[32][MAXF + 1];
  double acc[EPT];
#pragma unroll
  for (int q = 0; q < EPT; q++) acc[q] = 0.0;
  const long s0 = (long)blockIdx.x * chunk, s1 = s0 + chunk < n_samples ? s0 + chunk : n_samples;
  for (long base = s0; base < s1; base += 32) {
    const int cnt = (int)(s1 - base < 32 ? s1 - base : 32);
    __syncthreads();
    if (threadIdx.x < cnt) {
      const long smp = base + threadIdx.x;
      baseline_features(obs + smp * odim, odim, idx[smp], sf[threadIdx.x]);
      sf[threadIdx.x][D] = ret[smp];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < EPT; q++) {
      const int p = threadIdx.x + 256 * q;
      if (p < n_ent) {
        int i, j;  // entry p -> (i, j): packed rows of the upper triangle, then the F'y column (j = D)
        if (p < D * (D + 1) / 2) {
          i = 0; int rem = p;
          while (rem >= D - i) { rem -= D - i; i++; }
          j = i + rem;
        } else { i = p - D * (D + 1) / 2; j = D; }
        double sacc = 0.0;
        for (int c = 0; c < cnt; c++) sacc += (double)sf[c][i] * (double)sf[c][j];
        acc[q] += sacc;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < EPT; q++) {
    const int p = threadIdx.x + 256 * q;
    if (p < n_ent) atomicAdd(out + p, acc[q]);
  }
}

template <typename T, int MAXF>
__global__ void __launch_bounds__(128) k_advantages(const T* __restrict__ obs, const T* __restrict__ rew,
                                                    const uint8_t* __restrict__ done, const int32_t* __restrict__ idx,
                                                    const T* __restrict__ coeffs, int odim, T gamma, T lambda, int T_steps, int n,
                                                    T* __restrict__ adv, T* __restrict__ value) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const int D = 2 * odim + 4;
  T f[MAXF];
  T v_next = T(0), a_next = T(0);
  for (int t = T_steps - 1; t >= 0; t--) {
    const size_t i = (size_t)t * n + e;
    baseline_features(obs + i * odim, odim, idx[i], f);
    T v = T(0);
    for (int c = 0; c < D; c++) v += f[c] * coeffs[c];
    if (done[i]) { v_next = T(0); a_next = T(0); }   // np.append(baseline, 0): nothing beyond a path end
    const T delta = rew[i] + gamma * v_next - v;
    const T a = delta + gamma * lambda * a_next;
    adv[i] = a;
    if (value) value[i] = v;
    v_next = v; a_next = a;
  }
}

template <typename T, int MAXF, int EPT>
cudaError_t launch_baseline_moments(const BaselineArgs& a, cudaStream_t s) {
  k_path_index<T><<<grid_for(a.n, 128), 128, 0, s>>>(a.done, a.T_steps, a.n, a.start, a.idx);
  const long n_samples = (long)a.T_steps * a.n;
  const int chunk = 4096;
  const int D = 2 * a.odim + 4;
  cudaError_t e = cudaMemsetAsync(a.moments, 0, sizeof(double) * (D * (D + 1) / 2 + D), s);
  if (e != cudaSuccess) return e;
  k_baseline_moments<T, MAXF, EPT><<<(unsigned)((n_samples + chunk - 1) / chunk), 256, 0, s>>>((const T*)a.obs, (const T*)a.ret, a.idx, a.odim,
                                                                                  n_samples, chunk, a.moments);
  count_launch(); count_launch();
  return cudaGetLastError();
}
template <typename T, int MAXF>
cudaError_t launch_advantages(const BaselineArgs& a, cudaStream_t s) {
  k_advantages<T, MAXF><<<grid_for(a.n, 128), 128, 0, s>>>((const T*)a.obs, (const T*)a.rew, a.done, a.idx, (const T*)a.coeffs, a.odim,
                                                    (T)a.gamma, (T)a.lambda, a.T_steps, a.n, (T*)a.adv, (T*)a.value);
  count_launch();
  return cudaGetLastError();
}
// the planar observations (batch_state.h)
template <typename T>
cudaError_t launch_baseline_moments(const BaselineArgs& a, cudaStream_t s) {
  return launch_baseline_moments<T, kMaxFeat, kMomentsPerThread>(a, s);
}
template <typename T>
cudaError_t launch_advantages(const BaselineArgs& a, cudaStream_t s) {
  return launch_advantages<T, kMaxFeat>(a, s);
}

template <typename T>
RolloutDev<T> make_rollout_dev(const RolloutArgs& a) {
  RolloutDev<T> d;
  d.task = a.task; d.flags = a.flags; d.n_sub = a.n_substeps; d.T_steps = a.T_steps; d.max_path_length = a.max_path_length;
  d.normalize = a.normalize; d.seed = a.seed; d.env0 = a.env0;
  d.mlp_tc = 0;
  d.params = (const T*)a.params; d.obs = (T*)a.obs; d.act = (T*)a.act; d.mean = (T*)a.mean; d.rew = (T*)a.rew; d.done = a.done;
  for (int i = 0; i < 7; i++) { d.act_lo[i] = (T)a.act_lo[i]; d.act_hi[i] = (T)a.act_hi[i]; }
  const double qi[26] = {0.0, 0.939, 0.0, 0.0, 0.0, 0.0, 0.68111815, -1.40730357, 1.62972042, -1.77611107, -0.61968407,
                         0.0, 0.0, 0.0, 0.0, 0.0, 0.68111815, -1.40730357, 1.62972042, -1.77611107, -0.61968407,
                         0.0, 0.0, 0.0, 0.0, 0.0};
  for (int i = 0; i < 26; i++) d.reset_state[i] = (T)qi[i];
  return d;
}
// thread-per-env launcher (rollout_launch.cuh picks between this and the quad engine's)
template <typename T>
cudaError_t thread_rollout(const ModelPair<T>& mp, const BatchView<T>& v, const RolloutArgs& a, cudaStream_t s) {
  const RolloutDev<T> d = make_rollout_dev<T>(a);
  const int odim = a.task == kTaskStand ? 17 : 26, adim = action_dim(a.mode);
  const int n_params = odim * kHidden + kHidden + kHidden * kHidden + kHidden + kHidden * adim + adim + adim;
  RolloutDev<T> dd = d;
  if (const char* e = getenv("CASSIE_MLP")) dd.mlp_tc = (strcmp(e, "tc") == 0 && sizeof(T) == 4 && v.n % 32 == 0) ? 1 : 0;
  const size_t smem = sizeof(T) * (size_t)(n_params + (26 + 32) * kBlock);
  const unsigned g = grid_for(v.n, kBlock);
  switch (a.mode) {
    case kModeTorque: k_rollout<T, kModeTorque><<<g, kBlock, smem, s>>>(mp, v, dd); break;
    case kModePd: k_rollout<T, kModePd><<<g, kBlock, smem, s>>>(mp, v, dd); break;
    case kModeOsc: k_rollout<T, kModeOsc><<<g, kBlock, smem, s>>>(mp, v, dd); break;
    default: return cudaErrorInvalidValue;
  }
  count_launch();
  return cudaGetLastError();
}

}  // namespace cassie
