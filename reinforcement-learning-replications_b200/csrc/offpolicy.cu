// Off-policy update engine: DDPG / TD3 train() on device-resident minibatches.
//
// Replaces (reference: /root/reference/src/rl_replicas/): algorithms/td3.py:214-358 (train, train_policy,
// compute_targets, train_q_function), algorithms/ddpg.py:195-293, q_function.py:20-32, policies/
// deterministic_policy.py:23-32, utils.py:47-57 (polyak_average), and the torch.optim.Adam steps inside them.
//
// Regime: minibatch B ~ 100-256 rows, 256-wide ReLU MLPs (~70k parameters each): ~0.5 GFLOP per train step, i.e.
// launch-latency bound, not throughput bound (SURVEY 7.3-8).  The design therefore minimises host involvement:
// ALL `num_train_steps` minibatches (and the target-smoothing noise) are uploaded once, every step runs as a fixed
// sequence of small fp32 kernels with no host synchronisation, and losses / Q-values are read back once at the end.
// GEMMs are one generic 32x32x32 shared-memory-tiled fp32 kernel in three operand arrangements (forward NT, dX NN,
// dW TN) with the activation derivative fused into the operand load, so activations are never rewritten; torch.cat of
// [s | a] is a split operand, the target-smoothing noise an epilogue.  File map: tile function and elementwise kernels;
// the opt-in persistent step kernel (offpolicy_mega_kernel) and its program builder; the engine (one state slab);
// enqueue_steps = the S steps as a four-stream dependency graph (captured once, replayed); the three entry points
// train (host-staged minibatches), train_gather (host-drawn indices, device gather), train_gather_rng (device draws).
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace b200rl {

constexpr int GT = 32;   // output tile (256x256 outputs -> 64 CTAs; the batch is small, parallelism matters more than reuse)
constexpr int GK = 32;   // k tile
constexpr int GTHREADS = 256;

__device__ __forceinline__ float op_act(float z, int kind) {
  if (kind == B200RL_ACT_TANH) return tanhf(z);
  if (kind == B200RL_ACT_RELU) return fmaxf(z, 0.f);
  return z;
}
__device__ __forceinline__ float op_act_prime(float y, int kind) {  // derivative from the activation OUTPUT
  if (kind == B200RL_ACT_TANH) return 1.f - y * y;
  if (kind == B200RL_ACT_RELU) return y > 0.f ? 1.f : 0.f;
  return 1.f;
}

// a' = clamp(a + clamp(sigma * eps, -c, c), -limit, limit)   (td3.py:326-332)
__device__ __forceinline__ float smooth_target_action(float a, float eps, float sigma, float clipv, float limit) {
  float e = sigma * eps;
  e = fminf(fmaxf(e, -clipv), clipv);
  return fminf(fmaxf(a + e, -limit), limit);
}

// MODE 0 (NT): C[M,N] = act(A[M,K] * B[N,K]^T + bias[N])              forward: A = X, B = W [out,in]
// MODE 1 (NN): C[M,N] = (A (.) act'(Y))[M,K] * B[K,N]                  dX = dZ * W,   A = dY, Y = layer output
// MODE 2 (TN): C[M,N] = (A (.) act'(Y))[K,M]^T * B[K,N]                dW = dZ^T * X, A = dY [rows, out];
//              and, when dbias is set, dbias[M] = column sums of (A (.) act'(Y)) -- the bias gradient rides along
// All matrices row-major with explicit leading dimensions.  Y (same shape / ld as A) may be NULL (no derivative).
struct GemmArgs {
  const float* A; int lda;
  const float* B; int ldb;
  float* C; int ldc;
  const float* bias;
  const float* Y; int ldy; int act;  // MODE 0: output activation; MODE 1/2: activation whose derivative gates A
  int M, N, K;
  float* dbias;                      // MODE 2 only
  // MODE 0 extras (the persistent step kernel fuses the small elementwise kernels into its GEMMs):
  const float* A2; int lda2; int ksplit;  // A2 != NULL: columns >= ksplit of A (MODE 0) / of B (MODE 2) come from
                                          // A2[:, col - ksplit]: the operand is torch.cat([left, A2], -1), never built
  const float* eps; float sigma, clipv, limit;  // eps != NULL: target-policy smoothing on the output (td3.py:326-332)
};

// These GEMMs are tiny (256 x 256 x 256) and sit on a long dependency chain, so latency is what counts: the operands are
// fetched into registers (coalesced along the contiguous dimension of each operand) eight k-tiles at a time and
// multiplied out of shared memory tile by tile.
typedef float GemmTile[GK][GT + 2];

template <int MODE, int KT>  // KT = k-tiles fetched ahead (registers: 8 per k-tile)
__device__ __forceinline__ void gemm_tile(const GemmArgs& g, int bx, int by, GemmTile& As, GemmTile& Bs) {
  const int tid = threadIdx.x;
  const int m0 = by * GT, n0 = bx * GT;
  const int tm = (tid / 16) * 2, tn = (tid % 16) * 2;  // 16 x 16 threads, 2 x 2 outputs each
  constexpr int PER = GK * GT / GTHREADS;               // elements of each operand tile per thread (4)
  float rab[KT][PER], rbb[KT][PER];
  // element e of a tile handled by this thread: idx = tid + e * GTHREADS; (hi, lo) = (idx / 32, idx % 32) with `lo`
  // running along the operand's contiguous dimension
  auto fetch = [&](int k0, float (&ra)[PER], float (&rb)[PER]) {
#pragma unroll
    for (int e = 0; e < PER; ++e) {
      const int idx = tid + e * GTHREADS, hi = idx >> 5, lo = idx & 31;
      {  // A
        const int k = MODE == 2 ? hi : lo, m = MODE == 2 ? lo : hi;
        const int gm = m0 + m, gk = k0 + k;
        float a = 0.f;
        if (gm < g.M && gk < g.K) {
          const size_t ia = MODE == 2 ? (size_t)gk * g.lda + gm : (size_t)gm * g.lda + gk;
          if (MODE == 0 && g.A2 != nullptr && gk >= g.ksplit) a = g.A2[(size_t)gm * g.lda2 + (gk - g.ksplit)];
          else a = g.A[ia];
          if (MODE != 0 && g.Y) a *= op_act_prime(g.Y[MODE == 2 ? (size_t)gk * g.ldy + gm : (size_t)gm * g.ldy + gk], g.act);
        }
        ra[e] = a;
      }
      {  // B
        const int k = MODE == 0 ? lo : hi, n = MODE == 0 ? hi : lo;
        const int gn = n0 + n, gk = k0 + k;
        float b = 0.f;
        if (gn < g.N && gk < g.K) {
          if (MODE == 2 && g.A2 != nullptr && gn >= g.ksplit) b = g.A2[(size_t)gk * g.lda2 + (gn - g.ksplit)];
          else b = MODE == 0 ? g.B[(size_t)gn * g.ldb + gk] : g.B[(size_t)gk * g.ldb + gn];
        }
        rb[e] = b;
      }
    }
  };
  auto stash = [&](const float (&ra)[PER], const float (&rb)[PER]) {
#pragma unroll
    for (int e = 0; e < PER; ++e) {
      const int idx = tid + e * GTHREADS, hi = idx >> 5, lo = idx & 31;
      if (MODE == 2) As[hi][lo] = ra[e]; else As[lo][hi] = ra[e];
      if (MODE == 0) Bs[lo][hi] = rb[e]; else Bs[hi][lo] = rb[e];
    }
  };
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  float colsum[2] = {0.f, 0.f};
  // All loads of up to KT k-tiles are issued back to back (one memory latency for the whole K = 256 product instead of
  // one per k-tile: these GEMMs sit on a dependency chain, their latency is the train step's); the tiles then go through
  // shared memory one after the other, k ascending, so every output's fma chain is the one of a plain k loop.
  for (int kb = 0; kb < g.K; kb += GK * KT) {
#pragma unroll
    for (int t = 0; t < KT; ++t)
      if (kb + t * GK < g.K) fetch(kb + t * GK, rab[t], rbb[t]);
#pragma unroll
    for (int t = 0; t < KT; ++t) {
      if (kb + t * GK < g.K) {  // block-uniform
        stash(rab[t], rbb[t]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GK; ++k) {
          const float2 av = *reinterpret_cast<const float2*>(&As[k][tm]);
          const float2 bv = *reinterpret_cast<const float2*>(&Bs[k][tn]);
          const float ar[2] = {av.x, av.y}, br[2] = {bv.x, bv.y};
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            if (MODE == 2) colsum[i] += ar[i];
#pragma unroll
            for (int j = 0; j < 2; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
          }
        }
        __syncthreads();
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int gm = m0 + tm + i, gn = n0 + tn + j;
      if (gm < g.M && gn < g.N) {
        float v = acc[i][j];
        if (MODE == 0) {
          v = op_act(v + (g.bias ? g.bias[gn] : 0.f), g.act);
          if (g.eps != nullptr) v = smooth_target_action(v, g.eps[(size_t)gm * g.N + gn], g.sigma, g.clipv, g.limit);
        }
        g.C[(size_t)gm * g.ldc + gn] = v;
      }
    }
  if (MODE == 2 && g.dbias != nullptr && bx == 0 && tn == 0) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (m0 + tm + i < g.M) g.dbias[m0 + tm + i] = colsum[i];
  }
}

template <int MODE>
__global__ void __launch_bounds__(GTHREADS) gemm_kernel(const GemmArgs g) {
  __shared__ GemmTile As, Bs;
  gemm_tile<MODE, 8>(g, blockIdx.x, blockIdx.y, As, Bs);  // K = 256 is ONE round of loads
}

// ---- device-side draws (opt-in; SURVEY 8f-4): Philox4x32-10, counter-based, so a (seed, call) pair names the whole
// [S, B] index block and the [S, B, A] noise block of one train() call whatever the launch geometry.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c.x, p1 = (unsigned long long)0xCD9E8D57u * c.z;
    c = make_uint4((unsigned)(p1 >> 32) ^ c.y ^ k.x, (unsigned)p1, (unsigned)(p0 >> 32) ^ c.w ^ k.y, (unsigned)p0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// idx[j] = physical row of a uniform draw over the `size` live rows of the ring (logical row u sits at
// (start + u) % capacity);  eps[j] = N(0, 1) by Box-Muller.  One thread = one Philox block = 4 values of each.
__global__ void draw_minibatches_kernel(long long* idx, long long n_idx, float* eps, long long n_eps,
                                        unsigned long long seed, unsigned long long call, long long start,
                                        long long size, long long capacity) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  if (4 * t < n_idx) {
    const uint4 r = philox4x32_10(make_uint4((unsigned)t, (unsigned)(t >> 32), (unsigned)call, 0x1D5u), key);
    const unsigned v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * t + j < n_idx) {
        const long long u = (long long)(((unsigned long long)v[j] * (unsigned long long)size) >> 32);  // [0, size)
        idx[4 * t + j] = (start + u) % capacity;
      }
  }
  if (eps != nullptr && 4 * t < n_eps) {
    const uint4 r = philox4x32_10(make_uint4((unsigned)t, (unsigned)(t >> 32), (unsigned)call, 0xE95u), key);
    const float u1 = ((float)r.x + 1.0f) * 2.3283064365386963e-10f, u2 = (float)r.y * 2.3283064365386963e-10f;
    const float u3 = ((float)r.z + 1.0f) * 2.3283064365386963e-10f, u4 = (float)r.w * 2.3283064365386963e-10f;
    const float m1 = sqrtf(-2.f * logf(u1)), m2 = sqrtf(-2.f * logf(u3));
    float s1, c1, s2, c2;
    sincospif(2.f * u2, &s1, &c1);
    sincospif(2.f * u4, &s2, &c2);
    const float z[4] = {m1 * c1, m1 * s1, m2 * c2, m2 * s2};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * t + j < n_eps) eps[4 * t + j] = z[j];
  }
}

// staged[i, :] = table[idx[i], :]  (replay-buffer gather; one launch per column)
__global__ void gather_rows_kernel(const float* table, const long long* idx, int width, long long n_out, float* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_out * width) return;
  const long long r = i / width;
  out[i] = table[idx[r] * width + (i - r * width)];
}

// y = r + gamma * (1 - d) * min(q1t, q2t)   (td3.py:337-339; ddpg.py:280: single target Q).  Every product and the sum
// rounded on its own, as the reference's float32 tensor ops do: written plainly, nvcc fuses the last two into an FFMA.
__device__ __forceinline__ float td_target(float rew, float done, float q1t, const float* q2t, int i, float gamma) {
  const float q = q2t ? fminf(q1t, q2t[i]) : q1t;
  return __fadd_rn(rew, __fmul_rn(__fmul_rn(gamma, 1.f - done), q));
}

// One CTA: the critic's loss with its TD target computed on the fly: y as above, loss = mean((q - y)^2),
// dq = 2 (q - y) / B (F.mse_loss + backward), q_copy = q (the logged Q-values);  rew == NULL: the policy loss
// -mean(q), dq = -1/B
__global__ void __launch_bounds__(GTHREADS) q_loss_kernel(const float* q, const float* rew, const float* done,
                                                         const float* q1t, const float* q2t, float gamma, int n,
                                                         float* dq, float* loss_out, float* q_copy) {
  __shared__ double red[32];
  double acc = 0.0;
  const float inv = 1.0f / (float)n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float qi = q[i];
    if (q_copy) q_copy[i] = qi;
    if (rew) {
      const float d = qi - td_target(rew[i], done[i], q1t[i], q2t, i, gamma);
      acc += (double)d * (double)d;
      dq[i] = (2.f * d) * inv;
    } else {
      acc -= (double)qi;
      dq[i] = -inv;
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    *loss_out = (float)(t / (double)n);
  }
}

// target <- rho * target + (1 - rho) * param   (utils.py:47-57: f32 tensors tensor(rho), tensor(1 - rho)): two rounded
// products and a rounded sum, never an FFMA (the same rule as b200rl_polyak in utils_kernels.cu)
__device__ __forceinline__ float polyak(float rho, float target, float one_minus_rho, float param) {
  return __fadd_rn(__fmul_rn(rho, target), __fmul_rn(one_minus_rho, param));
}
struct PolyakArgs {
  float* target[3];
  const float* param[3];
  int n[3];
  int n_nets;
};
__global__ void polyak_kernel(const PolyakArgs a, float rho, float one_minus_rho) {  // every network in one launch
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (int k = 0; k < a.n_nets; ++k)
    if (i < a.n[k]) a.target[k][i] = polyak(rho, a.target[k][i], one_minus_rho, a.param[k][i]);
}

// ---------------------------------------------------------------------------------------------------------------
// The persistent step kernel.  A train() call of S steps is ~46 S small dependent kernels; even replayed as a CUDA
// graph each costs a launch-to-launch gap (~200 us per TD3 step at B = 256).  Here the SAME tile code runs as ONE
// cooperative launch: the host compiles the S steps into a program of ops grouped into PHASES (ops of a phase are
// independent: the four critics' forward passes of a layer, dW and dX of a layer, ...), every CTA walks the phases,
// takes virtual blocks `blockIdx.x, + gridDim.x, ...` of the phase's ops, and a grid barrier separates phases (~18 per
// TD3 step instead of ~46 launches).  The GEMM tiles are the functions above, so the arithmetic -- tile shapes,
// summation order, Adam's operation order -- is that of the launch-per-kernel path, which stays as the A/B reference
// (B200RL_OFFPOLICY_MEGAKERNEL=0) and must give bit-identical results.  concat / target smoothing are fused into the
// GEMMs' operand load and epilogue (GemmArgs: A2 / eps), the TD target into the loss op.
// ---------------------------------------------------------------------------------------------------------------
enum MkType : int { MK_GEMM_NT = 0, MK_GEMM_NN = 1, MK_GEMM_TN = 2, MK_TD_LOSS = 3, MK_POLICY_LOSS = 4, MK_ADAM = 5,
                    MK_POLYAK = 6, MK_FILL = 7 };

struct MkOp {
  int type;
  int n_vb;    // virtual blocks of this op
  int grid_x;  // GEMM: tiles along N (vb = by * grid_x + bx)
  int n;       // elementwise ops: element count
  GemmArgs g;
  // MK_TD_LOSS: q, rew, done, qt1, qt2 (NULL: single target critic) -> dq, loss_out, q_copy;  f0 = gamma
  // MK_POLICY_LOSS: q -> loss_out  (dq is the constant -1/B, filled once per program by MK_FILL)
  // MK_ADAM: params(o0) grad(p0) m(o1) v(o2), f0 = 1-b1, f1 = b2, f2 = 1-b2, f3 = eps, table + table_idx
  // MK_POLYAK: target(o0) param(p0), f0 = rho, f1 = 1 - rho;   MK_FILL: o0[0..n) = f0
  const float *p0, *p1, *p2, *p3, *p4;
  float *o0, *o1, *o2;
  float f0, f1, f2, f3;
  const float2* table;
  int table_idx;
  int pad;
};

struct MkPhase {
  int op0, n_ops, total_vb, pad;
};
// The program in device memory: one fixed-size block per phase, so that a CTA can stage the NEXT phase's descriptors
// into shared memory with cp.async while it works on the current one (descriptor reads are off the critical path).
constexpr int MK_MAX_OPS = 8;
struct __align__(16) MkBlock {
  MkPhase hdr;
  MkOp ops[MK_MAX_OPS];
};
static_assert(sizeof(MkBlock) % 16 == 0, "MkBlock is copied in 16-byte pieces");

// mean((q - y)^2) / -mean(q) exactly as q_loss_kernel sums them: per-thread partial over a stride of the block size, a
// shuffle tree per warp, the warp totals in warp order
__device__ __forceinline__ void mk_block_mean(double acc, int n, float* loss_out, double* red) {
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    *loss_out = (float)(t / (double)n);
  }
}

__global__ void __launch_bounds__(GTHREADS, 2) offpolicy_mega_kernel(const MkBlock* __restrict__ prog, int n_phases,
                                                                      unsigned* bar) {
  __shared__ GemmTile As, Bs;
  __shared__ double red[32];
  __shared__ MkBlock s_blk[2];
  const unsigned n_cta = gridDim.x;
  constexpr int PIECES = (int)(sizeof(MkBlock) / 16);
  auto stage = [&](int ph) {  // asynchronous: lands while this CTA works; completed before the phase barrier
    if (ph < n_phases) {
      const char* src = reinterpret_cast<const char*>(prog + ph);
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&s_blk[ph & 1]);
      for (int i = threadIdx.x; i < PIECES; i += GTHREADS)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i), "l"(src + 16 * i) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  stage(0);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  for (int ph = 0; ph < n_phases; ++ph) {
    const MkBlock& blk = s_blk[ph & 1];
    stage(ph + 1);
    const int total_vb = blk.hdr.total_vb;
    for (int vb = blockIdx.x; vb < total_vb; vb += (int)n_cta) {
      int o = 0, local = vb;
      while (local >= blk.ops[o].n_vb) {
        local -= blk.ops[o].n_vb;
        ++o;
      }
      const MkOp& op = blk.ops[o];
      const int type = op.type;
      if (type <= MK_GEMM_TN) {
        const int bx = local % op.grid_x, by = local / op.grid_x;
        // four k-tiles ahead: two CTAs per SM leave 128 registers per thread
        if (type == MK_GEMM_NT) gemm_tile<0, 4>(op.g, bx, by, As, Bs);
        else if (type == MK_GEMM_NN) gemm_tile<1, 4>(op.g, bx, by, As, Bs);
        else gemm_tile<2, 4>(op.g, bx, by, As, Bs);
      } else if (type == MK_TD_LOSS) {  // q_loss_kernel of one critic
        const int n = op.n;
        const float inv = 1.0f / (float)n;
        double acc = 0.0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
          const float qi = op.p0[i];
          op.o2[i] = qi;
          const float d = qi - td_target(op.p1[i], op.p2[i], op.p3[i], op.p4, i, op.f0);
          acc += (double)d * (double)d;
          op.o0[i] = (2.f * d) * inv;
        }
        mk_block_mean(acc, n, op.o1, red);
      } else if (type == MK_POLICY_LOSS) {
        double acc = 0.0;
        for (int i = threadIdx.x; i < op.n; i += blockDim.x) acc -= (double)op.p0[i];
        mk_block_mean(acc, op.n, op.o1, red);
      } else if (type == MK_ADAM) {
        const int i = local * GTHREADS + threadIdx.x;
        if (i < op.n) {
          const float2 t = op.table[op.table_idx];
          const float g = op.p0[i];
          float m = op.o1[i], v = op.o2[i];
          m = m + op.f0 * (g - m);                       // the arithmetic of adam_step_kernel (adam.cu)
          v = v * op.f1 + op.f2 * (g * g);
          const float denom = sqrtf(v) / t.y + op.f3;
          op.o1[i] = m;
          op.o2[i] = v;
          op.o0[i] = op.o0[i] - t.x * (m / denom);
        }
      } else if (type == MK_POLYAK) {
        const int i = local * GTHREADS + threadIdx.x;
        if (i < op.n) op.o0[i] = polyak(op.f0, op.o0[i], op.f1, op.p0[i]);
      } else {  // MK_FILL
        const int i = local * GTHREADS + threadIdx.x;
        if (i < op.n) op.o0[i] = op.f0;
      }
      __syncthreads();  // the tiles / the reduction scratch are reused by the next virtual block
    }
    // grid barrier: a monotonically increasing ticket counter (every CTA is resident: cooperative launch)
    asm volatile("cp.async.wait_group 0;" ::: "memory");  // the next phase's descriptors have landed
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned target = (unsigned)(ph + 1) * n_cta;
      atomicAdd(bar, 1u);
      unsigned seen;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(bar) : "memory");
      } while (seen < target);
    }
    __syncthreads();
  }
}

}  // namespace b200rl

using namespace b200rl;

// ---------------------------------------------------------------------------------------------------------------
struct NetBuf {
  b200rl_mlp_desc d;
  int64_t P = 0;
  float* params = nullptr;
  float *m = nullptr, *v = nullptr;  // Adam state (trainable nets only)
  float* grad = nullptr;
  bool present = false;
  int64_t step = 0;
  int w_off[B200RL_MAX_LAYERS], b_off[B200RL_MAX_LAYERS];
};

struct b200rl_offpolicy {
  b200rl_offpolicy_config cfg;
  NetBuf net[6];  // 0 pi, 1 Q1, 2 Q2, 3 pi_targ, 4 Q1_targ, 5 Q2_targ
  int O = 0, A = 0, maxw = 0;
  // staged minibatches [S,B,*]
  float *obs = nullptr, *act = nullptr, *rew = nullptr, *nobs = nullptr, *done = nullptr, *eps = nullptr;
  // per-step workspace
  float* acts[5][B200RL_MAX_LAYERS + 1];  // activation stacks [B, width]: 0 scratch/target (Q1 side), 1 Q1, 2 policy,
                                          // 3 target Q2, 4 Q2 (the twin critic runs on a second stream)
  float* acts_tq[B200RL_MAX_LAYERS + 1];  // the persistent kernel: Q1's target critic gets a stack of its own (there the
                                          // critics' first layers run beside the target policy's, which owns stack 0)
  float *x_cat = nullptr, *x_cat2 = nullptr, *qt1 = nullptr, *qt2 = nullptr, *dq = nullptr;
  float *dbuf0 = nullptr, *dbuf1 = nullptr;  // gradient ping-pong [B, maxw]
  float *dbuf2 = nullptr, *dbuf3 = nullptr, *dq2 = nullptr;  // the same for the twin critic's branch
  cudaStream_t s2 = nullptr;                // side stream of the twin critic (forked / joined with events)
  cudaStream_t s3 = nullptr, s4 = nullptr;  // the critics' forward passes on [s | a] beside the target path; the
                                            // weight-gradient products beside the dX chains
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_side = nullptr;
  // outputs
  float *out_q1 = nullptr, *out_q2 = nullptr, *out_l1 = nullptr, *out_l2 = nullptr, *out_lp = nullptr;
  // CUDA graph of the S-step loop: node arguments are fixed per (S, B, hyper-parameters); what changes between calls
  // (minibatch contents, Adam bias-correction scalars) lives in device buffers refreshed before each launch
  long long* idx = nullptr;      // [max_steps * max_minibatch] replay rows of train_gather
  float2* adam_tab = nullptr;    // [3][max_steps] {lr / (1 - beta1^t), sqrt(1 - beta2^t)} for policy, Q1, Q2
  float2* h_adam_tab = nullptr;  // pinned mirror
  cudaStream_t gs = nullptr;     // internal stream (the caller's may be the legacy default stream: not capturable)
  cudaEvent_t ev = nullptr;
  cudaGraphExec_t graph = nullptr;
  b200rl_offpolicy_hparams graph_hp;
  int graph_S = -1, graph_B = -1, graph_npol = 0, graph_launches = 0;
  // the persistent step kernel's program for (S, B, hyper-parameters), see offpolicy_mega_kernel
  MkBlock* mk_prog = nullptr;
  unsigned* mk_bar = nullptr;
  float* dq_pol = nullptr;  // [max_minibatch] the constant -1/B gradient of the policy loss
  b200rl_offpolicy_hparams mk_hp;
  int mk_S = -1, mk_B = -1, mk_npol = 0, mk_n_phases = 0, mk_grid = 0;
  size_t mk_prog_cap = 0;
  float* state = nullptr;  // parameters + Adam state of every network, blob order (see b200rl_offpolicy_create)
  int64_t state_n = 0;
  std::vector<void*> allocs;
};

namespace {

inline int64_t state_pad(int64_t n) { return (n + 63) & ~(int64_t)63; }

template <typename T>
int oalloc(b200rl_offpolicy* h, T** p, size_t count) {
  void* q = nullptr;
  B200RL_CUDA(cudaMalloc(&q, (count ? count : 1) * sizeof(T)));
  B200RL_CUDA(cudaMemset(q, 0, (count ? count : 1) * sizeof(T)));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return 0;
}

template <int MODE>
int gemm(const GemmArgs& g, cudaStream_t s) {
  dim3 grid((g.N + GT - 1) / GT, (g.M + GT - 1) / GT);
  gemm_kernel<MODE><<<grid, GTHREADS, 0, s>>>(g);
  B200RL_CUDA(cudaGetLastError());
  count_launch(1);
  return 0;
}

// forward through one network: acts[0] = input [rows, n0] (ld = n0); acts[l+1] = layer outputs.
// in_b != NULL: the input is torch.cat([acts[0] (ksplit columns), in_b (ld_b)], -1), read in place by the first layer
// (q_function.py:30); eps != NULL: target-policy smoothing on the output (td3.py:326-332)
int net_forward(const NetBuf& nb, float* const* acts, int rows, cudaStream_t s, const float* in_b = nullptr, int ld_b = 0,
                int ksplit = 0, const float* eps = nullptr, const b200rl_offpolicy_hparams* hp = nullptr) {
  const int L = nb.d.n_layers;
  for (int l = 0; l < L; ++l) {
    GemmArgs g{};
    g.A = acts[l]; g.lda = nb.d.sizes[l];
    if (l == 0 && in_b != nullptr) {
      g.lda = ksplit;
      g.A2 = in_b; g.lda2 = ld_b; g.ksplit = ksplit;
    }
    if (l == L - 1 && eps != nullptr) {
      g.eps = eps;
      g.sigma = (float)hp->target_noise_scale;
      g.clipv = (float)hp->target_noise_clip;
      g.limit = (float)hp->action_limit;
    }
    g.B = nb.params + nb.w_off[l]; g.ldb = nb.d.sizes[l];
    g.C = acts[l + 1]; g.ldc = nb.d.sizes[l + 1];
    g.bias = nb.params + nb.b_off[l];
    g.act = (l == L - 1) ? nb.d.out_act : nb.d.hidden_act;
    g.M = rows; g.N = nb.d.sizes[l + 1]; g.K = nb.d.sizes[l];
    if (gemm<0>(g, s)) return 1;
  }
  return 0;
}

// backward: dOut = gradient w.r.t. the network OUTPUT (after the output activation) [rows, nL] with ld ld_dout.
// want_param_grads: write nb.grad (flat).  dx_out (optional): gradient w.r.t. the input [rows, n0].
// s_dw != NULL (and at most 3 layers: the two ping-pong buffers then never see a writer while a reader is pending): the
// weight-gradient products go to that stream, behind the gradient they read, and the dX chain -- the critical path --
// stays on `s`; both are joined before returning.
int net_backward(b200rl_offpolicy* h, const NetBuf& nb, float* const* acts, const float* dOut, int ld_dout, int rows,
                 bool want_param_grads, float* dx_out, cudaStream_t s, bool twin_branch = false,
                 const float* in_b = nullptr, int ld_b = 0, int ksplit = 0, cudaStream_t s_dw = nullptr) {
  const int L = nb.d.n_layers;
  const bool side = s_dw != nullptr && want_param_grads && L <= 3;
  const float* dY = dOut;
  int ldd = ld_dout;
  float* pp[2] = {twin_branch ? h->dbuf2 : h->dbuf0, twin_branch ? h->dbuf3 : h->dbuf1};
  for (int l = L - 1; l >= 0; --l) {
    const int nout = nb.d.sizes[l + 1], nin = nb.d.sizes[l];
    const int act = (l == L - 1) ? nb.d.out_act : nb.d.hidden_act;
    const float* Y = acts[l + 1];
    if (want_param_grads) {
      GemmArgs g{};  // dW[nout, nin] = (dY . act'(Y))^T [nout, rows] * X[rows, nin]
      g.A = dY; g.lda = ldd; g.Y = Y; g.ldy = nout; g.act = act;
      g.B = acts[l]; g.ldb = nin;
      if (l == 0 && in_b != nullptr) {  // the layer's input is [acts[0] | in_b], never materialised
        g.ldb = ksplit;
        g.A2 = in_b; g.lda2 = ld_b; g.ksplit = ksplit;
      }
      g.C = nb.grad + nb.w_off[l]; g.ldc = nin;
      g.M = nout; g.N = nin; g.K = rows;
      g.dbias = nb.grad + nb.b_off[l];  // db = column sums of dZ, accumulated by the same kernel
      if (side) {  // dY of this layer is complete on `s` at this point
        B200RL_CUDA(cudaEventRecord(h->ev_side, s));
        B200RL_CUDA(cudaStreamWaitEvent(s_dw, h->ev_side, 0));
      }
      if (gemm<2>(g, side ? s_dw : s)) return 1;
    }
    if (l > 0 || dx_out) {
      float* dst = (l == 0) ? dx_out : pp[l & 1];
      GemmArgs g{};  // dX[rows, nin] = (dY . act'(Y))[rows, nout] * W[nout, nin]
      g.A = dY; g.lda = ldd; g.Y = Y; g.ldy = nout; g.act = act;
      g.B = nb.params + nb.w_off[l]; g.ldb = nin;
      g.C = dst; g.ldc = nin;
      g.M = rows; g.N = nin; g.K = nout;
      if (gemm<1>(g, s)) return 1;
      dY = dst;
      ldd = nin;
    }
  }
  if (side) {
    B200RL_CUDA(cudaEventRecord(h->ev_side, s_dw));
    B200RL_CUDA(cudaStreamWaitEvent(s, h->ev_side, 0));
  }
  return 0;
}

int adam_net(NetBuf& nb, const float2* table, int idx, double b1, double b2, double eps, cudaStream_t s) {
  return adam_step_table(nb.params, nb.grad, nb.m, nb.v, nb.P, table, idx, b1, b2, eps, s);
}

}  // namespace

extern "C" int b200rl_offpolicy_create(const b200rl_offpolicy_config* cfg, b200rl_offpolicy** out) {
  B200RL_REQUIRE(cfg && out, "offpolicy_create: NULL argument");
  B200RL_REQUIRE(cfg->n_q == 1 || cfg->n_q == 2, "offpolicy_create: n_q must be 1 (DDPG) or 2 (TD3)");
  B200RL_REQUIRE(cfg->max_minibatch >= 1 && cfg->max_minibatch <= 65536 && cfg->max_steps >= 1,
                 "offpolicy_create: bad capacities");
  const int64_t Pp = b200rl_mlp_param_count(&cfg->policy), Pq = b200rl_mlp_param_count(&cfg->q);
  B200RL_REQUIRE(Pp > 0 && Pq > 0, "offpolicy_create: invalid MLP description");
  const int O = cfg->policy.sizes[0], A = cfg->policy.sizes[cfg->policy.n_layers];
  B200RL_REQUIRE(cfg->q.sizes[0] == O + A && cfg->q.sizes[cfg->q.n_layers] == 1,
                 "offpolicy_create: Q network must map [obs %d + act %d] -> 1", O, A);
  B200RL_REQUIRE(device_sm_count() > 0, "offpolicy_create: no CUDA device");
  b200rl_offpolicy* h = new b200rl_offpolicy();
  h->cfg = *cfg;
  h->O = O;
  h->A = A;
  int rc = 0;
  int maxw = O + A;
  for (int i = 0; i < 6; ++i) {
    NetBuf& nb = h->net[i];
    nb.d = (i == 0 || i == 3) ? cfg->policy : cfg->q;
    nb.P = (i == 0 || i == 3) ? Pp : Pq;
    int off = 0;
    for (int l = 0; l < nb.d.n_layers; ++l) {
      nb.w_off[l] = off;
      off += nb.d.sizes[l + 1] * nb.d.sizes[l];
      nb.b_off[l] = off;
      off += nb.d.sizes[l + 1];
      maxw = nb.d.sizes[l + 1] > maxw ? nb.d.sizes[l + 1] : maxw;
    }
    if (cfg->n_q == 1 && (i == 2 || i == 5)) continue;
    nb.present = true;
    if (i < 3) rc |= oalloc(h, &nb.grad, (size_t)nb.P);
  }
  // parameters and Adam state live in ONE slab in the order of the state blob (b200rl_offpolicy_get_state): the
  // parameters of networks 0..5, then exp_avg / exp_avg_sq of optimizers 0..2, every segment padded to 64 floats
  {
    int64_t n = 0;
    for (int i = 0; i < 6; ++i)
      if (h->net[i].present) n += state_pad(h->net[i].P);
    for (int i = 0; i < 3; ++i)
      if (h->net[i].present) n += 2 * state_pad(h->net[i].P);
    h->state_n = n;
    rc |= oalloc(h, &h->state, (size_t)n);
    if (rc == 0) {
      float* q = h->state;
      for (int i = 0; i < 6; ++i)
        if (h->net[i].present) {
          h->net[i].params = q;
          q += state_pad(h->net[i].P);
        }
      for (int i = 0; i < 3; ++i)
        if (h->net[i].present) {
          h->net[i].m = q;
          q += state_pad(h->net[i].P);
          h->net[i].v = q;
          q += state_pad(h->net[i].P);
        }
    }
  }
  h->maxw = maxw;
  const size_t B = (size_t)cfg->max_minibatch, S = (size_t)cfg->max_steps;
  rc |= oalloc(h, &h->obs, S * B * O);
  rc |= oalloc(h, &h->act, S * B * A);
  rc |= oalloc(h, &h->rew, S * B);
  rc |= oalloc(h, &h->nobs, S * B * O);
  rc |= oalloc(h, &h->done, S * B);
  rc |= oalloc(h, &h->eps, S * B * A);
  for (int k = 0; k < 5; ++k)
    for (int l = 0; l <= B200RL_MAX_LAYERS; ++l) rc |= oalloc(h, &h->acts[k][l], B * (size_t)maxw);
  for (int l = 0; l <= B200RL_MAX_LAYERS; ++l) rc |= oalloc(h, &h->acts_tq[l], B * (size_t)maxw);
  rc |= oalloc(h, &h->x_cat, B * (size_t)(O + A));
  rc |= oalloc(h, &h->x_cat2, B * (size_t)(O + A));
  rc |= oalloc(h, &h->qt1, B);
  rc |= oalloc(h, &h->qt2, B);
  rc |= oalloc(h, &h->dq, B);
  rc |= oalloc(h, &h->dbuf0, B * (size_t)maxw);
  rc |= oalloc(h, &h->dbuf1, B * (size_t)maxw);
  rc |= oalloc(h, &h->dbuf2, B * (size_t)maxw);
  rc |= oalloc(h, &h->dbuf3, B * (size_t)maxw);
  rc |= oalloc(h, &h->dq2, B);
  rc |= oalloc(h, &h->dq_pol, B);
  rc |= oalloc(h, &h->mk_bar, 1);
  rc |= oalloc(h, &h->out_q1, S * B);
  rc |= oalloc(h, &h->out_q2, S * B);
  rc |= oalloc(h, &h->out_l1, S);
  rc |= oalloc(h, &h->out_l2, S);
  rc |= oalloc(h, &h->out_lp, S);
  rc |= oalloc(h, &h->adam_tab, 3 * S);
  rc |= oalloc(h, &h->idx, S * B);
  if (!rc && cudaMallocHost(reinterpret_cast<void**>(&h->h_adam_tab), 3 * S * sizeof(float2)) != cudaSuccess) rc = 1;
  if (!rc && cudaStreamCreateWithFlags(&h->gs, cudaStreamNonBlocking) != cudaSuccess) rc = 1;
  if (!rc && cudaEventCreateWithFlags(&h->ev, cudaEventDisableTiming) != cudaSuccess) rc = 1;
  if (!rc && cudaStreamCreateWithFlags(&h->s2, cudaStreamNonBlocking) != cudaSuccess) rc = 1;
  if (!rc && cudaStreamCreateWithFlags(&h->s3, cudaStreamNonBlocking) != cudaSuccess) rc = 1;
  if (!rc && cudaStreamCreateWithFlags(&h->s4, cudaStreamNonBlocking) != cudaSuccess) rc = 1;
  if (!rc && cudaEventCreateWithFlags(&h->ev_side, cudaEventDisableTiming) != cudaSuccess) rc = 1;
  if (!rc && cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess) rc = 1;
  if (!rc && cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) rc = 1;
  if (rc) {
    b200rl_offpolicy_destroy(h);
    return 1;
  }
  *out = h;
  return 0;
}

extern "C" void b200rl_offpolicy_destroy(b200rl_offpolicy* h) {
  if (!h) return;
  if (h->graph) cudaGraphExecDestroy(h->graph);
  if (h->mk_prog) cudaFree(h->mk_prog);
  if (h->ev) cudaEventDestroy(h->ev);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_side) cudaEventDestroy(h->ev_side);
  if (h->s2) cudaStreamDestroy(h->s2);
  if (h->s3) cudaStreamDestroy(h->s3);
  if (h->s4) cudaStreamDestroy(h->s4);
  if (h->gs) cudaStreamDestroy(h->gs);
  if (h->h_adam_tab) cudaFreeHost(h->h_adam_tab);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
}

extern "C" int b200rl_offpolicy_set_params(b200rl_offpolicy* h, int which, const float* host_flat, int64_t n,
                                           void* stream) {
  B200RL_REQUIRE(h && host_flat && which >= 0 && which < 6 && h->net[which].params, "offpolicy_set_params: bad net");
  B200RL_REQUIRE(n == h->net[which].P, "offpolicy_set_params: expects %lld floats", (long long)h->net[which].P);
  B200RL_CUDA(cudaMemcpyAsync(h->net[which].params, host_flat, (size_t)n * 4, cudaMemcpyHostToDevice,
                              static_cast<cudaStream_t>(stream)));
  return 0;
}

extern "C" int b200rl_offpolicy_get_params(b200rl_offpolicy* h, int which, float* host_flat, int64_t n, void* stream) {
  B200RL_REQUIRE(h && host_flat && which >= 0 && which < 6 && h->net[which].params, "offpolicy_get_params: bad net");
  B200RL_REQUIRE(n == h->net[which].P, "offpolicy_get_params: expects %lld floats", (long long)h->net[which].P);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  B200RL_CUDA(cudaMemcpyAsync(host_flat, h->net[which].params, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaStreamSynchronize(s));
  return 0;
}

extern "C" int b200rl_offpolicy_set_adam(b200rl_offpolicy* h, int which, const float* exp_avg, const float* exp_avg_sq,
                                         int64_t n, int64_t step, void* stream) {
  B200RL_REQUIRE(h && which >= 0 && which < 3 && h->net[which].m, "offpolicy_set_adam: bad net");
  NetBuf& nb = h->net[which];
  B200RL_REQUIRE(n == nb.P && step >= 0, "offpolicy_set_adam: expects %lld floats", (long long)nb.P);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (exp_avg) B200RL_CUDA(cudaMemcpyAsync(nb.m, exp_avg, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  else B200RL_CUDA(cudaMemsetAsync(nb.m, 0, (size_t)n * 4, s));
  if (exp_avg_sq) B200RL_CUDA(cudaMemcpyAsync(nb.v, exp_avg_sq, (size_t)n * 4, cudaMemcpyHostToDevice, s));
  else B200RL_CUDA(cudaMemsetAsync(nb.v, 0, (size_t)n * 4, s));
  nb.step = step;
  return 0;
}

extern "C" int b200rl_offpolicy_get_adam(b200rl_offpolicy* h, int which, float* exp_avg, float* exp_avg_sq, int64_t n,
                                         int64_t* step, void* stream) {
  B200RL_REQUIRE(h && which >= 0 && which < 3 && h->net[which].m && exp_avg && exp_avg_sq && step,
                 "offpolicy_get_adam: bad arguments");
  NetBuf& nb = h->net[which];
  B200RL_REQUIRE(n == nb.P, "offpolicy_get_adam: expects %lld floats", (long long)nb.P);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  B200RL_CUDA(cudaMemcpyAsync(exp_avg, nb.m, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaMemcpyAsync(exp_avg_sq, nb.v, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaStreamSynchronize(s));
  *step = nb.step;
  return 0;
}

// Whole learner state in ONE call and ONE synchronisation: blob = for every present network 0..5 its parameters, then
// for every optimizer 0..2 (policy, Q1, Q2) exp_avg and exp_avg_sq; steps[3] = Adam step counts.
static int64_t state_floats(const b200rl_offpolicy* h) { return h->state_n; }

extern "C" int64_t b200rl_offpolicy_state_floats(b200rl_offpolicy* h) { return h ? state_floats(h) : -1; }

// One copy each way: the slab IS the blob.  With a page-locked `blob` the copy is a plain DMA transfer.
extern "C" int b200rl_offpolicy_get_state(b200rl_offpolicy* h, float* blob, int64_t n_floats, int64_t* steps,
                                          void* stream) {
  B200RL_REQUIRE(h && blob && steps && n_floats == state_floats(h), "offpolicy_get_state: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  B200RL_CUDA(cudaMemcpyAsync(blob, h->state, (size_t)h->state_n * 4, cudaMemcpyDeviceToHost, s));
  for (int i = 0; i < 3; ++i) steps[i] = h->net[i].m ? h->net[i].step : 0;
  B200RL_CUDA(cudaStreamSynchronize(s));
  return 0;
}

extern "C" int b200rl_offpolicy_set_state(b200rl_offpolicy* h, const float* blob, int64_t n_floats, const int64_t* steps,
                                          void* stream) {
  B200RL_REQUIRE(h && blob && steps && n_floats == state_floats(h), "offpolicy_set_state: bad arguments");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int i = 0; i < 3; ++i)
    if (h->net[i].m) B200RL_REQUIRE(steps[i] >= 0, "offpolicy_set_state: negative step count");
  B200RL_CUDA(cudaMemcpyAsync(h->state, blob, (size_t)h->state_n * 4, cudaMemcpyHostToDevice, s));
  for (int i = 0; i < 3; ++i)
    if (h->net[i].m) h->net[i].step = steps[i];
  B200RL_CUDA(cudaStreamSynchronize(s));  // `blob` may be reused by the caller right away
  return 0;
}

// Enqueue the S train steps on `s` (plain launches or under stream capture).  Everything that varies between calls
// with the same (S, B, hyper-parameters) is read from device buffers: staged minibatches, Adam scalar tables.
static int enqueue_steps(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int S, int B, cudaStream_t s,
                         int* n_pol_out) {
  const bool td3 = h->cfg.n_q == 2;
  const int O = h->O, A = h->A;
  const int maxS = h->cfg.max_steps;
  NetBuf &pi = h->net[0], &q1 = h->net[1], &q2 = h->net[2], &pit = h->net[3], &q1t = h->net[4], &q2t = h->net[5];
  const int Lq = q1.d.n_layers, Lp = pi.d.n_layers;
  const int ew = 256;
  cudaStream_t s2 = h->s2, s3 = h->s3, s4 = h->s4;
  // work queued on `to` from here on waits for everything queued on `from` so far (a graph edge under capture)
  auto edge = [&](cudaStream_t from, cudaStream_t to) -> int {
    B200RL_CUDA(cudaEventRecord(h->ev_fork, from));
    B200RL_CUDA(cudaStreamWaitEvent(to, h->ev_fork, 0));
    return 0;
  };
  int n_pol = 0;
  // A step is a dependency graph, not a sequence; the branches below are what the kernels actually need:
  //   s  : target policy -> Q1 target ---------+-> Q1 loss -> Q1 dX chain -----+-> Adam(Q1) -> [policy step] -> polyak
  //   s2 :               -> Q2 target ---------+-> Q2 loss -> Q2 dX chain -----+-> Adam(Q2)
  //   s3 : Q1 forward on [s | a] (independent of the targets) ..... Q1's dW products (pi's in the policy step)
  //   s4 : Q2 forward on [s | a] .................................. Q2's dW products
  // Critical path per step: 6 + 1 + 3 + 1 kernels (was 7 + 10 in a single chain), policy steps 14 more (was 19).
  for (int st = 0; st < S; ++st) {
    const float* s_obs = h->obs + (size_t)st * B * O;
    const float* s_act = h->act + (size_t)st * B * A;
    const float* s_rew = h->rew + (size_t)st * B;
    const float* s_nobs = h->nobs + (size_t)st * B * O;
    const float* s_done = h->done + (size_t)st * B;
    // ---- the critics' forward passes on [s | a]: their values are also the logged Q-values (td3.py:231-235) ----
    float* qa[2][B200RL_MAX_LAYERS + 1];
    for (int qi = 0; qi < (td3 ? 2 : 1); ++qi) {
      qa[qi][0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lq; ++l) qa[qi][l] = h->acts[qi == 0 ? 1 : 4][l];
      cudaStream_t qs = qi == 0 ? s3 : s4;
      if (edge(s, qs)) return 1;
      if (net_forward(qi == 0 ? q1 : q2, qa[qi], B, qs, s_act, A, O)) return 1;
    }
    // ---- targets (td3.py:325-341 / ddpg.py:275-282): the smoothing noise rides on the last layer's epilogue;
    //      [s' | a'] is read in place by the target critics' first layer ----
    float* ta[B200RL_MAX_LAYERS + 1];
    ta[0] = const_cast<float*>(s_nobs);
    for (int l = 1; l <= Lp; ++l) ta[l] = h->acts[0][l];
    if (net_forward(pit, ta, B, s, nullptr, 0, 0, hp->use_target_noise ? h->eps + (size_t)st * B * A : nullptr, hp))
      return 1;
    float* tq[B200RL_MAX_LAYERS + 1];
    tq[0] = const_cast<float*>(s_nobs);
    for (int l = 1; l < Lq; ++l) tq[l] = h->acts_tq[l];  // apart from the target policy's stack, whose output it reads
    tq[Lq] = h->qt1;
    if (td3) {
      if (edge(s, s2)) return 1;
      float* tq2[B200RL_MAX_LAYERS + 1];
      tq2[0] = const_cast<float*>(s_nobs);
      for (int l = 1; l < Lq; ++l) tq2[l] = h->acts[3][l];
      tq2[Lq] = h->qt2;
      if (net_forward(q2t, tq2, B, s2, ta[Lp], A, O)) return 1;
    }
    if (net_forward(q1t, tq, B, s, ta[Lp], A, O)) return 1;
    if (td3 && edge(s2, s)) return 1;  // both target values are complete on `s`
    // ---- Q steps (td3.py:343-358): TD target + MSE + dq in one kernel, backward, Adam ----
    if (td3) {
      if (edge(s, s2)) return 1;   // the targets
      if (edge(s4, s2)) return 1;  // Q2's forward pass
    }
    if (edge(s3, s)) return 1;     // Q1's forward pass
    for (int qi = (td3 ? 1 : 0); qi >= 0; --qi) {
      NetBuf& qn = qi == 0 ? q1 : q2;
      cudaStream_t qs = qi == 0 ? s : s2;
      float* dq = qi == 0 ? h->dq : h->dq2;
      q_loss_kernel<<<1, GTHREADS, 0, qs>>>(qa[qi][Lq], s_rew, s_done, h->qt1, td3 ? h->qt2 : nullptr, (float)hp->gamma, B,
                                            dq, (qi == 0 ? h->out_l1 : h->out_l2) + st,
                                            (qi == 0 ? h->out_q1 : h->out_q2) + (size_t)st * B);
      B200RL_CUDA(cudaGetLastError());
      count_launch(1);
      if (net_backward(h, qn, qa[qi], dq, 1, B, true, nullptr, qs, qi != 0, s_act, A, O, qi == 0 ? s3 : s4)) return 1;
      if (adam_net(qn, h->adam_tab + (size_t)(1 + qi) * maxS, st, hp->q_beta1, hp->q_beta2, hp->q_eps, qs)) return 1;
    }
    if (td3 && edge(s2, s)) return 1;
    // ---- delayed policy step + polyak (td3.py:244-263, 301-323; ddpg: every step) ----
    if (st % hp->policy_delay == 0) {
      float* pa[B200RL_MAX_LAYERS + 1];
      pa[0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lp; ++l) pa[l] = h->acts[2][l];
      if (net_forward(pi, pa, B, s)) return 1;
      float* qp[B200RL_MAX_LAYERS + 1];
      qp[0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lq; ++l) qp[l] = h->acts[1][l];
      if (net_forward(q1, qp, B, s, pa[Lp], A, O)) return 1;  // Q1 with its freshly updated parameters (td3.py:309)
      q_loss_kernel<<<1, GTHREADS, 0, s>>>(qp[Lq], nullptr, nullptr, nullptr, nullptr, 0.f, B, h->dq, h->out_lp + n_pol,
                                           nullptr);
      B200RL_CUDA(cudaGetLastError());
      count_launch(1);
      // gradient w.r.t. Q1's input; its action columns are the gradient w.r.t. pi(s) (Q parameters frozen)
      if (net_backward(h, q1, qp, h->dq, 1, B, false, h->x_cat, s)) return 1;
      if (net_backward(h, pi, pa, h->x_cat + O, O + A, B, true, nullptr, s, false, nullptr, 0, 0, s3)) return 1;
      if (adam_net(pi, h->adam_tab, n_pol, hp->policy_beta1, hp->policy_beta2, hp->policy_eps, s)) return 1;
      PolyakArgs pk{};
      pk.n_nets = td3 ? 3 : 2;
      int nmax = 0;
      for (int k = 0; k < pk.n_nets; ++k) {
        pk.target[k] = h->net[3 + k].params;
        pk.param[k] = h->net[k].params;
        pk.n[k] = (int)h->net[k].P;
        nmax = pk.n[k] > nmax ? pk.n[k] : nmax;
      }
      polyak_kernel<<<(nmax + ew - 1) / ew, ew, 0, s>>>(pk, (float)hp->polyak_rho, (float)(1.0 - hp->polyak_rho));
      B200RL_CUDA(cudaGetLastError());
      count_launch(1);
      ++n_pol;
    }
  }
  *n_pol_out = n_pol;
  return 0;
}

// ---- the program of the persistent step kernel: enqueue_steps restated as ops in dependency phases ----------------
namespace {
struct MkBuilder {
  std::vector<MkOp> ops;
  std::vector<MkPhase> phases;
  int op0 = 0;
  void end_phase() {
    if ((int)ops.size() == op0) return;
    MkPhase p{};
    p.op0 = op0;
    p.n_ops = (int)ops.size() - op0;
    for (int i = op0; i < (int)ops.size(); ++i) p.total_vb += ops[i].n_vb;
    phases.push_back(p);
    op0 = (int)ops.size();
  }
  void gemm(int mode, const GemmArgs& g) {
    MkOp o{};
    o.type = mode;
    o.g = g;
    o.grid_x = (g.N + GT - 1) / GT;
    o.n_vb = o.grid_x * ((g.M + GT - 1) / GT);
    ops.push_back(o);
  }
  void elementwise(MkOp o, int n) {
    o.n = n;
    o.n_vb = (n + GTHREADS - 1) / GTHREADS;
    ops.push_back(o);
  }
  void single(MkOp o, int n) {
    o.n = n;
    o.n_vb = 1;
    ops.push_back(o);
  }
};

// forward layer l of a network; input = acts[0] (or the torch.cat of in_a | in_b when in_b != NULL)
void mk_forward_layer(MkBuilder& b, const NetBuf& nb, float* const* acts, int l, int rows, const float* in_b = nullptr,
                      int ld_b = 0, int ksplit = 0, const float* eps = nullptr, const b200rl_offpolicy_hparams* hp = nullptr) {
  const int L = nb.d.n_layers;
  GemmArgs g{};
  g.A = acts[l];
  g.lda = nb.d.sizes[l];
  if (l == 0 && in_b != nullptr) {
    g.lda = ksplit;  // acts[0] is the left block [rows, ksplit]
    g.A2 = in_b;
    g.lda2 = ld_b;
    g.ksplit = ksplit;
  }
  g.B = nb.params + nb.w_off[l];
  g.ldb = nb.d.sizes[l];
  g.C = acts[l + 1];
  g.ldc = nb.d.sizes[l + 1];
  g.bias = nb.params + nb.b_off[l];
  g.act = (l == L - 1) ? nb.d.out_act : nb.d.hidden_act;
  g.M = rows;
  g.N = nb.d.sizes[l + 1];
  g.K = nb.d.sizes[l];
  if (l == L - 1 && eps != nullptr) {
    g.eps = eps;
    g.sigma = (float)hp->target_noise_scale;
    g.clipv = (float)hp->target_noise_clip;
    g.limit = (float)hp->action_limit;
  }
  b.gemm(MK_GEMM_NT, g);
}

// backward layer l (net_backward's loop body): dY / ldd = the gradient entering the layer, pp = ping-pong buffers
void mk_backward_layer(MkBuilder& b, const NetBuf& nb, float* const* acts, int l, const float* dY, int ldd, int rows,
                       bool want_param_grads, float* dst_dx) {
  const int L = nb.d.n_layers;
  const int nout = nb.d.sizes[l + 1], nin = nb.d.sizes[l];
  const int act = (l == L - 1) ? nb.d.out_act : nb.d.hidden_act;
  const float* Y = acts[l + 1];
  if (want_param_grads) {
    GemmArgs g{};
    g.A = dY; g.lda = ldd; g.Y = Y; g.ldy = nout; g.act = act;
    g.B = acts[l]; g.ldb = nin;
    g.C = nb.grad + nb.w_off[l]; g.ldc = nin;
    g.M = nout; g.N = nin; g.K = rows;
    g.dbias = nb.grad + nb.b_off[l];
    b.gemm(MK_GEMM_TN, g);
  }
  if (dst_dx != nullptr) {
    GemmArgs g{};
    g.A = dY; g.lda = ldd; g.Y = Y; g.ldy = nout; g.act = act;
    g.B = nb.params + nb.w_off[l]; g.ldb = nin;
    g.C = dst_dx; g.ldc = nin;
    g.M = rows; g.N = nin; g.K = nout;
    b.gemm(MK_GEMM_NN, g);
  }
}

void mk_adam(MkBuilder& b, NetBuf& nb, const float2* table, int idx, double b1, double b2, double eps) {
  MkOp o{};
  o.type = MK_ADAM;
  o.o0 = nb.params; o.p0 = nb.grad; o.o1 = nb.m; o.o2 = nb.v;
  o.f0 = (float)(1.0 - b1); o.f1 = (float)b2; o.f2 = (float)(1.0 - b2); o.f3 = (float)eps;
  o.table = table;
  o.table_idx = idx;
  b.elementwise(o, (int)nb.P);
}
}  // namespace

static int build_program(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int S, int B, int* n_pol_out,
                         cudaStream_t s) {
  const bool td3 = h->cfg.n_q == 2;
  const int O = h->O, A = h->A;
  const int maxS = h->cfg.max_steps;
  NetBuf &pi = h->net[0], &q1 = h->net[1], &q2 = h->net[2], &pit = h->net[3], &q1t = h->net[4], &q2t = h->net[5];
  const int Lq = q1.d.n_layers, Lp = pi.d.n_layers;
  const int nq = td3 ? 2 : 1;
  MkBuilder b;
  {  // the policy loss's gradient w.r.t. Q is the constant -1/B (q_loss_kernel with y == NULL)
    MkOp o{};
    o.type = MK_FILL;
    o.o0 = h->dq_pol;
    o.f0 = -(1.0f / (float)B);
    b.elementwise(o, B);
    b.end_phase();
  }
  int n_pol = 0;
  for (int st = 0; st < S; ++st) {
    const float* s_obs = h->obs + (size_t)st * B * O;
    const float* s_act = h->act + (size_t)st * B * A;
    const float* s_rew = h->rew + (size_t)st * B;
    const float* s_nobs = h->nobs + (size_t)st * B * O;
    const float* s_done = h->done + (size_t)st * B;
    // ---- target action (td3.py:325-332): the smoothing noise rides on the last layer's epilogue ----
    float* ta[B200RL_MAX_LAYERS + 1];
    ta[0] = const_cast<float*>(s_nobs);
    for (int l = 1; l <= Lp; ++l) ta[l] = h->acts[0][l];
    // the critics' forward passes on [s | a] do not depend on the targets: their layers share the phases
    float* qa[2][B200RL_MAX_LAYERS + 1];
    for (int qi = 0; qi < nq; ++qi) {
      qa[qi][0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lq; ++l) qa[qi][l] = h->acts[qi == 0 ? 1 : 4][l];
    }
    float* tq[2][B200RL_MAX_LAYERS + 1];
    for (int qi = 0; qi < nq; ++qi) {
      tq[qi][0] = const_cast<float*>(s_nobs);
      // the target critics' hidden activations: stack 3 for the twin, and a stack of their own for Q1's target (stack 0
      // holds the target policy's activations, which layer 0 still reads)
      for (int l = 1; l < Lq; ++l) tq[qi][l] = qi == 0 ? h->acts_tq[l] : h->acts[3][l];
      tq[qi][Lq] = qi == 0 ? h->qt1 : h->qt2;
    }
    const int lead = Lp < Lq ? Lp : Lq;  // the critics' first layers run beside the target policy's layers
    for (int l = 0; l < Lp; ++l) {
      mk_forward_layer(b, pit, ta, l, B, nullptr, 0, 0,
                       (l == Lp - 1 && hp->use_target_noise) ? h->eps + (size_t)st * B * A : nullptr, hp);
      if (l < lead)
        for (int qi = 0; qi < nq; ++qi) mk_forward_layer(b, qi == 0 ? q1 : q2, qa[qi], l, B, s_act, A, O);
      b.end_phase();
    }
    for (int l = 0; l < Lq; ++l) {
      for (int qi = 0; qi < nq; ++qi) mk_forward_layer(b, qi == 0 ? q1t : q2t, tq[qi], l, B, ta[Lp], A, O);
      if (l + lead < Lq)
        for (int qi = 0; qi < nq; ++qi) mk_forward_layer(b, qi == 0 ? q1 : q2, qa[qi], l + lead, B, s_act, A, O);
      b.end_phase();
    }
    // ---- TD target + MSE + dq (td3.py:337-339, 343-358) ----
    for (int qi = 0; qi < nq; ++qi) {
      MkOp o{};
      o.type = MK_TD_LOSS;
      o.p0 = qa[qi][Lq]; o.p1 = s_rew; o.p2 = s_done; o.p3 = h->qt1; o.p4 = td3 ? h->qt2 : nullptr;
      o.f0 = (float)hp->gamma;
      o.o0 = qi == 0 ? h->dq : h->dq2;
      o.o1 = (qi == 0 ? h->out_l1 : h->out_l2) + st;
      o.o2 = (qi == 0 ? h->out_q1 : h->out_q2) + (size_t)st * B;
      b.single(o, B);
    }
    b.end_phase();
    // ---- critics' backward: dW and dX of a layer side by side, both critics ----
    {
      const float* dY[2] = {h->dq, h->dq2};
      int ldd[2] = {1, 1};
      for (int l = Lq - 1; l >= 0; --l) {
        for (int qi = 0; qi < nq; ++qi) {
          float* pp[2] = {qi == 0 ? h->dbuf0 : h->dbuf2, qi == 0 ? h->dbuf1 : h->dbuf3};
          float* dst = l > 0 ? pp[l & 1] : nullptr;
          // layer 0 reads the concatenated input: dW0 = dZ0^T [s | a]  ->  the B operand of the TN product is split too
          mk_backward_layer(b, qi == 0 ? q1 : q2, qa[qi], l, dY[qi], ldd[qi], B, true, dst);
          if (l == 0) {
            GemmArgs& g = b.ops.back().g;  // the TN op just added (no dX at layer 0): its B operand is [s | a]
            g.ldb = O;
            g.A2 = s_act;
            g.lda2 = A;
            g.ksplit = O;
          }
          if (dst) {
            dY[qi] = dst;
            ldd[qi] = q1.d.sizes[l];
          }
        }
        b.end_phase();
      }
    }
    for (int qi = 0; qi < nq; ++qi)
      mk_adam(b, qi == 0 ? q1 : q2, h->adam_tab + (size_t)(1 + qi) * maxS, st, hp->q_beta1, hp->q_beta2, hp->q_eps);
    b.end_phase();
    // ---- delayed policy step + polyak (td3.py:244-263, 301-323) ----
    if (st % hp->policy_delay == 0) {
      float* pa[B200RL_MAX_LAYERS + 1];
      pa[0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lp; ++l) pa[l] = h->acts[2][l];
      for (int l = 0; l < Lp; ++l) {
        mk_forward_layer(b, pi, pa, l, B);
        b.end_phase();
      }
      float* qp[B200RL_MAX_LAYERS + 1];
      qp[0] = const_cast<float*>(s_obs);
      for (int l = 1; l <= Lq; ++l) qp[l] = h->acts[1][l];
      for (int l = 0; l < Lq; ++l) {
        mk_forward_layer(b, q1, qp, l, B, pa[Lp], A, O);  // Q1 with its freshly updated parameters (td3.py:309)
        b.end_phase();
      }
      {  // -mean(Q1(s, pi(s))) is only logged; its gradient is the constant filled above
        MkOp o{};
        o.type = MK_POLICY_LOSS;
        o.p0 = qp[Lq];
        o.o1 = h->out_lp + n_pol;
        b.single(o, B);
      }
      const float* dY = h->dq_pol;
      int ldd = 1;
      for (int l = Lq - 1; l >= 0; --l) {  // gradient w.r.t. Q1's input, parameters frozen
        float* pp[2] = {h->dbuf0, h->dbuf1};
        float* dst = l == 0 ? h->x_cat2 : pp[l & 1];
        mk_backward_layer(b, q1, qp, l, dY, ldd, B, false, dst);
        b.end_phase();
        dY = dst;
        ldd = q1.d.sizes[l];
      }
      dY = h->x_cat2 + O;  // the action columns of dQ/d[s | a]
      ldd = O + A;
      for (int l = Lp - 1; l >= 0; --l) {
        float* pp[2] = {h->dbuf0, h->dbuf1};
        float* dst = l > 0 ? pp[l & 1] : nullptr;
        mk_backward_layer(b, pi, pa, l, dY, ldd, B, true, dst);
        b.end_phase();
        if (dst) {
          dY = dst;
          ldd = pi.d.sizes[l];
        }
      }
      mk_adam(b, pi, h->adam_tab, n_pol, hp->policy_beta1, hp->policy_beta2, hp->policy_eps);
      b.end_phase();
      for (int k = 0; k < (td3 ? 3 : 2); ++k) {
        MkOp o{};
        o.type = MK_POLYAK;
        o.o0 = h->net[3 + k].params;
        o.p0 = h->net[k].params;
        o.f0 = (float)hp->polyak_rho;
        o.f1 = (float)(1.0 - hp->polyak_rho);
        b.elementwise(o, (int)h->net[k].P);
      }
      b.end_phase();
      ++n_pol;
    }
  }
  *n_pol_out = n_pol;
  // upload: one fixed-size block per phase
  std::vector<MkBlock> prog(b.phases.size());
  for (size_t i = 0; i < b.phases.size(); ++i) {
    const MkPhase& ph = b.phases[i];
    B200RL_REQUIRE(ph.n_ops <= MK_MAX_OPS, "offpolicy_train: a phase of %d ops exceeds the block size", ph.n_ops);
    memset(&prog[i], 0, sizeof(MkBlock));
    prog[i].hdr = ph;
    for (int k = 0; k < ph.n_ops; ++k) prog[i].ops[k] = b.ops[ph.op0 + k];
    for (int k = ph.n_ops; k < MK_MAX_OPS; ++k) prog[i].ops[k].n_vb = 0x7fffffff;  // the op search stops here at the latest
  }
  if (prog.size() > h->mk_prog_cap) {
    if (h->mk_prog) cudaFree(h->mk_prog);
    h->mk_prog = nullptr;
    h->mk_prog_cap = 0;
    B200RL_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->mk_prog), prog.size() * sizeof(MkBlock)));
    h->mk_prog_cap = prog.size();
  }
  B200RL_CUDA(cudaMemcpyAsync(h->mk_prog, prog.data(), prog.size() * sizeof(MkBlock), cudaMemcpyHostToDevice, s));
  B200RL_CUDA(cudaStreamSynchronize(s));  // the host vectors go away; the launches behind are ordered on `s` anyway
  h->mk_n_phases = (int)b.phases.size();
  return 0;
}

// Runs the S steps on minibatches ALREADY staged in h->obs ... h->eps (stream h->gs) and reads the logs back.
static int run_staged(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int32_t S, int32_t B, float* q1_values,
                      float* q2_values, float* q1_losses, float* q2_losses, float* policy_losses,
                      int32_t* n_policy_updates) {
  const bool td3 = h->cfg.n_q == 2;
  cudaStream_t s = h->gs;
  const size_t SB = (size_t)S * B;

  // Adam's step-dependent scalars for the steps of this call (torch's host-side double arithmetic), one small upload
  const int maxS = h->cfg.max_steps;
  const int n_pol_expected = (S + hp->policy_delay - 1) / hp->policy_delay;
  for (int k = 0; k < n_pol_expected; ++k)
    adam_scalars(h->net[0].step + k + 1, hp->policy_lr, hp->policy_beta1, hp->policy_beta2, &h->h_adam_tab[k].x,
                 &h->h_adam_tab[k].y);
  for (int qi = 0; qi < (td3 ? 2 : 1); ++qi)
    for (int k = 0; k < S; ++k)
      adam_scalars(h->net[1 + qi].step + k + 1, qi == 0 ? hp->q1_lr : hp->q2_lr, hp->q_beta1, hp->q_beta2,
                   &h->h_adam_tab[(size_t)(1 + qi) * maxS + k].x, &h->h_adam_tab[(size_t)(1 + qi) * maxS + k].y);
  B200RL_CUDA(cudaMemcpyAsync(h->adam_tab, h->h_adam_tab, 3 * (size_t)maxS * sizeof(float2), cudaMemcpyHostToDevice, s));

  int n_pol = 0;
  // opt-in: measured 12.1 ms per 50 TD3 steps against 11.1 ms for the graph replay (B = 256, 256-wide nets) -- the
  // 32 x 32 fp32 tiles themselves, two per SM in the phases that merge four networks, are the cost, not the launches
  const char* menv = getenv("B200RL_OFFPOLICY_MEGAKERNEL");
  const bool use_mega = menv != nullptr && menv[0] == '1';
  const char* genv = getenv("B200RL_OFFPOLICY_GRAPH");
  const bool use_graph = !(genv != nullptr && genv[0] == '0');
  if (use_mega) {
    // ONE cooperative launch runs all S steps (see offpolicy_mega_kernel); the program is rebuilt only when the shape
    // or the hyper-parameters change -- minibatches and Adam's scalars are read from device buffers
    if (h->mk_S != S || h->mk_B != B || memcmp(&h->mk_hp, hp, sizeof(*hp)) != 0) {
      B200RL_CUDA(cudaStreamSynchronize(s));  // the previous program may still be in use
      if (build_program(h, hp, S, B, &n_pol, s)) return 1;
      h->mk_S = S;
      h->mk_B = B;
      h->mk_hp = *hp;
      h->mk_npol = n_pol;
      if (h->mk_grid == 0) {
        int per_sm = 0;
        B200RL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, offpolicy_mega_kernel, GTHREADS, 0));
        B200RL_REQUIRE(per_sm >= 1, "offpolicy_train: the step kernel does not fit an SM");
        h->mk_grid = (per_sm > 2 ? 2 : per_sm) * device_sm_count();
      }
    }
    n_pol = h->mk_npol;
    B200RL_CUDA(cudaMemsetAsync(h->mk_bar, 0, sizeof(unsigned), s));
    const MkBlock* prog = h->mk_prog;
    int n_phases = h->mk_n_phases;
    unsigned* bar = h->mk_bar;
    void* kargs[] = {&prog, &n_phases, &bar};
    B200RL_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(offpolicy_mega_kernel), dim3(h->mk_grid),
                                            dim3(GTHREADS), kargs, 0, s));
    count_launch(1);
  } else if (!use_graph) {
    if (enqueue_steps(h, hp, S, B, s, &n_pol)) return 1;
  } else {
    if (h->graph == nullptr || h->graph_S != S || h->graph_B != B || memcmp(&h->graph_hp, hp, sizeof(*hp)) != 0) {
      if (h->graph) {
        cudaGraphExecDestroy(h->graph);
        h->graph = nullptr;
      }
      const int64_t l0 = launches_total();
      B200RL_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      const int rc = enqueue_steps(h, hp, S, B, s, &n_pol);
      cudaGraph_t g = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(s, &g);
      if (rc || ce != cudaSuccess || g == nullptr) {
        if (g) cudaGraphDestroy(g);
        if (!rc) set_error("offpolicy_train: stream capture failed: %s", cudaGetErrorString(ce));
        return 1;
      }
      const cudaError_t ie = cudaGraphInstantiate(&h->graph, g, 0);
      cudaGraphDestroy(g);
      if (ie != cudaSuccess) {
        h->graph = nullptr;
        set_error("offpolicy_train: cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
        return 1;
      }
      h->graph_launches = (int)(launches_total() - l0);
      count_launch(-h->graph_launches);  // counted per replay below
      h->graph_S = S;
      h->graph_B = B;
      h->graph_hp = *hp;
      h->graph_npol = n_pol;
    }
    n_pol = h->graph_npol;
    B200RL_CUDA(cudaGraphLaunch(h->graph, s));
    count_launch(h->graph_launches);
  }
  h->net[0].step += n_pol;
  h->net[1].step += S;
  if (td3) h->net[2].step += S;
  // one device -> host read of everything train() logs
  B200RL_CUDA(cudaMemcpyAsync(q1_values, h->out_q1, SB * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaMemcpyAsync(q1_losses, h->out_l1, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
  if (td3) {
    B200RL_CUDA(cudaMemcpyAsync(q2_values, h->out_q2, SB * 4, cudaMemcpyDeviceToHost, s));
    B200RL_CUDA(cudaMemcpyAsync(q2_losses, h->out_l2, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
  }
  if (n_pol > 0) B200RL_CUDA(cudaMemcpyAsync(policy_losses, h->out_lp, (size_t)n_pol * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaStreamSynchronize(s));
  *n_policy_updates = n_pol;
  return 0;
}

extern "C" int b200rl_offpolicy_train(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int32_t S, int32_t B,
                                      const float* obs, const float* act, const float* rew, const float* next_obs,
                                      const float* done, const float* noise, float* q1_values, float* q2_values,
                                      float* q1_losses, float* q2_losses, float* policy_losses,
                                      int32_t* n_policy_updates, void* stream) {
  B200RL_REQUIRE(h && hp && obs && act && rew && next_obs && done && q1_values && q1_losses && policy_losses &&
                     n_policy_updates, "offpolicy_train: NULL argument");
  B200RL_REQUIRE(S >= 0 && S <= h->cfg.max_steps && B >= 1 && B <= h->cfg.max_minibatch,
                 "offpolicy_train: S=%d B=%d exceed the capacities", S, B);
  const bool td3 = h->cfg.n_q == 2;
  B200RL_REQUIRE(!td3 || (q2_values && q2_losses), "offpolicy_train: TD3 needs the Q2 outputs");
  B200RL_REQUIRE(!hp->use_target_noise || noise, "offpolicy_train: target noise requested but no noise given");
  B200RL_REQUIRE(hp->policy_delay >= 1, "offpolicy_train: policy_delay must be >= 1");
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  cudaStream_t s = h->gs;  // everything runs on the engine's stream, ordered after the caller's
  const int O = h->O, A = h->A;
  const size_t SB = (size_t)S * B;
  *n_policy_updates = 0;
  if (S == 0) return 0;
  B200RL_CUDA(cudaEventRecord(h->ev, user));
  B200RL_CUDA(cudaStreamWaitEvent(s, h->ev, 0));
  // one host -> device upload of every minibatch of this train() call
  B200RL_CUDA(cudaMemcpyAsync(h->obs, obs, SB * O * 4, cudaMemcpyHostToDevice, s));
  B200RL_CUDA(cudaMemcpyAsync(h->act, act, SB * A * 4, cudaMemcpyHostToDevice, s));
  B200RL_CUDA(cudaMemcpyAsync(h->rew, rew, SB * 4, cudaMemcpyHostToDevice, s));
  B200RL_CUDA(cudaMemcpyAsync(h->nobs, next_obs, SB * O * 4, cudaMemcpyHostToDevice, s));
  B200RL_CUDA(cudaMemcpyAsync(h->done, done, SB * 4, cudaMemcpyHostToDevice, s));
  if (hp->use_target_noise) B200RL_CUDA(cudaMemcpyAsync(h->eps, noise, SB * A * 4, cudaMemcpyHostToDevice, s));


  return run_staged(h, hp, S, B, q1_values, q2_values, q1_losses, q2_losses, policy_losses, n_policy_updates);
}

extern "C" int b200rl_offpolicy_train_gather(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int32_t S,
                                             int32_t B, const float* d_obs, const float* d_act, const float* d_rew,
                                             const float* d_next_obs, const float* d_done, int64_t rows,
                                             const int64_t* idx, const float* noise, float* q1_values,
                                             float* q2_values, float* q1_losses, float* q2_losses,
                                             float* policy_losses, int32_t* n_policy_updates, void* stream) {
  B200RL_REQUIRE(h && hp && d_obs && d_act && d_rew && d_next_obs && d_done && idx && q1_values && q1_losses &&
                     policy_losses && n_policy_updates, "offpolicy_train_gather: NULL argument");
  B200RL_REQUIRE(S >= 0 && S <= h->cfg.max_steps && B >= 1 && B <= h->cfg.max_minibatch,
                 "offpolicy_train_gather: S=%d B=%d exceed the capacities", S, B);
  const bool td3 = h->cfg.n_q == 2;
  B200RL_REQUIRE(!td3 || (q2_values && q2_losses), "offpolicy_train_gather: TD3 needs the Q2 outputs");
  B200RL_REQUIRE(!hp->use_target_noise || noise, "offpolicy_train_gather: target noise requested but no noise given");
  B200RL_REQUIRE(hp->policy_delay >= 1, "offpolicy_train_gather: policy_delay must be >= 1");
  const size_t SB = (size_t)S * B;
  for (size_t i = 0; i < SB; ++i)
    B200RL_REQUIRE(idx[i] >= 0 && idx[i] < rows, "offpolicy_train_gather: index %lld outside the %lld replay rows",
                   (long long)idx[i], (long long)rows);
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  cudaStream_t s = h->gs;
  const int O = h->O, A = h->A;
  *n_policy_updates = 0;
  if (S == 0) return 0;
  B200RL_CUDA(cudaEventRecord(h->ev, user));
  B200RL_CUDA(cudaStreamWaitEvent(s, h->ev, 0));
  // the minibatches are gathered on the device from the replay columns: only the indices (and noise) cross PCIe
  B200RL_CUDA(cudaMemcpyAsync(h->idx, idx, SB * sizeof(long long), cudaMemcpyHostToDevice, s));
  if (hp->use_target_noise) B200RL_CUDA(cudaMemcpyAsync(h->eps, noise, SB * A * 4, cudaMemcpyHostToDevice, s));
  const struct { const float* src; float* dst; int w; } cols[5] = {
      {d_obs, h->obs, O}, {d_act, h->act, A}, {d_rew, h->rew, 1}, {d_next_obs, h->nobs, O}, {d_done, h->done, 1}};
  for (const auto& c : cols) {
    const long long n = (long long)SB * c.w;
    gather_rows_kernel<<<(int)((n + 255) / 256), 256, 0, s>>>(c.src, h->idx, c.w, (long long)SB, c.dst);
    B200RL_CUDA(cudaGetLastError());
    count_launch(1);
  }
  return run_staged(h, hp, S, B, q1_values, q2_values, q1_losses, q2_losses, policy_losses, n_policy_updates);
}

/* Opt-in: the minibatch indices and the target-smoothing noise are DRAWN ON THE DEVICE (Philox4x32-10 keyed by `seed`,
 * block `call`), so nothing but the hyper-parameters crosses PCIe on the way in.  The streams are not the reference's
 * (numpy's MT19937 / torch's CPU generator): same distributions, different numbers -- callers that need the reference's
 * draws use b200rl_offpolicy_train_gather.  The ring: `size` live rows, logical row u at physical (start + u) % rows. */
extern "C" int b200rl_offpolicy_train_gather_rng(b200rl_offpolicy* h, const b200rl_offpolicy_hparams* hp, int32_t S,
                                                 int32_t B, const float* d_obs, const float* d_act, const float* d_rew,
                                                 const float* d_next_obs, const float* d_done, int64_t rows,
                                                 int64_t ring_start, int64_t ring_size, uint64_t seed, uint64_t call,
                                                 float* q1_values, float* q2_values, float* q1_losses,
                                                 float* q2_losses, float* policy_losses, int32_t* n_policy_updates,
                                                 void* stream) {
  B200RL_REQUIRE(h && hp && d_obs && d_act && d_rew && d_next_obs && d_done && q1_values && q1_losses &&
                     policy_losses && n_policy_updates, "offpolicy_train_gather_rng: NULL argument");
  B200RL_REQUIRE(S >= 0 && S <= h->cfg.max_steps && B >= 1 && B <= h->cfg.max_minibatch,
                 "offpolicy_train_gather_rng: S=%d B=%d exceed the capacities", S, B);
  B200RL_REQUIRE(rows >= 1 && ring_size >= 1 && ring_size <= rows && ring_start >= 0 && ring_start < rows,
                 "offpolicy_train_gather_rng: bad ring (rows %lld, start %lld, size %lld)", (long long)rows,
                 (long long)ring_start, (long long)ring_size);
  const bool td3 = h->cfg.n_q == 2;
  B200RL_REQUIRE(!td3 || (q2_values && q2_losses), "offpolicy_train_gather_rng: TD3 needs the Q2 outputs");
  B200RL_REQUIRE(hp->policy_delay >= 1, "offpolicy_train_gather_rng: policy_delay must be >= 1");
  cudaStream_t user = static_cast<cudaStream_t>(stream);
  cudaStream_t s = h->gs;
  const int O = h->O, A = h->A;
  const long long SB = (long long)S * B;
  *n_policy_updates = 0;
  if (S == 0) return 0;
  B200RL_CUDA(cudaEventRecord(h->ev, user));
  B200RL_CUDA(cudaStreamWaitEvent(s, h->ev, 0));
  const long long n_eps = hp->use_target_noise ? SB * A : 0;
  const long long n_thr = ((SB > n_eps ? SB : n_eps) + 3) / 4;
  draw_minibatches_kernel<<<(int)((n_thr + 255) / 256), 256, 0, s>>>(h->idx, SB, n_eps ? h->eps : nullptr, n_eps, seed, call,
                                                                    ring_start, ring_size, rows);
  B200RL_CUDA(cudaGetLastError());
  count_launch(1);
  const struct { const float* src; float* dst; int w; } cols[5] = {
      {d_obs, h->obs, O}, {d_act, h->act, A}, {d_rew, h->rew, 1}, {d_next_obs, h->nobs, O}, {d_done, h->done, 1}};
  for (const auto& c : cols) {
    const long long n = SB * c.w;
    gather_rows_kernel<<<(int)((n + 255) / 256), 256, 0, s>>>(c.src, h->idx, c.w, SB, c.dst);
    B200RL_CUDA(cudaGetLastError());
    count_launch(1);
  }
  return run_staged(h, hp, S, B, q1_values, q2_values, q1_losses, q2_losses, policy_losses, n_policy_updates);
}

/* The draws of the last train_gather / train_gather_rng call (physical rows [S*B], noise [S*B*A] or NULL): what a test
 * replays through the oracle. */
extern "C" int b200rl_offpolicy_get_draws(b200rl_offpolicy* h, int32_t S, int32_t B, int64_t* idx, float* noise,
                                          void* stream) {
  B200RL_REQUIRE(h && idx && S >= 0 && S <= h->cfg.max_steps && B >= 1 && B <= h->cfg.max_minibatch,
                 "offpolicy_get_draws: bad arguments");
  cudaStream_t s = h->gs;
  (void)stream;
  const size_t SB = (size_t)S * B;
  static_assert(sizeof(long long) == sizeof(int64_t), "index width");
  B200RL_CUDA(cudaMemcpyAsync(idx, h->idx, SB * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  if (noise) B200RL_CUDA(cudaMemcpyAsync(noise, h->eps, SB * h->A * 4, cudaMemcpyDeviceToHost, s));
  B200RL_CUDA(cudaStreamSynchronize(s));
  return 0;
}
