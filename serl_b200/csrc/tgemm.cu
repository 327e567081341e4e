// Heads of the 16-bit builds, round 2: single-pass TF32 GEMM on the 5th-gen tensor cores whose operands go from the fp32
// tensors in HBM / L2 STRAIGHT into the MMA - no conversion pass, no threads in the main loop:
//   * both operands are staged by TMA (cp.async.bulk.tensor.3d, 128-byte swizzles, out-of-range rows / columns / k zero-filled by
//     the hardware; element type TFLOAT32, i.e. the copy engine rounds fp32 -> tf32) and consumed by tcgen05.mma kind::tf32;
//   * either operand may be K-major (k contiguous) or MN-major (m / n contiguous): the instruction descriptor's a_major /
//     b_major bits select the layout, so X @ W (W stored (K,N) row-major: MN-major B), dZ @ W^T (K-major B) and X^T @ dZ
//     (both MN-major) - forward, input gradient and weight gradient of a Dense layer (networks/mlp.py:22-31 and its jax.grad
//     transposes) - all read the same row-major fp32 arrays the rest of the step uses;
//   * one CTA per 128 x 256 output tile (x k-split x batch member): warp 0 = TMA producer, warp 1 = MMA issuer (whole warp
//     converged, one elected lane issues, uniform-register operands), warps 2-9 = epilogue (TMEM lane = output row, two warps per lane quarter);
//   * fused epilogues: bias; bias + LayerNorm(eps 1e-6, fast variance) + tanh with the statistics the backward pass needs
//     (an output row is one TMEM lane, so the row reductions are thread-local); + the value head (Q = h . w + b,
//     networks/actor_critic_nets.py:64-72) or the policy's mean / log-std heads with the tanh-Gaussian sample and its
//     log-probability (actor_critic_nets.py:187-227, 230-272) in the same pass;
//   * the reward classifier's hidden layer (networks/reward_classifier.py:22-28): bias + Dropout keep mask + LayerNorm + ReLU and
//     the Dense(1) logit head in one epilogue (LN_RELU_HEAD; train pass with the mask and eval pass without it = two problems).
// Accuracy: TF32 operands (10-bit mantissa, round to nearest), fp32 accumulation - what XLA's default matmul precision gives
// the reference on an NVIDIA GPU; the 16-bit builds are held to 1e-2 (north_star), the fp32 build keeps the SGEMM heads.
// Up to TG_MAXG problem groups (e.g. the three encoder passes x two cameras of a critic step) share one launch.
#include <cuda.h>

#include "gemm_common.cuh"
#include "serl_b200.h"

namespace serl {

constexpr int TG_BM = 128, TG_BN = 256, TG_BK = 32;           // 32 fp32 = 128 B = one swizzle row
constexpr int TG_STAGES = 4;
constexpr int TG_THREADS = 320;                               // TMA warp + MMA warp + 8 epilogue warps
constexpr int TG_EPI_THREADS = 256;
constexpr int TG_MAXG = SERL_TGEMM_MAX_PROBLEMS;
constexpr int TG_A_STAGE = TG_BM * 128, TG_B_STAGE = TG_BN * 128, TG_STAGE = TG_A_STAGE + TG_B_STAGE;
constexpr int TG_MAXHEAD = 8;
// epilogue vectors: bias, ln scale, ln bias (3 x 256), head weights (2 x 256 x 8), head biases (16)
constexpr int TG_SMEM = TG_STAGES * TG_STAGE + (3 * TG_BN + 2 * TG_BN * TG_MAXHEAD + 16) * 4 + 128 + 1024;

struct TgMaps { CUtensorMap a[TG_MAXG]; CUtensorMap b[TG_MAXG]; };

struct TgGroup {
  float* C; const float* bias; const float* ln_scale; const float* ln_bias; float* xhat; float* rstd;
  const float* head_w; const float* head_b; float* head_out;
  const float* head_w2; const float* head_b2; float* head_out2;
  const float* noise; float* act; float* logp; float* u_out; float* std_out;
  const uint8_t* keep_mask; float keep;
  long long sCz, sBiasZ, sLnZ, sXhatZ, sRstdZ, sHeadWz, sHeadBz, sHeadOutZ;
  int ldc, ld_head, ld_act, z0, Z, a_bcast, b_bcast;
};
struct TgArgs {
  TgGroup g[TG_MAXG];
  float* ws;
  int32_t* error;
  int G, M, N, K, S, kchunk, epi, a_mn, b_mn, accumulate, to_ws, head_n, deterministic;
  float eps, std_min, std_max;
};

__device__ inline uint32_t tg_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ inline bool tg_wait(uint64_t* bar, uint32_t parity, int32_t* error) {            // bounded: a protocol bug must not hang the box
  const uint32_t addr = tg_smem(bar);
  const long long t0 = clock64();
#pragma unroll 1
  for (;;) {
    uint32_t done;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    if (done) return true;
    if (clock64() - t0 > 2000000000ll) break;
  }
  if (error) atomicOr(error, 32);
  return false;
}
__device__ inline void tg_tma_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(dst), "l"(map), "r"(tg_smem(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// four k-steps (UMMA_K = 8 tf32) of one k-block in one statement, executed by the whole converged issuer warp with
// warp-uniform operands; one elected lane issues (see r3_mma_x4 in conv3x3_res.cu for why)
__device__ inline void tg_mma_x4(uint32_t tmem_d, uint64_t ad, uint64_t bd, uint64_t astep, uint64_t bstep, uint32_t idesc, uint32_t acc_first) {
  asm volatile("{\n .reg .pred p, t, e;\n .reg .b64 a1, a2, a3, b1, b2, b3;\n"
               " elect.sync _|e, 0xffffffff;\n"
               " setp.ne.b32 p, %6, 0;\n setp.eq.u32 t, 0, 0;\n"
               " add.u64 a1, %1, %3;\n add.u64 a2, a1, %3;\n add.u64 a3, a2, %3;\n"
               " add.u64 b1, %2, %4;\n add.u64 b2, b1, %4;\n add.u64 b3, b2, %4;\n"
               " @e tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %5, p;\n"
               " @e tcgen05.mma.cta_group::1.kind::tf32 [%0], a1, b1, %5, t;\n"
               " @e tcgen05.mma.cta_group::1.kind::tf32 [%0], a2, b2, %5, t;\n"
               " @e tcgen05.mma.cta_group::1.kind::tf32 [%0], a3, b3, %5, t;\n}"
               ::"r"(tmem_d), "l"(ad), "l"(bd), "l"(astep), "l"(bstep), "r"(idesc), "r"(acc_first) : "memory");
}
__device__ inline void tg_commit_w(uint64_t* bar) {
  asm volatile("{\n .reg .pred e;\n elect.sync _|e, 0xffffffff;\n"
               " @e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}" ::"r"(tg_smem(bar)) : "memory");
}
__device__ inline void tg_arrive_w(uint64_t* bar) {
  asm volatile("{\n .reg .pred e;\n elect.sync _|e, 0xffffffff;\n @e mbarrier.arrive.shared::cta.b64 _, [%0];\n}" ::"r"(tg_smem(bar)) : "memory");
}
__device__ inline void tg_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// tanh(x) = 1 - 2 / (exp(2x) + 1) on the special-function unit (ex2.approx + rcp.approx): absolute error < 3e-7, exact limits
__device__ inline float tg_tanh(float x) { return 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f); }
__device__ inline float tg_softplus(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

// kRelu: the LN_RELU_HEAD instantiation; every other epilogue runs the kRelu = false instantiation, whose code is the tanh epilogues' alone
template <bool kRelu>
__global__ void __launch_bounds__(TG_THREADS, 1) tgemm_tf32_kernel(const __grid_constant__ TgMaps maps, const __grid_constant__ TgArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sOp = smem;                                                   // TG_STAGES x [A 16 KB | B 32 KB]
  float* sVec = reinterpret_cast<float*>(smem + TG_STAGES * TG_STAGE);     // bias | ln scale | ln bias | head w | head w2 | head b, b2
  float* sBias = sVec, *sLs = sVec + TG_BN, *sLb = sVec + 2 * TG_BN, *sHw = sVec + 3 * TG_BN, *sHw2 = sHw + TG_BN * TG_MAXHEAD, *sHb = sHw2 + TG_BN * TG_MAXHEAD;
  uint64_t* full = reinterpret_cast<uint64_t*>(sHb + 16);
  uint64_t* empty = full + TG_STAGES;
  uint64_t* done = empty + TG_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int zz = blockIdx.z / a.S, ks = blockIdx.z - zz * a.S;
  int gi = 0;
#pragma unroll
  for (int i = 1; i < TG_MAXG; ++i) if (i < a.G && zz >= a.g[i].z0) gi = i;
  const TgGroup& g = a.g[gi];
  const int z = zz - g.z0;
  const int m0 = blockIdx.x * TG_BM, n0 = blockIdx.y * TG_BN;
  const int kbeg = ks * a.kchunk, kend = min(a.K, kbeg + a.kchunk);
  const int nk = kend > kbeg ? ceil_div(kend - kbeg, TG_BK) : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TG_STAGES; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tg_smem(&full[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tg_smem(&empty[s])));
    }
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tg_smem(done)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tg_smem(tmem_slot)), "r"((uint32_t)TG_BN) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.a[gi]) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.b[gi]) : "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;
  // Programmatic dependent launch: everything above (barriers, tensor-memory allocation, descriptor prefetch) touches no data
  // of the previous kernel and overlaps its tail; nothing below starts before that kernel has completed.
  pdl_prologue();

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      const int za = g.a_bcast ? 0 : z, zb = g.b_bcast ? 0 : z;
      bool ok = true;
      for (int kt = 0; kt < nk && ok; ++kt) {
        const int s = kt % TG_STAGES;
        ok = tg_wait(&empty[s], ((uint32_t)(kt / TG_STAGES) & 1u) ^ 1u, a.error);
        if (!ok) break;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tg_smem(&full[s])), "r"((uint32_t)TG_STAGE) : "memory");
        const uint32_t dA = tg_smem(sOp + s * TG_STAGE), dB = dA + TG_A_STAGE;
        const int k0 = kbeg + kt * TG_BK;
        if (!a.a_mn) tg_tma_3d(dA, &maps.a[gi], k0, m0, za, &full[s]);                               // box (32 k, 128 m)
        else {
#pragma unroll
          for (int j = 0; j < TG_BM / 32; ++j) tg_tma_3d(dA + j * 4096, &maps.a[gi], m0 + 32 * j, k0, za, &full[s]);   // box (32 m, 32 k)
        }
        if (!a.b_mn) tg_tma_3d(dB, &maps.b[gi], k0, n0, zb, &full[s]);                               // box (32 k, 256 n)
        else {
#pragma unroll
          for (int j = 0; j < TG_BN / 32; ++j) tg_tma_3d(dB + j * 4096, &maps.b[gi], n0 + 32 * j, k0, zb, &full[s]);   // box (32 n, 32 k)
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (whole warp, converged) ===============================
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(a.a_mn != 0) << 15) | ((uint32_t)(a.b_mn != 0) << 16) |
                           ((uint32_t)(TG_BN >> 3) << 17) | ((uint32_t)(TG_BM >> 4) << 24);
    // K-major, SWIZZLE_128B: SBO = 1024 B between 8-row groups, k-step (8 tf32 = 32 B) = +2 units of 16 B
    // MN-major 32-bit operands exist in ONE shared-memory layout, SWIZZLE_128B_BASE32B (layout type 1; TMA: SWIZZLE_128B_ATOM_32B):
    // rows of 128 B = 32 consecutive m / n for one k, 32-byte chunks XOR-ed with (k & 3); atom = 4 k-rows (512 B).
    // LBO = 4096 B between 32-element blocks along M / N, SBO = 512 B between 4-k groups, k-step (8 k-rows) = +64 units
    const uint64_t desc_k = (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
    const uint64_t desc_mn = (256ull << 16) | (32ull << 32) | (1ull << 46) | (1ull << 61);
    const uint64_t da_hi = a.a_mn ? desc_mn : desc_k, db_hi = a.b_mn ? desc_mn : desc_k;
    const uint64_t astep = a.a_mn ? 64ull : 2ull, bstep = a.b_mn ? 64ull : 2ull;
    bool ok = true;
    for (int kt = 0; kt < nk && ok; ++kt) {
      const int s = kt % TG_STAGES;
      ok = __all_sync(0xffffffffu, tg_wait(&full[s], (uint32_t)(kt / TG_STAGES) & 1u, a.error));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = tg_smem(sOp + s * TG_STAGE);
      const uint64_t ad = da_hi | (uint64_t)((sa & 0x3FFFF) >> 4), bd = db_hi | (uint64_t)(((sa + TG_A_STAGE) & 0x3FFFF) >> 4);
      if (ok) tg_mma_x4(tmem_d, ad, bd, astep, bstep, idesc, (uint32_t)(kt != 0));
      tg_commit_w(&empty[s]);
    }
    if (ok && nk > 0) tg_commit_w(done); else tg_arrive_w(done);
  } else {
    // =============================== epilogue: 8 warps, thread = (output row = TMEM lane, column half) ===============================
    // Two warps per TMEM lane quarter, 128 columns each: with one warp per scheduler the dependent chains of the LayerNorm /
    // tanh arithmetic ran at a fraction of the issue rate; the two halves of a row meet through shared memory.
    const int et = threadIdx.x - 64;                                     // 0..255
    const int q = warp & 3;                                              // TMEM lane quarter this warp may access
    const int hh = (warp - 2) >> 2;                                      // column half
    const int row = q * 32 + lane, m = m0 + row;
    const int c_lo = hh * (TG_BN / 2), c_hi = c_lo + TG_BN / 2;
    constexpr bool relu = kRelu;
    const bool ln = (a.epi >= SERL_TGEMM_EPI_LN_TANH && a.epi <= SERL_TGEMM_EPI_LN_TANH_POLICY) || relu;
    // stage the epilogue vectors while the main loop runs
    if (!a.to_ws) {
      const float* bias = g.bias ? g.bias + z * g.sBiasZ : nullptr;
      for (int c = et; c < TG_BN; c += TG_EPI_THREADS) {
        const int n = n0 + c;
        sBias[c] = (bias && n < a.N) ? bias[n] : 0.f;
        if (ln) { sLs[c] = g.ln_scale[z * g.sLnZ + n]; sLb[c] = g.ln_bias[z * g.sLnZ + n]; }
      }
      if (ln && a.epi >= SERL_TGEMM_EPI_LN_TANH_HEAD) {
        const float* hw = g.head_w + z * g.sHeadWz;
        for (int i = et; i < TG_BN * a.head_n; i += TG_EPI_THREADS) sHw[i] = hw[i];
        if (et < a.head_n) sHb[et] = g.head_b ? g.head_b[z * g.sHeadBz + et] : 0.f;
        if (a.epi == SERL_TGEMM_EPI_LN_TANH_POLICY) {
          for (int i = et; i < TG_BN * a.head_n; i += TG_EPI_THREADS) sHw2[i] = g.head_w2[i];
          if (et < a.head_n) sHb[8 + et] = g.head_b2 ? g.head_b2[et] : 0.f;
        }
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const bool ok = tg_wait(done, 0u, a.error);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tbase = tmem_d + ((uint32_t)(q * 32) << 16);
    const bool have = ok && nk > 0;
    // after `done` every MMA has read its operands and every TMA load has landed: the operand stages are free scratch
    float* sPart = reinterpret_cast<float*>(sOp);                        // [2 halves][128 rows][2]: sum, sum of squares
    float* sHeadPart = sPart + 2 * TG_BM * 2;                            // [128 rows][16]: half 1's head partial sums
    // Output rows leave through a per-warp staging tile (32 rows x 32 columns, 16-byte chunks XOR-swizzled by row): a thread owns
    // a ROW of the accumulator, so direct stores put the 32 lanes of an instruction on 32 different lines (measured: the
    // epilogue's time was these stores); staged, one instruction writes 4 rows x 128 contiguous bytes.
    float* sTile = reinterpret_cast<float*>(sOp + 16384) + (warp - 2) * 2048;   // two tiles per warp: activation | xhat
    const int row_w = m0 + q * 32;                                       // first global row of this warp
    auto stage = [&](float* tile, const float (&v)[32]) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(tile + lane * 32 + ((j ^ (lane & 7)) << 2)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    };
    auto flush = [&](const float* tile, float* gbase, long long ld, int col, bool acc, bool live) {
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = 4 * i + (lane >> 3), j = lane & 7;
        float4 o = *reinterpret_cast<const float4*>(tile + rr * 32 + ((j ^ (rr & 7)) << 2));
        if (live && row_w + rr < a.M) {
          float4* p = reinterpret_cast<float4*>(gbase + (size_t)(row_w + rr) * ld + col + 4 * j);
          if (acc) { const float4 old = *p; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
          *p = o;
        }
      }
      __syncwarp();
    };
    if (a.to_ws || !ln) {
      float* dst; long long ld;
      if (a.to_ws) { dst = a.ws + ((size_t)blockIdx.z * a.M) * a.N; ld = a.N; }
      else { dst = g.C + z * g.sCz; ld = g.ldc; }
      const bool vec = ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) && (ld % 4 == 0);
      const bool acc = !a.to_ws && a.accumulate;
#pragma unroll 1
      for (int c = c_lo; c < c_hi; c += 32) {
        if (n0 + c >= a.N) break;                                        // warp-uniform
        float v[32];
        if (have) tg_ld32(tbase + (uint32_t)c, v);
        else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (vec && n0 + c + 32 <= a.N) {                                 // warp-uniform
          if (!a.to_ws) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] += sBias[c + i];
          }
          stage(sTile, v);
          flush(sTile, dst, ld, n0 + c, acc, true);
        } else if (m < a.M) {
          float* rowp = dst + (size_t)m * ld + n0 + c;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (n0 + c + i < a.N) {
              float o = v[i] + (a.to_ws ? 0.f : sBias[c + i]);
              rowp[i] = acc ? rowp[i] + o : o;
            }
          }
        }
      }
    } else {
      // ---- bias [+ dropout] + LayerNorm + tanh | ReLU (N == 256: a row = this thread's 128 columns + its partner's) ----
      // LN_RELU_HEAD with a keep mask: d = mask ? (acc + bias) / keep : 0 (flax Dropout), applied before the statistics
      const uint8_t* mrow = (relu && g.keep_mask && m < a.M) ? g.keep_mask + (size_t)m * TG_BN : nullptr;
      auto drop = [&](float (&v)[32], int c) {
        if (relu && mrow) {
          const uint4 b0 = *reinterpret_cast<const uint4*>(mrow + c), b1 = *reinterpret_cast<const uint4*>(mrow + c + 16);
          const uint32_t w[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = ((w[i >> 2] >> (8 * (i & 3))) & 0xffu) ? v[i] / g.keep : 0.f;
        }
      };
      float s = 0.f, ss = 0.f;
#pragma unroll 1
      for (int c = c_lo; c < c_hi; c += 32) {
        float v[32];
        tg_ld32(tbase + (uint32_t)c, v);
        if constexpr (relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += sBias[c + i];
          drop(v, c);
#pragma unroll
          for (int i = 0; i < 32; ++i) { const float x = v[i]; s += x; ss += x * x; }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) { const float x = v[i] + sBias[c + i]; s += x; ss += x * x; }
        }
      }
      *reinterpret_cast<float2*>(sPart + (hh * TG_BM + row) * 2) = make_float2(s, ss);
      asm volatile("bar.sync 1, 256;" ::: "memory");
      {
        const float2 o = *reinterpret_cast<const float2*>(sPart + ((hh ^ 1) * TG_BM + row) * 2);
        // fixed summation order (half 0 + half 1) so that both threads of a row hold bit-identical statistics
        const float2 p0 = hh ? o : make_float2(s, ss), p1 = hh ? make_float2(s, ss) : o;
        s = p0.x + p1.x; ss = p0.y + p1.y;
      }
      const float mean = s * (1.f / TG_BN);
      const float var = fmaxf(ss * (1.f / TG_BN) - mean * mean, 0.f);
      const float rstd = rsqrtf(var + a.eps);
      float hacc[2 * TG_MAXHEAD];
#pragma unroll
      for (int i = 0; i < 2 * TG_MAXHEAD; ++i) hacc[i] = 0.f;
      float* hbase = g.C ? g.C + z * g.sCz : nullptr;
      float* xbase = g.xhat ? g.xhat + z * g.sXhatZ : nullptr;
      const bool hvec = hbase && ((reinterpret_cast<uintptr_t>(hbase) & 15) == 0) && (g.ldc % 4 == 0);
      const bool valid = have && m < a.M;
#pragma unroll 1
      for (int c = c_lo; c < c_hi; c += 32) {
        float v[32];
        tg_ld32(tbase + (uint32_t)c, v);
        float h[32];
        if constexpr (relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += sBias[c + i];
          drop(v, c);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float xh = (v[i] - mean) * rstd;
            v[i] = xh;
            h[i] = fmaxf(fmaf(xh, sLs[c + i], sLb[c + i]), 0.f);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float xh = (v[i] + sBias[c + i] - mean) * rstd;
            v[i] = xh;
            h[i] = tg_tanh(fmaf(xh, sLs[c + i], sLb[c + i]));
          }
        }
        if (hbase) {
          if (hvec) { stage(sTile, h); flush(sTile, hbase, g.ldc, c, false, have); }
          else if (valid) {
#pragma unroll
            for (int i = 0; i < 32; ++i) hbase[(size_t)m * g.ldc + c + i] = h[i];
          }
        }
        if (xbase) { stage(sTile + 1024, v); flush(sTile + 1024, xbase, TG_BN, c, false, have); }
        if (a.epi >= SERL_TGEMM_EPI_LN_TANH_HEAD) {
#pragma unroll
          for (int j = 0; j < TG_MAXHEAD; ++j) {
            if (j < a.head_n) {
              float t = hacc[j], t2 = hacc[TG_MAXHEAD + j];
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                t = fmaf(h[i], sHw[(c + i) * a.head_n + j], t);
                if (a.epi == SERL_TGEMM_EPI_LN_TANH_POLICY) t2 = fmaf(h[i], sHw2[(c + i) * a.head_n + j], t2);
              }
              hacc[j] = t; hacc[TG_MAXHEAD + j] = t2;
            }
          }
        }
      }
      if (valid && g.rstd && hh == 0) g.rstd[z * g.sRstdZ + m] = rstd;
      if (a.epi >= SERL_TGEMM_EPI_LN_TANH_HEAD) {
        // half 1 hands its partial head sums to half 0, which finishes the row
        if (hh == 1) {
#pragma unroll
          for (int j = 0; j < 2 * TG_MAXHEAD; ++j) sHeadPart[row * 16 + j] = hacc[j];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (hh == 0) {
#pragma unroll
          for (int j = 0; j < 2 * TG_MAXHEAD; ++j) hacc[j] += sHeadPart[row * 16 + j];
        }
      }
      if (valid && hh == 0) {
        if (a.epi == SERL_TGEMM_EPI_LN_TANH_HEAD || relu) {
          float* o = g.head_out + z * g.sHeadOutZ + (size_t)m * g.ld_head;
#pragma unroll
          for (int j = 0; j < TG_MAXHEAD; ++j) if (j < a.head_n) o[j] = hacc[j] + sHb[j];
        } else if (a.epi == SERL_TGEMM_EPI_LN_TANH_POLICY) {
          // means / log-stds -> tanh-Gaussian sample and its log-probability (same arithmetic as tanh_gaussian_fwd_kernel, sac_ops.cu)
          const int A = a.head_n;
          float lp = 0.f;
#pragma unroll
          for (int j = 0; j < TG_MAXHEAD; ++j) {
            if (j >= A) break;
            const float mu = hacc[j] + sHb[j], lsd = hacc[TG_MAXHEAD + j] + sHb[8 + j];
            if (g.head_out) g.head_out[(size_t)m * A + j] = mu;
            if (g.head_out2) g.head_out2[(size_t)m * A + j] = lsd;
            const float sd = fminf(fmaxf(expf(lsd), a.std_min), a.std_max);
            const float e = a.deterministic ? 0.f : g.noise[(size_t)m * A + j];
            const float u = mu + sd * e;
            const float zn = (u - mu) / sd;
            lp += -0.5f * zn * zn - logf(sd) - 0.918938533204672742f;
            lp -= 2.f * (0.693147180559945309f - u - tg_softplus(-2.f * u));
            g.act[(size_t)m * g.ld_act + j] = tanhf(u);
            if (g.u_out) g.u_out[(size_t)m * A + j] = u;
            if (g.std_out) g.std_out[(size_t)m * A + j] = sd;
          }
          if (g.logp) g.logp[m] = lp;
        }
      }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)TG_BN) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
typedef CUresult (*TgEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TgEncodeFn tg_get_encode() {
  static TgEncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<TgEncodeFn>(p);
  }
  return fn;
}

// Operand seen as (rows R, depth K) with element (r, k) at base + z*sZ + r*sR + k*sK (floats), one of sR / sK == 1.
// K-major (sK == 1): tensor (k, r, z), box (32, box_rows, 1).   MN-major (sR == 1): tensor (r, k, z), box (32, 32, 1).
static bool tg_operand_map(CUtensorMap* map, const float* base, int R, int K, int Z, long long sZ, long long sR, long long sK, int box_rows,
                           bool* mn, int* bcast) {
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return false;
  const bool kmaj = (sK == 1) && (sR % 4 == 0) && sR >= K;
  const bool mmaj = (sR == 1) && (sK % 4 == 0) && sK >= R;
  if (!kmaj && !mmaj) return false;
  *mn = !kmaj;
  *bcast = (Z > 1 && sZ == 0) ? 1 : 0;
  const int zdim = (*bcast || Z < 1) ? 1 : Z;
  if (zdim > 1 && sZ % 4 != 0) return false;
  const long long inner = kmaj ? K : R, outer = kmaj ? R : K, so = kmaj ? sR : sK;
  // the z stride of a single-member tensor is never used for addressing; any legal value will do
  const long long sz = zdim > 1 ? sZ : ((outer * so + 3) / 4) * 4;
  const cuuint64_t gdim[3] = {(cuuint64_t)inner, (cuuint64_t)outer, (cuuint64_t)zdim};
  const cuuint64_t gstr[2] = {(cuuint64_t)so * 4, (cuuint64_t)(sz > 0 ? sz : 4) * 4};
  const cuuint32_t box[3] = {32u, (cuuint32_t)(kmaj ? box_rows : 32), 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return tg_get_encode()(map, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 3, const_cast<float*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         kmaj ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace serl

using namespace serl;

extern "C" int serl_tgemm_tf32(const serl_tgemm_desc* d, void* stream) {
  if (!d || !d->problems || d->num_problems < 1 || d->num_problems > TG_MAXG || d->M < 1 || d->N < 1 || d->K < 1) {
    set_last_error("serl_tgemm_tf32: invalid descriptor"); return SERL_ERR_INVALID;
  }
  if (!tg_get_encode()) { set_last_error("serl_tgemm_tf32: cuTensorMapEncodeTiled unavailable"); return SERL_ERR_CUDA; }
  static bool attr_done = false;
  if (!attr_done) {
    if (cudaFuncSetAttribute(tgemm_tf32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM) != cudaSuccess ||
        cudaFuncSetAttribute(tgemm_tf32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TG_SMEM) != cudaSuccess) {
      set_last_error("serl_tgemm_tf32: cannot reserve %d bytes of shared memory", TG_SMEM); return SERL_ERR_CUDA;
    }
    attr_done = true;
  }
  const bool relu = d->epilogue == SERL_TGEMM_EPI_LN_RELU_HEAD;
  const bool ln = (d->epilogue >= SERL_TGEMM_EPI_LN_TANH && d->epilogue <= SERL_TGEMM_EPI_LN_TANH_POLICY) || relu;
  const bool partial = d->epilogue == SERL_TGEMM_EPI_PARTIAL;
  if (d->epilogue < 0 || d->epilogue > SERL_TGEMM_EPI_LN_RELU_HEAD) { set_last_error("serl_tgemm_tf32: unknown epilogue %d", d->epilogue); return SERL_ERR_INVALID; }
  if (ln && (d->N != TG_BN || d->reduce_z || d->splits > 1)) { set_last_error("serl_tgemm_tf32: LayerNorm epilogues need N == 256, no k-split, no reduce_z"); return SERL_ERR_UNSUPPORTED; }
  if (ln && d->epilogue >= SERL_TGEMM_EPI_LN_TANH_HEAD && (d->head_n < 1 || d->head_n > TG_MAXHEAD)) { set_last_error("serl_tgemm_tf32: head_n in [1, 8]"); return SERL_ERR_UNSUPPORTED; }
  TgMaps maps;
  TgArgs a{};
  a.G = d->num_problems; a.M = d->M; a.N = d->N; a.K = d->K; a.epi = d->epilogue; a.accumulate = d->accumulate; a.head_n = d->head_n;
  a.eps = d->ln_eps; a.std_min = d->std_min; a.std_max = d->std_max; a.deterministic = d->deterministic; a.error = d->error;
  int ztotal = 0;
  for (int i = 0; i < d->num_problems; ++i) {
    const serl_tgemm_problem& p = d->problems[i];
    TgGroup& g = a.g[i];
    if (!p.A || !p.B || p.Z < 1) { set_last_error("serl_tgemm_tf32: problem %d: A, B, Z required", i); return SERL_ERR_INVALID; }
    bool amn = false, bmn = false;
    if (!tg_operand_map(&maps.a[i], p.A, d->M, d->K, p.Z, p.sAz, p.sAm, p.sAk, TG_BM, &amn, &g.a_bcast) ||
        !tg_operand_map(&maps.b[i], p.B, d->N, d->K, p.Z, p.sBz, p.sBn, p.sBk, TG_BN, &bmn, &g.b_bcast)) {
      set_last_error("serl_tgemm_tf32: problem %d: operands must be 16-byte aligned with one unit stride and the other a multiple of 4 floats", i);
      return SERL_ERR_UNSUPPORTED;
    }
    if (i == 0) { a.a_mn = amn; a.b_mn = bmn; }
    else if (a.a_mn != (int)amn || a.b_mn != (int)bmn) { set_last_error("serl_tgemm_tf32: all problems of a launch share the operand layouts"); return SERL_ERR_UNSUPPORTED; }
    g.C = p.C; g.bias = p.bias; g.ln_scale = p.ln_scale; g.ln_bias = p.ln_bias; g.xhat = p.xhat; g.rstd = p.rstd;
    g.head_w = p.head_w; g.head_b = p.head_b; g.head_out = p.head_out; g.head_w2 = p.head_w2; g.head_b2 = p.head_b2; g.head_out2 = p.head_out2;
    g.noise = p.noise; g.act = p.act; g.logp = p.logp; g.u_out = p.u_out; g.std_out = p.std_out;
    g.keep_mask = relu ? p.keep_mask : nullptr; g.keep = p.keep;
    if (g.keep_mask && (!(p.keep > 0.f) || (reinterpret_cast<uintptr_t>(p.keep_mask) & 15) || p.Z != 1)) {
      set_last_error("serl_tgemm_tf32: problem %d: keep_mask needs keep > 0, 16-byte alignment and Z == 1", i); return SERL_ERR_INVALID;
    }
    g.sCz = p.sCz; g.sBiasZ = p.sBiasZ; g.sLnZ = p.sLnZ; g.sXhatZ = p.sXhatZ; g.sRstdZ = p.sRstdZ; g.sHeadWz = p.sHeadWz; g.sHeadBz = p.sHeadBz;
    g.sHeadOutZ = p.sHeadOutZ; g.ldc = p.ldc; g.ld_head = p.ld_head; g.ld_act = p.ld_act; g.z0 = ztotal; g.Z = p.Z;
    if (!d->reduce_z && !p.C && !ln && !partial) { set_last_error("serl_tgemm_tf32: problem %d: C required", i); return SERL_ERR_INVALID; }
    if (ln && (!p.ln_scale || !p.ln_bias)) { set_last_error("serl_tgemm_tf32: problem %d: LayerNorm scale / bias required", i); return SERL_ERR_INVALID; }
    if (ln && d->epilogue >= SERL_TGEMM_EPI_LN_TANH_HEAD && (!p.head_w || !p.head_out)) { set_last_error("serl_tgemm_tf32: problem %d: head_w / head_out required", i); return SERL_ERR_INVALID; }
    if (d->epilogue == SERL_TGEMM_EPI_LN_TANH_POLICY && (!p.head_w2 || !p.act || (!d->deterministic && !p.noise) || p.Z != 1)) {
      set_last_error("serl_tgemm_tf32: problem %d: policy epilogue needs head_w2, act, noise and Z == 1", i); return SERL_ERR_INVALID;
    }
    ztotal += p.Z;
  }
  // k-splits: these GEMMs are tiny (<= 1 GFLOP); with fewer tiles than SMs split K until about one wave exists
  const int tiles = ceil_div(d->M, TG_BM) * ceil_div(d->N, TG_BN) * ztotal;
  int S = 1;
  if (!ln) {
    if (d->splits > 0) S = d->splits;
    else if (tiles < 74 && d->K >= 512) { S = 148 / tiles; if (S > d->K / 128) S = d->K / 128; if (S < 1) S = 1; }
  }
  const size_t part = (size_t)d->M * d->N * sizeof(float);
  if (partial) {
    // the caller reduces: partial products of split s of member zz (counted across the problems) at workspace[(zz * S + s)][M][N]
    S = d->splits > 0 ? d->splits : 1;
    if (d->reduce_z || !d->workspace) { set_last_error("serl_tgemm_tf32: the PARTIAL epilogue needs a workspace and no reduce_z"); return SERL_ERR_INVALID; }
    const int kc = ceil_div(ceil_div(d->K, S), TG_BK) * TG_BK;
    if (ceil_div(d->K, kc) != S) { set_last_error("serl_tgemm_tf32: %d splits of K = %d leave empty splits", S, d->K); return SERL_ERR_INVALID; }
    if (part * (size_t)ztotal * S > d->workspace_bytes) { set_last_error("serl_tgemm_tf32: PARTIAL needs %zu workspace bytes", part * (size_t)ztotal * S); return SERL_ERR_INVALID; }
  } else if (d->reduce_z || S > 1) {
    if (d->num_problems != 1) { set_last_error("serl_tgemm_tf32: k-split / reduce_z launches take one problem"); return SERL_ERR_UNSUPPORTED; }
    while (S > 1 && part * (size_t)ztotal * S > d->workspace_bytes) --S;
    if (!d->workspace || part * (size_t)ztotal * S > d->workspace_bytes) {
      if (d->reduce_z) { set_last_error("serl_tgemm_tf32: reduce_z needs %zu workspace bytes", part * (size_t)ztotal); return SERL_ERR_INVALID; }
      S = 1;
    }
  }
  a.kchunk = ceil_div(ceil_div(d->K, S), TG_BK) * TG_BK;
  S = ceil_div(d->K, a.kchunk);
  a.S = S;
  a.to_ws = (partial || d->reduce_z || S > 1) ? 1 : 0;
  a.ws = d->workspace;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid(ceil_div(d->M, TG_BM), ceil_div(d->N, TG_BN), ztotal * S);
  if (relu) launch_k(tgemm_tf32_kernel<true>, grid, TG_THREADS, TG_SMEM, st, maps, a);
  else launch_k(tgemm_tf32_kernel<false>, grid, TG_THREADS, TG_SMEM, st, maps, a);
  if (int e = check_launch("tgemm_tf32_kernel")) return e;
  if (a.to_ws && !partial) {
    const serl_tgemm_problem& p = d->problems[0];
    GemmArgs r{};
    r.C = p.C; r.bias = p.bias; r.ws = d->workspace; r.M = d->M; r.N = d->N; r.K = d->K; r.Z = p.Z; r.S = S;
    r.sCz = p.sCz; r.sBiasZ = p.sBiasZ; r.ldc = p.ldc; r.accumulate = d->accumulate;
    return launch_gemm_reduce(r, d->reduce_z, st);
  }
  return SERL_OK;
}
