// Replay minibatch sampler for the HBM-resident frame-dedup ring.
//
// ONE kernel per (buffer, step): draws uniform indices (Philox4x32-10 + Lemire, bounded redraw on
// invalid slots), gathers (s, a, r, s', mask, done) and the T+1 adjacent camera frames, and applies
// the DrQ random shift (edge-replicating crop) on the way out.  Frames are staged global->shared with
// a TMA bulk copy (cp.async.bulk, 16-byte aligned row ranges) and written back with 128-bit stores.
//
// Replaces (reference, relative to serl_launcher/serl_launcher):
//   data/memory_efficient_replay_buffer.py:91-164  sample()      (host python loop + numpy gather)
//   data/replay_buffer.py:77-90                    get_iterator  (host->device copy of the batch)
//   utils/train_utils.py:44-66                     _unpack
//   vision/data_augmentations.py:7-36 + agents/continuous/drq.py:244-253  batched_random_crop
// Semantics are restated in oracle/replay.py (draw_indices, gather_packed, random_shift) and
// oracle/jax_prng.py (crop_offsets).
#include "common.cuh"
#include "serl_b200.h"

namespace serl {

constexpr int kBandRows = 32;
constexpr int kSamplerThreads = 128;
constexpr int kMaxDrawAttempts = 64;

struct SamplerArgs {
  serl_replay_view rv;
  // draw
  uint64_t seed, step;
  const uint64_t* step_dev;      // optional device counter overriding `step` (CUDA-graph replays)
  const int32_t* size_dev;       // optional device fill level overriding rv.size
  uint32_t lane_offset;          // philox lane of row 0 (independent of out_row_offset)
  const int32_t* explicit_idx;   // optional (B): skip the draw
  // crop
  const uint32_t* key_obs;       // device, 2 words: JAX key whose split(key, crop_total)[g] seeds frame g
  const uint32_t* key_next;
  const int32_t* explicit_off_obs;   // optional (crop_total, 2) [cy, cx]
  const int32_t* explicit_off_next;
  int crop_total;                // total frames in the (possibly concatenated) batch = B_total * T
  int out_row_offset;            // first output row of this launch inside the B_total-row outputs
  int padding;
  // outputs (B_total rows each)
  uint8_t* obs_pix[SERL_MAX_CAMS];    // (B_total, T, H, W, C)
  uint8_t* next_pix[SERL_MAX_CAMS];
  float* obs_state; float* next_state; float* actions; float* rewards; float* masks;
  uint8_t* dones; int32_t* idx_out; int32_t* off_obs_out; int32_t* off_next_out;   // off_*: (B_total*T, 2)
  int32_t* status;               // device int, OR-ed with 1 when a draw fails
  int batch;                     // rows produced by this launch
  int one_side;                  // 0: obs and next frames; 1: obs frames only; 2: next frames only (the other side's pointers are NULL)
};

__device__ inline int draw_index(const SamplerArgs& a, uint32_t lane) {
  const uint32_t size = (uint32_t)(a.size_dev ? *a.size_dev : a.rv.size);
  const uint64_t step = a.step_dev ? *a.step_dev : a.step;
  if (size == 0) return -1;
  const uint32_t thresh = (uint32_t)((0x100000000ull - size) % size);
  for (int att = 0; att < kMaxDrawAttempts; ++att) {
    u32x4 r = philox4x32_10(u32x4{lane, (uint32_t)att, (uint32_t)step, (uint32_t)(step >> 32)},
                            (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
    uint64_t m = (uint64_t)r.x * size;
    if ((uint32_t)m < thresh) continue;
    uint32_t idx = (uint32_t)(m >> 32);
    if (a.rv.valid[idx]) return (int)idx;
  }
  return -1;
}

__device__ inline void crop_offset_for(const uint32_t* key, const int32_t* expl, int crop_total, int g,
                                       int span, int* cy, int* cx) {
  if (expl) { *cy = expl[2 * g]; *cx = expl[2 * g + 1]; return; }
  u32x2 k = jax_split_at(u32x2{key[0], key[1]}, (uint32_t)crop_total, (uint32_t)g);
  jax_randint2(k, (uint32_t)span, cy, cx);
}

__device__ inline void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ inline void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ inline void mbar_wait(uint64_t* bar, uint32_t phase) {
  uint32_t addr = (uint32_t)__cvta_generic_to_shared(bar), done = 0;
  while (!done) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(addr), "r"(phase) : "memory");
  }
}
__device__ inline void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(bytes),
                 "r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}

// grid: x = band, y = (cam, which, t) flattened, z = row i.   kFast: row_bytes % 16 == 0.
template <bool kFast>
__global__ void __launch_bounds__(kSamplerThreads) sample_gather_crop_kernel(const SamplerArgs a) {
  pdl_prologue();
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ int s_idx, s_cy, s_cx;

  const serl_replay_view& rv = a.rv;
  const int T = rv.num_stack, H = rv.height, W = rv.width, C = rv.channels;
  const int row_bytes = W * C;
  const int band = blockIdx.x;
  int yz = blockIdx.y;
  const int t = yz % T; yz /= T;
  const int which = a.one_side ? a.one_side - 1 : (yz & 1);
  if (!a.one_side) yz >>= 1;
  const int cam = yz;
  const int i = blockIdx.z;
  const int out_row = a.out_row_offset + i;
  const int g = out_row * T + t;                         // frame index inside the batch
  const int y0 = band * kBandRows;
  const int rows = min(kBandRows, H - y0);
  const bool leader = (cam == 0 && (which == 0 || a.one_side) && t == 0 && band == 0);

  if (threadIdx.x == 0) {
    int idx = a.explicit_idx ? a.explicit_idx[i] : draw_index(a, a.lane_offset + (uint32_t)i);
    int cy = a.padding, cx = a.padding;
    if (rv.num_cams > 0)
      crop_offset_for(which ? a.key_next : a.key_obs, which ? a.explicit_off_next : a.explicit_off_obs,
                      a.crop_total, g, 2 * a.padding + 1, &cy, &cx);
    s_idx = idx; s_cy = cy; s_cx = cx;
    if (idx < 0) atomicOr(a.status, 1);
    if (cam == 0 && band == 0 && rv.num_cams > 0) {       // record offsets once per (which, t)
      int32_t* o = which ? a.off_next_out : a.off_obs_out;
      if (o) { o[2 * g] = cy; o[2 * g + 1] = cx; }
    }
    if (kFast) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  }
  __syncthreads();
  const int idx = s_idx, cy = s_cy, cx = s_cx;
  if (idx < 0) return;

  // ---- small fields: one CTA per row ---------------------------------------------------------
  if (leader) {
    const int ns = T * rv.state_dim;
    for (int k = threadIdx.x; k < ns; k += blockDim.x) {
      a.obs_state[(size_t)out_row * ns + k] = rv.state[(size_t)idx * ns + k];
      a.next_state[(size_t)out_row * ns + k] = rv.next_state[(size_t)idx * ns + k];
    }
    for (int k = threadIdx.x; k < rv.action_dim; k += blockDim.x)
      a.actions[(size_t)out_row * rv.action_dim + k] = rv.actions[(size_t)idx * rv.action_dim + k];
    if (threadIdx.x == 0) {
      a.rewards[out_row] = rv.rewards[idx];
      a.masks[out_row] = rv.masks[idx];
      a.dones[out_row] = rv.dones[idx];
      if (a.idx_out) a.idx_out[out_row] = idx;
    }
  }

  if (rv.num_cams == 0) return;                          // state-only ring (data/replay_buffer.py:40-75)

  // ---- frame band: slot idx - T + t + which, rows clamp(y + cy - pad) ---------------------------
  const size_t frame_bytes = (size_t)H * row_bytes;
  // window idx - T of numpy's sliding_window_view over the (capacity) slot axis; the reference indexes it with idx - T as is, so a
  // valid slot idx < T (first transition of an episode whose filler frame sits at the END of the ring) gets numpy's negative-index
  // window = the LAST one, slots capacity-T-1 .. capacity-1 (memory_efficient_replay_buffer.py:148-151; pinned by tests/golden/replay_wrap_first.npz)
  const int w0 = idx - T + ((idx - T) < 0 ? rv.capacity - T : 0);
  const int slot = w0 + t + which;
  const uint8_t* src = rv.frames[cam] + (size_t)slot * frame_bytes;
  uint8_t* dst = (which ? a.next_pix[cam] : a.obs_pix[cam]) + ((size_t)g * H + y0) * row_bytes;
  const int dy = cy - a.padding;
  const int sh = (cx - a.padding) * C;                   // byte shift inside a row
  const int r_lo = min(max(y0 + dy, 0), H - 1);
  const int r_hi = min(max(y0 + rows - 1 + dy, 0), H - 1);

  if (kFast) {
    const uint32_t nbytes = (uint32_t)(r_hi - r_lo + 1) * row_bytes;
    if (threadIdx.x == 0) {
      mbar_expect_tx(&bar, nbytes);
      bulk_g2s(smem, src + (size_t)r_lo * row_bytes, nbytes, &bar);
    }
    mbar_wait(&bar, 0);
    const int cpr = row_bytes >> 4;                      // 16-byte chunks per row
    const uint32_t* s32 = reinterpret_cast<const uint32_t*>(smem);
    for (int q = threadIdx.x; q < rows * cpr; q += blockDim.x) {
      const int yl = q / cpr, j = q - yl * cpr;
      const int r = min(max(y0 + yl + dy, 0), H - 1) - r_lo;
      const int b0 = j * 16;
      const int a0 = b0 + sh;                            // first source byte if no clamping
      uint4 v;
      if (a0 >= 0 && a0 + 16 <= row_bytes) {
        const int base = r * row_bytes + a0;
        const int wi = base >> 2, bs = (base & 3) * 8;
        uint32_t w0 = s32[wi], w1 = s32[wi + 1], w2 = s32[wi + 2], w3 = s32[wi + 3], w4 = s32[wi + 4];
        v.x = __funnelshift_r(w0, w1, bs); v.y = __funnelshift_r(w1, w2, bs);
        v.z = __funnelshift_r(w2, w3, bs); v.w = __funnelshift_r(w3, w4, bs);
      } else {
        uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
        for (int b = 0; b < 16; ++b) {
          const int ob = b0 + b;
          const int x = ob / C, ch = ob - x * C;
          const int xs = min(max(x + cx - a.padding, 0), W - 1);
          o[b >> 2] |= (uint32_t)smem[r * row_bytes + xs * C + ch] << ((b & 3) * 8);
        }
        v = make_uint4(o[0], o[1], o[2], o[3]);
      }
      asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (size_t)yl * row_bytes + b0),
                   "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    }
  } else {
    for (int q = threadIdx.x; q < rows * row_bytes; q += blockDim.x) {
      const int yl = q / row_bytes, ob = q - yl * row_bytes;
      const int r = min(max(y0 + yl + dy, 0), H - 1);
      const int x = ob / C, ch = ob - x * C;
      const int xs = min(max(x + cx - a.padding, 0), W - 1);
      dst[(size_t)yl * row_bytes + ob] = src[(size_t)r * row_bytes + xs * C + ch];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Fast path (row_bytes % 16 == 0): ONE CTA per (row, camera, obs|next) streams its whole frame(s).
// The serial preamble runs once per frame instead of once per band and is spread over two warps (warp 0: Philox index
// draw; warp 1: the threefry crop-key chain, two lanes wide, three evaluations deep); the 32-row bands of a frame are then
// all fetched at once (one TMA bulk copy + mbarrier per band, 48 KiB of shared memory per CTA) and shifted / written back
// in arrival order, so a CTA pays one memory round trip per frame instead of one per band.
// ---------------------------------------------------------------------------------------------
constexpr int kFrameThreads = 256;
constexpr int kMaxBands = 8;             // frames up to 256 rows

// crop offsets for frame g, computed cooperatively by lanes 0/1 of a full warp (all 32 lanes must call)
__device__ inline void crop_offset_warp(const uint32_t* key, const int32_t* expl, int crop_total, int g, int span, int lane,
                                        int* cy, int* cx) {
  if (expl) { *cy = expl[2 * g]; *cx = expl[2 * g + 1]; return; }
  const uint32_t n = (uint32_t)crop_total;
  // level 1: key_g = split(key, n)[g] = (flat[2g], flat[2g+1])
  const uint32_t pos = 2u * (uint32_t)g + (uint32_t)(lane & 1);
  const uint32_t j = pos < n ? pos : pos - n;
  const u32x2 y1 = threefry2x32(u32x2{key[0], key[1]}, j, n + j);
  const uint32_t f = pos < n ? y1.x : y1.y;
  const u32x2 k{__shfl_sync(0xffffffffu, f, 0), __shfl_sync(0xffffffffu, f, 1)};
  // level 2: k1, k2 = split(key_g, 2): flat = [a0, a1, b0, b1] with (a_j, b_j) = TF(key_g, j, 2 + j)
  const u32x2 y2 = threefry2x32(k, (uint32_t)(lane & 1), 2u + (uint32_t)(lane & 1));
  const uint32_t a0 = __shfl_sync(0xffffffffu, y2.x, 0), a1 = __shfl_sync(0xffffffffu, y2.x, 1);
  const uint32_t b0 = __shfl_sync(0xffffffffu, y2.y, 0), b1 = __shfl_sync(0xffffffffu, y2.y, 1);
  // level 3: higher bits = random_bits(k1, (2,)), lower bits = random_bits(k2, (2,))
  const u32x2 y3 = threefry2x32((lane & 1) ? u32x2{b0, b1} : u32x2{a0, a1}, 0u, 1u);
  const uint32_t hb0 = __shfl_sync(0xffffffffu, y3.x, 0), hb1 = __shfl_sync(0xffffffffu, y3.y, 0);
  const uint32_t lb0 = __shfl_sync(0xffffffffu, y3.x, 1), lb1 = __shfl_sync(0xffffffffu, y3.y, 1);
  const uint32_t sp = (uint32_t)span;
  uint32_t mult = 65536u % sp; mult = (mult * mult) % sp;
  *cy = (int)(((hb0 % sp) * mult + (lb0 % sp)) % sp);
  *cx = (int)(((hb1 % sp) * mult + (lb1 % sp)) % sp);
}

// grid: x = cam*2 + which (one-sided: x = cam), y = row i.
__global__ void __launch_bounds__(kFrameThreads) sample_frames_kernel(const SamplerArgs a) {
  pdl_prologue();
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar[kMaxBands];
  __shared__ int s_idx, s_cy[8], s_cx[8];

  const serl_replay_view& rv = a.rv;
  const int T = rv.num_stack, H = rv.height, W = rv.width, C = rv.channels;
  const int row_bytes = W * C;
  const int which = a.one_side ? a.one_side - 1 : (blockIdx.x & 1), cam = a.one_side ? blockIdx.x : (blockIdx.x >> 1);
  const int i = blockIdx.y;
  const int out_row = a.out_row_offset + i;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool leader = (cam == 0 && (which == 0 || a.one_side));
  const int band_bytes = kBandRows * row_bytes + 32;

  if (threadIdx.x == 0) {
    const int idx = a.explicit_idx ? a.explicit_idx[i] : draw_index(a, a.lane_offset + (uint32_t)i);
    s_idx = idx;
    if (idx < 0) atomicOr(a.status, 1);
    for (int b = 0; b < kMaxBands; ++b) mbar_init(&bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    for (int t = 0; t < T; ++t) {
      const int g = out_row * T + t;
      int cy, cx;
      crop_offset_warp(which ? a.key_next : a.key_obs, which ? a.explicit_off_next : a.explicit_off_obs, a.crop_total, g,
                       2 * a.padding + 1, lane, &cy, &cx);
      if (lane == 0) {
        s_cy[t] = cy; s_cx[t] = cx;
        if (cam == 0) { int32_t* o = which ? a.off_next_out : a.off_obs_out; if (o) { o[2 * g] = cy; o[2 * g + 1] = cx; } }
      }
    }
  }
  __syncthreads();
  const int idx = s_idx;
  if (idx < 0) return;

  if (leader) {                                            // small fields: one CTA per row
    const int ns = T * rv.state_dim;
    for (int k = threadIdx.x; k < ns; k += blockDim.x) {
      a.obs_state[(size_t)out_row * ns + k] = rv.state[(size_t)idx * ns + k];
      a.next_state[(size_t)out_row * ns + k] = rv.next_state[(size_t)idx * ns + k];
    }
    for (int k = threadIdx.x; k < rv.action_dim; k += blockDim.x)
      a.actions[(size_t)out_row * rv.action_dim + k] = rv.actions[(size_t)idx * rv.action_dim + k];
    if (threadIdx.x == 0) {
      a.rewards[out_row] = rv.rewards[idx]; a.masks[out_row] = rv.masks[idx]; a.dones[out_row] = rv.dones[idx];
      if (a.idx_out) a.idx_out[out_row] = idx;
    }
  }

  const size_t frame_bytes = (size_t)H * row_bytes;
  const int nb = ceil_div(H, kBandRows);                   // <= kMaxBands, all in flight at once
  const int cpr = row_bytes >> 4;
  for (int t = 0; t < T; ++t) {
    const int cy = s_cy[t], cx = s_cx[t];
    const int dy = cy - a.padding, sh = (cx - a.padding) * C;
    if (threadIdx.x == 0) {                                // one TMA bulk copy per band, each with its own mbarrier
      const int w0 = idx - T + ((idx - T) < 0 ? rv.capacity - T : 0);                 // negative window index: numpy semantics (see sample_gather_crop_kernel)
      const uint8_t* fsrc = rv.frames[cam] + (size_t)(w0 + t + which) * frame_bytes;
      for (int band = 0; band < nb; ++band) {
        const int y0 = band * kBandRows, rows = min(kBandRows, H - y0);
        const int r_lo = min(max(y0 + dy, 0), H - 1), r_hi = min(max(y0 + rows - 1 + dy, 0), H - 1);
        const uint32_t nbytes = (uint32_t)(r_hi - r_lo + 1) * row_bytes;
        mbar_expect_tx(&bar[band], nbytes);
        bulk_g2s(smem + band * band_bytes, fsrc + (size_t)r_lo * row_bytes, nbytes, &bar[band]);
      }
    }
    const int g = out_row * T + t;
    for (int band = 0; band < nb; ++band) {
      mbar_wait(&bar[band], (uint32_t)t & 1u);
      const int y0 = band * kBandRows, rows = min(kBandRows, H - y0);
      const int r_lo = min(max(y0 + dy, 0), H - 1);
      const uint8_t* sb = smem + band * band_bytes;
      uint8_t* dst = (which ? a.next_pix[cam] : a.obs_pix[cam]) + ((size_t)g * H + y0) * row_bytes;
      // interior chunks: a row-shifted copy with ONE aligned 128-bit shared load per lane.  A warp takes whole rows; lane l
      // loads the aligned 16-byte chunk (l + kq) of the source row (conflict-free: consecutive lanes, consecutive chunks),
      // gets the next chunk from lane l+1 by shuffle, and funnels the two by the byte shift (uniform per frame).  Round 1
      // read five 32-bit words per lane at a 16-byte lane stride: 4-way bank conflicts on 85 % of the shared wavefronts
      // (profiles/r01_ncu_sampler_stem_full.md).  The <= 1 chunk per row that touches the clamped edge is handled by the
      // compact bytewise loop below.
      {
        const int kqg = (sh >= 0) ? (sh >> 4) : -((-sh + 15) >> 4);   // floor(sh / 16)
        const int bsh = sh - 16 * kqg;                         // 0..15
        const int wsft = bsh >> 2, bits = (bsh & 3) * 8;
        const uint4* s128 = reinterpret_cast<const uint4*>(sb);
        const int cpr4 = row_bytes >> 4;
        for (int yl = warp; yl < rows; yl += (kFrameThreads >> 5)) {
          const int r = min(max(y0 + yl + dy, 0), H - 1) - r_lo;
          for (int j0 = 0; j0 < cpr; j0 += 31) {              // 31 output chunks per pass (lane 31 only supplies its neighbour)
            const int jj = j0 + lane, c = jj + kqg;
            uint4 A = make_uint4(0u, 0u, 0u, 0u);
            if (c >= 0 && c < cpr4) A = s128[r * cpr4 + c];
            uint4 Bn;
            Bn.x = __shfl_down_sync(0xffffffffu, A.x, 1); Bn.y = __shfl_down_sync(0xffffffffu, A.y, 1);
            Bn.z = __shfl_down_sync(0xffffffffu, A.z, 1); Bn.w = __shfl_down_sync(0xffffffffu, A.w, 1);
            const int a0 = jj * 16 + sh;
            if (lane < 31 && jj < cpr && a0 >= 0 && a0 + 16 <= row_bytes) {
              uint32_t w0, w1, w2, w3, w4;                     // the five words starting at word offset wsft of (A, Bn)
              switch (wsft) {
                case 0: w0 = A.x; w1 = A.y; w2 = A.z; w3 = A.w; w4 = Bn.x; break;
                case 1: w0 = A.y; w1 = A.z; w2 = A.w; w3 = Bn.x; w4 = Bn.y; break;
                case 2: w0 = A.z; w1 = A.w; w2 = Bn.x; w3 = Bn.y; w4 = Bn.z; break;
                default: w0 = A.w; w1 = Bn.x; w2 = Bn.y; w3 = Bn.z; w4 = Bn.w; break;
              }
              asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (size_t)yl * row_bytes + jj * 16),
                           "r"(__funnelshift_r(w0, w1, bits)), "r"(__funnelshift_r(w1, w2, bits)), "r"(__funnelshift_r(w2, w3, bits)),
                           "r"(__funnelshift_r(w3, w4, bits)) : "memory");
            }
          }
        }
      }
      const int ne_l = sh < 0 ? min(cpr, (-sh + 15) >> 4) : 0, ne_r = sh > 0 ? min(cpr - ne_l, (sh + 15) >> 4) : 0;
      const int ne = ne_l + ne_r;
      for (int e = threadIdx.x; e < rows * ne; e += blockDim.x) {
        const int yl = e / ne, k = e - yl * ne;
        const int jj = k < ne_l ? k : cpr - ne_r + (k - ne_l);
        const int r = min(max(y0 + yl + dy, 0), H - 1) - r_lo;
        const int b0 = jj * 16;
        uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
        for (int b = 0; b < 16; ++b) {
          const int ob = b0 + b;
          const int x = (C == 3 && ob < 65536) ? (int)(((uint32_t)ob * 43691u) >> 17) : ob / C;
          const int ch = ob - x * C;
          const int xs = min(max(x + cx - a.padding, 0), W - 1);
          o[b >> 2] |= (uint32_t)sb[r * row_bytes + xs * C + ch] << ((b & 3) * 8);
        }
        asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (size_t)yl * row_bytes + b0),
                     "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
      }
    }
    __syncthreads();                                       // every band buffer is free again for the next stacked frame
  }
}

// ---------------------------------------------------------------------------------------------
// Persistent variant of the fast path (round 2, frame stack T == 1): CTAs walk the (row, camera, obs|next) frames of the
// launch with a two-deep shared-memory pipeline.  Round 1's one-CTA-per-frame kernel ran as a single wave whose CTAs all
// did preamble -> load -> shift -> store in lock step: 0.35 of the HBM roofline with 7.9 warps per issue stalled on the TMA
// barrier.  Here
//   * the whole preamble of a CTA (Philox draw + validity lookups, threefry crop-key chains) runs ONCE, for all of its
//     frames in parallel (thread per frame for the draw, warp per frame for the crop offsets);
//   * the four band copies of frame k+1 are issued before frame k is shifted and written back, so every CTA always has a
//     48 KiB frame in flight (2 CTAs per SM: ~96 KiB of loads outstanding per SM - what 6.5 TB/s x ~2 us needs).
// Same arithmetic, same outputs as sample_frames_kernel (bit-exact tests cover both through SERL_SAMPLER_PERSISTENT).
// ---------------------------------------------------------------------------------------------
constexpr int kPersistMaxItems = 16;     // frames per CTA (grid is sized so that this is never exceeded)

__device__ inline void shift_store_band(const uint8_t* sb, uint8_t* dst, int rows, int y0, int r_lo, int dy, int sh, int cx, int padding,
                                        int H, int W, int C, int row_bytes, int warp, int lane) {
  const int cpr = row_bytes >> 4;
  const int kqg = (sh >= 0) ? (sh >> 4) : -((-sh + 15) >> 4);   // floor(sh / 16)
  const int bsh = sh - 16 * kqg;
  const int wsft = bsh >> 2, bits = (bsh & 3) * 8;
  const uint4* s128 = reinterpret_cast<const uint4*>(sb);
  for (int yl = warp; yl < rows; yl += (kFrameThreads >> 5)) {
    const int r = min(max(y0 + yl + dy, 0), H - 1) - r_lo;
    for (int j0 = 0; j0 < cpr; j0 += 31) {
      const int jj = j0 + lane, c = jj + kqg;
      uint4 A = make_uint4(0u, 0u, 0u, 0u);
      if (c >= 0 && c < cpr) A = s128[r * cpr + c];
      uint4 Bn;
      Bn.x = __shfl_down_sync(0xffffffffu, A.x, 1); Bn.y = __shfl_down_sync(0xffffffffu, A.y, 1);
      Bn.z = __shfl_down_sync(0xffffffffu, A.z, 1); Bn.w = __shfl_down_sync(0xffffffffu, A.w, 1);
      const int a0 = jj * 16 + sh;
      if (lane < 31 && jj < cpr && a0 >= 0 && a0 + 16 <= row_bytes) {
        uint32_t w0, w1, w2, w3, w4;
        switch (wsft) {
          case 0: w0 = A.x; w1 = A.y; w2 = A.z; w3 = A.w; w4 = Bn.x; break;
          case 1: w0 = A.y; w1 = A.z; w2 = A.w; w3 = Bn.x; w4 = Bn.y; break;
          case 2: w0 = A.z; w1 = A.w; w2 = Bn.x; w3 = Bn.y; w4 = Bn.z; break;
          default: w0 = A.w; w1 = Bn.x; w2 = Bn.y; w3 = Bn.z; w4 = Bn.w; break;
        }
        asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (size_t)yl * row_bytes + jj * 16),
                     "r"(__funnelshift_r(w0, w1, bits)), "r"(__funnelshift_r(w1, w2, bits)), "r"(__funnelshift_r(w2, w3, bits)),
                     "r"(__funnelshift_r(w3, w4, bits)) : "memory");
      }
    }
  }
  // the <= 1 chunk per row that touches the clamped left / right edge: bytewise
  const int ne_l = sh < 0 ? min(cpr, (-sh + 15) >> 4) : 0, ne_r = sh > 0 ? min(cpr - ne_l, (sh + 15) >> 4) : 0;
  const int ne = ne_l + ne_r;
  for (int e = threadIdx.x; e < rows * ne; e += blockDim.x) {
    const int yl = e / ne, k = e - yl * ne;
    const int jj = k < ne_l ? k : cpr - ne_r + (k - ne_l);
    const int r = min(max(y0 + yl + dy, 0), H - 1) - r_lo;
    const int b0 = jj * 16;
    uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
    for (int b = 0; b < 16; ++b) {
      const int ob = b0 + b;
      const int x = (C == 3 && ob < 65536) ? (int)(((uint32_t)ob * 43691u) >> 17) : ob / C;
      const int ch = ob - x * C;
      const int xs = min(max(x + cx - padding, 0), W - 1);
      o[b >> 2] |= (uint32_t)sb[r * row_bytes + xs * C + ch] << ((b & 3) * 8);
    }
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + (size_t)yl * row_bytes + b0),
                 "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
  }
}

// grid: persistent, item q = blockIdx.x + k * gridDim.x over (row i, cam*2 + which), q = i * (2*ncam) + cw.   T == 1.
__global__ void __launch_bounds__(kFrameThreads, 2) sample_frames_persistent_kernel(const SamplerArgs a, int n_items) {
  pdl_prologue();
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar[2][kMaxBands];
  __shared__ int s_idx[kPersistMaxItems], s_cy[kPersistMaxItems], s_cx[kPersistMaxItems];

  const serl_replay_view& rv = a.rv;
  const int H = rv.height, W = rv.width, C = rv.channels;
  const int row_bytes = W * C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int band_bytes = kBandRows * row_bytes + 32;
  const int nb = ceil_div(H, kBandRows);
  const int frame_smem = nb * band_bytes;
  const int per_row = 2 * rv.num_cams;
  const int mine = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;      // items of this CTA (>= 1)
  const size_t frame_bytes = (size_t)H * row_bytes;

  // ---- preamble, once: all of this CTA's draws and crop offsets in parallel ----
  if (threadIdx.x == 0) {
    for (int b = 0; b < 2 * kMaxBands; ++b) mbar_init(&bar[0][0] + b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if ((int)threadIdx.x < mine) {
    const int q = blockIdx.x + threadIdx.x * gridDim.x, i = q / per_row;
    const int idx = a.explicit_idx ? a.explicit_idx[i] : draw_index(a, a.lane_offset + (uint32_t)i);
    s_idx[threadIdx.x] = idx;
    if (idx < 0) atomicOr(a.status, 1);
  }
  for (int k = warp; k < mine; k += (kFrameThreads >> 5)) {
    const int q = blockIdx.x + k * gridDim.x, i = q / per_row, cw = q % per_row, which = cw & 1, cam = cw >> 1;
    const int g = a.out_row_offset + i;                    // frame index inside the batch (T == 1)
    int cy, cx;
    crop_offset_warp(which ? a.key_next : a.key_obs, which ? a.explicit_off_next : a.explicit_off_obs, a.crop_total, g,
                     2 * a.padding + 1, lane, &cy, &cx);
    if (lane == 0) {
      s_cy[k] = cy; s_cx[k] = cx;
      if (cam == 0) { int32_t* o = which ? a.off_next_out : a.off_obs_out; if (o) { o[2 * g] = cy; o[2 * g + 1] = cx; } }
    }
  }
  __syncthreads();

  auto issue = [&](int k) {                                 // one TMA bulk copy per band of item k into buffer k & 1
    const int q = blockIdx.x + k * gridDim.x, i = q / per_row, cw = q % per_row, which = cw & 1, cam = cw >> 1;
    const int idx = s_idx[k];
    if (idx < 0) {                                            // failed draw (status flagged): keep the barrier phases in step
      for (int band = 0; band < nb; ++band) mbar_expect_tx(&bar[k & 1][band], 0u);
      return;
    }
    const int dy = s_cy[k] - a.padding;
    const uint8_t* fsrc = rv.frames[cam] + (size_t)((idx > 0 ? idx - 1 : rv.capacity - 2) + which) * frame_bytes;   // idx == 0: numpy's window -1
    (void)i;
    for (int band = 0; band < nb; ++band) {
      const int y0 = band * kBandRows, rows = min(kBandRows, H - y0);
      const int r_lo = min(max(y0 + dy, 0), H - 1), r_hi = min(max(y0 + rows - 1 + dy, 0), H - 1);
      const uint32_t nbytes = (uint32_t)(r_hi - r_lo + 1) * row_bytes;
      mbar_expect_tx(&bar[k & 1][band], nbytes);
      bulk_g2s(smem + (k & 1) * frame_smem + band * band_bytes, fsrc + (size_t)r_lo * row_bytes, nbytes, &bar[k & 1][band]);
    }
  };
  if (threadIdx.x == 0) issue(0);
  for (int k = 0; k < mine; ++k) {
    if (threadIdx.x == 0 && k + 1 < mine) issue(k + 1);     // buffer (k+1)&1 was drained by item k-1 (barrier at the end of that iteration)
    const int q = blockIdx.x + k * gridDim.x, i = q / per_row, cw = q % per_row, which = cw & 1, cam = cw >> 1;
    const int out_row = a.out_row_offset + i;
    const int idx = s_idx[k];
    if (idx >= 0) {
      if (cw == 0) {                                        // small fields: once per row
        const int ns = rv.state_dim;
        for (int e = threadIdx.x; e < ns; e += blockDim.x) {
          a.obs_state[(size_t)out_row * ns + e] = rv.state[(size_t)idx * ns + e];
          a.next_state[(size_t)out_row * ns + e] = rv.next_state[(size_t)idx * ns + e];
        }
        for (int e = threadIdx.x; e < rv.action_dim; e += blockDim.x)
          a.actions[(size_t)out_row * rv.action_dim + e] = rv.actions[(size_t)idx * rv.action_dim + e];
        if (threadIdx.x == 0) {
          a.rewards[out_row] = rv.rewards[idx]; a.masks[out_row] = rv.masks[idx]; a.dones[out_row] = rv.dones[idx];
          if (a.idx_out) a.idx_out[out_row] = idx;
        }
      }
      const int cy = s_cy[k], cx = s_cx[k];
      const int dy = cy - a.padding, sh = (cx - a.padding) * C;
      const uint32_t ph = (uint32_t)(k >> 1) & 1u;          // buffer k & 1 is on its (k >> 1)-th use
      for (int band = 0; band < nb; ++band) {
        mbar_wait(&bar[k & 1][band], ph);
        const int y0 = band * kBandRows, rows = min(kBandRows, H - y0);
        const int r_lo = min(max(y0 + dy, 0), H - 1);
        uint8_t* dst = (which ? a.next_pix[cam] : a.obs_pix[cam]) + ((size_t)out_row * H + y0) * row_bytes;
        shift_store_band(smem + (k & 1) * frame_smem + band * band_bytes, dst, rows, y0, r_lo, dy, sh, cx, a.padding, H, W, C, row_bytes, warp, lane);
      }
    }
    __syncthreads();                                        // buffer k & 1 is free for item k + 2
  }
}

// ---------------------------------------------------------------------------------------------
// Replay ring writes (insert path).  The ring bookkeeping (cursor, episode-start fillers, validity)
// is host logic mirroring data/memory_efficient_replay_buffer.py:53-89; these kernels apply a batch
// of slot writes staged in device memory.
// ---------------------------------------------------------------------------------------------
struct ScatterArgs {
  serl_replay_view rv;           // frames etc. are written (const_cast on the device side)
  int n;                         // slot writes
  const int32_t* dst_slot;       // (n)
  const int32_t* src_slot;       // (n) >= 0: copy from ring slot; < 0: from staging row k
  const uint8_t* st_frames[SERL_MAX_CAMS];   // (n, frame_bytes)
  const float* st_state; const float* st_next_state; const float* st_actions;
  const float* st_rewards; const float* st_masks; const uint8_t* st_dones; const uint8_t* st_valid;
  long long row_stride;          // 0: every staging field is a packed (n, ...) array; else: byte distance between rows k, k+1
};

// staging row k of a field: packed arrays, or fields interleaved in one record per row (one H2D copy per flush)
template <class T>
__device__ inline const T* st_row(const T* base, int k, size_t packed_elems, long long stride) {
  return stride ? reinterpret_cast<const T*>(reinterpret_cast<const uint8_t*>(base) + (size_t)k * (size_t)stride) : base + (size_t)k * packed_elems;
}

// grid: x = chunk of the frame, y = cam, z = write k.  Ordered writes: launch once per dependency level.
__global__ void __launch_bounds__(256) replay_scatter_kernel(const ScatterArgs a) {
  pdl_prologue();
  const serl_replay_view& rv = a.rv;
  const int k = blockIdx.z, cam = blockIdx.y;
  const int dst = *st_row(a.dst_slot, k, 1, a.row_stride), ss = *st_row(a.src_slot, k, 1, a.row_stride);
  const size_t fb = (size_t)rv.height * rv.width * rv.channels;
  if (cam < rv.num_cams) {
    const uint8_t* s = ss >= 0 ? rv.frames[cam] + (size_t)ss * fb : st_row(a.st_frames[cam], k, fb, a.row_stride);
    uint8_t* d = const_cast<uint8_t*>(rv.frames[cam]) + (size_t)dst * fb;
    if ((fb & 15) == 0 && ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
      const uint4* s4 = reinterpret_cast<const uint4*>(s);
      uint4* d4 = reinterpret_cast<uint4*>(d);
      for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < (fb >> 4); q += (size_t)gridDim.x * blockDim.x)
        d4[q] = s4[q];
    } else {
      for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < fb; q += (size_t)gridDim.x * blockDim.x)
        d[q] = s[q];
    }
  }
  if (cam == 0 && blockIdx.x == 0) {
    const int ns = rv.num_stack * rv.state_dim;
    float* st = const_cast<float*>(rv.state); float* nst = const_cast<float*>(rv.next_state);
    float* ac = const_cast<float*>(rv.actions);
    const float* s_st = st_row(a.st_state, k, ns, a.row_stride); const float* s_nst = st_row(a.st_next_state, k, ns, a.row_stride);
    const float* s_ac = st_row(a.st_actions, k, rv.action_dim, a.row_stride);
    for (int e = threadIdx.x; e < ns; e += blockDim.x) {
      st[(size_t)dst * ns + e] = ss >= 0 ? rv.state[(size_t)ss * ns + e] : s_st[e];
      nst[(size_t)dst * ns + e] = ss >= 0 ? rv.next_state[(size_t)ss * ns + e] : s_nst[e];
    }
    for (int e = threadIdx.x; e < rv.action_dim; e += blockDim.x)
      ac[(size_t)dst * rv.action_dim + e] = ss >= 0 ? rv.actions[(size_t)ss * rv.action_dim + e] : s_ac[e];
    if (threadIdx.x == 0) {
      const_cast<float*>(rv.rewards)[dst] = ss >= 0 ? rv.rewards[ss] : *st_row(a.st_rewards, k, 1, a.row_stride);
      const_cast<float*>(rv.masks)[dst] = ss >= 0 ? rv.masks[ss] : *st_row(a.st_masks, k, 1, a.row_stride);
      const_cast<uint8_t*>(rv.dones)[dst] = ss >= 0 ? rv.dones[ss] : *st_row(a.st_dones, k, 1, a.row_stride);
      const_cast<uint8_t*>(rv.valid)[dst] = *st_row(a.st_valid, k, 1, a.row_stride);
    }
  }
}

__global__ void counter_add_kernel(uint64_t* ctr, uint64_t inc) {
  pdl_prologue(); if (threadIdx.x == 0 && blockIdx.x == 0) *ctr += inc; }

__global__ void replay_set_valid_kernel(uint8_t* valid, const int32_t* slots, const uint8_t* vals, int n, int32_t* size_dev, int32_t size) {
  pdl_prologue();
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) valid[slots[k]] = vals[k];
  if (k == 0 && size_dev) *size_dev = size;
}

}  // namespace serl

using namespace serl;

static int check_view(const serl_replay_view* rv) {
  if (!rv || rv->num_cams < 0 || rv->num_cams > SERL_MAX_CAMS || rv->num_stack < 1 || rv->size < 0 ||
      rv->size > rv->capacity || rv->height < 1 || rv->width < 1 || rv->channels < 1) {
    set_last_error("serl_replay: invalid replay view");
    return SERL_ERR_INVALID;
  }
  return SERL_OK;
}

extern "C" int serl_replay_sample_crop(const serl_replay_view* rv, const serl_sample_request* rq,
                                       const serl_batch_out* out, void* stream) {
  if (int e = check_view(rv)) return e;
  if (!rq || !out || rq->batch < 1 || rq->crop_total < (rq->out_row_offset + rq->batch) * rv->num_stack) {
    set_last_error("serl_replay_sample_crop: invalid request (batch=%d crop_total=%d)", rq ? rq->batch : -1,
                   rq ? rq->crop_total : -1);
    return SERL_ERR_INVALID;
  }
  if (!rq->explicit_idx && rv->size <= rv->num_stack) {
    set_last_error("serl_replay_sample_crop: buffer holds %d slots, need > num_stack", rv->size);
    return SERL_ERR_INVALID;
  }
  // one-sided output: every obs_pix (or every next_pix) pointer NULL -> only the other view is gathered and cropped, one CTA per
  // (row, camera) instead of two (the reward classifier's batch uses the positive rows' next frames and the negative rows' frames)
  int one_side = 0;
  if (rv->num_cams > 0) {
    bool any_obs = false, any_next = false;
    for (int c = 0; c < rv->num_cams; ++c) { any_obs |= out->obs_pix[c] != nullptr; any_next |= out->next_pix[c] != nullptr; }
    if (!any_obs && !any_next) { set_last_error("serl_replay_sample_crop: no frame output"); return SERL_ERR_INVALID; }
    one_side = any_obs && any_next ? 0 : (any_obs ? 1 : 2);
    for (int c = 0; c < rv->num_cams; ++c)
      if ((one_side != 2 && !out->obs_pix[c]) || (one_side != 1 && !out->next_pix[c])) {
        set_last_error("serl_replay_sample_crop: camera %d: frame output missing", c); return SERL_ERR_INVALID;
      }
    const bool obs_ok = rq->key_obs || rq->explicit_off_obs, next_ok = rq->key_next || rq->explicit_off_next;
    const bool two_ok = (rq->key_obs && rq->key_next) || (rq->explicit_off_obs && rq->explicit_off_next);
    if (one_side == 0 ? !two_ok : (one_side == 1 ? !obs_ok : !next_ok)) {
      set_last_error("serl_replay_sample_crop: need crop keys or explicit offsets");
      return SERL_ERR_INVALID;
    }
  }
  SamplerArgs a{};
  a.rv = *rv;
  a.seed = rq->seed; a.step = rq->step; a.step_dev = rq->step_dev; a.size_dev = rq->size_dev; a.lane_offset = rq->lane_offset; a.explicit_idx = rq->explicit_idx;
  a.key_obs = rq->key_obs; a.key_next = rq->key_next;
  a.explicit_off_obs = rq->explicit_off_obs; a.explicit_off_next = rq->explicit_off_next;
  a.crop_total = rq->crop_total; a.out_row_offset = rq->out_row_offset; a.padding = rq->padding;
  for (int c = 0; c < rv->num_cams; ++c) { a.obs_pix[c] = out->obs_pix[c]; a.next_pix[c] = out->next_pix[c]; }
  a.obs_state = out->obs_state; a.next_state = out->next_state; a.actions = out->actions;
  a.rewards = out->rewards; a.masks = out->masks; a.dones = out->dones; a.idx_out = out->idx;
  a.off_obs_out = out->off_obs; a.off_next_out = out->off_next; a.status = out->status; a.batch = rq->batch;
  a.one_side = one_side;
  const int sides = one_side ? 1 : 2;

  const int row_bytes = rv->width * rv->channels;
  const bool fast = rv->num_cams > 0 && (row_bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(rv->frames[0]) & 15) == 0);
  dim3 grid(ceil_div(rv->height, kBandRows), rv->num_cams * sides * rv->num_stack, rq->batch);
  if (rv->num_cams == 0) grid = dim3(1, 1, rq->batch);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (fast && rv->num_stack <= 8 && ceil_div(rv->height, kBandRows) <= kMaxBands &&
      (size_t)ceil_div(rv->height, kBandRows) * ((size_t)kBandRows * row_bytes + 32) <= 96 * 1024) {
    const size_t smem = (size_t)ceil_div(rv->height, kBandRows) * ((size_t)kBandRows * row_bytes + 32);
    static size_t configured = 0;
    if (smem > configured) {
      if (cudaFuncSetAttribute(sample_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch("cudaFuncSetAttribute(sample_frames)");
      configured = smem;
    }
    static int persistent = -1;
    if (persistent < 0) { const char* e = getenv("SERL_SAMPLER_PERSISTENT"); persistent = (e && atoi(e) != 0) ? 1 : 0; }
    if (persistent && !one_side && rv->num_stack == 1 && 2 * smem <= 112 * 1024) {
      static int sms = 0;
      if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
      const int n_items = rq->batch * rv->num_cams * 2;
      int grid = n_items < 2 * sms ? n_items : 2 * sms;
      if (ceil_div(n_items, grid) > kPersistMaxItems) grid = ceil_div(n_items, kPersistMaxItems);
      static size_t pconf = 0;
      if (2 * smem > pconf) {
        if (cudaFuncSetAttribute(sample_frames_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * smem)) != cudaSuccess) return check_launch("cudaFuncSetAttribute(sample_frames_persistent)");
        pconf = 2 * smem;
      }
      launch_k(sample_frames_persistent_kernel, grid, kFrameThreads, 2 * smem, st, a, n_items);
      return check_launch("sample_frames_persistent_kernel");
    }
    dim3 fgrid(rv->num_cams * sides, rq->batch);
    launch_k(sample_frames_kernel, fgrid, kFrameThreads, smem, st, a);
    return check_launch("sample_frames_kernel");
  } else if (fast) {
    size_t smem = (size_t)kBandRows * row_bytes + 32;
    launch_k(sample_gather_crop_kernel<true>, grid, kSamplerThreads, smem, st, a);
  } else {
    launch_k(sample_gather_crop_kernel<false>, grid, kSamplerThreads, 0, st, a);
  }
  return check_launch("sample_gather_crop_kernel");
}

extern "C" int serl_replay_scatter(const serl_replay_view* rv, const serl_scatter_request* rq, void* stream) {
  if (int e = check_view(rv)) return e;
  if (!rq || rq->n < 0) { set_last_error("serl_replay_scatter: invalid request"); return SERL_ERR_INVALID; }
  if (rq->n == 0) return SERL_OK;
  ScatterArgs a{};
  a.rv = *rv; a.n = rq->n; a.dst_slot = rq->dst_slot; a.src_slot = rq->src_slot;
  for (int c = 0; c < rv->num_cams; ++c) a.st_frames[c] = rq->frames[c];
  a.st_state = rq->state; a.st_next_state = rq->next_state; a.st_actions = rq->actions;
  a.st_rewards = rq->rewards; a.st_masks = rq->masks; a.st_dones = rq->dones; a.st_valid = rq->valid;
  a.row_stride = rq->row_stride;
  const size_t fb = (size_t)rv->height * rv->width * rv->channels;
  int chunks = (int)((fb / 16 + 255) / 256); if (chunks < 1) chunks = 1; if (chunks > 16) chunks = 16;
  dim3 grid(chunks, rv->num_cams > 0 ? rv->num_cams : 1, rq->n);
  launch_k(replay_scatter_kernel, grid, 256, 0, static_cast<cudaStream_t>(stream), a);
  return check_launch("replay_scatter_kernel");
}

extern "C" int serl_replay_set_valid(uint8_t* valid, const int32_t* slots, const uint8_t* vals, int n, void* stream) {
  if (n <= 0) return SERL_OK;
  launch_k(replay_set_valid_kernel, ceil_div(n, 128), 128, 0, static_cast<cudaStream_t>(stream), valid, slots, vals, n, nullptr, 0);
  return check_launch("replay_set_valid_kernel");
}

extern "C" int serl_replay_commit(uint8_t* valid, const int32_t* slots, const uint8_t* vals, int n, int32_t* size_dev, int32_t size, void* stream) {
  if (n < 0 || !size_dev) { set_last_error("serl_replay_commit: invalid arguments"); return SERL_ERR_INVALID; }
  launch_k(replay_set_valid_kernel, n > 0 ? ceil_div(n, 128) : 1, 128, 0, static_cast<cudaStream_t>(stream), valid, slots, vals, n, size_dev, size);
  return check_launch("replay_set_valid_kernel");
}

extern "C" int serl_counter_add(uint64_t* counter, uint64_t inc, void* stream) {
  launch_k(counter_add_kernel, 1, 32, 0, static_cast<cudaStream_t>(stream), counter, inc);
  return check_launch("counter_add_kernel");
}

// Host-side mirrors of the integer RNG specs (no GPU needed): used by CPU tests to pin the device
// functions (same __host__ __device__ code) against oracle/jax_prng.py and oracle/replay.py.
extern "C" int serl_host_crop_offsets(const uint32_t key[2], int n_frames, int padding, int32_t* out) {
  for (int g = 0; g < n_frames; ++g) {
    u32x2 k = jax_split_at(u32x2{key[0], key[1]}, (uint32_t)n_frames, (uint32_t)g);
    int cy, cx; jax_randint2(k, (uint32_t)(2 * padding + 1), &cy, &cx);
    out[2 * g] = cy; out[2 * g + 1] = cx;
  }
  return SERL_OK;
}

extern "C" int serl_host_draw_indices(uint64_t seed, uint64_t step, uint32_t lane_offset, int batch, int size,
                                      const uint8_t* valid, int32_t* out) {
  if (size < 1) return SERL_ERR_INVALID;
  const uint32_t thresh = (uint32_t)((0x100000000ull - (uint32_t)size) % (uint32_t)size);
  for (int i = 0; i < batch; ++i) {
    out[i] = -1;
    for (int att = 0; att < kMaxDrawAttempts; ++att) {
      u32x4 r = philox4x32_10(u32x4{lane_offset + (uint32_t)i, (uint32_t)att, (uint32_t)step, (uint32_t)(step >> 32)},
                              (uint32_t)seed, (uint32_t)(seed >> 32));
      uint64_t m = (uint64_t)r.x * (uint32_t)size;
      if ((uint32_t)m < thresh) continue;
      uint32_t idx = (uint32_t)(m >> 32);
      if (valid[idx]) { out[i] = (int)idx; break; }
    }
  }
  return SERL_OK;
}

extern "C" int serl_host_threefry_split(const uint32_t key[2], int n, uint32_t* out) {
  for (int i = 0; i < n; ++i) { u32x2 k = jax_split_at(u32x2{key[0], key[1]}, (uint32_t)n, (uint32_t)i); out[2 * i] = k.x; out[2 * i + 1] = k.y; }
  return SERL_OK;
}

extern "C" int serl_host_random_bits(const uint32_t key[2], int size, uint32_t* out) {
  for (int j = 0; j < size; ++j) out[j] = jax_random_bits_at(u32x2{key[0], key[1]}, (uint32_t)size, (uint32_t)j);
  return SERL_OK;
}
