// tcgen05 kind::tf32 tap-GEMM of TFL_PRECISION_TF32: the TapGemm contract of tap_gemm_kernel (kernels_f32.cuh) on the
// tensor core.  The ConvSwiGLU FFN of the tf32 mode keeps the fp32 mode's dataflow and workspace (norm_launch -> g1 with
// EpiSwiGLU into `hid` -> g2 with EpiResidual, tfl_api.cu: ffn_f32) and runs both GEMMs here:
//
//   * Rows are laid on a stream of period P = max(Sout, Sin + padL, Sout + taps - 1 - padL): output row (s, j) is stream
//     row s * P + j, and stream row s * P + o holds input row (s, o - padL), zero outside [0, Sin).  Output row q then
//     reads stream rows q .. q + taps - 1, so the taps are row-shifted descriptors onto ONE staged A tile of 128 + taps - 1
//     rows (tc_common.cuh), also across sequence boundaries.  For the conv1d (padL = taps - 1) P = Sout; for the
//     transposed conv (padL = 0, Sin = Sout + taps - 1) P = Sin and the taps - 1 stream rows past Sout are not written.
//   * One CTA computes 128 stream rows x Nt (<= 256) output columns.  Per pipeline stage it stages 8 input channels:
//     the A rows through SeqMap (sequence padding stays exact zeros) and the taps x Nt weight columns read from the fp32
//     tap-major pack [tap][Kc][N], both rounded with cvt.rna.tf32.f32 into the canonical no-swizzle K-major layout
//     (core matrix = 8 rows x 4 tf32: byte(r, c) = ((c / 4) * R + r) * 16 + (c % 4) * 4).  No tf32 weight image is
//     packed: the rounding and the transpose happen while staging, so the packed buffer is the same in every mode.
//   * One elected lane of warp 0 issues taps tcgen05.mma.cta_group::1.kind::tf32 (M 128, K 8) per stage into an fp32
//     TMEM accumulator; the stage's empty barrier is the MMAs' commit.  The accumulator is <= 256 columns, and the
//     shared-memory request (sized from the device's shared memory per SM) makes exactly 512 / columns CTAs resident
//     per SM -- two at 256 columns: two accumulators per SM, one CTA's epilogue beside the other's MMAs.
//   * Epilogue: each thread owns one TMEM lane (= one output row) and hands 8 columns at a time, + bias, to the fp32
//     path's functors, so the SwiGLU and the residual add are the fp32 mode's arithmetic on a tf32 product.
#pragma once
#include "common.cuh"
#include "tc_common.cuh"
#include "kernels_f32.cuh"
#include "kernels_tc.cuh"

namespace tfl {

constexpr int TF_KC = 8;             // input channels per stage: one K = 8 kind::tf32 MMA per tap
constexpr int TF_THREADS = 256;
constexpr int TF_STAGES = 3;
constexpr int TF_TAP_COLS = 1024;    // taps * Nt per stage: the weight stage stays <= 32 KB

struct TapGemmTf32Geom {
  int P, nseq, AR, Nt, n_ntiles, tmem_cols;
  long long n_mtiles;
  uint32_t a_bytes, b_tap_bytes, stage_bytes, off_tab, off_bar, smem;
};

// kind::tf32 instruction descriptor: tf32 x tf32 -> fp32, both operands K-major, M x N tile
__host__ __device__ constexpr uint32_t tf32_instr_desc(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}

__device__ __forceinline__ float4 tf32_round4(float4 v) {
  return make_float4(__uint_as_float(to_tf32(v.x)), __uint_as_float(to_tf32(v.y)), __uint_as_float(to_tf32(v.z)),
                     __uint_as_float(to_tf32(v.w)));
}

// Host: the tile geometry of one call, or an error naming the limit the shape exceeds.
inline int tap_gemm_tf32_geometry(const TapGemm& g, TapGemmTf32Geom* o) {
  TFL_CHECK(g.Kc % TF_KC == 0 && g.N >= 1 && g.Sout >= 1 && g.M % g.Sout == 0,
            "tf32 tap-GEMM needs input channels %% 8 == 0 (got Kc %d, N %d)", g.Kc, g.N);
  TFL_CHECK(g.taps >= 1 && 16 * g.taps <= TF_TAP_COLS,
            "tf32 tap-GEMM supports at most %d taps (got %d)", TF_TAP_COLS / 16, g.taps);
  o->nseq = (int)(g.M / g.Sout);
  int P = g.Sout;
  if (g.Sin + g.padL > P) P = g.Sin + g.padL;
  if (g.Sout + g.taps - 1 - g.padL > P) P = g.Sout + g.taps - 1 - g.padL;
  o->P = P;
  o->AR = 128 + g.taps - 1;
  const int n16 = (g.N + 15) / 16 * 16;
  int nmax = TF_TAP_COLS / g.taps / 16 * 16;
  if (nmax > 256) nmax = 256;
  o->n_ntiles = (n16 + nmax - 1) / nmax;
  o->Nt = ((n16 + o->n_ntiles - 1) / o->n_ntiles + 15) / 16 * 16;
  o->tmem_cols = 32;
  while (o->tmem_cols < o->Nt) o->tmem_cols <<= 1;
  // stream rows after the last output row, (nseq - 1) * P + Sout - 1, are never written: no tile for them
  o->n_mtiles = ((long long)(o->nseq - 1) * P + g.Sout + 127) / 128;
  TFL_CHECK(o->n_mtiles * o->n_ntiles < (1LL << 31), "tf32 tap-GEMM grid too large (%lld row tiles)", o->n_mtiles);
  o->a_bytes = ((uint32_t)o->AR * TF_KC * 4 + 127) & ~127u;
  o->b_tap_bytes = (uint32_t)o->Nt * TF_KC * 4;
  o->stage_bytes = (o->a_bytes + g.taps * o->b_tap_bytes + 127) & ~127u;
  o->off_tab = TF_STAGES * o->stage_bytes;
  o->off_bar = o->off_tab + (((uint32_t)o->AR * 8 + 15) & ~15u);
  uint32_t smem = o->off_bar + 8 * (2 * TF_STAGES + 2);
  // at most 512 / tmem_cols CTAs may hold an accumulator on one SM at a time: size the request from the device's
  // shared memory per SM and per-block reservation so that no more are resident (a further CTA would wait in
  // tcgen05.alloc, which has no bounded wait); at 256 columns that is two CTAs, one's epilogue beside the other's MMAs
  int dev = 0, sm_smem = 0, reserved = 0;
  TFL_CUDA(cudaGetDevice(&dev));
  TFL_CUDA(cudaDeviceGetAttribute(&sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  TFL_CUDA(cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev));
  const uint32_t per_sm = (uint32_t)(512 / o->tmem_cols);
  const long long floor_bytes = (long long)sm_smem / (per_sm + 1) + 1 - reserved;
  if ((long long)smem < floor_bytes) smem = (uint32_t)floor_bytes;
  TFL_CHECK(smem <= (uint32_t)TC_SMEM_MAX, "tf32 tap-GEMM stages need %u bytes of shared memory (> %d)", smem, TC_SMEM_MAX);
  o->smem = smem;
  return 0;
}

template <class Epi>
__global__ void __launch_bounds__(TF_THREADS) tap_gemm_tf32_kernel(TapGemm p, Epi epi, TapGemmTf32Geom g) {
  using namespace tc;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long mt = (long long)blockIdx.x / g.n_ntiles;
  const int nt = (int)(blockIdx.x - mt * g.n_ntiles);
  const long long q0 = mt * 128;
  const int n0 = nt * g.Nt;
  long long* row_off = reinterpret_cast<long long*>(smem + g.off_tab);
  const uint32_t bar0 = smem_u32(smem + g.off_bar);
  auto FULL = [&](int i) { return bar0 + 8u * i; };
  auto EMPTY = [&](int i) { return bar0 + 8u * (TF_STAGES + i); };
  const uint32_t DONE = bar0 + 8u * (2 * TF_STAGES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + g.off_bar + 8 * (2 * TF_STAGES + 1));

  // element offset of every A row of the tile (-1: a zero row -- sequence padding or past the last sequence)
  for (int i = tid; i < g.AR; i += TF_THREADS) {
    const long long q = q0 + i;
    const int s = (int)(q / g.P), pos = (int)(q - (long long)s * g.P) - p.padL;
    row_off[i] = (s < g.nseq && pos >= 0 && pos < p.Sin) ? p.amap.base(s) + (long long)pos * p.amap.pos_stride : -1;
  }
  if (tid == 0) {
    for (int i = 0; i < TF_STAGES; ++i) { mbar_init(FULL(i), TF_THREADS); mbar_init(EMPTY(i), 1); }
    mbar_init(DONE, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), g.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int n_steps = p.Kc / TF_KC;
  const int b_items = p.taps * 2 * g.Nt;   // (tap, channel quad, column) -> one 16-byte core-matrix row
  const uint32_t idesc = tf32_instr_desc(128, g.Nt);
  for (int k = 0; k < n_steps; ++k) {
    const int slot = k % TF_STAGES;
    const uint32_t ph = (uint32_t)(k / TF_STAGES) & 1u;
    if (k >= TF_STAGES) mbar_wait(EMPTY(slot), ph ^ 1u);   // the MMAs of stage k - TF_STAGES are done with the slot
    uint8_t* sa = smem + (size_t)slot * g.stage_bytes;
    uint8_t* sb = sa + g.a_bytes;
    const int c0 = k * TF_KC;
    for (int i = tid; i < 2 * g.AR; i += TF_THREADS) {
      const int h = i >= g.AR, row = i - h * g.AR;
      const long long off = row_off[row];
      const float4 v = off >= 0 ? __ldg(reinterpret_cast<const float4*>(p.A + off + c0 + 4 * h)) : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(sa + ((size_t)h * g.AR + row) * 16) = tf32_round4(v);
    }
    // weights: four loads down the channel axis (each coalesced along N across the warp) make one K-major core-matrix row
    for (int i0 = tid; i0 < b_items; i0 += 4 * TF_THREADS) {
      float4 v[4];
      int dst[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * TF_THREADS;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        dst[u] = -1;
        if (i < b_items) {
          const int tq = i / g.Nt, n = i - tq * g.Nt, tap = tq >> 1, h = tq & 1;
          dst[u] = (int)(tap * g.b_tap_bytes) + (h * g.Nt + n) * 16;
          if (n0 + n < p.N) {
            const float* w = p.W + ((size_t)tap * p.Kc + c0 + 4 * h) * p.N + n0 + n;
            v[u] = make_float4(__ldg(w), __ldg(w + p.N), __ldg(w + 2 * p.N), __ldg(w + 3 * p.N));
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (dst[u] >= 0) *reinterpret_cast<float4*>(sb + dst[u]) = tf32_round4(v[u]);
    }
    fence_proxy_async();
    mbar_arrive(FULL(slot));
    if (warp == 0) {
      mbar_wait(FULL(slot), ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(sa), b_addr = smem_u32(sb);
        for (int tap = 0; tap < p.taps; ++tap)
          mma_tf32(tmem, smem_desc(a_addr + tap * 16, g.AR * 16, 128), smem_desc(b_addr + tap * g.b_tap_bytes, g.Nt * 16, 128),
                   idesc, (k | tap) != 0);
        mma_commit(EMPTY(slot));
        if (k == n_steps - 1) mma_commit(DONE);
      }
      __syncwarp();
    }
  }

  mbar_wait(DONE, 0);
  tc_fence_after();
  const int quarter = warp & 3;
  const long long q = q0 + quarter * 32 + lane;
  const int s = (int)(q / g.P), j = (int)(q - (long long)s * g.P);
  const bool valid = s < g.nseq && j < p.Sout;
  const long long r = (long long)s * p.Sout + j;
  for (int cg = warp >> 2; cg < g.Nt / 16; cg += 2) {   // warps w and w + 4 share a lane quarter, alternate 16 columns
    uint32_t acc[16];
    tmem_ld16(tmem + ((uint32_t)(quarter * 32) << 16) + cg * 16, acc);
    tc_wait_ld();
    if (valid) {
#pragma unroll
      for (int e = 0; e < 16; e += 8) {
        const int n = n0 + cg * 16 + e;
        if (n >= p.N) break;
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
          v[u] = __uint_as_float(acc[e + u]) + ((p.bias != nullptr && n + u < p.N) ? __ldg(&p.bias[n + u]) : 0.f);
        epi(s, j, r, n, p.N, v);
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, g.tmem_cols);
}

template <class Epi>
inline int tap_gemm_tf32_launch(const TapGemm& gm, const Epi& epi, cudaStream_t st) {
  TapGemmTf32Geom g;
  if (tap_gemm_tf32_geometry(gm, &g)) return -1;
  TFL_CUDA(opt_in_smem(tap_gemm_tf32_kernel<Epi>, g.smem));
  tap_gemm_tf32_kernel<Epi><<<(unsigned)(g.n_mtiles * g.n_ntiles), TF_THREADS, g.smem, st>>>(gm, epi, g);
  TFL_LAUNCH_CHECK();
  return 0;
}

// ---- self-test mode 3: D[128, N] = sum_tap A[m + tap, :] . B[tap][n, :] through tap_gemm_tf32_kernel ----------------
struct EpiStore {   // D[r][n]
  float* d;
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
    for (int i = 0; i < 8 && n0 + i < N; ++i) d[r * N + n0 + i] = v[i];
  }
};

__global__ void tf32_selftest_transpose_kernel(const float* __restrict__ B, float* __restrict__ W, int N, int Kd, int taps) {
  // B [taps][N][Kd] -> W [taps][Kd][N] (the tap-major layout of the packed FFN weights)
  const int total = taps * N * Kd;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int t = i / (N * Kd), n = (i / Kd) % N, c = i % Kd;
    W[((size_t)t * Kd + c) * N + n] = B[i];
  }
}

inline int tf32_selftest(const float* A, const float* B, float* D, void* scratch, int N, int Kd, int taps, cudaStream_t st) {
  float* W = (float*)scratch;
  tf32_selftest_transpose_kernel<<<64, 256, 0, st>>>(B, W, N, Kd, taps);
  TFL_LAUNCH_CHECK();
  // one sequence of 128 + taps - 1 rows, 128 outputs, no padding: row m reads rows m .. m + taps - 1
  const TapGemm gm{A, make_dense_map(0, Kd), 128 + taps - 1, 128, 0, taps, Kd, W, nullptr, N, 128};
  return tap_gemm_tf32_launch(gm, EpiStore{D}, st);
}

}  // namespace tfl
