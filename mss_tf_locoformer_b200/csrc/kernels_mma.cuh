// tf32 tensor-core variants of the fp32 tap-GEMM (kernels_f32.cuh) and of the weight-gradient GEMM (kernels_bwd.cuh) for
// the TRAINING step: mma.sync m16n8k8, tf32 operands (cvt.rna: 2^-11 per operand), fp32 accumulation -- the arithmetic
// the reference trains in at best (configs/musdb18_rtx5090_xlarge.yaml:136 `tf32: true`, under bf16 autocast).  Same
// parameters, same 128 x 128 x 8 block tiles and the same epilogue functors (through their two-column `pair` form: an
// accumulator fragment holds adjacent column pairs).  The fp32 inference / parity mode never runs these kernels.
//   block = 8 warps as 2 (m) x 4 (n); warp tile 64 x 32 = 4 x 4 fragments, 16 MMAs per 8-deep k step and 24 shared loads (tf32)
//   or 6 ldmatrix.x4 per 16-deep step (bf16 forms further down).
//   shared tiles are k-major with a pitch of 136 floats: fragment loads (k = t or t + 4, m / n = g) hit 32 distinct banks.
#pragma once
#include "kernels_bwd.cuh"

namespace tfl {

constexpr int MMA_PITCH = GBM + 8;
constexpr int MMA_BK = 16;   // k depth per barrier round (two m16n8k8 steps): the 8-deep version ran latency-bound (r02: 89 TFLOP/s)

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ uint32_t pack2_bf16(float lo, float hi) {   // low half = the lower k index
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// one 8-deep step (m16n8k8) of the warp's 64 x 32 tile over an [8][MMA_PITCH] tile pair holding tf32 bit patterns
__device__ __forceinline__ void mma_warp_step(const uint32_t* As, const uint32_t* Bs, float (&acc)[4][4][4], int wm, int wn, int g, int t) {
  uint32_t a[4][4], b[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = wm * 64 + i * 16 + g;
    a[i][0] = As[t * MMA_PITCH + m]; a[i][1] = As[t * MMA_PITCH + m + 8];
    a[i][2] = As[(t + 4) * MMA_PITCH + m]; a[i][3] = As[(t + 4) * MMA_PITCH + m + 8];
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = wn * 32 + j * 8 + g;
    b[j][0] = Bs[t * MMA_PITCH + n]; b[j][1] = Bs[(t + 4) * MMA_PITCH + n];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) mma_tf32(acc[i][j], a[i], b[j]);
}

template <class Epi>
__global__ void __launch_bounds__(256, 2) tap_gemm_mma_kernel(TapGemm p, Epi epi) {
  __shared__ __align__(16) uint32_t As[2][MMA_BK][MMA_PITCH];
  __shared__ __align__(16) uint32_t Bs[2][MMA_BK][MMA_PITCH];
  __shared__ long long row_base[GBM];
  __shared__ int row_j[GBM], row_s[GBM];
  const int tid = threadIdx.x;
  const long long m0 = (long long)blockIdx.x * GBM;
  const int n0 = blockIdx.y * GBN;
  if (tid < GBM) {
    const long long r = m0 + tid;
    if (r < p.M) {
      const int s = (int)(r / p.Sout), j = (int)(r - (long long)s * p.Sout);
      row_s[tid] = s; row_j[tid] = j; row_base[tid] = p.amap.base(s);
    } else { row_s[tid] = -1; row_j[tid] = 0; row_base[tid] = 0; }
  }
  __syncthreads();
  const int a_row = tid >> 1, a_kq = (tid & 1) << 2;       // A: row a_row, k = a_kq .. +3 and a_kq + 8 .. +11
  const int b_row = tid >> 5, b_col = (tid & 31) << 2;    // B: k rows b_row and b_row + 8, columns b_col .. +3
  const int kt_per_tap = p.Kc / MMA_BK, n_kt = p.taps * kt_per_tap;
  const int my_s = row_s[a_row], my_j = row_j[a_row];
  const long long my_base = row_base[a_row];
  auto load_a = [&](int kt, float4 (&a)[2]) {
    const int tap = kt / kt_per_tap, c0 = (kt - tap * kt_per_tap) * MMA_BK;
    const int pos = my_j + tap - p.padL;
    if (my_s < 0 || pos < 0 || pos >= p.Sin) { a[0] = a[1] = make_float4(0.f, 0.f, 0.f, 0.f); return; }
    const float* src = p.A + my_base + (long long)pos * p.amap.pos_stride + c0 + a_kq;
    a[0] = __ldg(reinterpret_cast<const float4*>(src));
    a[1] = __ldg(reinterpret_cast<const float4*>(src + 8));
  };
  auto load_b = [&](int kt, float4 (&b)[2]) {
    const int n = n0 + b_col;
    if (n >= p.N) { b[0] = b[1] = make_float4(0.f, 0.f, 0.f, 0.f); return; }
    const float* src = p.W + ((size_t)kt * MMA_BK + b_row) * p.N + n;
    b[0] = __ldg(reinterpret_cast<const float4*>(src));
    b[1] = __ldg(reinterpret_cast<const float4*>(src + (size_t)8 * p.N));
  };
  auto stash = [&](int buf, const float4 (&a)[2], const float4 (&b)[2]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      As[buf][8 * h + a_kq + 0][a_row] = to_tf32(a[h].x); As[buf][8 * h + a_kq + 1][a_row] = to_tf32(a[h].y);
      As[buf][8 * h + a_kq + 2][a_row] = to_tf32(a[h].z); As[buf][8 * h + a_kq + 3][a_row] = to_tf32(a[h].w);
      *reinterpret_cast<uint4*>(&Bs[buf][8 * h + b_row][b_col]) = make_uint4(to_tf32(b[h].x), to_tf32(b[h].y), to_tf32(b[h].z), to_tf32(b[h].w));
    }
  };
  float acc[4][4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
  float4 na[2], nb[2];
  load_a(0, na); load_b(0, nb);
  stash(0, na, nb);
  __syncthreads();
  for (int kt = 0; kt < n_kt; ++kt) {
    const int cur = kt & 1;
    const bool more = kt + 1 < n_kt;
    if (more) { load_a(kt + 1, na); load_b(kt + 1, nb); }
    mma_warp_step(&As[cur][0][0], &Bs[cur][0][0], acc, wm, wn, g, t);
    mma_warp_step(&As[cur][8][0], &Bs[cur][8][0], acc, wm, wn, g, t);
    if (more) stash(cur ^ 1, na, nb);
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + wn * 32 + j * 8 + 2 * t;
    if (n >= p.N) continue;
    const float b0 = p.bias != nullptr ? __ldg(&p.bias[n]) : 0.f, b1 = p.bias != nullptr ? __ldg(&p.bias[n + 1]) : 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int rl = wm * 64 + i * 16 + g + 8 * h;
        const int s = row_s[rl];
        if (s < 0) continue;
        epi.pair(s, row_j[rl], m0 + rl, n, p.N, acc[i][j][2 * h] + b0, acc[i][j][2 * h + 1] + b1);
      }
    }
  }
}

template <bool DET>
__global__ void __launch_bounds__(256, 2) tap_wgrad_mma_kernel(TapWgrad p) {
  __shared__ __align__(16) uint32_t As[2][MMA_BK][MMA_PITCH];
  __shared__ __align__(16) uint32_t Bs[2][MMA_BK][MMA_PITCH];
  const int tid = threadIdx.x;
  const int tiles_i = (p.Kc + GBM - 1) / GBM, tiles_n = (p.N + GBN - 1) / GBN;
  int bx = blockIdx.x;
  const int tn = bx % tiles_n; bx /= tiles_n;
  const int ti = bx % tiles_i; bx /= tiles_i;
  const int tap = bx;
  const int i0 = ti * GBM, n0 = tn * GBN;
  const long long r_lo = (long long)blockIdx.y * p.rows_per_split;
  const long long r_hi = r_lo + p.rows_per_split < p.R ? r_lo + p.rows_per_split : p.R;
  if (r_lo >= r_hi) return;
  const int l_row = tid >> 5, l_col = (tid & 31) << 2;     // rows l_row and l_row + 8 of the round, columns l_col .. + 3
  // The (sequence, position) of the thread's FIRST row is carried from round to round (the rows advance by MMA_BK): the
  // 64-bit divisions of a per-load r / Sout and the SeqMap bases were most of this kernel's instructions (ncu r02: issue
  // 52 % active against a tensor pipe at 17 %).
  long long row_first = r_lo + l_row;
  int s_first = (int)(row_first / p.Sout), j_first = (int)(row_first - (long long)s_first * p.Sout);
  long long abase = p.amap.base(s_first), bbase = p.bmap.base(s_first);
  auto advance = [&]() {
    row_first += MMA_BK; j_first += MMA_BK;
    if (j_first >= p.Sout) {
      do { j_first -= p.Sout; ++s_first; } while (j_first >= p.Sout);
      abase = p.amap.base(s_first); bbase = p.bmap.base(s_first);
    }
  };
  auto load = [&](float4 (&a)[2], float4 (&b)[2]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      a[h] = make_float4(0.f, 0.f, 0.f, 0.f); b[h] = a[h];
      if (row_first + 8 * h >= r_hi) continue;
      int j = j_first + 8 * h;
      long long ab = abase, bb = bbase;
      if (j >= p.Sout) {                                    // this row belongs to a later sequence (rare)
        int sq = s_first;
        do { j -= p.Sout; ++sq; } while (j >= p.Sout);
        ab = p.amap.base(sq); bb = p.bmap.base(sq);
      }
      const int pos = j + tap - p.padL;
      if (pos >= 0 && pos < p.Sin && i0 + l_col < p.Kc)
        a[h] = __ldg(reinterpret_cast<const float4*>(p.A + ab + (long long)pos * p.amap.pos_stride + i0 + l_col));
      if (n0 + l_col < p.N)
        b[h] = __ldg(reinterpret_cast<const float4*>(p.B + bb + (long long)j * p.bmap.pos_stride + n0 + l_col));
    }
  };
  auto stash = [&](int buf, const float4 (&a)[2], const float4 (&b)[2]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      *reinterpret_cast<uint4*>(&As[buf][l_row + 8 * h][l_col]) = make_uint4(to_tf32(a[h].x), to_tf32(a[h].y), to_tf32(a[h].z), to_tf32(a[h].w));
      *reinterpret_cast<uint4*>(&Bs[buf][l_row + 8 * h][l_col]) = make_uint4(to_tf32(b[h].x), to_tf32(b[h].y), to_tf32(b[h].z), to_tf32(b[h].w));
    }
  };
  float acc[4][4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
  float4 a[2], b[2];
  load(a, b);
  stash(0, a, b);
  __syncthreads();
  int cur = 0;
  for (long long r0 = r_lo; r0 < r_hi; r0 += MMA_BK) {
    const bool more = r0 + MMA_BK < r_hi;
    if (more) { advance(); load(a, b); }
    mma_warp_step(&As[cur][0][0], &Bs[cur][0][0], acc, wm, wn, g, t);
    mma_warp_step(&As[cur][8][0], &Bs[cur][8][0], acc, wm, wn, g, t);
    if (more) stash(cur ^ 1, a, b);
    __syncthreads();
    cur ^= 1;
  }
  float* o = wgrad_out<DET>(p, tap);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int ii = i0 + wm * 64 + i * 16 + g + 8 * h;
      if (ii >= p.Kc) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int nn = n0 + wn * 32 + j * 8 + 2 * t;
        if (nn < p.N) wgrad_put2<DET>(&o[(size_t)ii * p.N + nn], acc[i][j][2 * h], acc[i][j][2 * h + 1]);
      }
    }
}


// =========================================================================================================================
// bf16 forms of the two GEMMs with ldmatrix fragment loads (TFL_OPT_TRAIN_MODE 2).  The k-major word tiles above cost 24
// scalar shared loads per 16 MMAs; here the tiles are bf16 in the layouts ldmatrix wants -- A [m][k] (80-byte pitch),
// B [k][n] (272-byte pitch, read transposed), the weight gradient's A [k = row][m] (transposed too) -- and a 16-deep step of
// a warp's 64 x 32 tile is 4 + 2 ldmatrix.x4 for 16 MMAs.  Conversion fp32 -> bf16 happens once, on the way into shared
// memory.  (Measured: 261 -> 254 ms per Variant-D step -- the kernels stay bound by the latency of the next round's global
// loads at two blocks per SM, ncu r02; a producer / consumer split like the tcgen05 kernels' is what would lift that.)
// =========================================================================================================================
constexpr int BF_AP = 40;    // A tile pitch in bf16 (32 k + 8): rows 80 bytes apart -> 8 consecutive rows hit 8 distinct 16-byte banks
constexpr int BF_BP = 136;   // [k][n] tile pitch in bf16 (128 + 8): rows 272 bytes apart

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_row);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_row) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_row);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ uint2 pack4_bf16(const float4& v) { return make_uint2(pack2_bf16(v.x, v.y), pack2_bf16(v.z, v.w)); }

// B fragments of the warp's four 8-wide n tiles for one 16-deep step, from a [k][n] bf16 tile (rows k0 .. k0 + 15)
__device__ __forceinline__ void load_b_frags(uint32_t (&b)[4][2], const __nv_bfloat16* Bs, int k0, int n_base, int lane) {
#pragma unroll
  for (int jp = 0; jp < 2; ++jp) {
    uint32_t r[4];
    ldmatrix_x4_trans(r, Bs + (size_t)(k0 + (lane & 7) + 8 * ((lane >> 3) & 1)) * BF_BP + n_base + jp * 16 + 8 * (lane >> 4));
    b[2 * jp][0] = r[0]; b[2 * jp][1] = r[1]; b[2 * jp + 1][0] = r[2]; b[2 * jp + 1][1] = r[3];
  }
}

template <class Epi>
__global__ void __launch_bounds__(256, 2) tap_gemm_bf16_kernel(TapGemm p, Epi epi) {
  __shared__ __align__(16) __nv_bfloat16 As[2][GBM][BF_AP];
  __shared__ __align__(16) __nv_bfloat16 Bs[2][32][BF_BP];
  __shared__ long long row_base[GBM];
  __shared__ int row_j[GBM], row_s[GBM];
  const int tid = threadIdx.x;
  const long long m0 = (long long)blockIdx.x * GBM;
  const int n0 = blockIdx.y * GBN;
  if (tid < GBM) {
    const long long r = m0 + tid;
    if (r < p.M) {
      const int s = (int)(r / p.Sout), j = (int)(r - (long long)s * p.Sout);
      row_s[tid] = s; row_j[tid] = j; row_base[tid] = p.amap.base(s);
    } else { row_s[tid] = -1; row_j[tid] = 0; row_base[tid] = 0; }
  }
  __syncthreads();
  // per round (k = 32) and thread: A row a_row, k = 16 a_half .. + 15;  B k rows 4 b_row4 .. + 3, columns b_col .. + 3
  const int a_row = tid >> 1, a_half = tid & 1;
  const int b_row4 = tid >> 5, b_col = (tid & 31) << 2;
  const int kt_per_tap = p.Kc / 32, n_kt = p.taps * kt_per_tap;
  const int my_s = row_s[a_row], my_j = row_j[a_row];
  const long long my_base = row_base[a_row];
  auto load_a = [&](int kt, float4 (&a)[4]) {
    const int tap = kt / kt_per_tap, c0 = (kt - tap * kt_per_tap) * 32;
    const int pos = my_j + tap - p.padL;
    if (my_s < 0 || pos < 0 || pos >= p.Sin) {
#pragma unroll
      for (int h = 0; h < 4; ++h) a[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      return;
    }
    const float* src = p.A + my_base + (long long)pos * p.amap.pos_stride + c0 + 16 * a_half;
#pragma unroll
    for (int h = 0; h < 4; ++h) a[h] = __ldg(reinterpret_cast<const float4*>(src + 4 * h));
  };
  auto load_b = [&](int kt, float4 (&b)[4]) {
    const int n = n0 + b_col;
    if (n >= p.N) {
#pragma unroll
      for (int h = 0; h < 4; ++h) b[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      return;
    }
    const float* src = p.W + ((size_t)kt * 32 + 4 * b_row4) * p.N + n;
#pragma unroll
    for (int h = 0; h < 4; ++h) b[h] = __ldg(reinterpret_cast<const float4*>(src + (size_t)h * p.N));
  };
  auto stash = [&](int buf, const float4 (&a)[4], const float4 (&b)[4]) {
    const uint2 p0 = pack4_bf16(a[0]), p1 = pack4_bf16(a[1]), p2 = pack4_bf16(a[2]), p3 = pack4_bf16(a[3]);
    *reinterpret_cast<uint4*>(&As[buf][a_row][16 * a_half]) = make_uint4(p0.x, p0.y, p1.x, p1.y);
    *reinterpret_cast<uint4*>(&As[buf][a_row][16 * a_half + 8]) = make_uint4(p2.x, p2.y, p3.x, p3.y);
#pragma unroll
    for (int h = 0; h < 4; ++h) *reinterpret_cast<uint2*>(&Bs[buf][4 * b_row4 + h][b_col]) = pack4_bf16(b[h]);
  };
  float acc[4][4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
  float4 na[4], nb[4];
  load_a(0, na); load_b(0, nb);
  stash(0, na, nb);
  __syncthreads();
  for (int kt = 0; kt < n_kt; ++kt) {
    const int cur = kt & 1;
    const bool more = kt + 1 < n_kt;
    if (more) { load_a(kt + 1, na); load_b(kt + 1, nb); }
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t a[4][4], b[4][2];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        ldmatrix_x4(a[i], &As[cur][wm * 64 + i * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)][ks * 16 + 8 * (lane >> 4)]);
      load_b_frags(b, &Bs[cur][0][0], ks * 16, wn * 32, lane);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) mma_bf16(acc[i][j], a[i], b[j]);
    }
    if (more) stash(cur ^ 1, na, nb);
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int n = n0 + wn * 32 + j * 8 + 2 * t;
    if (n >= p.N) continue;
    const float b0 = p.bias != nullptr ? __ldg(&p.bias[n]) : 0.f, b1 = p.bias != nullptr ? __ldg(&p.bias[n + 1]) : 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int rl = wm * 64 + i * 16 + g + 8 * h;
        const int s = row_s[rl];
        if (s < 0) continue;
        epi.pair(s, row_j[rl], m0 + rl, n, p.N, acc[i][j][2 * h] + b0, acc[i][j][2 * h + 1] + b1);
      }
    }
  }
}

template <bool DET>
__global__ void __launch_bounds__(256, 2) tap_wgrad_bf16_kernel(TapWgrad p) {
  __shared__ __align__(16) __nv_bfloat16 As[2][32][BF_BP];   // [k = row][m = i]
  __shared__ __align__(16) __nv_bfloat16 Bs[2][32][BF_BP];   // [k = row][n]
  const int tid = threadIdx.x;
  const int tiles_i = (p.Kc + GBM - 1) / GBM, tiles_n = (p.N + GBN - 1) / GBN;
  int bx = blockIdx.x;
  const int tn = bx % tiles_n; bx /= tiles_n;
  const int ti = bx % tiles_i; bx /= tiles_i;
  const int tap = bx;
  const int i0 = ti * GBM, n0 = tn * GBN;
  const long long r_lo = (long long)blockIdx.y * p.rows_per_split;
  const long long r_hi = r_lo + p.rows_per_split < p.R ? r_lo + p.rows_per_split : p.R;
  if (r_lo >= r_hi) return;
  const int l_row4 = tid >> 5, l_col = (tid & 31) << 2;    // rows 4 l_row4 .. + 3 of the round, columns l_col .. + 3
  // (sequence, position) of the thread's first row, carried from round to round (rows advance by 32)
  long long row_first = r_lo + 4 * l_row4;
  int s_first = (int)(row_first / p.Sout), j_first = (int)(row_first - (long long)s_first * p.Sout);
  long long abase = p.amap.base(s_first), bbase = p.bmap.base(s_first);
  auto advance = [&]() {
    row_first += 32; j_first += 32;
    if (j_first >= p.Sout) {
      do { j_first -= p.Sout; ++s_first; } while (j_first >= p.Sout);
      abase = p.amap.base(s_first); bbase = p.bmap.base(s_first);
    }
  };
  auto load = [&](float4 (&a)[4], float4 (&b)[4]) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      a[h] = make_float4(0.f, 0.f, 0.f, 0.f); b[h] = a[h];
      if (row_first + h >= r_hi) continue;
      int j = j_first + h;
      long long ab = abase, bb = bbase;
      if (j >= p.Sout) {                                    // this row belongs to a later sequence (rare)
        int sq = s_first;
        do { j -= p.Sout; ++sq; } while (j >= p.Sout);
        ab = p.amap.base(sq); bb = p.bmap.base(sq);
      }
      const int pos = j + tap - p.padL;
      if (pos >= 0 && pos < p.Sin && i0 + l_col < p.Kc)
        a[h] = __ldg(reinterpret_cast<const float4*>(p.A + ab + (long long)pos * p.amap.pos_stride + i0 + l_col));
      if (n0 + l_col < p.N)
        b[h] = __ldg(reinterpret_cast<const float4*>(p.B + bb + (long long)j * p.bmap.pos_stride + n0 + l_col));
    }
  };
  auto stash = [&](int buf, const float4 (&a)[4], const float4 (&b)[4]) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      *reinterpret_cast<uint2*>(&As[buf][4 * l_row4 + h][l_col]) = pack4_bf16(a[h]);
      *reinterpret_cast<uint2*>(&Bs[buf][4 * l_row4 + h][l_col]) = pack4_bf16(b[h]);
    }
  };
  float acc[4][4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = acc[i][j][2] = acc[i][j][3] = 0.f;
  const int warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
  float4 a4[4], b4[4];
  load(a4, b4);
  stash(0, a4, b4);
  __syncthreads();
  int cur = 0;
  for (long long r0 = r_lo; r0 < r_hi; r0 += 32) {
    const bool more = r0 + 32 < r_hi;
    if (more) { advance(); load(a4, b4); }
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t a[4][4], b[4][2];
#pragma unroll
      for (int i = 0; i < 4; ++i)   // A^T: matrices (k 0-7, m 0-7), (k 0-7, m 8-15), (k 8-15, m 0-7), (k 8-15, m 8-15) = a0 .. a3
        ldmatrix_x4_trans(a[i], &As[cur][ks * 16 + (lane & 7) + 8 * (lane >> 4)][wm * 64 + i * 16 + 8 * ((lane >> 3) & 1)]);
      load_b_frags(b, &Bs[cur][0][0], ks * 16, wn * 32, lane);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) mma_bf16(acc[i][j], a[i], b[j]);
    }
    if (more) stash(cur ^ 1, a4, b4);
    __syncthreads();
    cur ^= 1;
  }
  float* o = wgrad_out<DET>(p, tap);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int ii = i0 + wm * 64 + i * 16 + g + 8 * h;
      if (ii >= p.Kc) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int nn = n0 + wn * 32 + j * 8 + 2 * t;
        if (nn < p.N) wgrad_put2<DET>(&o[(size_t)ii * p.N + nn], acc[i][j][2 * h], acc[i][j][2 * h + 1]);
      }
    }
}

// =========================================================================================================================
// Attention backward on mma.sync m16n8k8 (tf32 operands, fp32 accumulation): the tensor-core form of attn_bwd_dq_kernel /
// attn_bwd_dkv_kernel (kernels_bwd.cuh; same buffers, same math).  A warp owns 16 queries (dq) or 16 keys (dk, dv); the other
// side is staged 64 rows at a time in shared memory as tf32 [row][HD + 4] (every fragment load below hits 32 distinct
// banks).  Per 8-wide tile of the other side:
//   S   = Q K^T and dP = dO V^T       A = own rows (registers, loaded once), B = staged rows: b = X[n = g][k = 8 ks + t (+4)]
//   P   = exp(S - lse),  dS = P (dP - D)          in the accumulator layout: (row g, cols 2t, 2t+1), (row g + 8, same cols)
//   dQ += dS K   (dV += P^T dO, dK += dS^T Q)     the accumulator IS the A fragment once k slot t is read as column 2t and
//                                                 slot t + 4 as column 2t + 1 (the order of k inside an MMA is free as long
//                                                 as B uses the same one: b = X[2t (+1)][n = 8 j + g]) -- no shuffles.
// =========================================================================================================================
template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dq_mma_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                              const float* __restrict__ v, const float* __restrict__ o,
                                                              const float* __restrict__ dO, const float* __restrict__ lse,
                                                              float* __restrict__ dq, float* __restrict__ Dbuf,
                                                              int L, int hd, int heads, float scale) {
  constexpr int TK = 64, PITCH = HD + 4, KS = HD / 8;
  __shared__ uint32_t ks_[TK][PITCH], vs_[TK][PITCH];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;          // this lane's two query rows
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  uint32_t aq[KS][4], ado[KS][4];
  float D0 = 0.f, D1 = 0.f;
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = (e & 1) ? r1 : r0, d = 8 * ks + t + ((e & 2) ? 4 : 0);
      const bool ok = r < L && d < hd;
      const float qv = ok ? q[base + (size_t)r * hd + d] * scale : 0.f;
      const float gv = ok ? dO[((size_t)s * L + r) * A + (size_t)head * hd + d] : 0.f;
      const float ov = ok ? o[((size_t)s * L + r) * A + (size_t)head * hd + d] : 0.f;
      aq[ks][e] = to_tf32(qv); ado[ks][e] = to_tf32(gv);
      if (e & 1) D1 = fmaf(gv, ov, D1); else D0 = fmaf(gv, ov, D0);
    }
  }
  D0 += __shfl_xor_sync(0xffffffffu, D0, 1); D0 += __shfl_xor_sync(0xffffffffu, D0, 2);
  D1 += __shfl_xor_sync(0xffffffffu, D1, 1); D1 += __shfl_xor_sync(0xffffffffu, D1, 2);
  const size_t lrow = ((size_t)s * heads + head) * L;
  const float l0 = r0 < L ? lse[lrow + r0] : 0.f, l1 = r1 < L ? lse[lrow + r1] : 0.f;
  if (t == 0) {
    if (r0 < L) Dbuf[lrow + r0] = D0;
    if (r1 < L) Dbuf[lrow + r1] = D1;
  }
  float acc[KS][4];
#pragma unroll
  for (int j = 0; j < KS; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (int j0 = 0; j0 < L; j0 += TK) {
    __syncthreads();
    for (int e = threadIdx.x; e < TK * HD; e += blockDim.x) {
      const int jj = e / HD, d = e - jj * HD;
      const bool ok = (j0 + jj < L) && (d < hd);
      ks_[jj][d] = to_tf32(ok ? k[base + (size_t)(j0 + jj) * hd + d] : 0.f);
      vs_[jj][d] = to_tf32(ok ? v[base + (size_t)(j0 + jj) * hd + d] : 0.f);
    }
    __syncthreads();
#pragma unroll 2
    for (int nt = 0; nt < TK / 8; ++nt) {
      const int key0 = nt * 8;
      if (j0 + key0 >= L) break;
      float S[4] = {0.f, 0.f, 0.f, 0.f}, dP[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t bk[2] = {ks_[key0 + g][8 * ks + t], ks_[key0 + g][8 * ks + t + 4]};
        const uint32_t bv[2] = {vs_[key0 + g][8 * ks + t], vs_[key0 + g][8 * ks + t + 4]};
        mma_tf32(S, aq[ks], bk);
        mma_tf32(dP, ado[ks], bv);
      }
      const bool v0 = j0 + key0 + 2 * t < L, v1 = j0 + key0 + 2 * t + 1 < L;
      const float p0 = v0 ? __expf(S[0] - l0) : 0.f, p1 = v1 ? __expf(S[1] - l0) : 0.f;
      const float p2 = v0 ? __expf(S[2] - l1) : 0.f, p3 = v1 ? __expf(S[3] - l1) : 0.f;
      // A fragment of dS: (row g, slot t = key 2t), (row g + 8, slot t), (row g, slot t + 4 = key 2t + 1), (row g + 8, slot t + 4)
      const uint32_t ads[4] = {to_tf32(p0 * (dP[0] - D0)), to_tf32(p2 * (dP[2] - D1)), to_tf32(p1 * (dP[1] - D0)), to_tf32(p3 * (dP[3] - D1))};
#pragma unroll
      for (int j = 0; j < KS; ++j) {
        const uint32_t b[2] = {ks_[key0 + 2 * t][8 * j + g], ks_[key0 + 2 * t + 1][8 * j + g]};
        mma_tf32(acc[j], ads, b);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < KS; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {
      if (r0 < L) *reinterpret_cast<float2*>(dq + base + (size_t)r0 * hd + d) = make_float2(acc[j][0] * scale, acc[j][1] * scale);
      if (r1 < L) *reinterpret_cast<float2*>(dq + base + (size_t)r1 * hd + d) = make_float2(acc[j][2] * scale, acc[j][3] * scale);
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dkv_mma_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                               const float* __restrict__ v, const float* __restrict__ dO,
                                                               const float* __restrict__ lse, const float* __restrict__ Dbuf,
                                                               float* __restrict__ dk, float* __restrict__ dv,
                                                               int L, int hd, int heads, float scale) {
  constexpr int TQ = 64, PITCH = HD + 4, KS = HD / 8;
  __shared__ uint32_t qs_[TQ][PITCH], dos_[TQ][PITCH];
  __shared__ float ls_[TQ], Ds_[TQ];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;          // this lane's two key rows
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  const size_t lrow = ((size_t)s * heads + head) * L;
  uint32_t ak[KS][4], av[KS][4];
#pragma unroll
  for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = (e & 1) ? r1 : r0, d = 8 * ks + t + ((e & 2) ? 4 : 0);
      const bool ok = r < L && d < hd;
      ak[ks][e] = to_tf32(ok ? k[base + (size_t)r * hd + d] : 0.f);
      av[ks][e] = to_tf32(ok ? v[base + (size_t)r * hd + d] : 0.f);
    }
  }
  float dK[KS][4], dV[KS][4];
#pragma unroll
  for (int j = 0; j < KS; ++j) {
    dK[j][0] = dK[j][1] = dK[j][2] = dK[j][3] = 0.f;
    dV[j][0] = dV[j][1] = dV[j][2] = dV[j][3] = 0.f;
  }
  for (int i0 = 0; i0 < L; i0 += TQ) {
    __syncthreads();
    for (int e = threadIdx.x; e < TQ * HD; e += blockDim.x) {
      const int ii = e / HD, d = e - ii * HD;
      const bool ok = (i0 + ii < L) && (d < hd);
      qs_[ii][d] = to_tf32(ok ? q[base + (size_t)(i0 + ii) * hd + d] * scale : 0.f);
      dos_[ii][d] = to_tf32(ok ? dO[((size_t)s * L + i0 + ii) * A + (size_t)head * hd + d] : 0.f);
    }
    for (int e = threadIdx.x; e < TQ; e += blockDim.x) {
      const bool ok = i0 + e < L;
      ls_[e] = ok ? lse[lrow + i0 + e] : INFINITY;                       // exp(S - inf) = 0: queries beyond the sequence
      Ds_[e] = ok ? Dbuf[lrow + i0 + e] : 0.f;
    }
    __syncthreads();
#pragma unroll 2
    for (int nt = 0; nt < TQ / 8; ++nt) {
      const int qq0 = nt * 8;
      if (i0 + qq0 >= L) break;
      float ST[4] = {0.f, 0.f, 0.f, 0.f}, dPT[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t bq[2] = {qs_[qq0 + g][8 * ks + t], qs_[qq0 + g][8 * ks + t + 4]};
        const uint32_t bd[2] = {dos_[qq0 + g][8 * ks + t], dos_[qq0 + g][8 * ks + t + 4]};
        mma_tf32(ST, ak[ks], bq);
        mma_tf32(dPT, av[ks], bd);
      }
      const float la = ls_[qq0 + 2 * t], lb = ls_[qq0 + 2 * t + 1], da = Ds_[qq0 + 2 * t], db = Ds_[qq0 + 2 * t + 1];
      const float p0 = __expf(ST[0] - la), p1 = __expf(ST[1] - lb), p2 = __expf(ST[2] - la), p3 = __expf(ST[3] - lb);
      const uint32_t ap[4] = {to_tf32(p0), to_tf32(p2), to_tf32(p1), to_tf32(p3)};
      const uint32_t ads[4] = {to_tf32(p0 * (dPT[0] - da)), to_tf32(p2 * (dPT[2] - da)), to_tf32(p1 * (dPT[1] - db)), to_tf32(p3 * (dPT[3] - db))};
#pragma unroll
      for (int j = 0; j < KS; ++j) {
        const uint32_t bo[2] = {dos_[qq0 + 2 * t][8 * j + g], dos_[qq0 + 2 * t + 1][8 * j + g]};
        const uint32_t bq[2] = {qs_[qq0 + 2 * t][8 * j + g], qs_[qq0 + 2 * t + 1][8 * j + g]};
        mma_tf32(dV[j], ap, bo);
        mma_tf32(dK[j], ads, bq);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < KS; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {   // qs_ carries the softmax scale already: dK_j = sum_i dS_ij * (scale * Q_i)
      if (r0 < L) {
        *reinterpret_cast<float2*>(dk + base + (size_t)r0 * hd + d) = make_float2(dK[j][0], dK[j][1]);
        *reinterpret_cast<float2*>(dv + base + (size_t)r0 * hd + d) = make_float2(dV[j][0], dV[j][1]);
      }
      if (r1 < L) {
        *reinterpret_cast<float2*>(dk + base + (size_t)r1 * hd + d) = make_float2(dK[j][2], dK[j][3]);
        *reinterpret_cast<float2*>(dv + base + (size_t)r1 * hd + d) = make_float2(dV[j][2], dV[j][3]);
      }
    }
  }
}

// ---- bf16 forms of the two backward kernels (TFL_OPT_TRAIN_MODE 2): m16n8k16, the staged side as bf16 [row][HD + 8]
// tiles read with ldmatrix (plain for the S / dP operands, transposed for the dQ / dK / dV operands) -- 12 (dq) and 16
// (dk, dv) MMAs per 16 rows of the other side instead of 24 and 32, and the own-side fragments take half the registers.
// P and dS are rounded to bf16 before their MMA (as in the forward tcgen05 kernel); accumulation stays fp32.
template <int HD>
__device__ __forceinline__ void stage_bf16_rows(__nv_bfloat16 (*tile)[HD + 8], const float* __restrict__ src, size_t row_stride,
                                                int row0, int L, int hd, float mul) {
  for (int e = threadIdx.x; e < 64 * (HD / 2); e += blockDim.x) {
    const int rr = e / (HD / 2), d = 2 * (e - rr * (HD / 2));
    float2 v = make_float2(0.f, 0.f);
    if (row0 + rr < L && d < hd) v = *reinterpret_cast<const float2*>(src + (size_t)(row0 + rr) * row_stride + d);
    *reinterpret_cast<uint32_t*>(&tile[rr][d]) = pack2_bf16(v.x * mul, v.y * mul);
  }
}
// own-side A fragments (16 rows x HD) from fp32 rows r0 / r1: [ks][0..3] = (r0, 2t), (r1, 2t), (r0, 2t + 8), (r1, 2t + 8) pairs
template <int HD>
__device__ __forceinline__ void load_a_rows_bf16(uint32_t (&a)[HD / 16][4], const float* __restrict__ src, size_t row_stride,
                                                 int r0, int r1, int L, int hd, int t, float mul) {
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = (e & 1) ? r1 : r0, d = 16 * ks + 2 * t + ((e & 2) ? 8 : 0);
      float2 v = make_float2(0.f, 0.f);
      if (r < L && d < hd) v = *reinterpret_cast<const float2*>(src + (size_t)r * row_stride + d);
      a[ks][e] = pack2_bf16(v.x * mul, v.y * mul);
    }
}

template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dq_bf16_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                               const float* __restrict__ v, const float* __restrict__ o,
                                                               const float* __restrict__ dO, const float* __restrict__ lse,
                                                               float* __restrict__ dq, float* __restrict__ Dbuf,
                                                               int L, int hd, int heads, float scale) {
  constexpr int TK = 64, KS = HD / 16, NT = HD / 8;
  __shared__ __align__(16) __nv_bfloat16 ks_[TK][HD + 8], vs_[TK][HD + 8];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  const float* dO_h = dO + (size_t)s * L * A + (size_t)head * hd;     // row stride A
  const float* o_h = o + (size_t)s * L * A + (size_t)head * hd;
  uint32_t aq[KS][4], ado[KS][4];
  load_a_rows_bf16<HD>(aq, q + base, hd, r0, r1, L, hd, t, scale);
  load_a_rows_bf16<HD>(ado, dO_h, A, r0, r1, L, hd, t, 1.f);
  float D0 = 0.f, D1 = 0.f;                                             // D = dO . O from the fp32 values
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = (e & 1) ? r1 : r0, d = 16 * ks + 2 * t + ((e & 2) ? 8 : 0);
      if (r < L && d < hd) {
        const float2 gv = *reinterpret_cast<const float2*>(dO_h + (size_t)r * A + d);
        const float2 ov = *reinterpret_cast<const float2*>(o_h + (size_t)r * A + d);
        const float dd = gv.x * ov.x + gv.y * ov.y;
        if (e & 1) D1 += dd; else D0 += dd;
      }
    }
  D0 += __shfl_xor_sync(0xffffffffu, D0, 1); D0 += __shfl_xor_sync(0xffffffffu, D0, 2);
  D1 += __shfl_xor_sync(0xffffffffu, D1, 1); D1 += __shfl_xor_sync(0xffffffffu, D1, 2);
  const size_t lrow = ((size_t)s * heads + head) * L;
  const float l0 = r0 < L ? lse[lrow + r0] : 0.f, l1 = r1 < L ? lse[lrow + r1] : 0.f;
  if (t == 0) {
    if (r0 < L) Dbuf[lrow + r0] = D0;
    if (r1 < L) Dbuf[lrow + r1] = D1;
  }
  float acc[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (int j0 = 0; j0 < L; j0 += TK) {
    __syncthreads();
    stage_bf16_rows<HD>(ks_, k + base, hd, j0, L, hd, 1.f);
    stage_bf16_rows<HD>(vs_, v + base, hd, j0, L, hd, 1.f);
    __syncthreads();
#pragma unroll 2
    for (int kb = 0; kb < TK / 16; ++kb) {
      const int key0 = kb * 16;
      if (j0 + key0 >= L) break;
      float S[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, dP[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {   // matrices (keys 0-7 | 8-15) x (dims 16 ks .. +7 | +8 .. +15): b0, b1 of n-tile 0 then of n-tile 1
        uint32_t bk[4], bv[4];
        ldmatrix_x4(bk, &ks_[key0 + (lane & 7) + 8 * (lane >> 4)][16 * ks + 8 * ((lane >> 3) & 1)]);
        ldmatrix_x4(bv, &vs_[key0 + (lane & 7) + 8 * (lane >> 4)][16 * ks + 8 * ((lane >> 3) & 1)]);
        const uint32_t bk0[2] = {bk[0], bk[1]}, bk1[2] = {bk[2], bk[3]}, bv0[2] = {bv[0], bv[1]}, bv1[2] = {bv[2], bv[3]};
        mma_bf16(S[0], aq[ks], bk0); mma_bf16(S[1], aq[ks], bk1);
        mma_bf16(dP[0], ado[ks], bv0); mma_bf16(dP[1], ado[ks], bv1);
      }
      float ds[2][4];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        const bool v0 = j0 + key0 + 8 * n + 2 * t < L, v1 = j0 + key0 + 8 * n + 2 * t + 1 < L;
        ds[n][0] = v0 ? __expf(S[n][0] - l0) * (dP[n][0] - D0) : 0.f;
        ds[n][1] = v1 ? __expf(S[n][1] - l0) * (dP[n][1] - D0) : 0.f;
        ds[n][2] = v0 ? __expf(S[n][2] - l1) * (dP[n][2] - D1) : 0.f;
        ds[n][3] = v1 ? __expf(S[n][3] - l1) * (dP[n][3] - D1) : 0.f;
      }
      const uint32_t ads[4] = {pack2_bf16(ds[0][0], ds[0][1]), pack2_bf16(ds[0][2], ds[0][3]),
                               pack2_bf16(ds[1][0], ds[1][1]), pack2_bf16(ds[1][2], ds[1][3])};
#pragma unroll
      for (int jp = 0; jp < NT / 2; ++jp) {   // K^T operand: matrices (keys 0-7 | 8-15) x (dims 16 jp .. +7 | +8 .. +15), transposed
        uint32_t b[4];
        ldmatrix_x4_trans(b, &ks_[key0 + (lane & 7) + 8 * ((lane >> 3) & 1)][16 * jp + 8 * (lane >> 4)]);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16(acc[2 * jp], ads, b0); mma_bf16(acc[2 * jp + 1], ads, b1);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {
      if (r0 < L) *reinterpret_cast<float2*>(dq + base + (size_t)r0 * hd + d) = make_float2(acc[j][0] * scale, acc[j][1] * scale);
      if (r1 < L) *reinterpret_cast<float2*>(dq + base + (size_t)r1 * hd + d) = make_float2(acc[j][2] * scale, acc[j][3] * scale);
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dkv_bf16_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                                const float* __restrict__ v, const float* __restrict__ dO,
                                                                const float* __restrict__ lse, const float* __restrict__ Dbuf,
                                                                float* __restrict__ dk, float* __restrict__ dv,
                                                                int L, int hd, int heads, float scale) {
  constexpr int TQ = 64, KS = HD / 16, NT = HD / 8;
  __shared__ __align__(16) __nv_bfloat16 qs_[TQ][HD + 8], dos_[TQ][HD + 8];
  __shared__ float ls_[TQ], Ds_[TQ];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;          // this lane's two key rows
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  const size_t lrow = ((size_t)s * heads + head) * L;
  const float* dO_h = dO + (size_t)s * L * A + (size_t)head * hd;
  uint32_t ak[KS][4], av[KS][4];
  load_a_rows_bf16<HD>(ak, k + base, hd, r0, r1, L, hd, t, 1.f);
  load_a_rows_bf16<HD>(av, v + base, hd, r0, r1, L, hd, t, 1.f);
  float dK[NT][4], dV[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    dK[j][0] = dK[j][1] = dK[j][2] = dK[j][3] = 0.f;
    dV[j][0] = dV[j][1] = dV[j][2] = dV[j][3] = 0.f;
  }
  for (int i0 = 0; i0 < L; i0 += TQ) {
    __syncthreads();
    stage_bf16_rows<HD>(qs_, q + base, hd, i0, L, hd, scale);
    stage_bf16_rows<HD>(dos_, dO_h, A, i0, L, hd, 1.f);
    for (int e = threadIdx.x; e < TQ; e += blockDim.x) {
      const bool ok = i0 + e < L;
      ls_[e] = ok ? lse[lrow + i0 + e] : INFINITY;                       // exp(S - inf) = 0: queries beyond the sequence
      Ds_[e] = ok ? Dbuf[lrow + i0 + e] : 0.f;
    }
    __syncthreads();
#pragma unroll 2
    for (int qb = 0; qb < TQ / 16; ++qb) {
      const int qq0 = qb * 16;
      if (i0 + qq0 >= L) break;
      float ST[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, dPT[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t bq[4], bd[4];
        ldmatrix_x4(bq, &qs_[qq0 + (lane & 7) + 8 * (lane >> 4)][16 * ks + 8 * ((lane >> 3) & 1)]);
        ldmatrix_x4(bd, &dos_[qq0 + (lane & 7) + 8 * (lane >> 4)][16 * ks + 8 * ((lane >> 3) & 1)]);
        const uint32_t bq0[2] = {bq[0], bq[1]}, bq1[2] = {bq[2], bq[3]}, bd0[2] = {bd[0], bd[1]}, bd1[2] = {bd[2], bd[3]};
        mma_bf16(ST[0], ak[ks], bq0); mma_bf16(ST[1], ak[ks], bq1);
        mma_bf16(dPT[0], av[ks], bd0); mma_bf16(dPT[1], av[ks], bd1);
      }
      float pt[2][4], ds[2][4];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        const int c = qq0 + 8 * n + 2 * t;
        const float la = ls_[c], lb = ls_[c + 1], da = Ds_[c], db = Ds_[c + 1];
        pt[n][0] = __expf(ST[n][0] - la); pt[n][1] = __expf(ST[n][1] - lb);
        pt[n][2] = __expf(ST[n][2] - la); pt[n][3] = __expf(ST[n][3] - lb);
        ds[n][0] = pt[n][0] * (dPT[n][0] - da); ds[n][1] = pt[n][1] * (dPT[n][1] - db);
        ds[n][2] = pt[n][2] * (dPT[n][2] - da); ds[n][3] = pt[n][3] * (dPT[n][3] - db);
      }
      const uint32_t ap[4] = {pack2_bf16(pt[0][0], pt[0][1]), pack2_bf16(pt[0][2], pt[0][3]),
                              pack2_bf16(pt[1][0], pt[1][1]), pack2_bf16(pt[1][2], pt[1][3])};
      const uint32_t ads[4] = {pack2_bf16(ds[0][0], ds[0][1]), pack2_bf16(ds[0][2], ds[0][3]),
                               pack2_bf16(ds[1][0], ds[1][1]), pack2_bf16(ds[1][2], ds[1][3])};
#pragma unroll
      for (int jp = 0; jp < NT / 2; ++jp) {
        uint32_t bo[4], bq[4];
        ldmatrix_x4_trans(bo, &dos_[qq0 + (lane & 7) + 8 * ((lane >> 3) & 1)][16 * jp + 8 * (lane >> 4)]);
        ldmatrix_x4_trans(bq, &qs_[qq0 + (lane & 7) + 8 * ((lane >> 3) & 1)][16 * jp + 8 * (lane >> 4)]);
        const uint32_t bo0[2] = {bo[0], bo[1]}, bo1[2] = {bo[2], bo[3]}, bq0[2] = {bq[0], bq[1]}, bq1[2] = {bq[2], bq[3]};
        mma_bf16(dV[2 * jp], ap, bo0); mma_bf16(dV[2 * jp + 1], ap, bo1);
        mma_bf16(dK[2 * jp], ads, bq0); mma_bf16(dK[2 * jp + 1], ads, bq1);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {   // qs_ carries the softmax scale already: dK_j = sum_i dS_ij * (scale * Q_i)
      if (r0 < L) {
        *reinterpret_cast<float2*>(dk + base + (size_t)r0 * hd + d) = make_float2(dK[j][0], dK[j][1]);
        *reinterpret_cast<float2*>(dv + base + (size_t)r0 * hd + d) = make_float2(dV[j][0], dV[j][1]);
      }
      if (r1 < L) {
        *reinterpret_cast<float2*>(dk + base + (size_t)r1 * hd + d) = make_float2(dK[j][2], dK[j][3]);
        *reinterpret_cast<float2*>(dv + base + (size_t)r1 * hd + d) = make_float2(dV[j][2], dV[j][3]);
      }
    }
  }
}

// bf16 form of the forward-with-lse kernel below (the backward pass's recompute in mode 2): 64 keys per stage, S of the
// whole stage first (8 n-tiles = 4 ldmatrix.x4 per 16 dims), one online-softmax update per stage, P V with V read transposed.
template <int HD>
__global__ void __launch_bounds__(128) attn_fwd_bf16_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                            const float* __restrict__ v, float* __restrict__ o,
                                                            int L, int hd, int heads, float scale, float* __restrict__ lse) {
  constexpr int TK = 64, KS = HD / 16, NT = HD / 8;
  __shared__ __align__(16) __nv_bfloat16 ks_[TK][HD + 8], vs_[TK][HD + 8];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  uint32_t aq[KS][4];
  load_a_rows_bf16<HD>(aq, q + base, hd, r0, r1, L, hd, t, scale);
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  float acc[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (int j0 = 0; j0 < L; j0 += TK) {
    __syncthreads();
    stage_bf16_rows<HD>(ks_, k + base, hd, j0, L, hd, 1.f);
    stage_bf16_rows<HD>(vs_, v + base, hd, j0, L, hd, 1.f);
    __syncthreads();
    float S[TK / 8][4];
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int kb = 0; kb < TK / 16; ++kb) {
#pragma unroll
      for (int n = 0; n < 2; ++n) S[2 * kb + n][0] = S[2 * kb + n][1] = S[2 * kb + n][2] = S[2 * kb + n][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t bk[4];
        ldmatrix_x4(bk, &ks_[kb * 16 + (lane & 7) + 8 * (lane >> 4)][16 * ks + 8 * ((lane >> 3) & 1)]);
        const uint32_t b0[2] = {bk[0], bk[1]}, b1[2] = {bk[2], bk[3]};
        mma_bf16(S[2 * kb], aq[ks], b0); mma_bf16(S[2 * kb + 1], aq[ks], b1);
      }
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        const int nt = 2 * kb + n, c0 = j0 + nt * 8 + 2 * t;
        if (c0 >= L) { S[nt][0] = -INFINITY; S[nt][2] = -INFINITY; }
        if (c0 + 1 >= L) { S[nt][1] = -INFINITY; S[nt][3] = -INFINITY; }
        mx0 = fmaxf(mx0, fmaxf(S[nt][0], S[nt][1]));
        mx1 = fmaxf(mx1, fmaxf(S[nt][2], S[nt][3]));
      }
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float n0 = fmaxf(m0, mx0), n1 = fmaxf(m1, mx1);        // finite: every stage holds at least one key < L
    const float a0 = __expf(m0 - n0), a1 = __expf(m1 - n1);
    l0 *= a0; l1 *= a1;
#pragma unroll
    for (int j = 0; j < NT; ++j) { acc[j][0] *= a0; acc[j][1] *= a0; acc[j][2] *= a1; acc[j][3] *= a1; }
    m0 = n0; m1 = n1;
#pragma unroll
    for (int kb = 0; kb < TK / 16; ++kb) {
      float pr[2][4];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        const int nt = 2 * kb + n;
        pr[n][0] = __expf(S[nt][0] - n0); pr[n][1] = __expf(S[nt][1] - n0);
        pr[n][2] = __expf(S[nt][2] - n1); pr[n][3] = __expf(S[nt][3] - n1);
        l0 += pr[n][0] + pr[n][1]; l1 += pr[n][2] + pr[n][3];
      }
      const uint32_t ap[4] = {pack2_bf16(pr[0][0], pr[0][1]), pack2_bf16(pr[0][2], pr[0][3]),
                              pack2_bf16(pr[1][0], pr[1][1]), pack2_bf16(pr[1][2], pr[1][3])};
#pragma unroll
      for (int jp = 0; jp < NT / 2; ++jp) {
        uint32_t b[4];
        ldmatrix_x4_trans(b, &vs_[kb * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)][16 * jp + 8 * (lane >> 4)]);
        const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
        mma_bf16(acc[2 * jp], ap, b0); mma_bf16(acc[2 * jp + 1], ap, b1);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {
      if (r0 < L) *reinterpret_cast<float2*>(o + ((size_t)s * L + r0) * A + (size_t)head * hd + d) = make_float2(acc[j][0] * i0, acc[j][1] * i0);
      if (r1 < L) *reinterpret_cast<float2*>(o + ((size_t)s * L + r1) * A + (size_t)head * hd + d) = make_float2(acc[j][2] * i1, acc[j][3] * i1);
    }
  }
  if (lse != nullptr && t == 0) {
    const size_t lrow = ((size_t)s * heads + head) * L;
    if (r0 < L) lse[lrow + r0] = m0 + logf(l0);
    if (r1 < L) lse[lrow + r1] = m1 + logf(l1);
  }
}

// Forward attention with the log-sum-exp kept (training forward in TFL_OPT_TRAIN_MODE 1 and the recompute of the backward
// pass): the mma form of attn_f32_kernel.  16 queries per warp, 64 keys per stage; S of the whole stage first (8 tiles),
// one online-softmax update per stage, then P V with the accumulator-as-A-fragment trick above.
template <int HD>
__global__ void __launch_bounds__(128) attn_fwd_mma_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                           const float* __restrict__ v, float* __restrict__ o,
                                                           int L, int hd, int heads, float scale, float* __restrict__ lse) {
  constexpr int TK = 64, PITCH = HD + 4, KS = HD / 8;
  __shared__ uint32_t ks_[TK][PITCH], vs_[TK][PITCH];
  const int head = blockIdx.y, s = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = blockIdx.x * 64 + warp * 16 + g, r1 = r0 + 8;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const size_t A = (size_t)heads * hd;
  uint32_t aq[KS][4];
#pragma unroll
  for (int ks = 0; ks < KS; ++ks)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = (e & 1) ? r1 : r0, d = 8 * ks + t + ((e & 2) ? 4 : 0);
      aq[ks][e] = to_tf32((r < L && d < hd) ? q[base + (size_t)r * hd + d] * scale : 0.f);
    }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  float acc[KS][4];
#pragma unroll
  for (int j = 0; j < KS; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  for (int j0 = 0; j0 < L; j0 += TK) {
    __syncthreads();
    for (int e = threadIdx.x; e < TK * HD; e += blockDim.x) {
      const int jj = e / HD, d = e - jj * HD;
      const bool ok = (j0 + jj < L) && (d < hd);
      ks_[jj][d] = to_tf32(ok ? k[base + (size_t)(j0 + jj) * hd + d] : 0.f);
      vs_[jj][d] = to_tf32(ok ? v[base + (size_t)(j0 + jj) * hd + d] : 0.f);
    }
    __syncthreads();
    float S[TK / 8][4];
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < TK / 8; ++nt) {
      S[nt][0] = S[nt][1] = S[nt][2] = S[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const uint32_t bk[2] = {ks_[nt * 8 + g][8 * ks + t], ks_[nt * 8 + g][8 * ks + t + 4]};
        mma_tf32(S[nt], aq[ks], bk);
      }
      const int c0 = j0 + nt * 8 + 2 * t;
      if (c0 >= L) { S[nt][0] = -INFINITY; S[nt][2] = -INFINITY; }
      if (c0 + 1 >= L) { S[nt][1] = -INFINITY; S[nt][3] = -INFINITY; }
      mx0 = fmaxf(mx0, fmaxf(S[nt][0], S[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(S[nt][2], S[nt][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float n0 = fmaxf(m0, mx0), n1 = fmaxf(m1, mx1);        // finite: every stage holds at least one key < L
    const float a0 = __expf(m0 - n0), a1 = __expf(m1 - n1);
    l0 *= a0; l1 *= a1;
#pragma unroll
    for (int j = 0; j < KS; ++j) { acc[j][0] *= a0; acc[j][1] *= a0; acc[j][2] *= a1; acc[j][3] *= a1; }
    m0 = n0; m1 = n1;
#pragma unroll
    for (int nt = 0; nt < TK / 8; ++nt) {
      const float p0 = __expf(S[nt][0] - n0), p1 = __expf(S[nt][1] - n0), p2 = __expf(S[nt][2] - n1), p3 = __expf(S[nt][3] - n1);
      l0 += p0 + p1; l1 += p2 + p3;
      const uint32_t ap[4] = {to_tf32(p0), to_tf32(p2), to_tf32(p1), to_tf32(p3)};
#pragma unroll
      for (int j = 0; j < KS; ++j) {
        const uint32_t b[2] = {vs_[nt * 8 + 2 * t][8 * j + g], vs_[nt * 8 + 2 * t + 1][8 * j + g]};
        mma_tf32(acc[j], ap, b);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
#pragma unroll
  for (int j = 0; j < KS; ++j) {
    const int d = 8 * j + 2 * t;
    if (d < hd) {
      if (r0 < L) *reinterpret_cast<float2*>(o + ((size_t)s * L + r0) * A + (size_t)head * hd + d) = make_float2(acc[j][0] * i0, acc[j][1] * i0);
      if (r1 < L) *reinterpret_cast<float2*>(o + ((size_t)s * L + r1) * A + (size_t)head * hd + d) = make_float2(acc[j][2] * i1, acc[j][3] * i1);
    }
  }
  if (lse != nullptr && t == 0) {
    const size_t lrow = ((size_t)s * heads + head) * L;
    if (r0 < L) lse[lrow + r0] = m0 + logf(l0);
    if (r1 < L) lse[lrow + r1] = m1 + logf(l1);
  }
}

}  // namespace tfl
