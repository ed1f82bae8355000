// K8  Band-split encoder / band-wise decoder of BS-Locoformer
// (standalone/bslocoformer_separator.py:186-270), fp32 CUDA-core kernels.  The reference runs
// 62 x (GroupNorm + 1x1 conv) and 62 x (GroupNorm + 3 x 1x1 conv + tanh + GLU) tiny module calls;
// here each stage is ONE launch with a CTA per (band, frame tile, batch element).
//
// Weights live in one caller-packed fp32 buffer `w`; `table` (device, int64) holds per band b
//   table[b*16 + 0]  = first bin f0          table[b*16 + 1]  = width w_b
//   split : [2] gn_w  [3] gn_b  [4] Wt [K_b][C] (transposed 1x1 conv)  [5] bias [C]      K_b = w_b * 2M
//   decode: [6] gn_w  [7] gn_b  [8] W1t [C][4C]  [9] b1  [10] W3t [4C][4C]  [11] b3  [12] W4t [4C][O_b]  [13] b4
//   O_b = w_b * S * 2M * 2 (pre-GLU).
#pragma once
#include "common.cuh"

namespace tfl {

constexpr int BS_TT = 16;  // frames per CTA tile

__device__ __forceinline__ float2 block_sum2(float a, float b, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  __syncthreads();
  if (lane == 0) { red[warp * 2] = a; red[warp * 2 + 1] = b; }
  __syncthreads();
  float sa = 0.f, sb = 0.f;
  for (int i = 0; i < nw; ++i) { sa += red[i * 2]; sb += red[i * 2 + 1]; }
  return make_float2(sa, sb);
}

// spec [B, M, T, F, 2] -> x [B, T, nb, C].  Band channel index k = f_local * 2M + ch, ch = (re_0..re_{M-1}, im_0..)
// (:163-164, :247-252).  GroupNorm(1, K_b) statistics run over (K_b, T) per batch element.
__global__ void __launch_bounds__(256) bs_split_kernel(const float* __restrict__ spec, int M, int T, int F, int C, int nb,
                                                       const long long* __restrict__ table, const float* __restrict__ w,
                                                       float* __restrict__ x, float eps) {
  extern __shared__ float sm[];           // xn [K_b][BS_TT] + reduction scratch
  const int band = blockIdx.x, b = blockIdx.z;
  const long long* tb = table + band * 16;
  const int f0 = (int)tb[0], wb = (int)tb[1], K = wb * 2 * M;
  const float* gw = w + tb[2]; const float* gb = w + tb[3]; const float* Wt = w + tb[4]; const float* bias = w + tb[5];
  float* red = sm + (size_t)K * BS_TT;
  const float* sp = spec + (size_t)b * M * T * F * 2;
  auto feat = [&](int k, int t) -> float {      // k = fl * 2M + ch
    const int fl = k / (2 * M), ch = k - fl * 2 * M, m = ch % M, ri = ch / M;
    return __ldg(&sp[(((size_t)m * T + t) * F + f0 + fl) * 2 + ri]);
  };
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < K * T; i += blockDim.x) { const float v = feat(i % K, i / K); s1 += v; s2 += v * v; }
  const float2 tot = block_sum2(s1, s2, red);
  const float mean = tot.x / (float)(K * T);
  const float rstd = rsqrtf(fmaxf(tot.y / (float)(K * T) - mean * mean, 0.f) + eps);
  const int t0 = blockIdx.y * BS_TT;
  __syncthreads();
  for (int i = threadIdx.x; i < K * BS_TT; i += blockDim.x) {
    const int k = i / BS_TT, tt = i - k * BS_TT;
    sm[i] = t0 + tt < T ? (feat(k, t0 + tt) - mean) * rstd * gw[k] + gb[k] : 0.f;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc[BS_TT];
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = bias[c];
    for (int k = 0; k < K; ++k) {
      const float wv = __ldg(&Wt[(size_t)k * C + c]);
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = fmaf(wv, sm[k * BS_TT + tt], acc[tt]);
    }
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt)
      if (t0 + tt < T) x[(((size_t)b * T + t0 + tt) * nb + band) * C + c] = acc[tt];
  }
}

// x [B, T, nb, C] -> est [B, S, M, T, F, 2] (= input * mask when masking).  Per band: GroupNorm(1, C) over (C, T),
// Conv1d(C, 4C) -> tanh -> Conv1d(4C, 4C) -> Conv1d(4C, O_b) -> GLU (:221-236, :256-270, :175-182).
__global__ void __launch_bounds__(256) bs_decode_kernel(const float* __restrict__ x, const float* __restrict__ spec, int M,
                                                        int T, int F, int C, int nb, int S,
                                                        const long long* __restrict__ table, const float* __restrict__ w,
                                                        float* __restrict__ est, int masking, float eps) {
  extern __shared__ float sm[];           // xn [C][TT] | h1 [4C][TT] | h2 [4C][TT] | red
  const int band = blockIdx.x, b = blockIdx.z;
  const long long* tb = table + band * 16;
  const int f0 = (int)tb[0], wb = (int)tb[1];
  const int C4 = 4 * C, Q = wb * S * 2 * M;      // Q post-GLU channels, O = 2Q pre-GLU
  const float* gw = w + tb[6]; const float* gb = w + tb[7];
  const float* W1 = w + tb[8]; const float* b1 = w + tb[9];
  const float* W3 = w + tb[10]; const float* b3 = w + tb[11];
  const float* W4 = w + tb[12]; const float* b4 = w + tb[13];
  float* xn = sm; float* h1 = xn + (size_t)C * BS_TT; float* h2 = h1 + (size_t)C4 * BS_TT; float* red = h2 + (size_t)C4 * BS_TT;
  const float* xb = x + (size_t)b * T * nb * C + (size_t)band * C;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < C * T; i += blockDim.x) {
    const float v = __ldg(&xb[(size_t)(i / C) * nb * C + (i % C)]);
    s1 += v; s2 += v * v;
  }
  const float2 tot = block_sum2(s1, s2, red);
  const float mean = tot.x / (float)(C * T);
  const float rstd = rsqrtf(fmaxf(tot.y / (float)(C * T) - mean * mean, 0.f) + eps);
  const int t0 = blockIdx.y * BS_TT;
  __syncthreads();
  for (int i = threadIdx.x; i < C * BS_TT; i += blockDim.x) {
    const int c = i % C, tt = i / C;
    xn[c * BS_TT + tt] = t0 + tt < T ? (__ldg(&xb[(size_t)(t0 + tt) * nb * C + c]) - mean) * rstd * gw[c] + gb[c] : 0.f;
  }
  __syncthreads();
  auto dense = [&](const float* in, int K, const float* Wt, const float* bias, int N, float* out, bool tanh_act) {
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
      float acc[BS_TT];
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = bias[n];
      for (int k = 0; k < K; ++k) {
        const float wv = __ldg(&Wt[(size_t)k * N + n]);
#pragma unroll
        for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = fmaf(wv, in[k * BS_TT + tt], acc[tt]);
      }
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) out[n * BS_TT + tt] = tanh_act ? tanhf(acc[tt]) : acc[tt];
    }
    __syncthreads();
  };
  dense(xn, C, W1, b1, C4, h1, true);
  dense(h1, C4, W3, b3, C4, h2, false);
  // last layer + GLU + complex mask, one thread per (source, channel, bin): needs the re and im channels and their gates
  const int P = S * M * wb;
  for (int pidx = threadIdx.x; pidx < P; pidx += blockDim.x) {
    const int fl = pidx % wb, m = (pidx / wb) % M, s = pidx / (wb * M);
    const int q_re = ((0 * S + s) * M + m) * wb + fl, q_im = ((1 * S + s) * M + m) * wb + fl;
    float a_re[BS_TT], a_im[BS_TT], g_re[BS_TT], g_im[BS_TT];
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt) { a_re[tt] = b4[q_re]; a_im[tt] = b4[q_im]; g_re[tt] = b4[Q + q_re]; g_im[tt] = b4[Q + q_im]; }
    for (int k = 0; k < C4; ++k) {
      const float* wr = W4 + (size_t)k * 2 * Q;
      const float w0 = __ldg(&wr[q_re]), w1 = __ldg(&wr[q_im]), w2 = __ldg(&wr[Q + q_re]), w3 = __ldg(&wr[Q + q_im]);
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) {
        const float hv = h2[k * BS_TT + tt];
        a_re[tt] = fmaf(w0, hv, a_re[tt]); a_im[tt] = fmaf(w1, hv, a_im[tt]);
        g_re[tt] = fmaf(w2, hv, g_re[tt]); g_im[tt] = fmaf(w3, hv, g_im[tt]);
      }
    }
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt) {
      const int t = t0 + tt;
      if (t >= T) break;
      float re = a_re[tt] / (1.f + expf(-g_re[tt])), im = a_im[tt] / (1.f + expf(-g_im[tt]));   // GLU(dim=1)
      if (masking) {
        const float2 in = *reinterpret_cast<const float2*>(&spec[((((size_t)b * M + m) * T + t) * F + f0 + fl) * 2]);
        const float r2 = in.x * re - in.y * im, i2 = in.x * im + in.y * re;
        re = r2; im = i2;
      }
      *reinterpret_cast<float2*>(&est[(((((size_t)b * S + s) * M + m) * T + t) * F + f0 + fl) * 2]) = make_float2(re, im);
    }
  }
}

// ---- backward (training through autograd) ---------------------------------------------------------------------------
// Rows r = b * T + t of one band are stored densely per band in the backward workspace; the weight gradients are dense
// products over those B * T rows, one CTA per output tile (no atomics, deterministic), batched over the bands
// (grid.z = band).  An operand of band `band` (first bin f0, width w) starts at p + band * per_band + f0 * per_bin and
// has row stride ld0 + ldw * w.
struct BandMat {
  const float* p; long long per_band, per_bin; int ld0, ldw;
  __device__ __forceinline__ const float* base(int band, int f0) const { return p + band * per_band + (long long)f0 * per_bin; }
  __device__ __forceinline__ int ld(int w) const { return ld0 + ldw * w; }
};

// Recompute of the band decoder per (band, frame tile, sample) -- GroupNorm, W1 + tanh, W3, W4, GLU -- storing the rows of
// xn, h1 = tanh(.), h2 for the weight gradients, and dz = dL/d(W4 output) from dEst through the complex mask and the GLU.
__global__ void __launch_bounds__(256) bs_decode_bwd_rows_kernel(
    const float* __restrict__ x, const float* __restrict__ spec, const float* __restrict__ dest, int M, int T, int F, int C,
    int nb, int S, const long long* __restrict__ table, const float* __restrict__ w, int masking, float eps,
    float* __restrict__ xn_rows, float* __restrict__ h1_rows, float* __restrict__ h2_rows, float* __restrict__ dz_rows) {
  extern __shared__ float sm[];           // xn [C][TT] | h1 [4C][TT] | h2 [4C][TT] | red
  const int band = blockIdx.x, b = blockIdx.z;
  const long long* tb = table + band * 16;
  const int f0 = (int)tb[0], wb = (int)tb[1];
  const int C4 = 4 * C, Q = wb * S * 2 * M, O = 2 * Q;
  const long long R = (long long)gridDim.z * T;
  const float* gw = w + tb[6]; const float* gb = w + tb[7];
  const float* W1 = w + tb[8]; const float* b1 = w + tb[9];
  const float* W3 = w + tb[10]; const float* b3 = w + tb[11];
  const float* W4 = w + tb[12]; const float* b4 = w + tb[13];
  float* xn = sm; float* h1 = xn + (size_t)C * BS_TT; float* h2 = h1 + (size_t)C4 * BS_TT; float* red = h2 + (size_t)C4 * BS_TT;
  const float* xb = x + (size_t)b * T * nb * C + (size_t)band * C;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < C * T; i += blockDim.x) {
    const float v = __ldg(&xb[(size_t)(i / C) * nb * C + (i % C)]);
    s1 += v; s2 += v * v;
  }
  const float2 tot = block_sum2(s1, s2, red);
  const float mean = tot.x / (float)(C * T);
  const float rstd = rsqrtf(fmaxf(tot.y / (float)(C * T) - mean * mean, 0.f) + eps);
  const int t0 = blockIdx.y * BS_TT;
  const int nt = T - t0 < BS_TT ? T - t0 : BS_TT;
  const long long row0 = (long long)b * T + t0;
  __syncthreads();
  for (int i = threadIdx.x; i < C * BS_TT; i += blockDim.x) {
    const int c = i % C, tt = i / C;
    const float v = tt < nt ? (__ldg(&xb[(size_t)(t0 + tt) * nb * C + c]) - mean) * rstd * gw[c] + gb[c] : 0.f;
    xn[c * BS_TT + tt] = v;
    if (tt < nt) xn_rows[((size_t)band * R + row0 + tt) * C + c] = v;
  }
  __syncthreads();
  auto dense = [&](const float* in, int K, const float* Wt, const float* bias, int N, float* out, bool tanh_act, float* rows) {
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
      float acc[BS_TT];
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = bias[n];
      for (int k = 0; k < K; ++k) {
        const float wv = __ldg(&Wt[(size_t)k * N + n]);
#pragma unroll
        for (int tt = 0; tt < BS_TT; ++tt) acc[tt] = fmaf(wv, in[k * BS_TT + tt], acc[tt]);
      }
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) {
        const float v = tanh_act ? tanhf(acc[tt]) : acc[tt];
        out[n * BS_TT + tt] = v;
        if (tt < nt) rows[((size_t)band * R + row0 + tt) * N + n] = v;
      }
    }
    __syncthreads();
  };
  dense(xn, C, W1, b1, C4, h1, true, h1_rows);
  dense(h1, C4, W3, b3, C4, h2, false, h2_rows);
  float* dzb = dz_rows + R * (long long)f0 * S * 4 * M;    // this band's [R][O] block
  const int P = S * M * wb;
  for (int pidx = threadIdx.x; pidx < P; pidx += blockDim.x) {
    const int fl = pidx % wb, m = (pidx / wb) % M, s = pidx / (wb * M);
    const int q_re = ((0 * S + s) * M + m) * wb + fl, q_im = ((1 * S + s) * M + m) * wb + fl;
    float a_re[BS_TT], a_im[BS_TT], g_re[BS_TT], g_im[BS_TT];
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt) { a_re[tt] = b4[q_re]; a_im[tt] = b4[q_im]; g_re[tt] = b4[Q + q_re]; g_im[tt] = b4[Q + q_im]; }
    for (int k = 0; k < C4; ++k) {
      const float* wr = W4 + (size_t)k * 2 * Q;
      const float w0 = __ldg(&wr[q_re]), w1 = __ldg(&wr[q_im]), w2 = __ldg(&wr[Q + q_re]), w3 = __ldg(&wr[Q + q_im]);
#pragma unroll
      for (int tt = 0; tt < BS_TT; ++tt) {
        const float hv = h2[k * BS_TT + tt];
        a_re[tt] = fmaf(w0, hv, a_re[tt]); a_im[tt] = fmaf(w1, hv, a_im[tt]);
        g_re[tt] = fmaf(w2, hv, g_re[tt]); g_im[tt] = fmaf(w3, hv, g_im[tt]);
      }
    }
#pragma unroll
    for (int tt = 0; tt < BS_TT; ++tt) {
      if (tt >= nt) break;
      const int t = t0 + tt;
      const float2 g = *reinterpret_cast<const float2*>(&dest[(((((size_t)b * S + s) * M + m) * T + t) * F + f0 + fl) * 2]);
      float dr = g.x, di = g.y;
      if (masking) {            // est = in * y (complex): dy = conj(in) * dest
        const float2 in = *reinterpret_cast<const float2*>(&spec[((((size_t)b * M + m) * T + t) * F + f0 + fl) * 2]);
        const float r2 = in.x * dr + in.y * di, i2 = in.x * di - in.y * dr;
        dr = r2; di = i2;
      }
      const float sr = 1.f / (1.f + expf(-g_re[tt])), si = 1.f / (1.f + expf(-g_im[tt]));   // GLU: y = a * sigmoid(g)
      float* dzr = dzb + (row0 + tt) * O;
      dzr[q_re] = dr * sr; dzr[Q + q_re] = dr * a_re[tt] * sr * (1.f - sr);
      dzr[q_im] = di * si; dzr[Q + q_im] = di * a_im[tt] * si * (1.f - si);
    }
  }
}

// Data gradient of a band's 1x1 conv: D[r][k] = sum_n G[r][n] * Wt[k][n]  (Wt = the packed, transposed weight [K][N] at
// table entry widx), times (1 - H[r][k]^2) when H is given (through tanh).  K = k0 + kw * w, N = n0 + nw * w.
struct BsGemm { BandMat g, d, h; int k0, kw, n0, nw, widx; long long R; };
__global__ void __launch_bounds__(256) bs_gemm_nt_kernel(BsGemm p, const long long* __restrict__ table, const float* __restrict__ w) {
  __shared__ float Gs[16][65];
  __shared__ float Ws[16][65];
  const int band = blockIdx.z;
  const int f0 = (int)table[band * 16], wb = (int)table[band * 16 + 1];
  const int K = p.k0 + p.kw * wb, N = p.n0 + p.nw * wb;
  const int kb = blockIdx.y * 64;
  if (kb >= K) return;
  const long long rb = (long long)blockIdx.x * 64;
  const float* G = p.g.base(band, f0); const int ldg = p.g.ld(wb);
  float* D = const_cast<float*>(p.d.base(band, f0)); const int ldd = p.d.ld(wb);
  const float* Wt = w + table[band * 16 + p.widx];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  float acc[4][4] = {};
  for (int n0 = 0; n0 < N; n0 += 16) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = tid + 256 * q, rr = idx >> 4, nn = idx & 15;
      const long long r = rb + rr;
      Gs[nn][rr] = (r < p.R && n0 + nn < N) ? G[r * ldg + n0 + nn] : 0.f;
      Ws[nn][rr] = (kb + rr < K && n0 + nn < N) ? __ldg(&Wt[(size_t)(kb + rr) * N + n0 + nn]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int nn = 0; nn < 16; ++nn) {
      float a[4], bw[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = Gs[nn][ty * 4 + i]; bw[i] = Ws[nn][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bw[j], acc[i][j]);
    }
    __syncthreads();
  }
  const float* H = p.h.p ? p.h.base(band, f0) : nullptr; const int ldh = p.h.ld(wb);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long r = rb + ty * 4 + i;
    if (r >= p.R) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = kb + tx * 4 + j;
      if (k >= K) continue;
      float v = acc[i][j];
      if (H) { const float hv = H[r * ldh + k]; v *= 1.f - hv * hv; }
      D[r * ldd + k] = v;
    }
  }
}

// Weight gradient of a band's 1x1 conv over all B * T rows: dWt[k][n] = sum_r A[r][k] * G[r][n] (the packed transposed
// layout, table entry oidx) and the bias gradient db[n] = sum_r G[r][n] (entry bidx).  One CTA per 64 x 64 output tile.
struct BsWgrad { BandMat a, g; int k0, kw, n0, nw, oidx, bidx; long long R; };
__global__ void __launch_bounds__(256) bs_wgrad_kernel(BsWgrad p, const long long* __restrict__ table, float* __restrict__ dw) {
  __shared__ float As[16][64];
  __shared__ float Gs[16][64];
  const int band = blockIdx.z;
  const int f0 = (int)table[band * 16], wb = (int)table[band * 16 + 1];
  const int K = p.k0 + p.kw * wb, N = p.n0 + p.nw * wb;
  const int kb = blockIdx.y * 64, nb0 = blockIdx.x * 64;
  if (kb >= K || nb0 >= N) return;
  const float* A = p.a.base(band, f0); const int lda = p.a.ld(wb);
  const float* G = p.g.base(band, f0); const int ldg = p.g.ld(wb);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const bool bias_row = blockIdx.y == 0 && ty == 0;
  float acc[4][4] = {}, bacc[4] = {};
  for (long long r0 = 0; r0 < p.R; r0 += 16) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = tid + 256 * q, rr = idx >> 6, cc = idx & 63;
      const long long r = r0 + rr;
      As[rr][cc] = (r < p.R && kb + cc < K) ? A[r * lda + kb + cc] : 0.f;
      Gs[rr][cc] = (r < p.R && nb0 + cc < N) ? G[r * ldg + nb0 + cc] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < 16; ++rr) {
      float a[4], g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[rr][ty * 4 + i]; g[i] = Gs[rr][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], g[j], acc[i][j]);
      if (bias_row) {
#pragma unroll
        for (int j = 0; j < 4; ++j) bacc[j] += g[j];
      }
    }
    __syncthreads();
  }
  float* out = dw + table[band * 16 + p.oidx];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = kb + ty * 4 + i;
    if (k >= K) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = nb0 + tx * 4 + j;
      if (n < N) out[(size_t)k * N + n] = acc[i][j];
    }
  }
  if (bias_row) {
    float* ob = dw + table[band * 16 + p.bidx];
#pragma unroll
    for (int j = 0; j < 4; ++j) if (nb0 + tx * 4 + j < N) ob[nb0 + tx * 4 + j] = bacc[j];
  }
}

// GroupNorm(1, K) over (K, T) per (sample, band), y = xhat * gw + gb.  Pass 1, one CTA per (band, sample): mean / rstd of
// X and, when dY is given, S1 = sum dY * gw and S2 = sum dY * gw * xhat (double).  K = k0 + kw * w.
struct BsNorm { BandMat x, dy; int k0, kw, gidx; int T; };
__global__ void __launch_bounds__(256) bs_gn_sums_kernel(BsNorm p, const long long* __restrict__ table, const float* __restrict__ w,
                                                         float eps, float* __restrict__ stats /*[B][nb][2]*/,
                                                         double* __restrict__ sums /*[B][nb][2]*/) {
  __shared__ float red[64];
  __shared__ double dred[2][8];
  const int band = blockIdx.x, b = blockIdx.y, nbands = gridDim.x;
  const int f0 = (int)table[band * 16], wb = (int)table[band * 16 + 1];
  const int K = p.k0 + p.kw * wb;
  const float* X = p.x.base(band, f0) + (long long)b * p.T * p.x.ld(wb); const int ldx = p.x.ld(wb);
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < K * p.T; i += blockDim.x) { const float v = X[(long long)(i / K) * ldx + i % K]; s1 += v; s2 += v * v; }
  const float2 tot = block_sum2(s1, s2, red);
  const float mean = tot.x / (float)(K * p.T);
  const float rstd = rsqrtf(fmaxf(tot.y / (float)(K * p.T) - mean * mean, 0.f) + eps);
  if (threadIdx.x == 0) { stats[(b * nbands + band) * 2] = mean; stats[(b * nbands + band) * 2 + 1] = rstd; }
  if (p.dy.p == nullptr) return;
  const float* dY = p.dy.base(band, f0) + (long long)b * p.T * p.dy.ld(wb); const int ldy = p.dy.ld(wb);
  const float* gw = w + table[band * 16 + p.gidx];
  double a1 = 0.0, a2 = 0.0;
  for (int i = threadIdx.x; i < K * p.T; i += blockDim.x) {
    const int k = i % K; const long long t = i / K;
    const float d = dY[t * ldy + k] * gw[k], xh = (X[t * ldx + k] - mean) * rstd;
    a1 += d; a2 += (double)d * xh;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
  if ((threadIdx.x & 31) == 0) { dred[0][threadIdx.x >> 5] = a1; dred[1][threadIdx.x >> 5] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { t1 += dred[0][i]; t2 += dred[1][i]; }
    sums[(b * nbands + band) * 2] = t1; sums[(b * nbands + band) * 2 + 1] = t2;
  }
}

// Pass 2, a CTA per (band, 32 channels), 8 row lanes: dgw[k] = sum_r dY * xhat, dgb[k] = sum_r dY (entries gidx, gidx + 1),
// and, when dX is given, dX = rstd * (dY * gw - S1 / n - xhat * S2 / n), n = K * T.
__global__ void __launch_bounds__(256) bs_gn_bwd_kernel(BsNorm p, BandMat dxm, int B, const long long* __restrict__ table,
                                                        const float* __restrict__ w, const float* __restrict__ stats,
                                                        const double* __restrict__ sums, float* __restrict__ dw) {
  __shared__ float rw[8][33], rb[8][33];
  const int band = blockIdx.x, nbands = gridDim.x;
  const int f0 = (int)table[band * 16], wb = (int)table[band * 16 + 1];
  const int K = p.k0 + p.kw * wb;
  const int k = blockIdx.y * 32 + threadIdx.x;
  if (blockIdx.y * 32 >= K) return;
  const float* X = p.x.base(band, f0); const int ldx = p.x.ld(wb);
  const float* dY = p.dy.base(band, f0); const int ldy = p.dy.ld(wb);
  float* dX = dxm.p ? const_cast<float*>(dxm.base(band, f0)) : nullptr; const int ldd = dxm.ld(wb);
  const float gwk = k < K ? w[table[band * 16 + p.gidx] + k] : 0.f;
  const double n = (double)K * p.T;
  float aw = 0.f, ab = 0.f;
  if (k < K) {
    for (long long r = threadIdx.y; r < (long long)B * p.T; r += blockDim.y) {
      const int b = (int)(r / p.T);
      const float mean = stats[(b * nbands + band) * 2], rstd = stats[(b * nbands + band) * 2 + 1];
      const float xh = (X[r * ldx + k] - mean) * rstd, d = dY[r * ldy + k];
      aw = fmaf(d, xh, aw); ab += d;
      if (dX) {
        const float m1 = (float)(sums[(b * nbands + band) * 2] / n), m2 = (float)(sums[(b * nbands + band) * 2 + 1] / n);
        dX[r * ldd + k] = rstd * (d * gwk - m1 - xh * m2);
      }
    }
  }
  rw[threadIdx.y][threadIdx.x] = aw; rb[threadIdx.y][threadIdx.x] = ab;
  __syncthreads();
  if (threadIdx.y == 0 && k < K) {
    float sw = 0.f, sb = 0.f;
    for (int i = 0; i < (int)blockDim.y; ++i) { sw += rw[i][threadIdx.x]; sb += rb[i][threadIdx.x]; }
    dw[table[band * 16 + p.gidx] + k] = sw;
    dw[table[band * 16 + p.gidx + 1] + k] = sb;
  }
}

// Band-split input features, one CTA per (band, sample): xs[band block][r][k] = spec feature k = f_local * 2M + ch of
// frame t (row r = b * T + t), and xn = GroupNorm output (xhat * gw + gb) with the statistics of bs_gn_sums_kernel.
__global__ void __launch_bounds__(256) bs_split_rows_kernel(const float* __restrict__ spec, int M, int T, int F,
                                                            const long long* __restrict__ table, const float* __restrict__ w,
                                                            const float* __restrict__ stats, float* __restrict__ xs,
                                                            float* __restrict__ xn) {
  const int band = blockIdx.x, b = blockIdx.y, nbands = gridDim.x;
  const int f0 = (int)table[band * 16], wb = (int)table[band * 16 + 1], K = wb * 2 * M;
  const long long R = (long long)gridDim.y * T;
  const float* sp = spec + (size_t)b * M * T * F * 2;
  const float* gw = w + table[band * 16 + 2]; const float* gb = w + table[band * 16 + 3];
  float* xsb = xs + R * (long long)f0 * 2 * M + (long long)b * T * K;
  float* xnb = xn + R * (long long)f0 * 2 * M + (long long)b * T * K;
  for (int i = threadIdx.x; i < K * T; i += blockDim.x) {
    const int k = i % K, t = i / K;
    const int fl = k / (2 * M), ch = k - fl * 2 * M, m = ch % M, ri = ch / M;
    const float v = __ldg(&sp[(((size_t)m * T + t) * F + f0 + fl) * 2 + ri]);
    xsb[i] = v;
    if (stats) xnb[i] = (v - stats[(b * nbands + band) * 2]) * stats[(b * nbands + band) * 2 + 1] * gw[k] + gb[k];
  }
}

}  // namespace tfl
