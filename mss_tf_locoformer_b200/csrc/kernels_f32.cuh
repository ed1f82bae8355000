// fp32 CUDA-core kernels: the bandwidth-bound stages (STFT, encoder conv + gLN,
// RMSGroupNorm, decoder, iSTFT + OLA, segment stitch) used in BOTH precision modes, plus
// the fp32 tap-GEMM / attention kernels that make up TFL_PRECISION_FP32 (the <= 1e-4
// parity mode).  References are to /root/reference/models/mss_tflocoformer.py.
#pragma once
#include "common.cuh"

namespace tfl {

// ======================================================================================
// Shared-memory radix-2 FFT (decimation in time on bit-reversed input).
// tw[k] = exp(-2 pi i k / N), k < N/2.  All threads of the CTA participate.
// ======================================================================================
template <bool INVERSE>
__device__ __forceinline__ void fft_smem(float2* buf, const float2* __restrict__ tw, int n, int log_n) {
  for (int s = 1; s <= log_n; ++s) {
    const int half = 1 << (s - 1);
    for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
      const int j = i & (half - 1);
      const int a = ((i >> (s - 1)) << s) + j;
      const int b = a + half;
      float2 w = __ldg(&tw[j << (log_n - s)]);
      if (INVERSE) w.y = -w.y;
      const float2 u = buf[a], v = buf[b];
      const float tr = v.x * w.x - v.y * w.y, ti = v.x * w.y + v.y * w.x;
      buf[a] = make_float2(u.x + tr, u.y + ti);
      buf[b] = make_float2(u.x - tr, u.y - ti);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ int bitrev(int i, int log_n) { return (int)(__brev((unsigned)i) >> (32 - log_n)); }

// --------------------------------------------------------------------------------------
// K1 stft: reflect pad + periodic Hann + FFT, one CTA per frame; writes channels-last
// (re, im) so the reference's stack + transpose (:207-214) never exist.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stft_kernel(const float* __restrict__ audio, int n_samples, int n_fft,
                                                   int log_n, int hop, int n_frames,
                                                   const float2* __restrict__ tw, const float* __restrict__ win,
                                                   float* __restrict__ spec) {
  extern __shared__ float2 fbuf[];
  const int t = blockIdx.x, b = blockIdx.y;
  const float* a = audio + (size_t)b * n_samples;
  const int pad = n_fft >> 1;
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    int n = t * hop + i - pad;
    if (n < 0) n = -n;
    if (n >= n_samples) n = 2 * (n_samples - 1) - n;
    fbuf[bitrev(i, log_n)] = make_float2(__ldg(&a[n]) * __ldg(&win[i]), 0.f);
  }
  __syncthreads();
  fft_smem<false>(fbuf, tw, n_fft, log_n);
  const int n_freq = pad + 1;
  float2* out = reinterpret_cast<float2*>(spec) + ((size_t)b * n_frames + t) * n_freq;
  for (int k = threadIdx.x; k < n_freq; k += blockDim.x) out[k] = fbuf[k];
}

// --------------------------------------------------------------------------------------
// K7 istft_ola: one CTA per (run of ISTFT_RUN hop blocks, source, batch).  For each frame overlapping the
// run: Hermitian-extend, inverse FFT in smem, window, accumulate; then divide by the sum of squared windows
// and store (:56-75).  Output audio[src][b][n].  The inverse real FFT is ONE complex FFT of n_fft/2 points (even /
// odd samples as real / imaginary parts) in radix-4 passes: 5 passes of 256 four-point butterflies at n_fft 2048
// where the full-size radix-2 version ran 11 passes of 1024 butterflies.  A run of 8 blocks needs 8 + n_fft/hop - 1 inverse FFTs
// (9 at hop = n_fft/2) where one CTA per block needed n_fft/hop each (16): the FFT passes were what the
// kernel spent its time on (ncu r02: shared-memory pipe 99 % busy).  Frames are added in increasing
// order: deterministic.  Twiddles are staged in shared memory once per CTA.
// --------------------------------------------------------------------------------------
constexpr int ISTFT_RUN = 8;   // hop blocks per CTA (fewer when shared memory is short: very large hop_length)
template <bool INVERSE>
__device__ __forceinline__ void fft_smem_tw(float2* buf, const float2* tws, int n, int log_n) {
  for (int s = 1; s <= log_n; ++s) {
    const int half = 1 << (s - 1);
    for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
      const int j = i & (half - 1);
      const int a = ((i >> (s - 1)) << s) + j;
      const int b = a + half;
      float2 w = tws[j << (log_n - s)];
      if (INVERSE) w.y = -w.y;
      const float2 u = buf[a], v = buf[b];
      const float tr = v.x * w.x - v.y * w.y, ti = v.x * w.y + v.y * w.x;
      buf[a] = make_float2(u.x + tr, u.y + ti);
      buf[b] = make_float2(u.x - tr, u.y - ti);
    }
    __syncthreads();
  }
}

// Radix-4 decimation-in-time passes over bit-reversed input (two radix-2 stages per pass in registers: half the
// shared-memory traffic and barriers, 3 instead of 4 twiddle products per 4 points; one leading radix-2 pass when
// log_n is odd).  tws[m] = exp(-2 pi i m / (n << tw_shift)), first half of the circle.
template <bool INVERSE>
__device__ __forceinline__ void fft_smem_r4(float2* buf, const float2* tws, int n, int log_n, int tw_shift) {
  int s = 1;
  if (log_n & 1) {
    for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
      const float2 u = buf[2 * i], v = buf[2 * i + 1];
      buf[2 * i] = make_float2(u.x + v.x, u.y + v.y);
      buf[2 * i + 1] = make_float2(u.x - v.x, u.y - v.y);
    }
    __syncthreads();
    s = 2;
  }
  for (; s < log_n; s += 2) {                              // stages s and s + 1
    const int h = 1 << (s - 1);
    for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) {
      const int j = i & (h - 1);
      const int i0 = ((i >> (s - 1)) << (s + 1)) + j;
      float2 w = tws[(j << (log_n - s)) << tw_shift];      // exp(-2 pi i j / 2^s)
      float2 v = tws[(j << (log_n - s - 1)) << tw_shift];  // exp(-2 pi i j / 2^(s+1))
      if (INVERSE) { w.y = -w.y; v.y = -v.y; }
      const float2 x0 = buf[i0], x1 = buf[i0 + h], x2 = buf[i0 + 2 * h], x3 = buf[i0 + 3 * h];
      const float2 t1 = make_float2(x1.x * w.x - x1.y * w.y, x1.x * w.y + x1.y * w.x);
      const float2 t3 = make_float2(x3.x * w.x - x3.y * w.y, x3.x * w.y + x3.y * w.x);
      const float2 u0 = make_float2(x0.x + t1.x, x0.y + t1.y), u1 = make_float2(x0.x - t1.x, x0.y - t1.y);
      const float2 u2 = make_float2(x2.x + t3.x, x2.y + t3.y), u3 = make_float2(x2.x - t3.x, x2.y - t3.y);
      const float2 pp = make_float2(u2.x * v.x - u2.y * v.y, u2.x * v.y + u2.y * v.x);
      const float2 qq = make_float2(u3.x * v.x - u3.y * v.y, u3.x * v.y + u3.y * v.x);
      // second-stage twiddle of the odd pair: v * exp(-+ i pi / 2), i.e. qq * (-i) forward, qq * (+i) inverse
      const float2 q = INVERSE ? make_float2(-qq.y, qq.x) : make_float2(qq.y, -qq.x);
      buf[i0] = make_float2(u0.x + pp.x, u0.y + pp.y);
      buf[i0 + 2 * h] = make_float2(u0.x - pp.x, u0.y - pp.y);
      buf[i0 + h] = make_float2(u1.x + q.x, u1.y + q.y);
      buf[i0 + 3 * h] = make_float2(u1.x - q.x, u1.y - q.y);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) istft_ola_kernel(const float* __restrict__ est, int n_src, int n_frames,
                                                        int n_fft, int log_n, int hop, int n_samples,
                                                        const float2* __restrict__ tw,
                                                        const float* __restrict__ win, float* __restrict__ audio,
                                                        int batch, int run) {
  extern __shared__ float2 fbuf[];                       // n_fft | twiddles n_fft/2 | acc run*hop | env run*hop
  float2* tws = fbuf + n_fft;
  float* acc = reinterpret_cast<float*>(tws + (n_fft >> 1));
  const int span = run * hop;
  float* env = acc + span;
  const int m0 = blockIdx.x * run, src = blockIdx.y, b = blockIdx.z;
  const int pad = n_fft >> 1, n_freq = pad + 1;
  const int q_lo = m0 * hop + pad;                       // padded-signal coordinate of the run's first sample
  for (int i = threadIdx.x; i < (n_fft >> 1); i += blockDim.x) tws[i] = __ldg(&tw[i]);
  for (int i = threadIdx.x; i < span; i += blockDim.x) { acc[i] = 0.f; env[i] = 0.f; }
  int t_min = (q_lo - n_fft) / hop + 1;
  if (q_lo - n_fft < 0) t_min = 0;
  int t_max = (q_lo + span - 1) / hop;
  if (t_max > n_frames - 1) t_max = n_frames - 1;
  const float inv_n = 1.f / (float)n_fft;
  for (int t = t_min; t <= t_max; ++t) {
    const float2* x = reinterpret_cast<const float2*>(est) + (((size_t)b * n_src + src) * n_frames + t) * n_freq;
    __syncthreads();
    // Real output: one complex inverse FFT of HALF the size.  With E[k] = X[k] + conj(X[N/2 - k]) and
    // O[k] = (X[k] - conj(X[N/2 - k])) exp(+2 pi i k / N), z = IDFT_{N/2}(E + i O) holds z[n] = N (x[2n] + i x[2n+1]):
    // the frame's samples are the float view of fbuf.
    for (int k = threadIdx.x; k < pad; k += blockDim.x) {
      float2 a = __ldg(&x[k]), c = __ldg(&x[pad - k]);
      if (k == 0) { a.y = 0.f; c.y = 0.f; }                // irfft ignores the imaginary part of DC and Nyquist
      const float2 e = make_float2(a.x + c.x, a.y - c.y), d = make_float2(a.x - c.x, a.y + c.y);
      const float2 w = tws[k];                             // exp(-2 pi i k / N); O = d * conj(w)
      const float2 o = make_float2(d.x * w.x + d.y * w.y, d.y * w.x - d.x * w.y);
      fbuf[bitrev(k, log_n - 1)] = make_float2(e.x - o.y, e.y + o.x);
    }
    __syncthreads();
    fft_smem_r4<true>(fbuf, tws, pad, log_n - 1, 1);
    // samples of this frame that fall into the run: padded coordinate t * hop + off, off in [0, n_fft)
    const int lo = max(0, t * hop - q_lo), hi = min(span, t * hop + n_fft - q_lo);
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
      const int off = q_lo + i - t * hop;
      const float w = __ldg(&win[off]);
      acc[i] += reinterpret_cast<const float*>(fbuf)[off] * inv_n * w;
      env[i] += w * w;
    }
  }
  __syncthreads();
  float* out = audio + ((size_t)src * batch + b) * n_samples;
  for (int i = threadIdx.x; i < span; i += blockDim.x) {
    const int n = m0 * hop + i;
    if (n < n_samples) out[n] = acc[i] / env[i];
  }
}

// --------------------------------------------------------------------------------------
// K2 encoder: Conv2d(Cin, C, 3x3, pad 1) direct + per-sample sum / sum-of-squares
// partials (double) for the global layer norm (:141-146).  One thread per (position, 4
// channels); deterministic two-level reduction.
// --------------------------------------------------------------------------------------
template <int CIN>
__global__ void __launch_bounds__(256) enc_conv_kernel(const float* __restrict__ spec, int n_frames, int n_freq,
                                                       int C, const float* __restrict__ w /*[3][3][CIN][C]*/,
                                                       const float* __restrict__ bias, float* __restrict__ y,
                                                       double* __restrict__ partial /*[B][gridDim.x][2]*/) {
  extern __shared__ float wsm[];  // 9*CIN*C + C
  const int b = blockIdx.y;
  for (int i = threadIdx.x; i < 9 * CIN * C; i += blockDim.x) wsm[i] = w[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) wsm[9 * CIN * C + i] = bias[i];
  __syncthreads();
  const int c4n = C >> 2;
  const long long per_sample = (long long)n_frames * n_freq * c4n;
  const float* in = spec + (size_t)b * n_frames * n_freq * CIN;
  float* out = y + (size_t)b * n_frames * n_freq * C;
  double s1 = 0.0, s2 = 0.0;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < per_sample;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % c4n) << 2;
    const long long pos = idx / c4n;
    const int f = (int)(pos % n_freq), t = (int)(pos / n_freq);
    float4 a = *reinterpret_cast<const float4*>(&wsm[9 * CIN * C + c]);
#pragma unroll
    for (int dt = 0; dt < 3; ++dt) {
      const int tt = t + dt - 1;
      if (tt < 0 || tt >= n_frames) continue;
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        const int ff = f + df - 1;
        if (ff < 0 || ff >= n_freq) continue;
        const float* px = in + ((size_t)tt * n_freq + ff) * CIN;
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci) {
          const float xv = __ldg(&px[ci]);
          const float4 wv = *reinterpret_cast<const float4*>(&wsm[((dt * 3 + df) * CIN + ci) * C + c]);
          a.x = fmaf(xv, wv.x, a.x); a.y = fmaf(xv, wv.y, a.y);
          a.z = fmaf(xv, wv.z, a.z); a.w = fmaf(xv, wv.w, a.w);
        }
      }
    }
    *reinterpret_cast<float4*>(&out[pos * C + c]) = a;
    s1 += (double)a.x + (double)a.y + (double)a.z + (double)a.w;
    s2 += (double)a.x * a.x + (double)a.y * a.y + (double)a.z * a.z + (double)a.w * a.w;
  }
  __shared__ double r1[256], r2[256];
  r1[threadIdx.x] = s1; r2[threadIdx.x] = s2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) { r1[threadIdx.x] += r1[threadIdx.x + o]; r2[threadIdx.x] += r2[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2 + 0] = r1[0];
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2 + 1] = r2[0];
  }
}

// K2 (bf16 mode) on the warp-level tensor cores: M = 16 consecutive bins of a frame, N = C outputs in 8-wide
// n-tiles, K = 9 * CIN = 18 input taps padded to 24 (three m16n8k8 tf32 steps).  The CUDA-core kernel above issues
// 18 shared-memory weight reads per 72 FMAs and ran at 16 % of the HBM write peak (ncu r02); here a warp task costs
// ~50 MMAs and the kernel is bound by its 4 * N * C byte store.  tf32 rounding of the spectrogram and the weights
// (2^-11) -- TFL_PRECISION_BF16 only; the gLN statistics are accumulated in double from the fp32 accumulators.
// Weight rows in shared memory are padded to C + 8 floats: the four k rows a warp reads then fall into distinct banks.
// Two passes of the same kernel replace conv -> store -> gLN read-modify-write: PASS 0 only accumulates the statistics
// (nothing is stored: the conv costs ~50 MMAs per 16 bins), PASS 1 recomputes the conv and stores
// (v - mean) * rstd * gln_w + gln_b.  HBM traffic of the encoder: one 4 * N * C byte store instead of three passes.
template <int CIN, int PASS>
__global__ void __launch_bounds__(256) enc_conv_mma_kernel(const float* __restrict__ spec, int n_frames, int n_freq,
                                                           int C, const float* __restrict__ w /*[9*CIN][C]*/,
                                                           const float* __restrict__ bias, float* __restrict__ y,
                                                           double* __restrict__ partial /*[B][gridDim.x][2]*/,
                                                           const float* __restrict__ stats /*[B][2] mean, rstd*/,
                                                           const float* __restrict__ gw, const float* __restrict__ gb) {
  constexpr int KP = 24;                                      // 9 * CIN = 18 rounded up to a multiple of 8
  static_assert(9 * CIN <= KP, "tap count");
  extern __shared__ float wsm[];                              // [KP][C + 8] tf32-rounded, rows >= 9 * CIN zero; bias [C]; PASS 1: scale, shift [C]
  const int WP = C + 8;
  for (int i = threadIdx.x; i < KP * WP; i += blockDim.x) {
    const int k = i / WP, c = i - k * WP;
    wsm[i] = (k < 9 * CIN && c < C) ? __uint_as_float(to_tf32(w[k * C + c])) : 0.f;
  }
  float* bsm = wsm + KP * WP;
  const int b = blockIdx.y;
  float* scl = bsm + C;
  float* sft = scl + C;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    bsm[i] = bias[i];
    if (PASS == 1) { const float rstd = stats[b * 2 + 1]; scl[i] = rstd * gw[i]; sft[i] = gb[i] - stats[b * 2] * rstd * gw[i]; }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int g = lane >> 2, t4 = lane & 3;
  const int NG = (n_freq + 15) / 16;
  const long long n_tiles = (long long)n_frames * NG;
  const float* in = spec + (size_t)b * n_frames * n_freq * CIN;
  float* out = y + (size_t)b * n_frames * n_freq * C;
  double s1 = 0.0, s2 = 0.0;
  for (long long tile = (long long)blockIdx.x * wpb + warp; tile < n_tiles; tile += (long long)gridDim.x * wpb) {
    const int t = (int)(tile / NG), f0 = (int)(tile - (long long)t * NG) * 16;
    // A fragments: row position f0 + g (+ 8), k = 8 s + t4 (+ 4) -> tap k / CIN, channel k % CIN
    uint32_t a[3][4];
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int h = 0; h < 2; ++h) {                           // h: k-slot t4 / t4 + 4
        const int k = 8 * s + t4 + 4 * h;
        const int tap = k / CIN, ci = k - tap * CIN;
        const int dt = tap / 3, df = tap - dt * 3;
        const int tt = t + dt - 1;
#pragma unroll
        for (int r = 0; r < 2; ++r) {                         // r: tile row g / g + 8
          const int ff = f0 + g + 8 * r + df - 1;
          const bool ok = k < 9 * CIN && tt >= 0 && tt < n_frames && ff >= 0 && ff < n_freq;
          a[s][2 * h + r] = ok ? to_tf32(__ldg(&in[((size_t)tt * n_freq + ff) * CIN + ci])) : 0u;
        }
      }
    const bool va = f0 + g < n_freq, vb = f0 + g + 8 < n_freq;
    float* oa = out + ((size_t)t * n_freq + f0 + g) * C + 2 * t4;
    float* ob = oa + (size_t)8 * C;
    for (int j = 0; j < C / 8; ++j) {
      const float2 bb = *reinterpret_cast<const float2*>(bsm + 8 * j + 2 * t4);
      float acc[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const uint32_t b0 = __float_as_uint(wsm[(8 * s + t4) * WP + 8 * j + g]);
        const uint32_t b1 = __float_as_uint(wsm[(8 * s + t4 + 4) * WP + 8 * j + g]);
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
                     : "r"(a[s][0]), "r"(a[s][1]), "r"(a[s][2]), "r"(a[s][3]), "r"(b0), "r"(b1));
      }
      if (PASS == 0) {
        if (va) {
          s1 += (double)acc[0] + (double)acc[1];
          s2 += (double)acc[0] * acc[0] + (double)acc[1] * acc[1];
        }
        if (vb) {
          s1 += (double)acc[2] + (double)acc[3];
          s2 += (double)acc[2] * acc[2] + (double)acc[3] * acc[3];
        }
      } else {
        const float2 sc = *reinterpret_cast<const float2*>(scl + 8 * j + 2 * t4);
        const float2 sh = *reinterpret_cast<const float2*>(sft + 8 * j + 2 * t4);
        if (va) *reinterpret_cast<float2*>(oa + 8 * j) = make_float2(fmaf(acc[0], sc.x, sh.x), fmaf(acc[1], sc.y, sh.y));
        if (vb) *reinterpret_cast<float2*>(ob + 8 * j) = make_float2(fmaf(acc[2], sc.x, sh.x), fmaf(acc[3], sc.y, sh.y));
      }
    }
  }
  if (PASS != 0) return;
  __shared__ double r1[256], r2[256];
  r1[threadIdx.x] = s1; r2[threadIdx.x] = s2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) { r1[threadIdx.x] += r1[threadIdx.x + o]; r2[threadIdx.x] += r2[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2 + 0] = r1[0];
    partial[((size_t)b * gridDim.x + blockIdx.x) * 2 + 1] = r2[0];
  }
}

__global__ void gln_finalize_kernel(const double* __restrict__ partial, int n_part, double count, float eps,
                                    float* __restrict__ stats /*[B][2] mean, rstd*/) {
  const int b = blockIdx.x;
  __shared__ double r1[256], r2[256];
  double s1 = 0.0, s2 = 0.0;
  for (int i = threadIdx.x; i < n_part; i += blockDim.x) {
    s1 += partial[((size_t)b * n_part + i) * 2];
    s2 += partial[((size_t)b * n_part + i) * 2 + 1];
  }
  r1[threadIdx.x] = s1; r2[threadIdx.x] = s2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) { r1[threadIdx.x] += r1[threadIdx.x + o]; r2[threadIdx.x] += r2[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double mean = r1[0] / count;
    double var = r2[0] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    stats[b * 2] = (float)mean;
    stats[b * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
  }
}

__global__ void __launch_bounds__(256) gln_apply_kernel(float* __restrict__ x, long long per_sample4, int C,
                                                        const float* __restrict__ stats,
                                                        const float* __restrict__ gw, const float* __restrict__ gb) {
  const int b = blockIdx.y;
  const float mean = stats[b * 2], rstd = stats[b * 2 + 1];
  float4* p = reinterpret_cast<float4*>(x) + (size_t)b * per_sample4;
  const int c4n = C >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample4;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % c4n) << 2;
    float4 v = p[i];
    const float4 w = *reinterpret_cast<const float4*>(&gw[c]);
    const float4 bb = *reinterpret_cast<const float4*>(&gb[c]);
    v.x = (v.x - mean) * rstd * w.x + bb.x; v.y = (v.y - mean) * rstd * w.y + bb.y;
    v.z = (v.z - mean) * rstd * w.z + bb.z; v.w = (v.w - mean) * rstd * w.w + bb.w;
    p[i] = v;
  }
}

// --------------------------------------------------------------------------------------
// K3 rms_group_norm (:682-706): y = x / (||x_g|| * D^-1/2 + eps) * gamma.
// A sub-warp of W lanes owns one (row, group); each lane holds one 128-bit chunk.
// --------------------------------------------------------------------------------------
template <int W, typename OutT>
__global__ void __launch_bounds__(256) rms_group_norm_kernel(const float* __restrict__ x, OutT* __restrict__ y,
                                                             long long rows, int C, int G,
                                                             const float* __restrict__ gamma, float eps) {
  const int D = C / G, lanes = D >> 2;
  const float scale = rsqrtf((float)D);
  const int sub = threadIdx.x % W;
  const long long pairs = rows * G;
  const long long stride = (long long)gridDim.x * (blockDim.x / W);
  for (long long pr = (long long)blockIdx.x * (blockDim.x / W) + threadIdx.x / W;
       pr < ((pairs + stride - 1) / stride) * stride; pr += stride) {
    const bool active = pr < pairs && sub < lanes;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    long long off = 0;
    int c = 0;
    if (active) {
      const long long row = pr / G;
      c = (int)(pr % G) * D + (sub << 2);
      off = row * C + c;
      v = *reinterpret_cast<const float4*>(&x[off]);
    }
    float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
#pragma unroll
    for (int o = W >> 1; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o, W);
    if (active) {
      const float denom = sqrtf(ss) * scale + eps;
      const float4 g = *reinterpret_cast<const float4*>(&gamma[c]);
      const float o0 = v.x / denom * g.x, o1 = v.y / denom * g.y, o2 = v.z / denom * g.z, o3 = v.w / denom * g.w;
      if constexpr (sizeof(OutT) == 4) {
        *reinterpret_cast<float4*>(&y[off]) = make_float4(o0, o1, o2, o3);
      } else {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(&y[off]) = pk;
      }
    }
  }
}

// ======================================================================================
// fp32 tap-GEMM:  out[r, n] = bias[n] + sum_{tap, c} A[s, j + tap - padL, c] * W[tap][c][n]
// with flat row r = s * Sout + j and A rows outside [0, Sin) read as zero -- the exact
// zero padding the reference applies AFTER the norm (:640-644).  One kernel serves the
// conv1d (+SwiGLU epilogue), the transposed conv (+bias, +residual), the qkv projection
// (+RoPE epilogue) and the head-merge projection (+residual).
// ======================================================================================
struct TapGemm {
  const float* A; SeqMap amap; int Sin, Sout, padL, taps, Kc;
  const float* W; const float* bias; int N; long long M;
};

constexpr int GBM = 128, GBN = 128, GBK = 8;

struct EpiSwiGLU {  // columns are (value, gate) interleaved; writes hid[r][n/2]  (:648-649)
  float* hid; int H;
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float g = v[2 * i + 1]; o[i] = v[2 * i] * (g / (1.f + expf(-g))); }
    float* dst = hid + r * H + (n0 >> 1);
    if (n0 + 8 <= N) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
    else for (int i = 0; i < 4; ++i) if (n0 + 2 * i < N) dst[i] = o[i];
  }  // two adjacent columns (n even): the (value, gate) pair of one hidden channel -- the tf32 MMA kernel's epilogue unit
  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n < N) hid[r * H + (n >> 1)] = v0 * (v1 / (1.f + expf(-v1)));
  }
};

struct EpiResidual {  // x[s, j, n] += v   (:447, :456, :462)
  float* x; SeqMap omap;
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
    float* dst = x + omap.base(s) + (long long)j * omap.pos_stride + n0;
    if (n0 + 8 <= N) {
      float4 a = *reinterpret_cast<float4*>(dst), b = *reinterpret_cast<float4*>(dst + 4);
      a.x += v[0]; a.y += v[1]; a.z += v[2]; a.w += v[3];
      b.x += v[4]; b.y += v[5]; b.z += v[6]; b.w += v[7];
      *reinterpret_cast<float4*>(dst) = a; *reinterpret_cast<float4*>(dst + 4) = b;
    } else for (int i = 0; i < 8; ++i) if (n0 + i < N) dst[i] += v[i];
  }  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n >= N) return;
    float2* dst = reinterpret_cast<float2*>(x + omap.base(s) + (long long)j * omap.pos_stride + n);
    float2 a = *dst;
    a.x += v0; a.y += v1;
    *dst = a;
  }
};

struct EpiQkvRope {  // n -> (which, head, d); RoPE on q,k (interleaved pairs); out[which][s][head][j][d]
  float* qkv; int A, hd, heads, L, nseq; const float* freqs;  // freqs == nullptr -> "nope"
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      const int n = n0 + i;
      if (n >= N) break;
      const int which = n / A, rem = n - which * A, head = rem / hd, d = rem - head * hd;
      float a = v[i], b = v[i + 1];
      if (freqs != nullptr && which < 2) {
        const float ang = (float)j * __ldg(&freqs[d >> 1]);
        float sn, cs;
        sincosf(ang, &sn, &cs);
        const float ra = a * cs - b * sn, rb = b * cs + a * sn;
        a = ra; b = rb;
      }
      float* dst = qkv + ((((size_t)which * nseq + s) * heads + head) * L + j) * hd + d;
      *reinterpret_cast<float2*>(dst) = make_float2(a, b);
    }
  }  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n >= N) return;
    const int which = n / A, rem = n - which * A, head = rem / hd, d = rem - head * hd;
    float a = v0, b = v1;
    if (freqs != nullptr && which < 2) {
      float sn, cs;
      sincosf((float)j * __ldg(&freqs[d >> 1]), &sn, &cs);
      const float ra = a * cs - b * sn, rb = b * cs + a * sn;
      a = ra; b = rb;
    }
    *reinterpret_cast<float2*>(qkv + ((((size_t)which * nseq + s) * heads + head) * L + j) * hd + d) = make_float2(a, b);
  }
};

template <class Epi>
__global__ void __launch_bounds__(256) tap_gemm_kernel(TapGemm p, Epi epi) {
  __shared__ float As[2][GBK][GBM + 4];
  __shared__ float Bs[2][GBK][GBN];
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
  const int a_row = tid >> 1, a_kq = (tid & 1) << 2;
  const int b_row = tid >> 5, b_col = (tid & 31) << 2;
  const int kt_per_tap = p.Kc / GBK, n_kt = p.taps * kt_per_tap;
  const int my_s = row_s[a_row], my_j = row_j[a_row];
  const long long my_base = row_base[a_row];

  auto load_a = [&](int kt) -> float4 {
    const int tap = kt / kt_per_tap, c0 = (kt - tap * kt_per_tap) * GBK;
    const int pos = my_j + tap - p.padL;
    if (my_s < 0 || pos < 0 || pos >= p.Sin) return make_float4(0.f, 0.f, 0.f, 0.f);
    return __ldg(reinterpret_cast<const float4*>(p.A + my_base + (long long)pos * p.amap.pos_stride + c0 + a_kq));
  };
  auto load_b = [&](int kt) -> float4 {
    const int n = n0 + b_col;
    if (n >= p.N) return make_float4(0.f, 0.f, 0.f, 0.f);
    return __ldg(reinterpret_cast<const float4*>(p.W + ((size_t)kt * GBK + b_row) * p.N + n));
  };
  auto stash = [&](int buf, float4 a, float4 b) {
    As[buf][a_kq + 0][a_row] = a.x; As[buf][a_kq + 1][a_row] = a.y;
    As[buf][a_kq + 2][a_row] = a.z; As[buf][a_kq + 3][a_row] = a.w;
    *reinterpret_cast<float4*>(&Bs[buf][b_row][b_col]) = b;
  };

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const int ty = tid >> 4, tx = tid & 15;

  stash(0, load_a(0), load_b(0));
  __syncthreads();
  for (int kt = 0; kt < n_kt; ++kt) {
    const int cur = kt & 1;
    float4 na, nb;
    const bool more = kt + 1 < n_kt;
    if (more) { na = load_a(kt + 1); nb = load_b(kt + 1); }
#pragma unroll
    for (int k = 0; k < GBK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 8 + 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (more) stash(cur ^ 1, na, nb);
    __syncthreads();
  }
  const int nb0 = n0 + tx * 8;
  if (nb0 >= p.N) return;
  float bias[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) bias[j] = (p.bias != nullptr && nb0 + j < p.N) ? __ldg(&p.bias[nb0 + j]) : 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rl = ty * 8 + i;
    const int s = row_s[rl];
    if (s < 0) continue;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = acc[i][j] + bias[j];
    epi(s, row_j[rl], m0 + rl, nb0, p.N, v);
  }
}

// --------------------------------------------------------------------------------------
// fp32 attention (:523-531): softmax(q k^T / sqrt(hd)) v, online softmax, one thread per
// query, K/V tiles broadcast from shared memory.  q,k,v: [nseq][heads][L][hd].
// --------------------------------------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(128) attn_f32_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                       const float* __restrict__ v, float* __restrict__ o,
                                                       int L, int hd, int heads, float scale,
                                                       float* __restrict__ lse /* [nseq][heads][L] or nullptr (training) */) {
  constexpr int TK = 64, CH = 16;
  __shared__ float ks[TK][HD], vs[TK][HD];
  const int head = blockIdx.y, s = blockIdx.z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  float qr[HD], acc[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) { qr[d] = (i < L && d < hd) ? q[base + (size_t)i * hd + d] * scale : 0.f; acc[d] = 0.f; }
  float mx = -INFINITY, l = 0.f;
  for (int j0 = 0; j0 < L; j0 += TK) {
    __syncthreads();
    for (int e = threadIdx.x; e < TK * HD; e += blockDim.x) {
      const int jj = e / HD, d = e - jj * HD;
      const bool ok = (j0 + jj < L) && (d < hd);
      ks[jj][d] = ok ? k[base + (size_t)(j0 + jj) * hd + d] : 0.f;
      vs[jj][d] = ok ? v[base + (size_t)(j0 + jj) * hd + d] : 0.f;
    }
    __syncthreads();
    const int lim = min(TK, L - j0);
    for (int c0 = 0; c0 < lim; c0 += CH) {
      float sc[CH];
      float cm = -INFINITY;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        float dot = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) dot = fmaf(qr[d], ks[c0 + c][d], dot);
        sc[c] = (c0 + c < lim) ? dot : -INFINITY;
        cm = fmaxf(cm, sc[c]);
      }
      const float nm = fmaxf(mx, cm);
      const float corr = expf(mx - nm);
      l *= corr;
#pragma unroll
      for (int d = 0; d < HD; ++d) acc[d] *= corr;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const float pv = expf(sc[c] - nm);
        l += pv;
#pragma unroll
        for (int d = 0; d < HD; ++d) acc[d] = fmaf(pv, vs[c0 + c][d], acc[d]);
      }
      mx = nm;
    }
  }
  if (i < L) {
    const float inv = 1.f / l;
    float* dst = o + ((size_t)s * L + i) * ((size_t)heads * hd) + (size_t)head * hd;
#pragma unroll
    for (int d = 0; d < HD; ++d) if (d < hd) dst[d] = acc[d] * inv;
    if (lse != nullptr) lse[((size_t)s * heads + head) * L + i] = mx + logf(l);
  }
}

// --------------------------------------------------------------------------------------
// K6 decoder: ConvTranspose2d(C, 2S, 3x3, pad 1) as a 9-tap gather (:182).  One warp per group of
// DEC_P consecutive bins of one frame, lanes over channels: every weight vector read from shared
// memory (conflict-free float4) feeds DEC_P positions (the kernel was bound by those reads at one
// position per warp) and the three frequency taps share the DEC_P + 2 input columns.  The
// DEC_P * 8 partial sums per lane are reduced by a transposing butterfly (31 shuffles; lane l ends
// with the total of value l = position * 8 + output).  Writes est[b][src][t][f][re/im].
// wd layout: [9 taps][8 outputs][C] (tap = dt*3+df multiplies x[t+1-dt, f+1-df]).
// --------------------------------------------------------------------------------------
constexpr int DEC_P = 4;
__global__ void __launch_bounds__(256, 2) dec_conv_kernel(const float* __restrict__ x, int n_frames, int n_freq, int C,
                                                       int n_out, const float* __restrict__ wd,
                                                       const float* __restrict__ bias, float* __restrict__ est,
                                                       long long n_pos) {
  extern __shared__ float wsm[];  // 9*8*C
  for (int i = threadIdx.x; i < 9 * C * 8; i += blockDim.x) wsm[i] = wd[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int n_src = n_out >> 1;
  const int NG = (n_freq + DEC_P - 1) / DEC_P;                 // groups per frame
  const long long n_groups = (n_pos / n_freq) * NG;
  for (long long grp = (long long)blockIdx.x * wpb + warp; grp < n_groups; grp += (long long)gridDim.x * wpb) {
    const long long bt = grp / NG;
    const int f0 = (int)(grp - bt * NG) * DEC_P;
    const int t = (int)(bt % n_frames), b = (int)(bt / n_frames);
    float acc[DEC_P * 8];
#pragma unroll
    for (int k = 0; k < DEC_P * 8; ++k) acc[k] = 0.f;
    for (int c = lane << 2; c < C; c += 128) {
#pragma unroll
      for (int dt = 0; dt < 3; ++dt) {
        const int tt = t + 1 - dt;
        if (tt < 0 || tt >= n_frames) continue;
        const float* px = x + (((size_t)b * n_frames + tt) * n_freq) * C + c;
        float4 xv[DEC_P + 2];                                  // columns f0 - 1 .. f0 + DEC_P
#pragma unroll
        for (int j = 0; j < DEC_P + 2; ++j) {
          const int ff = f0 - 1 + j;
          xv[j] = (ff >= 0 && ff < n_freq) ? __ldg(reinterpret_cast<const float4*>(px + (size_t)ff * C))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int df = 0; df < 3; ++df) {
          const float* pw = wsm + (dt * 3 + df) * 8 * C + c;
#pragma unroll
          for (int o = 0; o < 8; ++o) {
            const float4 w = *reinterpret_cast<const float4*>(pw + o * C);
#pragma unroll
            for (int pi = 0; pi < DEC_P; ++pi) {               // position f0 + pi reads column f0 + pi + 1 - df
              const float4 v = xv[pi + 2 - df];
              acc[pi * 8 + o] = fmaf(v.x, w.x, fmaf(v.y, w.y, fmaf(v.z, w.z, fmaf(v.w, w.w, acc[pi * 8 + o]))));
            }
          }
        }
      }
    }
    // transposing butterfly: after the step with offset s, a lane keeps the half of its values whose index bit
    // log2(s) equals its own lane bit
#pragma unroll
    for (int s = 16, n = DEC_P * 8; s >= 1; s >>= 1, n >>= 1) {
      const bool up = (lane & s) != 0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (i < (n >> 1)) {
          const float keep = up ? acc[i + (n >> 1)] : acc[i];
          const float send = up ? acc[i] : acc[i + (n >> 1)];
          acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
      }
    }
    static_assert(DEC_P * 8 == 32, "one reduced value per lane");
    const int pi = lane >> 3, o = lane & 7, f = f0 + pi;
    if (f < n_freq && o < n_out) {
      const int src = o >> 1, ri = o & 1;
      est[(((((size_t)b * n_src + src) * n_frames + t) * n_freq + f) << 1) + ri] = acc[0] + __ldg(&bias[o]);
    }
  }
}

// --------------------------------------------------------------------------------------
// K6 (bf16 mode) decoder on the warp-level tensor cores: the transposed conv is an implicit GEMM with
// M = positions, N = 8 outputs, K = 9 taps x C -- N = 8 is exactly mma.sync m16n8k8 (tf32 operands, fp32
// accumulation), a shape the M >= 64 / N >= 16 tcgen05 path cannot use without 2-8x padding.  The CUDA-core
// kernel above is bound by its shared-memory weight reads and FMA issue together (1.6 ms, ncu r02); here a
// warp owns 16 consecutive bins of one frame and spends 2 global loads + 1 shared load per two MMAs.
// K order inside an MMA is free (a sum over channels): lane (g, t) feeds channels 4t .. 4t+3 of a
// 16-channel step as k-slots (t, t+4) of two MMAs, so x and w arrive as 128-bit loads.
// Operands are rounded to tf32 (cvt.rna): relative error 2^-11 per product, ~25 dB below the bf16 rounding of
// the blocks that feed this layer -- used in TFL_PRECISION_BF16 only; fp32 mode keeps dec_conv_kernel.
// wd layout: [9 taps][8 outputs][C] (tap = dt*3+df multiplies x[t+1-dt, f+1-df]).
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dec_conv_mma_kernel(const float* __restrict__ x, int n_frames, int n_freq, int C,
                                                           int n_out, const float* __restrict__ wd,
                                                           const float* __restrict__ bias, float* __restrict__ est,
                                                           long long n_rows /* B * Tf */) {
  extern __shared__ float wsm[];  // 9*8*C, tf32-rounded
  for (int i = threadIdx.x; i < 9 * C * 8; i += blockDim.x) wsm[i] = __uint_as_float(to_tf32(wd[i]));
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int g = lane >> 2, t4 = lane & 3;
  const int n_src = n_out >> 1;
  const int NG = (n_freq + 15) / 16;                           // 16-bin tiles per frame
  // A block works on a patch of wpb consecutive frames x 16 bins, one frame per warp: the three time taps of
  // neighbouring frames then hit the same SM's L1 (with frames spread over blocks every x row came from L2 three
  // times and the kernel was L2-bandwidth bound: 0.99 ms).
  const int TG = (n_frames + wpb - 1) / wpb;                   // frame groups per sample
  const long long n_patches = (n_rows / n_frames) * TG * NG;
  const float b0 = 2 * t4 < n_out ? __ldg(&bias[2 * t4]) : 0.f, b1 = 2 * t4 + 1 < n_out ? __ldg(&bias[2 * t4 + 1]) : 0.f;
  for (long long patch = blockIdx.x; patch < n_patches; patch += gridDim.x) {
    const int f0 = (int)(patch % NG) * 16;
    const long long r = patch / NG;
    const int t = (int)(r % TG) * wpb + warp, b = (int)(r / TG);
    if (t >= n_frames) continue;
    float acc[4] = {b0, b1, b0, b1};                           // rows g and g + 8, outputs 2 t4, 2 t4 + 1
#pragma unroll 1
    for (int dt = 0; dt < 3; ++dt) {
      const int tt = t + 1 - dt;
      if (tt < 0 || tt >= n_frames) continue;
      const float* prow = x + (((size_t)b * n_frames + tt) * n_freq) * C;
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        const int fa = f0 + g + 1 - df, fb = fa + 8;           // input bins of tile rows g and g + 8
        const bool va = fa >= 0 && fa < n_freq, vb = fb >= 0 && fb < n_freq;
        const float* pa = prow + (size_t)(va ? fa : 0) * C + 4 * t4;
        const float* pb = prow + (size_t)(vb ? fb : 0) * C + 4 * t4;
        const float* pw = wsm + ((dt * 3 + df) * 8 + g) * C + 4 * t4;
#pragma unroll 4
        for (int c0 = 0; c0 < C; c0 += 16) {
          const float4 xa = va ? __ldg(reinterpret_cast<const float4*>(pa + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
          const float4 xb = vb ? __ldg(reinterpret_cast<const float4*>(pb + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
          const float4 w = *reinterpret_cast<const float4*>(pw + c0);
          asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
                       : "r"(to_tf32(xa.x)), "r"(to_tf32(xb.x)), "r"(to_tf32(xa.y)), "r"(to_tf32(xb.y)),
                         "r"(__float_as_uint(w.x)), "r"(__float_as_uint(w.y)));
          asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(acc[0]), "+f"(acc[1]), "+f"(acc[2]), "+f"(acc[3])
                       : "r"(to_tf32(xa.z)), "r"(to_tf32(xb.z)), "r"(to_tf32(xa.w)), "r"(to_tf32(xb.w)),
                         "r"(__float_as_uint(w.z)), "r"(__float_as_uint(w.w)));
        }
      }
    }
    if (2 * t4 < n_out) {
      const int src = t4;                                      // outputs (2 src, 2 src + 1) = (re, im) of source src
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int f = f0 + g + 8 * h;
        if (f < n_freq)
          *reinterpret_cast<float2*>(est + ((((size_t)b * n_src + src) * n_frames + t) * n_freq + f) * 2) =
              make_float2(acc[2 * h], acc[2 * h + 1]);
      }
    }
  }
}

// --------------------------------------------------------------------------------------
// K6 (bf16 mode, C in {32, 64, 96, 128}) decoder in SCATTER form: every input position is read from HBM exactly once.
// A transposed conv is a scatter: position (ti, fi) sends P[(dt, df, o)] = W[tap = dt*3+df][o] . x[ti, fi, :] to
// output (ti - 1 + dt, fi - 1 + df, o).  P is one GEMM with M = positions, N = 72 (9 taps x 8 outputs), K = C:
// the same 144 mma.sync m16n8k8 (tf32) per 16 positions as the gather kernel above, but 16 instead of 144 128-bit
// global loads per thread -- the gather kernel fetched every x row for each of the 9 taps (L1 / L2 line lookups
// bound it at 0.97 ms for 1.09 GB).
// A block owns a strip of <= 126 output bins (128 input bins, one 16-bin tile per warp) and a run of output frames
// [ta, tb); it walks the input frames ta-1 .. tb in order and adds every warp's P into three rolling output-frame
// accumulators in shared memory ([frame % 3][source][bin], initialised to the bias).  One pass per frequency tap df
// (the three time taps of a pass land in different frames, so all targets of a pass are distinct; __syncthreads
// between passes), so the summation order of every output is fixed: input frames ascending, df ascending --
// deterministic and independent of the batch index and of how frames / bins were split into runs / strips.  After
// input frame ti the output frame ti - 1 is complete: written out ([B, S, Tf, F, 2], 8 bytes per lane, contiguous
// per source) and its accumulator reset.
// x rows are prefetched one frame ahead in 32-channel chunks (register ring of NCH = C / 32 chunks, refilled chunk
// by chunk as the MMAs consume them): 3/4 of a 16-bin tile (6 KB) is in flight per warp at any time.
// wd layout: [9 taps][8 outputs][C] as above; shared copy [72][C + 16] (the 16-word pad makes the 128-bit B-fragment
// loads of a quarter warp conflict-free).
// --------------------------------------------------------------------------------------
constexpr int DEC_WB = 132;   // accumulator bins per (frame, source): 130 used; 2 * DEC_WB % 32 == 8 keeps the RMW conflict-free
constexpr int DEC_WOUT = 126; // complete output bins of a 128-bin input strip
template <int NCH>
__global__ void __launch_bounds__(256, 2) dec_conv_scatter_kernel(const float* __restrict__ x, int n_batch, int n_frames,
                                                                  int n_freq, int n_out, const float* __restrict__ wd,
                                                                  const float* __restrict__ bias, float* __restrict__ est,
                                                                  int NS, int WOUT, int NR, int R) {
  constexpr int C = 32 * NCH, WS = C + 16;
  extern __shared__ float dsm[];
  float* wsm = dsm;                                            // [72][WS] tf32
  float2* accs = reinterpret_cast<float2*>(dsm + 72 * WS);     // [3][4][DEC_WB]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t4 = lane & 3;
  const int n_src = n_out >> 1;
  for (int i = tid; i < 72 * C; i += 256) wsm[(i / C) * WS + (i % C)] = __uint_as_float(to_tf32(wd[i]));
  // flush / reset mapping: thread (source fs, j) owns accumulator bins 2 + j and 66 + j (+ one of the four unused edge bins)
  const int fs = tid >> 6, fj = tid & 63;
  const float2 fbias = make_float2(2 * fs < n_out ? __ldg(&bias[2 * fs]) : 0.f, 2 * fs + 1 < n_out ? __ldg(&bias[2 * fs + 1]) : 0.f);
  for (int sl = 0; sl < 3; ++sl) {
    float2* a = accs + (sl * 4 + fs) * DEC_WB;
    a[2 + fj] = fbias; a[66 + fj] = fbias;
    if (fj < 4) a[fj < 2 ? fj : 128 + fj] = fbias;
  }
  __syncthreads();
  const long long n_items = (long long)n_batch * NS * NR;
  for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int run = (int)(item % NR), strip = (int)((item / NR) % NS), b = (int)(item / ((long long)NR * NS));
    const int ta = run * R, tb = min(ta + R, n_frames);
    if (ta >= n_frames) continue;
    const int o0 = strip * WOUT, wout = min(WOUT, n_freq - o0), i0 = o0 - 1;   // input bins i0 .. i0 + wout + 1
    if (wout <= 0) continue;
    const int ra = 16 * warp + g, rb = ra + 8;                 // tile rows of this lane; accumulator bin = row + df
    const int fa = i0 + ra, fb = i0 + rb;
    const bool va = fa >= 0 && fa < n_freq && ra < wout + 2, vb = fb >= 0 && fb < n_freq && rb < wout + 2;
    const bool active = 16 * warp < wout + 2 && i0 + 16 * warp < n_freq;      // warp-uniform
    const int t_first = max(ta - 1, 0), t_last = min(tb, n_frames - 1);
    const float* xa0 = x + (((size_t)b * n_frames) * n_freq + (va ? fa : 0)) * C + 4 * t4;
    const float* xb0 = x + (((size_t)b * n_frames) * n_freq + (vb ? fb : 0)) * C + 4 * t4;
    const size_t fstride = (size_t)n_freq * C;
    float4 X[NCH][4];                                          // [chunk][row a: 2 steps of 16 channels, row b: 2 steps]
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto ld_chunk = [&](int j, int ti) {
      const float* pa = xa0 + (size_t)ti * fstride + 32 * j;
      const float* pb = xb0 + (size_t)ti * fstride + 32 * j;
      X[j][0] = va ? __ldg(reinterpret_cast<const float4*>(pa)) : z4;
      X[j][1] = va ? __ldg(reinterpret_cast<const float4*>(pa + 16)) : z4;
      X[j][2] = vb ? __ldg(reinterpret_cast<const float4*>(pb)) : z4;
      X[j][3] = vb ? __ldg(reinterpret_cast<const float4*>(pb + 16)) : z4;
    };
    if (active) {
#pragma unroll
      for (int j = 0; j < NCH; ++j) ld_chunk(j, t_first);
    }
    for (int ti = t_first; ti <= t_last; ++ti) {
      bool use[3];                                             // output frame ti - 1 + dt belongs to this run
#pragma unroll
      for (int dt = 0; dt < 3; ++dt) use[dt] = ti - 1 + dt >= ta && ti - 1 + dt < tb;
      float acc[9][4];
#pragma unroll
      for (int nt = 0; nt < 9; ++nt) { acc[nt][0] = 0.f; acc[nt][1] = 0.f; acc[nt][2] = 0.f; acc[nt][3] = 0.f; }
      if (active) {
#pragma unroll
        for (int j = 0; j < NCH; ++j) {
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const float4 xa = X[j][s], xb = X[j][2 + s];
            const uint32_t a0 = to_tf32(xa.x), a1 = to_tf32(xb.x), a2 = to_tf32(xa.y), a3 = to_tf32(xb.y);
            const uint32_t c0 = to_tf32(xa.z), c1 = to_tf32(xb.z), c2 = to_tf32(xa.w), c3 = to_tf32(xb.w);
            const float* pw = wsm + g * WS + 32 * j + 16 * s + 4 * t4;
#pragma unroll
            for (int nt = 0; nt < 9; ++nt) {
              if (use[nt / 3]) {
                const float4 w = *reinterpret_cast<const float4*>(pw + nt * 8 * WS);
                asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                             : "+f"(acc[nt][0]), "+f"(acc[nt][1]), "+f"(acc[nt][2]), "+f"(acc[nt][3])
                             : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(__float_as_uint(w.x)), "r"(__float_as_uint(w.y)));
                asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                             : "+f"(acc[nt][0]), "+f"(acc[nt][1]), "+f"(acc[nt][2]), "+f"(acc[nt][3])
                             : "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(__float_as_uint(w.z)), "r"(__float_as_uint(w.w)));
              }
            }
          }
          if (ti < t_last) ld_chunk(j, ti + 1);                // refill the chunk just consumed with the next input frame
        }
      }
      // scatter: one pass per frequency tap; within a pass every (frame, source, bin) target is distinct
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        if (active) {
#pragma unroll
          for (int dt = 0; dt < 3; ++dt) {
            if (use[dt]) {
              float2* a = accs + (((ti + 2 + dt) % 3) * 4 + t4) * DEC_WB + df;   // frame ti - 1 + dt, source t4
              float2 u = a[ra], v = a[rb];
              u.x += acc[dt * 3 + df][0]; u.y += acc[dt * 3 + df][1];
              v.x += acc[dt * 3 + df][2]; v.y += acc[dt * 3 + df][3];
              a[ra] = u; a[rb] = v;
            }
          }
        }
        __syncthreads();
      }
      // output frame ti - 1 is complete (and output frame n_frames - 1 after the last input frame)
      for (int to = ti - 1; to <= (ti == n_frames - 1 ? ti : ti - 1); ++to) {
        if (to < ta || to >= tb) continue;
        float2* a = accs + ((to % 3) * 4 + fs) * DEC_WB;
        float* eo = est + ((((size_t)b * n_src + fs) * n_frames + to) * n_freq + o0) * 2;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int lo = fj + 64 * h;                          // output bin o0 + lo lives in accumulator bin 2 + lo
          const float2 v = a[2 + lo];
          if (lo < wout && fs < n_src) *reinterpret_cast<float2*>(eo + 2 * lo) = v;
          a[2 + lo] = fbias;
        }
        if (fj < 4) a[fj < 2 ? fj : 128 + fj] = fbias;
      }
      __syncthreads();
    }
  }
}

// --------------------------------------------------------------------------------------
// Full-track stitch: track[src][s0 + m] += w(m) * seg[src][b][m] (oracle/stitch.py; new
// behaviour, SURVEY.md F3).  Periodic-Hann cross-fade, flat outer edges.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) segment_ola_kernel(const float* __restrict__ seg, int n_src, int batch,
                                                          int seg_len, int seg_index0, int n_seg_total,
                                                          float* __restrict__ track, long long n_track,
                                                          long long track_origin) {
  const int b = blockIdx.y, src = blockIdx.z;
  const int gi = seg_index0 + b;
  const long long start = (long long)gi * (seg_len >> 1) - track_origin;   // `track` starts at sample track_origin
  const float* in = seg + ((size_t)src * batch + b) * seg_len;
  float* out = track + (size_t)src * n_track;
  const int half = seg_len >> 1;
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < seg_len; m += gridDim.x * blockDim.x) {
    const long long t = start + m;
    if (t >= n_track) break;
    if (t < 0) continue;
    float w = 0.5f - 0.5f * cospif(2.0f * (float)m / (float)seg_len);
    if ((gi == 0 && m < half) || (gi == n_seg_total - 1 && m >= half)) w = 1.f;
    atomicAdd(&out[t], w * in[m]);  // two addends per sample at most: order-independent in fp32
  }
}

// --------------------------------------------------------------------------------------
// Full-track stitch at any hop (oracle/stitch.py stitch_segments_hop), in gather form:
//   track[src][c][t] += sum_{i in this call, covering t} w_i(t - i*hop) * seg[src][(i - i0)*C + c][t - i*hop] / E(t),
//   E(t) = sum_{i covering t} w_i(t - i*hop) over the whole segment grid (closed form, <= ceil(L/hop) terms).
// One thread owns one output sample: it adds this call's segments in index order and writes once -- no
// atomics, so the result is bitwise reproducible for a given batch size at any overlap.  `seg` is the
// model's output [S][batch*C][L] read in place (row = segment * C + channel); `track` is [S][C][n_track]
// holding samples [track_origin, track_origin + n_track) of the full track.
// --------------------------------------------------------------------------------------
__device__ __forceinline__ float segment_window(long long i, int m, int seg_len, int n_seg) {
  if ((i == 0 && m < (seg_len >> 1)) || (i == n_seg - 1 && m >= (seg_len >> 1))) return 1.f;
  return 0.5f - 0.5f * cospif(2.0f * (float)m / (float)seg_len);
}

__global__ void __launch_bounds__(256) segment_ola_hop_kernel(const float* __restrict__ seg, int channels, int batch,
                                                              int seg_len, int hop, int seg_index0, int n_seg_total,
                                                              float* __restrict__ track, long long n_track,
                                                              long long track_origin, long long j0, long long j1) {
  const long long j = j0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= j1) return;
  const int src = blockIdx.y / channels, c = blockIdx.y - src * channels;
  const long long t = track_origin + j;
  const long long first = t >= seg_len ? (t - seg_len) / hop + 1 : 0;        // segments covering t: first .. last
  const long long last = min(t / hop, (long long)n_seg_total - 1);
  const float* in = seg + (size_t)src * batch * channels * seg_len;
  float e = 0.f, acc = 0.f;
  for (long long i = first; i <= last; ++i) {
    const int m = (int)(t - i * hop);
    const float w = segment_window(i, m, seg_len, n_seg_total);
    e += w;
    const long long k = i - seg_index0;
    if (k >= 0 && k < batch) acc += w * in[((size_t)k * channels + c) * seg_len + m];
  }
  float* out = track + ((size_t)src * channels + c) * n_track + j;
  *out += acc / e;
}

// --------------------------------------------------------------------------------------
// Pair statistics for the evaluation metrics (evaluation/metrics.py:14-168): per row r of two
// [rows, n] signals, out[r] = {sum e, sum t, sum e*e, sum t*t, sum e*t} in double.  Every metric of
// that file (SI-SDR, SDR, "SAR", "SIR") is a closed form of these five sums, so a track never has
// to leave the device to be scored.  Deterministic: fixed grid, block partials, ordered finish.
// --------------------------------------------------------------------------------------
constexpr int STATS_BLOCKS = 64;
__global__ void __launch_bounds__(256) pair_stats_partial_kernel(const float* __restrict__ est, const float* __restrict__ tgt,
                                                                 long long n, double* __restrict__ partial /*[rows][blocks][5]*/) {
  const int row = blockIdx.y;
  const float* e = est + (size_t)row * n;
  const float* t = tgt + (size_t)row * n;
  double s[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double a = (double)e[i], b = (double)t[i];
    s[0] += a; s[1] += b; s[2] += a * a; s[3] += b * b; s[4] += a * b;
  }
  __shared__ double red[5][256];
#pragma unroll
  for (int k = 0; k < 5; ++k) red[k][threadIdx.x] = s[k];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
#pragma unroll
      for (int k = 0; k < 5; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x < 5) partial[((size_t)row * gridDim.x + blockIdx.x) * 5 + threadIdx.x] = red[threadIdx.x][0];
}
__global__ void pair_stats_finish_kernel(const double* __restrict__ partial, int n_blocks, double* __restrict__ out /*[rows][5]*/) {
  const int row = blockIdx.x, k = threadIdx.x;
  if (k >= 5) return;
  double s = 0.0;
  for (int b = 0; b < n_blocks; ++b) s += partial[((size_t)row * n_blocks + b) * 5 + k];
  out[(size_t)row * 5 + k] = s;
}

}  // namespace tfl
