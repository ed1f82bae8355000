// Backward (training) kernels of the fp32 path: SURVEY.md section 8(f) row N1 -- the gradient of
// TFLocoformerMSS.forward + MSSLoss (/root/reference/training/train.py:68-172, /root/reference/models/mss_loss.py:18-244)
// as hand-written CUDA.  Every data-gradient GEMM reuses tap_gemm_kernel (kernels_f32.cuh) with a transposed weight
// and a new epilogue; the kernels here are what has no forward counterpart:
//   tap_wgrad_kernel          weight gradients: out[tap][i][n] += sum_rows A[row + tap][i] * B[row][n]
//   colsum_kernel             bias gradients
//   rms_group_norm_bwd_kernel RMSGroupNorm backward (+ gamma gradient), accumulating into the residual gradient
//   attn_bwd_dq / _dkv        softmax attention backward from the saved log-sum-exp (flash-attention style recompute)
//   qkv_unrope_kernel         inverse RoPE + regather of (dq, dk, dv) into GEMM rows
//   dec_dgrad / dec_wgrad     ConvTranspose2d decoder backward
//   enc_gln_bwd_* / enc_wgrad encoder GroupNorm(1, C) + Conv2d backward (weights only: the mixture needs no gradient)
//   istft_bwd_kernel          adjoint of iSTFT + overlap-add + envelope normalisation
//   loss kernels              SI-SDR + L1 + log-magnitude STFT loss and its gradient w.r.t. the separated audio
//   sqnorm / adamw            gradient clipping (torch.nn.utils.clip_grad_norm_) and torch.optim.AdamW
//   ordered_sum_kernel        second stage of every reduction of the deterministic mode
// All fp32 on CUDA cores.  By default the reductions over rows end in fp32 / double atomics, so their result depends on
// the order the blocks finish in (the last bits).  The kernels with a `DET` template switch (TFL_OPT_DETERMINISTIC)
// instead reduce inside a block in a fixed order and store one partial per block or row split; ordered_sum_kernel adds the
// partials in index order.  Every other reduction here is atomic-free and already fixed-order.
#pragma once
#include "kernels_f32.cuh"

namespace tfl {

// ---- tap-GEMM epilogues of the backward pass -------------------------------------------------------------------------
struct EpiStoreDense {  // out[r][n] = v
  float* out;
  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n < N) *reinterpret_cast<float2*>(out + r * N + n) = make_float2(v0, v1);
  }
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
    float* dst = out + r * N + n0;
    if (n0 + 8 <= N) {
      *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
    } else for (int i = 0; i < 8; ++i) if (n0 + i < N) dst[i] = v[i];
  }
};

struct EpiStoreMap {  // out[s, j, n] = v (rows addressed through a SeqMap, e.g. the channels-last residual layout)
  float* out; SeqMap omap;
  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n < N) *reinterpret_cast<float2*>(out + omap.base(s) + (long long)j * omap.pos_stride + n) = make_float2(v0, v1);
  }
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
    float* dst = out + omap.base(s) + (long long)j * omap.pos_stride + n0;
    if (n0 + 8 <= N) {
      *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
    } else for (int i = 0; i < 8; ++i) if (n0 + i < N) dst[i] = v[i];
  }
};

// Recomputes h = conv1d(norm(x)) (columns are (value, gate) interleaved) and, from dG = dL/d(value * silu(gate)):
//   hid[r][h] = value * silu(gate)                      (the hidden activation, for the transposed-conv weight gradient)
//   dh[r][2h] = dG * silu(gate),  dh[r][2h+1] = dG * value * silu'(gate)      (models/mss_tflocoformer.py:648-649)
struct EpiSwiGLUBwd {
  const float* dg; float* hid; float* dh; int H;
  __device__ __forceinline__ void pair(int s, int j, long long r, int n, int N, float v0, float v1) const {
    if (n >= N) return;
    const float sig = 1.f / (1.f + expf(-v1));
    const float silu = v1 * sig;
    const float d = dg[r * H + (n >> 1)];
    hid[r * H + (n >> 1)] = v0 * silu;
    *reinterpret_cast<float2*>(dh + r * N + n) = make_float2(d * silu, d * v0 * (sig * (1.f + v1 * (1.f - sig))));
  }
  __device__ __forceinline__ void operator()(int s, int j, long long r, int n0, int N, const float* v) const {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int n = n0 + 2 * i;
      if (n >= N) break;
      const float val = v[2 * i], gate = v[2 * i + 1];
      const float sig = 1.f / (1.f + expf(-gate));
      const float silu = gate * sig;
      const float d = dg[r * H + (n >> 1)];
      hid[r * H + (n >> 1)] = val * silu;
      dh[r * N + n] = d * silu;
      dh[r * N + n + 1] = d * val * (sig * (1.f + gate * (1.f - sig)));
    }
  }
};

// ---- deterministic mode: out[b][i] += sum over r = 0 .. n_rows - 1 of part[b][r][i], r ascending ----------------------
// One kernel serves every reduction of the mode: the per-split slabs of the weight-gradient GEMMs, the per-block partials
// of the bias, gamma, decoder and encoder gradients (float) and of the encoder statistics and loss rows (double).
template <class T>
__global__ void __launch_bounds__(256) ordered_sum_kernel(const T* __restrict__ part, int n_rows, long long row_stride,
                                                          long long width, long long part_bstride, T* __restrict__ out,
                                                          long long out_bstride) {
  const T* pb = part + (size_t)blockIdx.y * part_bstride;
  T* ob = out + (size_t)blockIdx.y * out_bstride;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < width; i += (long long)gridDim.x * blockDim.x) {
    T acc = 0;
    for (int r = 0; r < n_rows; ++r) acc += pb[(size_t)r * row_stride + i];
    ob[i] += acc;
  }
}

// ---- weight gradients ---------------------------------------------------------------------------------------------
// out[tap][i][n] += sum over rows r = (s, j), j in [0, Sout): A[s, j + tap - padL, i] * B[s, j, n]
// (A rows outside [0, Sin) are the zero padding).  Grid: x = tap * tiles_i * tiles_n, y = row splits; every block
// reduces its slice of the rows into a 128 x 128 register-tiled accumulator and adds it to `out` with fp32 atomics, or
// (DET) stores it into the slab of its split, out[split][tap][i][n], for ordered_sum_kernel.  Every split owns at least
// one row, so the splits of a tile together write every slab entry.
struct TapWgrad {
  const float* A; SeqMap amap; int Sin, padL, taps, Kc;
  const float* B; SeqMap bmap; int Sout, N;
  long long R;            // rows = nseq * Sout
  float* out;             // [taps][Kc][N]  (DET: [splits][taps][Kc][N])
  long long rows_per_split;
};

// the epilogue store of the three weight-gradient kernels: slab base of (split, tap), then add or store
template <bool DET>
__device__ __forceinline__ float* wgrad_out(const TapWgrad& p, int tap) {
  return p.out + ((size_t)(DET ? blockIdx.y * p.taps : 0) + tap) * p.Kc * p.N;
}
template <bool DET>
__device__ __forceinline__ void wgrad_put(float* o, float v) {
  if (DET) *o = v; else atomicAdd(o, v);
}
template <bool DET>
__device__ __forceinline__ void wgrad_put2(float* o, float v0, float v1) {   // o 8-byte aligned (n even, N % 4 == 0)
  if (DET) *reinterpret_cast<float2*>(o) = make_float2(v0, v1);
  else { atomicAdd(o, v0); atomicAdd(o + 1, v1); }
}

template <bool DET>
__global__ void __launch_bounds__(256) tap_wgrad_kernel(TapWgrad p) {
  __shared__ float As[2][GBK][GBM];
  __shared__ float Bs[2][GBK][GBN];
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
  const int l_row = tid >> 5, l_col = (tid & 31) << 2;   // this thread stages row l_row (of 8), columns l_col .. +3
  auto load = [&](long long r0, float4& a, float4& b) {
    a = make_float4(0.f, 0.f, 0.f, 0.f); b = a;
    const long long r = r0 + l_row;
    if (r >= r_hi) return;
    const int s = (int)(r / p.Sout), j = (int)(r - (long long)s * p.Sout);
    const int pos = j + tap - p.padL;
    if (pos >= 0 && pos < p.Sin && i0 + l_col < p.Kc)
      a = __ldg(reinterpret_cast<const float4*>(p.A + p.amap.base(s) + (long long)pos * p.amap.pos_stride + i0 + l_col));
    if (n0 + l_col < p.N)
      b = __ldg(reinterpret_cast<const float4*>(p.B + p.bmap.base(s) + (long long)j * p.bmap.pos_stride + n0 + l_col));
  };
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const int ty = tid >> 4, tx = tid & 15;
  float4 a, b;
  load(r_lo, a, b);
  *reinterpret_cast<float4*>(&As[0][l_row][l_col]) = a;
  *reinterpret_cast<float4*>(&Bs[0][l_row][l_col]) = b;
  __syncthreads();
  int cur = 0;
  for (long long r0 = r_lo; r0 < r_hi; r0 += GBK) {
    const bool more = r0 + GBK < r_hi;
    if (more) load(r0 + GBK, a, b);
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
    if (more) {
      *reinterpret_cast<float4*>(&As[cur ^ 1][l_row][l_col]) = a;
      *reinterpret_cast<float4*>(&Bs[cur ^ 1][l_row][l_col]) = b;
    }
    __syncthreads();
    cur ^= 1;
  }
  float* o = wgrad_out<DET>(p, tap);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ii = i0 + ty * 8 + i;
    if (ii >= p.Kc) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int nn = n0 + tx * 8 + j;
      if (nn < p.N) wgrad_put<DET>(&o[(size_t)ii * p.N + nn], acc[i][j]);
    }
  }
}

// out[n] += sum over rows (s, j) of B[s, j, n]   (bias gradients).  One thread per column group of 4, blocks over rows.
// DET: the rows_par row lanes of a block keep their sums apart in shared memory ([rows_par][N]), are added in lane order,
// and the block stores its column sums into out[block][n] for ordered_sum_kernel.
template <bool DET>
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ B, SeqMap bmap, int Sout, int N, long long R,
                                                     float* __restrict__ out) {
  extern __shared__ float cs_sm[];   // [N]  (DET: [rows_par][N])
  const int n4 = N >> 2;
  const int lanes = n4 < 256 ? n4 : 256;             // threads along the columns
  const int rows_par = 256 / lanes;                  // rows handled in parallel by one block
  for (int i = threadIdx.x; i < (DET ? rows_par : 1) * N; i += blockDim.x) cs_sm[i] = 0.f;
  __syncthreads();
  const int col = (threadIdx.x % lanes), rsub = threadIdx.x / lanes;
  // every block owns a contiguous run of rows; (sequence, position) is carried along it instead of divided out per row
  const long long chunk = (R + gridDim.x - 1) / gridDim.x;
  const long long r_lo = (long long)blockIdx.x * chunk, r_hi = r_lo + chunk < R ? r_lo + chunk : R;
  if (rsub < rows_par && r_lo + rsub < r_hi) {
    for (int c4 = col; c4 < n4; c4 += lanes) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      long long r = r_lo + rsub;
      int s = (int)(r / Sout), j = (int)(r - (long long)s * Sout);
      long long base = bmap.base(s);
      for (; r < r_hi; r += rows_par) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(B + base + (long long)j * bmap.pos_stride + 4 * c4));
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        j += rows_par;
        if (j >= Sout) {
          do { j -= Sout; ++s; } while (j >= Sout);
          base = bmap.base(s);
        }
      }
      if (DET) {
        *reinterpret_cast<float4*>(&cs_sm[(size_t)rsub * N + 4 * c4]) = acc;
      } else {
        atomicAdd(&cs_sm[4 * c4], acc.x); atomicAdd(&cs_sm[4 * c4 + 1], acc.y);
        atomicAdd(&cs_sm[4 * c4 + 2], acc.z); atomicAdd(&cs_sm[4 * c4 + 3], acc.w);
      }
    }
  }
  __syncthreads();
  if (DET) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      float s = 0.f;
      for (int q = 0; q < rows_par; ++q) s += cs_sm[(size_t)q * N + i];
      out[(size_t)blockIdx.x * N + i] = s;
    }
  } else {
    for (int i = threadIdx.x; i < N; i += blockDim.x) atomicAdd(&out[i], cs_sm[i]);
  }
}

// ---- RMSGroupNorm backward (models/mss_tflocoformer.py:682-706) ----------------------------------------------------
// y_c = x_c / r * gamma_c,  r = ||x_g|| / sqrt(D) + eps.  With dot = sum_c gamma_c dy_c x_c over the group:
//   dx_c = gamma_c dy_c / r - x_c * dot / (r^2 * ||x_g|| * sqrt(D)),   dgamma_c += dy_c x_c / r.
// dx_total (in place) += dx: the incoming gradient of the residual stream passes through unchanged.
// DET: the launcher makes the pair stride a multiple of G, so every slot of W threads keeps one group's channels in
// registers; the slots' sums meet in shared memory ([slots][D]) and are added in slot order into dgamma[block][C], the
// block's partial for ordered_sum_kernel.
template <int W, bool DET>
__global__ void __launch_bounds__(256) rms_group_norm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                                 float* __restrict__ dx_total, long long rows, int C, int G,
                                                                 const float* __restrict__ gamma, float eps,
                                                                 float* __restrict__ dgamma) {
  extern __shared__ float gsm[];   // [C]
  for (int i = threadIdx.x; i < C; i += blockDim.x) gsm[i] = 0.f;
  __syncthreads();
  const int D = C / G, lanes = D >> 2;
  const float rsD = rsqrtf((float)D);
  const int sub = threadIdx.x % W;
  const long long pairs = rows * G;
  const long long stride = (long long)gridDim.x * (blockDim.x / W);
  // a thread keeps the same channels for all of its rows when the stride is a multiple of G: gamma gradient in registers
  const bool fixed_c = stride % G == 0;
  float4 ga = make_float4(0.f, 0.f, 0.f, 0.f);
  int c_fixed = -1;
  for (long long pr = (long long)blockIdx.x * (blockDim.x / W) + threadIdx.x / W;
       pr < ((pairs + stride - 1) / stride) * stride; pr += stride) {
    const bool active = pr < pairs && sub < lanes;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f), d = v, g = v;
    long long off = 0;
    int c = 0;
    if (active) {
      const long long row = pr / G;
      c = (int)(pr % G) * D + (sub << 2);
      off = row * C + c;
      v = *reinterpret_cast<const float4*>(&x[off]);
      d = *reinterpret_cast<const float4*>(&dy[off]);
      g = *reinterpret_cast<const float4*>(&gamma[c]);
    }
    float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    float dot = g.x * d.x * v.x + g.y * d.y * v.y + g.z * d.z * v.z + g.w * d.w * v.w;
#pragma unroll
    for (int o = W >> 1; o > 0; o >>= 1) {
      ss += __shfl_xor_sync(0xffffffffu, ss, o, W);
      dot += __shfl_xor_sync(0xffffffffu, dot, o, W);
    }
    if (active) {
      const float nrm = sqrtf(ss);
      const float r = nrm * rsD + eps;
      const float inv_r = 1.f / r;
      const float k2 = nrm > 0.f ? dot * rsD / (r * r * nrm) : 0.f;
      float4 t = *reinterpret_cast<float4*>(&dx_total[off]);
      t.x += g.x * d.x * inv_r - v.x * k2; t.y += g.y * d.y * inv_r - v.y * k2;
      t.z += g.z * d.z * inv_r - v.z * k2; t.w += g.w * d.w * inv_r - v.w * k2;
      *reinterpret_cast<float4*>(&dx_total[off]) = t;
      if (fixed_c) {
        c_fixed = c;
        ga.x = fmaf(d.x * v.x, inv_r, ga.x); ga.y = fmaf(d.y * v.y, inv_r, ga.y);
        ga.z = fmaf(d.z * v.z, inv_r, ga.z); ga.w = fmaf(d.w * v.w, inv_r, ga.w);
      } else {
        atomicAdd(&gsm[c], d.x * v.x * inv_r); atomicAdd(&gsm[c + 1], d.y * v.y * inv_r);
        atomicAdd(&gsm[c + 2], d.z * v.z * inv_r); atomicAdd(&gsm[c + 3], d.w * v.w * inv_r);
      }
    }
  }
  if (DET) {
    const int slots = blockDim.x / W, slot = threadIdx.x / W;
    __syncthreads();
    if (sub < lanes) *reinterpret_cast<float4*>(&gsm[slot * D + (sub << 2)]) = ga;   // zero for a slot without rows
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
      const int grp = i / D;
      float s = 0.f;
      for (int q = 0; q < slots; ++q)
        if ((int)(((long long)blockIdx.x * slots + q) % G) == grp) s += gsm[q * D + i - grp * D];
      dgamma[(size_t)blockIdx.x * C + i] = s;
    }
    return;
  }
  if (c_fixed >= 0) {
    atomicAdd(&gsm[c_fixed], ga.x); atomicAdd(&gsm[c_fixed + 1], ga.y);
    atomicAdd(&gsm[c_fixed + 2], ga.z); atomicAdd(&gsm[c_fixed + 3], ga.w);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(&dgamma[i], gsm[i]);
}

// ---- attention backward (models/mss_tflocoformer.py:523-531) -----------------------------------------------------------
// q, k, v: [nseq][heads][L][hd] (q, k RoPE-rotated);  o, dO: [(s, i)][heads * hd];  lse[s][head][i] = log sum_j exp(s_ij),
// s_ij = scale * q_i . k_j.  With P_ij = exp(s_ij - lse_i), D_i = dO_i . O_i:
//   dV_j = sum_i P_ij dO_i,   dS_ij = P_ij (dO_i . V_j - D_i),   dQ_i = scale * sum_j dS_ij K_j,   dK_j = scale * sum_i dS_ij Q_i.
// One thread per query (dq kernel: also writes D) / per key (dkv kernel); the other side is staged in shared memory.
template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dq_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                          const float* __restrict__ v, const float* __restrict__ o,
                                                          const float* __restrict__ dO, const float* __restrict__ lse,
                                                          float* __restrict__ dq, float* __restrict__ Dbuf,
                                                          int L, int hd, int heads, float scale) {
  constexpr int TK = 64;
  __shared__ float ks[TK][HD], vs[TK][HD];
  const int head = blockIdx.y, s = blockIdx.z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const bool live = i < L;
  float qr[HD], dor[HD], acc[HD];
  float Di = 0.f, li = 0.f;
  {
    const size_t orow = ((size_t)s * L + (live ? i : 0)) * ((size_t)heads * hd) + (size_t)head * hd;
#pragma unroll
    for (int d = 0; d < HD; ++d) {
      const bool ok = live && d < hd;
      qr[d] = ok ? q[base + (size_t)i * hd + d] * scale : 0.f;
      dor[d] = ok ? dO[orow + d] : 0.f;
      const float ov = ok ? o[orow + d] : 0.f;
      Di = fmaf(dor[d], ov, Di);
      acc[d] = 0.f;
    }
    if (live) {
      li = lse[((size_t)s * heads + head) * L + i];
      Dbuf[((size_t)s * heads + head) * L + i] = Di;
    }
  }
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
    for (int c = 0; c < lim; ++c) {
      float sc = 0.f, dp = 0.f;
#pragma unroll
      for (int d = 0; d < HD; ++d) { sc = fmaf(qr[d], ks[c][d], sc); dp = fmaf(dor[d], vs[c][d], dp); }
      const float ds = expf(sc - li) * (dp - Di);
#pragma unroll
      for (int d = 0; d < HD; ++d) acc[d] = fmaf(ds, ks[c][d], acc[d]);
    }
  }
  if (live) {
#pragma unroll
    for (int d = 0; d < HD; ++d) if (d < hd) dq[base + (size_t)i * hd + d] = acc[d] * scale;
  }
}

template <int HD>
__global__ void __launch_bounds__(128) attn_bwd_dkv_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                           const float* __restrict__ v, const float* __restrict__ dO,
                                                           const float* __restrict__ lse, const float* __restrict__ Dbuf,
                                                           float* __restrict__ dk, float* __restrict__ dv,
                                                           int L, int hd, int heads, float scale) {
  constexpr int TQ = 64;
  __shared__ float qs[TQ][HD], dos[TQ][HD];
  __shared__ float ls[TQ], Ds[TQ];
  const int head = blockIdx.y, s = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const size_t base = ((size_t)s * heads + head) * (size_t)L * hd;
  const bool live = j < L;
  float kr[HD], vr[HD], dkr[HD], dvr[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) {
    const bool ok = live && d < hd;
    kr[d] = ok ? k[base + (size_t)j * hd + d] : 0.f;
    vr[d] = ok ? v[base + (size_t)j * hd + d] : 0.f;
    dkr[d] = 0.f; dvr[d] = 0.f;
  }
  for (int i0 = 0; i0 < L; i0 += TQ) {
    __syncthreads();
    for (int e = threadIdx.x; e < TQ * HD; e += blockDim.x) {
      const int ii = e / HD, d = e - ii * HD;
      const bool ok = (i0 + ii < L) && (d < hd);
      qs[ii][d] = ok ? q[base + (size_t)(i0 + ii) * hd + d] * scale : 0.f;
      dos[ii][d] = ok ? dO[((size_t)s * L + i0 + ii) * ((size_t)heads * hd) + (size_t)head * hd + d] : 0.f;
    }
    for (int e = threadIdx.x; e < TQ; e += blockDim.x) {
      const bool ok = i0 + e < L;
      ls[e] = ok ? lse[((size_t)s * heads + head) * L + i0 + e] : 0.f;
      Ds[e] = ok ? Dbuf[((size_t)s * heads + head) * L + i0 + e] : 0.f;
    }
    __syncthreads();
    const int lim = min(TQ, L - i0);
    for (int c = 0; c < lim; ++c) {
      float sc = 0.f, dp = 0.f;
#pragma unroll
      for (int d = 0; d < HD; ++d) { sc = fmaf(qs[c][d], kr[d], sc); dp = fmaf(dos[c][d], vr[d], dp); }
      const float pij = expf(sc - ls[c]);
      const float ds = pij * (dp - Ds[c]);
#pragma unroll
      for (int d = 0; d < HD; ++d) { dvr[d] = fmaf(pij, dos[c][d], dvr[d]); dkr[d] = fmaf(ds, qs[c][d], dkr[d]); }
    }
  }
  if (live) {
#pragma unroll
    for (int d = 0; d < HD; ++d)
      if (d < hd) {   // qs carries the softmax scale already: dK_j = sum_i dS_ij * (scale * Q_i)
        dk[base + (size_t)j * hd + d] = dkr[d];
        dv[base + (size_t)j * hd + d] = dvr[d];
      }
  }
}

// (dq, dk, dv)[which][s][head][j][d] -> rows of the q|k|v GEMM output gradient dQKV[(s, j)][which * A + head * hd + d],
// with the RoPE rotation of q and k undone (the transpose of a rotation: angle -> -angle; :550-559).
__global__ void __launch_bounds__(256) qkv_unrope_kernel(const float* __restrict__ dqkv_h, float* __restrict__ dqkv,
                                                         int nseq, int heads, int L, int hd, const float* __restrict__ freqs) {
  const int A = heads * hd;
  const long long total = (long long)3 * nseq * heads * L * (hd >> 1);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int dp = (int)(r % (hd >> 1)); r /= (hd >> 1);
    const int j = (int)(r % L); r /= L;
    const int head = (int)(r % heads); r /= heads;
    const int s = (int)(r % nseq);
    const int which = (int)(r / nseq);
    const float2 g = *reinterpret_cast<const float2*>(dqkv_h + 2 * idx);
    float a = g.x, b = g.y;
    if (freqs != nullptr && which < 2) {
      float sn, cs;
      sincosf((float)j * __ldg(&freqs[dp]), &sn, &cs);
      const float ra = a * cs + b * sn, rb = b * cs - a * sn;
      a = ra; b = rb;
    }
    *reinterpret_cast<float2*>(dqkv + ((size_t)s * L + j) * (3 * A) + (size_t)which * A + head * hd + 2 * dp) = make_float2(a, b);
  }
}

// ---- decoder backward (ConvTranspose2d(C, 2S, 3x3, pad 1), :182) -------------------------------------------------------
// forward: est[o][t, f] = b[o] + sum_{dt, df, c} wd[dt*3+df][o][c] * x[t+1-dt, f+1-df][c]
// dgrad:   dx[tt, ff][c] = sum_{dt, df, o} wd[dt*3+df][o][c] * dEst[o][tt-1+dt, ff-1+df]
__global__ void __launch_bounds__(256) dec_dgrad_kernel(const float* __restrict__ dest, int n_frames, int n_freq, int C, int n_out,
                                                        const float* __restrict__ wd, float* __restrict__ dx, long long n_pos) {
  extern __shared__ float wsm[];  // 9*8*C
  for (int i = threadIdx.x; i < 9 * C * 8; i += blockDim.x) wsm[i] = wd[i];
  __syncthreads();
  const int c4n = C >> 2, n_src = n_out >> 1;
  const long long total = n_pos * c4n;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % c4n) << 2;
    const long long pos = idx / c4n;
    const int ff = (int)(pos % n_freq);
    const long long bt = pos / n_freq;
    const int tt = (int)(bt % n_frames), b = (int)(bt / n_frames);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int dt = 0; dt < 3; ++dt) {
      const int t = tt - 1 + dt;
      if (t < 0 || t >= n_frames) continue;
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        const int f = ff - 1 + df;
        if (f < 0 || f >= n_freq) continue;
        for (int o = 0; o < n_out; ++o) {
          const float g = __ldg(&dest[(((((size_t)b * n_src + (o >> 1)) * n_frames + t) * n_freq + f) << 1) + (o & 1)]);
          const float4 w = *reinterpret_cast<const float4*>(&wsm[((dt * 3 + df) * 8 + o) * C + c]);
          a.x = fmaf(g, w.x, a.x); a.y = fmaf(g, w.y, a.y); a.z = fmaf(g, w.z, a.z); a.w = fmaf(g, w.w, a.w);
        }
      }
    }
    *reinterpret_cast<float4*>(&dx[pos * C + c]) = a;
  }
}

// wgrad: gw[dt*3+df][o][c] += sum_{b, tt, ff} x[tt, ff][c] * dEst[o][tt-1+dt, ff-1+df]
// Thread = channel (blockDim.x == C rounded up to a warp multiple), blocks over positions; 72 accumulators per thread.
// DET: gw is [blocks][9][8][C]; each block stores its sums there for ordered_sum_kernel.
template <bool DET>
__global__ void __launch_bounds__(256) dec_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dest, int n_frames,
                                                        int n_freq, int C, int n_out, long long n_pos,
                                                        float* __restrict__ gw /*[9][8][C]*/) {
  const int c = threadIdx.x;
  const int n_src = n_out >> 1;
  float acc[72];
#pragma unroll
  for (int i = 0; i < 72; ++i) acc[i] = 0.f;
  for (long long pos = blockIdx.x; pos < n_pos; pos += gridDim.x) {
    const int ff = (int)(pos % n_freq);
    const long long bt = pos / n_freq;
    const int tt = (int)(bt % n_frames), b = (int)(bt / n_frames);
    const float xv = c < C ? __ldg(&x[pos * C + c]) : 0.f;
#pragma unroll
    for (int dt = 0; dt < 3; ++dt) {
      const int t = tt - 1 + dt;
      if (t < 0 || t >= n_frames) continue;
#pragma unroll
      for (int df = 0; df < 3; ++df) {
        const int f = ff - 1 + df;
        if (f < 0 || f >= n_freq) continue;
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          if (o < n_out) {
            const float g = __ldg(&dest[(((((size_t)b * n_src + (o >> 1)) * n_frames + t) * n_freq + f) << 1) + (o & 1)]);
            acc[(dt * 3 + df) * 8 + o] = fmaf(xv, g, acc[(dt * 3 + df) * 8 + o]);
          }
        }
      }
    }
  }
  if (c < C) {
    float* g = gw + (DET ? (size_t)blockIdx.x * 72 * C : 0);
#pragma unroll
    for (int i = 0; i < 72; ++i) {
      if (DET) g[(size_t)i * C + c] = acc[i];
      else atomicAdd(&g[(size_t)i * C + c], acc[i]);
    }
  }
}

// gb[o] = sum over (b, t, f) of dEst[b][o >> 1][t][f][o & 1]: the terms largely cancel, so the sum is taken in double, one
// block per output, fixed order (deterministic).
__global__ void __launch_bounds__(256) dec_bias_grad_kernel(const float* __restrict__ dest, int batch, int n_src, long long per_src /* Tf * F */,
                                                            float* __restrict__ gb) {
  const int o = blockIdx.x, src = o >> 1, ri = o & 1;
  double acc = 0.0;
  for (int b = 0; b < batch; ++b) {
    const float* p = dest + (((size_t)b * n_src + src) * per_src << 1) + ri;
    for (long long i = threadIdx.x; i < per_src; i += blockDim.x) acc += (double)__ldg(&p[i << 1]);
  }
  __shared__ double red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) { if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k]; __syncthreads(); }
  if (threadIdx.x == 0) gb[o] = (float)red[0];
}

// ---- encoder backward: y = gLN(conv(spec)) = (v - mean) * rstd * gw_c + gb_c, statistics over (C, Tf, F) per sample ------
// pass 1: dgw_c += sum dy * vhat, dgb_c += sum dy, per-sample S1 = sum dy * gw_c, S2 = sum dy * gw_c * vhat (double).
// v is the conv output (pre-norm), recomputed by enc_conv_kernel.  Thread = channel, blocks over positions.
// DET: per (sample, block) partials -- dgw [B][blocks][2C] = (dgw, dgb), sums [B][blocks][2] -- for ordered_sum_kernel
// (dgb unused).
template <bool DET>
__global__ void __launch_bounds__(256) enc_gln_bwd_stats_kernel(const float* __restrict__ v, const float* __restrict__ dy,
                                                                long long per_sample_pos, int C, const float* __restrict__ stats,
                                                                const float* __restrict__ gw, float* __restrict__ dgw,
                                                                float* __restrict__ dgb, double* __restrict__ sums /*[B][2]*/) {
  const int b = blockIdx.y, c = threadIdx.x;
  const float mean = stats[b * 2], rstd = stats[b * 2 + 1];
  const float w = c < C ? gw[c] : 0.f;
  float a_w = 0.f, a_b = 0.f;
  double s1 = 0.0, s2 = 0.0;
  for (long long pos = blockIdx.x; pos < per_sample_pos; pos += gridDim.x) {
    if (c < C) {
      const size_t off = ((size_t)b * per_sample_pos + pos) * C + c;
      const float vh = (v[off] - mean) * rstd, d = dy[off];
      a_w = fmaf(d, vh, a_w); a_b += d;
      s1 += (double)(d * w); s2 += (double)(d * w * vh);
    }
  }
  const size_t part = (size_t)b * gridDim.x + blockIdx.x;
  if (c < C) {
    if (DET) { dgw[part * 2 * C + c] = a_w; dgw[part * 2 * C + C + c] = a_b; }
    else { atomicAdd(&dgw[c], a_w); atomicAdd(&dgb[c], a_b); }
  }
  __shared__ double r1[256], r2[256];
  r1[threadIdx.x] = s1; r2[threadIdx.x] = s2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o && threadIdx.x + o < blockDim.x) { r1[threadIdx.x] += r1[threadIdx.x + o]; r2[threadIdx.x] += r2[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (DET) { sums[part * 2] = r1[0]; sums[part * 2 + 1] = r2[0]; }
    else { atomicAdd(&sums[b * 2], r1[0]); atomicAdd(&sums[b * 2 + 1], r2[0]); }
  }
}

// pass 2: dv = rstd * (dy * gw_c - S1 / n - vhat * S2 / n);  conv weight gradient
//   gwc[(dt*3+df)][ci][c] += sum_pos dv[pos][c] * spec[t+dt-1, f+df-1][ci],  gbc[c] += sum dv.
// DET: gwc is [B][blocks][9 CIN + 1][C] (the bias row last; gbc unused), stored per (sample, block) for ordered_sum_kernel.
template <int CIN, bool DET>
__global__ void __launch_bounds__(256) enc_wgrad_kernel(const float* __restrict__ v, const float* __restrict__ dy,
                                                        const float* __restrict__ spec, int n_frames, int n_freq, int C,
                                                        const float* __restrict__ stats, const double* __restrict__ sums,
                                                        const float* __restrict__ gw, float* __restrict__ gwc,
                                                        float* __restrict__ gbc) {
  const int b = blockIdx.y, c = threadIdx.x;
  const long long per_sample_pos = (long long)n_frames * n_freq;
  const float mean = stats[b * 2], rstd = stats[b * 2 + 1];
  const double cnt = (double)per_sample_pos * C;
  const float m1 = (float)(sums[b * 2] / cnt), m2 = (float)(sums[b * 2 + 1] / cnt);
  const float w = c < C ? gw[c] : 0.f;
  float acc[9 * CIN];
#pragma unroll
  for (int i = 0; i < 9 * CIN; ++i) acc[i] = 0.f;
  float bacc = 0.f;
  const float* in = spec + (size_t)b * per_sample_pos * CIN;
  for (long long pos = blockIdx.x; pos < per_sample_pos; pos += gridDim.x) {
    const int f = (int)(pos % n_freq), t = (int)(pos / n_freq);
    float dv = 0.f;
    if (c < C) {
      const size_t off = ((size_t)b * per_sample_pos + pos) * C + c;
      const float vh = (v[off] - mean) * rstd;
      dv = rstd * (dy[off] * w - m1 - vh * m2);
    }
    bacc += dv;
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
        for (int ci = 0; ci < CIN; ++ci) acc[(dt * 3 + df) * CIN + ci] = fmaf(dv, __ldg(&px[ci]), acc[(dt * 3 + df) * CIN + ci]);
      }
    }
  }
  if (c < C && DET) {
    float* g = gwc + ((size_t)b * gridDim.x + blockIdx.x) * (9 * CIN + 1) * C;
#pragma unroll
    for (int i = 0; i < 9 * CIN; ++i) g[(size_t)i * C + c] = acc[i];
    g[(size_t)9 * CIN * C + c] = bacc;
  } else if (c < C) {
#pragma unroll
    for (int i = 0; i < 9 * CIN; ++i) atomicAdd(&gwc[(size_t)i * C + c], acc[i]);
    atomicAdd(&gbc[c], bacc);
  }
}

// pass 3 (input gradient, only when the caller wants d spec): dv as in pass 2, then the transposed 3x3 conv
//   dspec[t', f', i] = sum_{dt, df, c} dv[t' - dt + 1, f' - df + 1, c] * w[(dt*3+df)*CIN + i][c]   (zero outside the image)
// split as P[pos][j] = sum_c dv[pos][c] w[j][c] (j = (dt*3+df)*CIN + i; one warp per position, lanes over channels) and a
// 9-tap gather of P.  A CTA owns ENC_IG_TT frames x ENC_IG_FT bins; P of the tile plus a one-position halo lives in shared
// memory, so each v / dy row is read once per CTA that needs it (interior rows once, halo rows by two or four CTAs).
constexpr int ENC_IG_TT = 8, ENC_IG_FT = 32;
template <int CIN>
__global__ void __launch_bounds__(256) enc_input_grad_kernel(const float* __restrict__ v, const float* __restrict__ dy,
                                                             int n_frames, int n_freq, int C, const float* __restrict__ stats,
                                                             const double* __restrict__ sums, const float* __restrict__ gw,
                                                             const float* __restrict__ w /*[9][CIN][C]*/,
                                                             float* __restrict__ dspec /*[B][Tf][F][CIN]*/) {
  constexpr int J = 9 * CIN;
  static_assert(J <= 32, "one lane per tap-channel pair");
  constexpr int HT = ENC_IG_TT + 2, HF = ENC_IG_FT + 2;
  extern __shared__ float ig_sm[];            // wsm [J][C], then P [HT * HF][J]
  float* wsm = ig_sm;
  float* P = ig_sm + (size_t)J * C;
  const int b = blockIdx.z, t0 = blockIdx.y * ENC_IG_TT, f0 = blockIdx.x * ENC_IG_FT;
  for (int i = threadIdx.x; i < J * C; i += blockDim.x) wsm[i] = w[i];
  __syncthreads();
  const long long per_sample_pos = (long long)n_frames * n_freq;
  const float mean = stats[b * 2], rstd = stats[b * 2 + 1];
  const double cnt = (double)per_sample_pos * C;
  const float m1 = (float)(sums[b * 2] / cnt), m2 = (float)(sums[b * 2 + 1] / cnt);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  for (int hp = warp; hp < HT * HF; hp += n_warps) {
    const int t = t0 - 1 + hp / HF, f = f0 - 1 + hp % HF;
    float a[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) a[j] = 0.f;
    if (t >= 0 && t < n_frames && f >= 0 && f < n_freq) {
      const size_t row = ((size_t)b * per_sample_pos + (size_t)t * n_freq + f) * C;
      for (int c = lane; c < C; c += 32) {
        const float vh = (__ldg(&v[row + c]) - mean) * rstd;
        const float dv = rstd * (__ldg(&dy[row + c]) * __ldg(&gw[c]) - m1 - vh * m2);
#pragma unroll
        for (int j = 0; j < J; ++j) a[j] = fmaf(dv, wsm[j * C + c], a[j]);
      }
    }
    // transpose-reduce over the warp: after the step of width s, a lane keeps the half of its s-wide window selected by
    // its lane bit s; at the end lane l holds the warp total of value l
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
      const bool upper = (lane & s) != 0;
#pragma unroll
      for (int j = 0; j < s; ++j) {
        const float send = upper ? a[j] : a[j + s];
        const float keep = upper ? a[j + s] : a[j];
        a[j] = keep + __shfl_xor_sync(0xffffffffu, send, s);
      }
    }
    if (lane < J) P[hp * J + lane] = a[0];
  }
  __syncthreads();
  for (int o = threadIdx.x; o < ENC_IG_TT * ENC_IG_FT * CIN; o += blockDim.x) {
    const int i = o % CIN, q = o / CIN, lt = q / ENC_IG_FT, lf = q % ENC_IG_FT;
    const int t = t0 + lt, f = f0 + lf;
    if (t >= n_frames || f >= n_freq) continue;
    float acc = 0.f;
#pragma unroll
    for (int dt = 0; dt < 3; ++dt)
#pragma unroll
      for (int df = 0; df < 3; ++df)       // source position (t - dt + 1, f - df + 1) = halo cell (lt - dt + 2, lf - df + 2)
        acc += P[((lt - dt + 2) * HF + (lf - df + 2)) * J + (dt * 3 + df) * CIN + i];
    dspec[(((size_t)b * n_frames + t) * n_freq + f) * CIN + i] = acc;
  }
}

// ---- adjoint of reflect pad -> frame: dmix[b][n] = sum of the windowed frame adjoints (stft_adj_frames_kernel output)
// over every frame that covers padded coordinate n + pad, plus the reflected images pad - n (1 <= n <= pad) and
// pad + 2 (T - 1) - n (right pad).  The same fold as in loss_grad_kernel, for the model's own STFT.
__global__ void __launch_bounds__(256) stft_fold_kernel(const float* __restrict__ frames /*[b][t][n_fft]*/, int n_samples,
                                                        int n_fft, int hop, int n_frames, float* __restrict__ dmix /*[b][n]*/) {
  const int b = blockIdx.y, pad = n_fft >> 1;
  const float* fr = frames + (size_t)b * n_frames * n_fft;
  auto gather = [&](long long p) -> float {
    long long t_hi = p / hop;
    if (t_hi > n_frames - 1) t_hi = n_frames - 1;
    const long long t_lo = p - n_fft + 1 <= 0 ? 0 : (p - n_fft + hop) / hop;
    float acc = 0.f;
    for (long long tp = t_lo; tp <= t_hi; ++tp) acc += __ldg(&fr[tp * n_fft + (p - tp * hop)]);
    return acc;
  };
  const long long covered = (long long)(n_frames - 1) * hop + n_fft;
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_samples; n += (long long)gridDim.x * blockDim.x) {
    float g = gather(n + pad);
    if (n >= 1 && n <= pad) g += gather(pad - n);
    if (n <= n_samples - 2) {
      const long long p = pad + 2 * ((long long)n_samples - 1) - n;
      if (p < covered) g += gather(p);
    }
    dmix[(size_t)b * n_samples + n] = g;
  }
}

// ---- iSTFT backward: dEst[b][src][t][k] = (c_k / N) * rfft(w .* u[t * hop : t * hop + N])_k, u = dAudio / envelope on the
// valid samples and zero elsewhere (c_0 = c_{N/2} = 1, else 2; imaginary parts of DC / Nyquist get no gradient: :56-75) ----
__global__ void __launch_bounds__(256) istft_bwd_kernel(const float* __restrict__ daudio /*[src][b][n]*/, int n_src, int batch,
                                                        int n_samples, int n_fft, int log_n, int hop, int n_frames,
                                                        const float2* __restrict__ tw, const float* __restrict__ win,
                                                        float* __restrict__ dest /*[b][src][t][k][2]*/) {
  extern __shared__ float2 fbuf[];
  const int t = blockIdx.x, src = blockIdx.y, b = blockIdx.z;
  const float* g = daudio + ((size_t)src * batch + b) * n_samples;
  const int pad = n_fft >> 1;
  for (int i = threadIdx.x; i < n_fft; i += blockDim.x) {
    const int p = t * hop + i;          // padded-signal coordinate
    const int n = p - pad;
    float val = 0.f;
    if (n >= 0 && n < n_samples) {
      int t_lo = p - n_fft + 1 <= 0 ? 0 : (p - n_fft + hop) / hop;   // ceil((p - n_fft + 1) / hop)
      int t_hi = p / hop;
      if (t_hi > n_frames - 1) t_hi = n_frames - 1;
      float env = 0.f;
      for (int tp = t_lo; tp <= t_hi; ++tp) { const float w = __ldg(&win[p - tp * hop]); env += w * w; }
      val = __ldg(&g[n]) / env * __ldg(&win[i]);
    }
    fbuf[bitrev(i, log_n)] = make_float2(val, 0.f);
  }
  __syncthreads();
  fft_smem<false>(fbuf, tw, n_fft, log_n);
  const int n_freq = pad + 1;
  const float inv_n = 1.f / (float)n_fft;
  float2* out = reinterpret_cast<float2*>(dest) + (((size_t)b * n_src + src) * n_frames + t) * n_freq;
  for (int k = threadIdx.x; k < n_freq; k += blockDim.x) {
    float2 z = fbuf[k];
    if (k == 0 || k == pad) { z.x *= inv_n; z.y = 0.f; } else { z.x *= 2.f * inv_n; z.y *= 2.f * inv_n; }
    out[k] = z;
  }
}

// ---- loss (models/mss_loss.py:18-244) ---------------------------------------------------------------------------------
struct LossCfg {
  float w_sisdr, w_l1, w_spec, eps;
  int n_src, batch, n_samples;
  int l_fft, l_log, l_hop, l_frames;   // SpectralLoss STFT (n_fft 2048 / hop 1024 whatever the model uses, :184-193)
};

// SI-SDR per row (src, b) from the five sums of pair_stats: loss_row = -10 log10(sig / noise); gradient w.r.t. the
// estimate is affine in (est_i, tgt_i): coef[row] = {A, B, C0} with d loss / d est_i = A est_i + B tgt_i + C0 (mss_loss.py:141-168).
__global__ void sisdr_coef_kernel(const double* __restrict__ s5, LossCfg cfg, float* __restrict__ coef /*[rows][3]*/,
                                  double* __restrict__ loss_rows /*[rows]*/) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= cfg.n_src * cfg.batch) return;
  const double n = (double)cfg.n_samples, eps = (double)cfg.eps;
  const double Se = s5[row * 5], St = s5[row * 5 + 1], See = s5[row * 5 + 2], Stt = s5[row * 5 + 3], Set = s5[row * 5 + 4];
  const double me = Se / n, mt = St / n;
  const double dot = Set - n * me * mt, tt = Stt - n * mt * mt, ee = See - n * me * me;
  const double te = tt + eps, scale = dot / te;
  const double sig = scale * scale * tt + eps;
  const double noise = ee - 2.0 * scale * dot + scale * scale * tt + eps;
  const double sisdr = 10.0 * log10(sig / noise);
  loss_rows[row] = -sisdr;
  const double kf = -(double)cfg.w_sisdr * (10.0 / log(10.0)) / (double)cfg.batch;
  const double a_e = -2.0 * kf / noise;
  const double a_t = kf * (2.0 * scale * tt / (te * sig) + 2.0 * scale / noise + 2.0 * (dot - scale * tt) / (te * noise));
  coef[row * 3] = (float)a_e;
  coef[row * 3 + 1] = (float)a_t;
  coef[row * 3 + 2] = (float)(-a_e * me - a_t * mt);
}

// log-magnitude L1 between the loss spectrograms: partial sums per row, and dE written over E:
//   dE = w_spec / count * sign(log1p|E| - log1p|T|) / (1 + |E|) * E / |E|     (count = batch * bins * frames, per source)
// DET: sum_rows is [rows][blocks], one partial per block for ordered_sum_kernel.
template <bool DET>
__global__ void __launch_bounds__(256) spec_loss_kernel(float2* __restrict__ E, const float2* __restrict__ T, long long per_row,
                                                        float coef, double* __restrict__ sum_rows /*[rows]*/) {
  const int row = blockIdx.y;
  float2* e = E + (size_t)row * per_row;
  const float2* t = T + (size_t)row * per_row;
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_row; i += (long long)gridDim.x * blockDim.x) {
    const float2 ev = e[i], tv = t[i];
    const float me = sqrtf(ev.x * ev.x + ev.y * ev.y), mt = sqrtf(tv.x * tv.x + tv.y * tv.y);
    const float diff = log1pf(me) - log1pf(mt);
    acc += (double)fabsf(diff);
    const float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
    const float k = me > 0.f ? coef * sgn / ((1.f + me) * me) : 0.f;
    e[i] = make_float2(k * ev.x, k * ev.y);
  }
  __shared__ double red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) {
    if (DET) sum_rows[(size_t)row * gridDim.x + blockIdx.x] = red[0];
    else atomicAdd(&sum_rows[row], red[0]);
  }
}

// adjoint of the rfft of one windowed frame: frames[row][t][m] = w[m] * sum_k (dRe_k cos(2 pi k m / N) - dIm_k sin(...))
__global__ void __launch_bounds__(256) stft_adj_frames_kernel(const float2* __restrict__ dE /*[row][t][k]*/, int n_fft, int log_n,
                                                              int n_frames, const float2* __restrict__ tw,
                                                              const float* __restrict__ win, float* __restrict__ frames) {
  extern __shared__ float2 fbuf[];
  const int t = blockIdx.x, row = blockIdx.y;
  const int pad = n_fft >> 1, n_freq = pad + 1;
  const float2* x = dE + ((size_t)row * n_frames + t) * n_freq;
  for (int k = threadIdx.x; k < n_freq; k += blockDim.x) {
    const float2 v = __ldg(&x[k]);
    if (k == 0 || k == pad) {
      fbuf[bitrev(k, log_n)] = make_float2(v.x, 0.f);
    } else {
      fbuf[bitrev(k, log_n)] = make_float2(0.5f * v.x, 0.5f * v.y);
      fbuf[bitrev(n_fft - k, log_n)] = make_float2(0.5f * v.x, -0.5f * v.y);
    }
  }
  __syncthreads();
  fft_smem<true>(fbuf, tw, n_fft, log_n);
  float* out = frames + ((size_t)row * n_frames + t) * n_fft;
  for (int m = threadIdx.x; m < n_fft; m += blockDim.x) out[m] = fbuf[m].x * __ldg(&win[m]);
}

// d loss / d est[row][n] = SI-SDR (affine) + L1 sign + the adjoint of (reflect pad -> frame) applied to `frames`;
// also accumulates sum |est - tgt| per row for the reported L1 loss (DET: l1_rows is [rows][blocks] of block partials).
template <bool DET>
__global__ void __launch_bounds__(256) loss_grad_kernel(const float* __restrict__ est, const float* __restrict__ tgt,
                                                        const float* __restrict__ coef, const float* __restrict__ frames,
                                                        LossCfg cfg, float* __restrict__ dest, double* __restrict__ l1_rows) {
  const int row = blockIdx.y;
  const long long n_samples = cfg.n_samples;
  const float* e = est + (size_t)row * n_samples;
  const float* t = tgt + (size_t)row * n_samples;
  const float A = coef[row * 3], Bc = coef[row * 3 + 1], C0 = coef[row * 3 + 2];
  const float l1c = cfg.w_l1 / ((float)cfg.batch * (float)cfg.n_samples);
  const int N = cfg.l_fft, pad = N >> 1, hop = cfg.l_hop, TfL = cfg.l_frames;
  const float* fr = frames != nullptr ? frames + (size_t)row * TfL * N : nullptr;
  auto gather = [&](long long p) -> float {   // sum over the frames that cover padded coordinate p
    if (p < 0) return 0.f;
    long long t_hi = p / hop;
    if (t_hi > TfL - 1) t_hi = TfL - 1;
    long long t_lo = p - N + 1 <= 0 ? 0 : (p - N + hop) / hop;
    float acc = 0.f;
    for (long long tp = t_lo; tp <= t_hi; ++tp) acc += __ldg(&fr[tp * N + (p - tp * hop)]);
    return acc;
  };
  double l1 = 0.0;
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_samples; n += (long long)gridDim.x * blockDim.x) {
    const float ev = e[n], tv = t[n];
    const float diff = ev - tv;
    l1 += (double)fabsf(diff);
    float g = A * ev + Bc * tv + C0 + l1c * (diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f));
    if (fr != nullptr) {
      g += gather(n + pad);
      if (n >= 1 && n <= pad) g += gather(pad - n);                       // left reflection: padded p = pad - n
      if (n <= n_samples - 2) {                                           // right reflection: p = pad + 2 (T - 1) - n >= pad + T
        const long long p = pad + 2 * (n_samples - 1) - n;
        if (p < (long long)(TfL - 1) * hop + N) g += gather(p);
      }
    }
    dest[(size_t)row * n_samples + n] = g;
  }
  __shared__ double red[256];
  red[threadIdx.x] = l1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) {
    if (DET) l1_rows[(size_t)row * gridDim.x + blockIdx.x] = red[0];
    else atomicAdd(&l1_rows[row], red[0]);
  }
}

// loss_out[0] = total, then per source {si_sdr, l1, spectral} (means as the reference reports them)
__global__ void loss_finish_kernel(const double* __restrict__ sisdr_rows, const double* __restrict__ l1_rows,
                                   const double* __restrict__ spec_rows, LossCfg cfg, long long spec_count,
                                   float* __restrict__ loss_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double total = 0.0;
  for (int s = 0; s < cfg.n_src; ++s) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int i = 0; i < cfg.batch; ++i) {
      a += sisdr_rows[s * cfg.batch + i]; b += l1_rows[s * cfg.batch + i];
      if (spec_rows != nullptr) c += spec_rows[s * cfg.batch + i];
    }
    a /= cfg.batch; b /= (double)cfg.batch * cfg.n_samples; c /= (double)spec_count;
    loss_out[1 + 3 * s] = (float)a; loss_out[2 + 3 * s] = (float)b; loss_out[3 + 3 * s] = (float)c;
    total += cfg.w_sisdr * a + cfg.w_l1 * b + cfg.w_spec * c;
  }
  loss_out[0] = (float)total;
}

// ---- optimiser: clip_grad_norm_(max_norm) + AdamW (train.py:141-146, :351-357) --------------------------------------
__global__ void __launch_bounds__(256) sqnorm_partial_kernel(const float* __restrict__ g, long long n, double* __restrict__ partial) {
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc += (double)g[i] * (double)g[i];
  __shared__ double red[256];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}
// norm_out[0] = total L2 norm, norm_out[1] = clip coefficient min(1, max_norm / (norm + 1e-6))
__global__ void sqnorm_finish_kernel(const double* __restrict__ partial, int n_part, float max_norm, float* __restrict__ norm_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double s = 0.0;
  for (int i = 0; i < n_part; ++i) s += partial[i];
  const double nrm = sqrt(s);
  norm_out[0] = (float)nrm;
  const double coef = (double)max_norm / (nrm + 1e-6);
  norm_out[1] = (float)(coef < 1.0 ? coef : 1.0);
}
// acc += scale * g (gradient accumulation over micro-batches, train.py:117-146: loss / gradient_accumulation_steps)
__global__ void __launch_bounds__(256) grad_accumulate_kernel(float* __restrict__ acc, const float* __restrict__ g, long long n, float scale,
                                                              int overwrite) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    acc[i] = overwrite ? scale * g[i] : fmaf(scale, g[i], acc[i]);
}
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, long long n, const float* __restrict__ clip,
                                                    float lr, float beta1, float beta2, float eps, float wd, float bc1, float bc2_sqrt) {
  const float cc = clip != nullptr ? clip[1] : 1.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * cc;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    pi -= (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
    p[i] = pi;
  }
}

}  // namespace tfl
