// Host side of the training step (SURVEY.md section 8(f) N1): forward with saved sub-block inputs, MSSLoss, backward,
// gradient clipping and AdamW -- /root/reference/training/train.py:68-172, /root/reference/models/mss_loss.py:18-244.
// Included at the end of tfl_api.cu (same translation unit: it reuses gemm_launch / norm_launch / the fp32 forward).
//
// Gradients leave in ONE flat fp32 buffer, one slice per state_dict tensor in tfl_pack_weights order and in the
// reference's own tensor layout (conv1d.weight [2H, C, K], qkv.weight [3A, C], ...), so that param.grad of the
// reference model is the parity target, a data-parallel all-reduce is one NCCL call on the buffer, and clipping + AdamW
// are two kernels over it.
#pragma once

namespace tfl {

struct GradLayout {
  std::vector<long long> off;   // per weight tensor (tfl_pack_weights order): offset in floats, -1 = not trainable
  std::vector<long long> size;
  long long total;
};

static GradLayout grad_layout(const tfl_plan* pl) {
  const tfl_config& c = pl->cfg;
  GradLayout g;
  long long off = 0;
  auto add = [&](long long n, bool trainable = true) {
    g.off.push_back(trainable ? off : -1);
    g.size.push_back(n);
    if (trainable) off += (n + 63) / 64 * 64;
  };
  const long long C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel, S2 = c.n_src * 2;
  if (c.enc_in_ch > 0) { add(C * c.enc_in_ch * 9); add(C); add(C); add(C); }
  for (int layer = 0; layer < c.n_layers; ++layer)
    for (int axis = 0; axis < 2; ++axis) {
      for (int j = 0; j < pl->n_ffn; ++j) add(C);
      for (int j = 0; j < pl->n_ffn; ++j) {
        const long long H = j == 0 ? c.ffn_hidden0 : c.ffn_hidden1;
        add(2 * H * C * K); add(2 * H); add(H * C * K); add(C);
      }
      add(C);
      if (c.rope) add(pl->head_dim / 2, false);
      add(3 * A * C); add(C * A);
    }
  if (c.enc_in_ch > 0) { add(C * S2 * 9); add(S2); }
  g.total = off;
  return g;
}

// index of the first weight tensor of path (layer, axis) in tfl_pack_weights order
static int path_weight_index(const tfl_plan* pl, int layer, int axis) {
  const tfl_config& c = pl->cfg;
  const int per_path = pl->n_ffn + 4 * pl->n_ffn + 1 + (c.rope ? 1 : 0) + 2;
  return (c.enc_in_ch > 0 ? 4 : 0) + (layer * 2 + axis) * per_path;
}

struct TrainWs {
  Workspace fwd;             // the fp32 inference workspace sits at offset 0
  Workspace fwd16;           // bf16 workspace of the tcgen05 forward kernels (mixed mode), based at fwd16_base (0 = none)
  size_t fwd16_base;
  size_t ckpt, dx, dxn, scratch, lse, dbuf, nat, wt, dest, audio, daudio;
  size_t s5, stats_scratch, coef, loss_rows, l1_rows, spec_rows, ltab_tw, ltab_win, lspec_e, lspec_t, lframes, enc_sums;
  size_t dspec, adj_frames;  // saved mode with T > 0 (the MSS autograd pair): d spec [B][Tf][F][2], frame adjoints [B][Tf][n_fft]
  size_t det;                // TFL_OPT_DETERMINISTIC: partials of the reductions, sized for the largest one (0 = option off)
  size_t total;
  // inside `scratch` (FFN and attention backward never overlap in time)
  size_t dg, hid2, dh;       // FFN: dG, recomputed hidden, dH
  size_t dO, dqkv_h, dqkv;   // attention
  int n_sub, l_frames, l_freq;
};

// ---- deterministic mode (TFL_OPT_DETERMINISTIC) ----------------------------------------------------------------------
// Every reduction over rows of the backward pass stores one partial per block or row split and ordered_sum_kernel adds
// them in index order.  Its grids are sized for a 148-SM B200 whatever the device, so the order of each of these sums is a
// function of the shapes alone (DESIGN.md section 8b names the one forward reduction that still follows the SM count).
constexpr int DET_SMS = 148;

static float* det_ptr(const TrainWs& tw, char* wsp) { return tw.det != 0 ? (float*)(wsp + tw.det) : nullptr; }

template <class T>
static int ordered_sum(const T* part, int n_rows, long long row_stride, long long width, T* out, cudaStream_t st,
                       int batch = 1, long long part_bstride = 0, long long out_bstride = 0) {
  long long blocks = (width + 255) / 256;
  if (blocks > DET_SMS * 8) blocks = DET_SMS * 8;
  ordered_sum_kernel<T><<<dim3((unsigned)blocks, batch), 256, 0, st>>>(part, n_rows, row_stride, width, part_bstride, out,
                                                                       out_bstride);
  TFL_LAUNCH_CHECK();
  return 0;
}

// Row splits of a weight-gradient GEMM (sets rows_per_split): about four CTAs per SM, at least 256 rows per split.
static long long wgrad_splits(TapWgrad& g, int sm_count) {
  const int tiles = g.taps * ((g.Kc + GBM - 1) / GBM) * ((g.N + GBN - 1) / GBN);
  long long splits = ((long long)sm_count * 4 + tiles - 1) / tiles;
  const long long max_splits = (g.R + 255) / 256;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (splits > 65535) splits = 65535;
  g.rows_per_split = ((g.R + splits - 1) / splits + 31) / 32 * 32;
  return (g.R + g.rows_per_split - 1) / g.rows_per_split;
}
static long long wgrad_slab_bytes(int taps, int Kc, int N, long long R) {
  TapWgrad g{};
  g.taps = taps; g.Kc = Kc; g.N = N; g.R = R;
  return wgrad_splits(g, DET_SMS) * taps * Kc * N * (long long)sizeof(float);
}
static long long colsum_blocks(long long R, int sm_count) {
  const long long blocks = (R + 63) / 64;
  return blocks > (long long)sm_count * 4 ? (long long)sm_count * 4 : blocks;
}
// RMSGroupNorm backward: threads per (row, group) pair W and the block count; `det` rounds the blocks up to a multiple of
// G, which makes every slot of W threads keep one group for all of its rows
static long long norm_bwd_blocks(long long rows, int C, int G, int sm_count, bool det, int* W_out) {
  const int lanes = (C / G) / 4;
  int W = 1;
  while (W < lanes) W <<= 1;
  *W_out = W;
  const long long per_block = 256 / W;
  long long blocks = (rows * G + per_block - 1) / per_block;
  if (blocks > (long long)sm_count * 8) blocks = (long long)sm_count * 8;
  if (blocks < 1) blocks = 1;
  return det ? (blocks + G - 1) / G * G : blocks;
}
constexpr int DET_DEC_BLOCKS = DET_SMS * 4, DET_ENC_BLOCKS = DET_SMS * 2, DET_LOSS_BLOCKS = DET_SMS;

// The partials of the largest reduction of a step of this shape: every weight-gradient slab, bias, gamma, decoder and
// encoder partial, and (loss_rows > 0) the loss row sums.  One buffer serves them all: they are consumed in stream order.
static size_t det_scratch_bytes(const tfl_plan* pl, int B, int Tf, int F, int loss_rows) {
  const tfl_config& c = pl->cfg;
  const int C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel;
  const long long rows = (long long)B * Tf * F;
  long long need = 0;
  auto at_least = [&](long long bytes) { if (bytes > need) need = bytes; };
  for (int axis = 0; axis < 2; ++axis) {
    const long long S = axis == TFL_AXIS_FREQ ? F : Tf, nseq = rows / S, rows1 = nseq * (S + K - 1);
    for (int j = 0; j < pl->n_ffn; ++j) {
      const int H = j == 0 ? c.ffn_hidden0 : c.ffn_hidden1;
      at_least(wgrad_slab_bytes(K, H, C, rows));
      at_least(wgrad_slab_bytes(K, C, 2 * H, rows1));
      at_least(colsum_blocks(rows, DET_SMS) * C * 4);
      at_least(colsum_blocks(rows1, DET_SMS) * 2 * H * 4);
    }
    at_least(wgrad_slab_bytes(1, C, A, rows));
    at_least(wgrad_slab_bytes(1, 3 * A, C, rows));
  }
  int W;
  at_least(norm_bwd_blocks(rows, C, c.num_groups, DET_SMS, true, &W) * C * 4);
  if (c.enc_in_ch > 0) {
    at_least((long long)DET_DEC_BLOCKS * 72 * C * 4);
    const long long enc_parts = (long long)B * DET_ENC_BLOCKS;
    at_least(align_up(enc_parts * 2 * C * 4) + enc_parts * 2 * 8);          // enc_gln_bwd_stats_kernel
    at_least(enc_parts * (9 * c.enc_in_ch + 1) * C * 4);                     // enc_wgrad_kernel
  }
  at_least((long long)loss_rows * DET_SMS * 2 * 8);                          // loss_grad_kernel (spec_loss_kernel: half)
  return (size_t)need;
}

// (B, Tf, F) size the network buffers; T (audio samples, 0 = stage-level use) and the loss STFT size the rest.
// `saved`: the checkpoint slots of one saved forward, without the loss buffers.  T = 0: the separators' frames-only
// mode; T > 0: TFLocoformerMSS, plus the buffers of the mixture gradient (d spec and the adjoint STFT frames).
static TrainWs plan_train_ws(const tfl_plan* pl, int B, int Tf, int F, int T, int l_fft, int l_hop, bool saved = false) {
  const tfl_config& c = pl->cfg;
  TrainWs w{};
  const bool ckpt = T > 0 || saved;
  w.fwd = plan_workspace(pl, B, Tf, F, TFL_PRECISION_FP32);
  size_t off = align_up(w.fwd.total);
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  const size_t N = (size_t)B * Tf * F;
  const size_t C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel, S = c.n_src;
  const size_t Hmax = c.ffn_hidden0 > c.ffn_hidden1 ? c.ffn_hidden0 : c.ffn_hidden1;
  w.n_sub = ckpt ? c.n_layers * 2 * (pl->n_ffn + 1) : 0;
  w.ckpt = take((size_t)(w.n_sub > 0 ? w.n_sub + 1 : 0) * N * C * sizeof(float));   // x_0 .. x_n_sub (the residual stream itself)
  w.fwd16_base = 0;
  if (ckpt && attn_tc_supported((int)C, c.n_heads, pl->head_dim)) {
    w.fwd16 = plan_workspace(pl, B, Tf, F, TFL_PRECISION_BF16);
    w.fwd16_base = take(w.fwd16.total);
  }
  w.dx = take(N * C * sizeof(float));
  w.dxn = take(N * C * sizeof(float));
  const size_t rows_f = (size_t)B * Tf * (F + K - 1), rows_t = (size_t)B * F * (Tf + K - 1);
  const size_t rows1 = rows_f > rows_t ? rows_f : rows_t;
  const size_t ffn_bytes = align_up(rows1 * Hmax * 4) * 2 + align_up(rows1 * 2 * Hmax * 4);
  const size_t attn_bytes = align_up(N * A * 4) + 2 * align_up(N * 3 * A * 4);
  w.scratch = take(ffn_bytes > attn_bytes ? ffn_bytes : attn_bytes);
  w.dg = w.scratch; w.hid2 = w.dg + align_up(rows1 * Hmax * 4); w.dh = w.hid2 + align_up(rows1 * Hmax * 4);
  w.dO = w.scratch; w.dqkv_h = w.dO + align_up(N * A * 4); w.dqkv = w.dqkv_h + align_up(N * 3 * A * 4);
  w.lse = take(N * c.n_heads * sizeof(float));
  w.dbuf = take(N * c.n_heads * sizeof(float));
  // natural-layout weight-gradient scratch (largest: conv1d [K][C][2H] + [2H] + transposed conv [K][H][C]; decoder [9][8][C] + 8)
  size_t nat = K * C * 2 * Hmax + 2 * Hmax + K * Hmax * C + 64;
  if (nat < 9 * 8 * C + 64) nat = 9 * 8 * C + 64;
  w.nat = take(nat * sizeof(float));
  // transposed weights of the data-gradient GEMMs of one FFN: [K][C][H] and [K][2H][C]
  w.wt = take((K * C * Hmax + K * 2 * Hmax * C) * sizeof(float));
  w.dest = take(N * 2 * S * sizeof(float));
  const size_t rows = S * B;
  if (!saved) {
    w.audio = take(S * B * (size_t)T * sizeof(float));
    w.daudio = take(S * B * (size_t)T * sizeof(float));
    w.s5 = take(rows * 5 * sizeof(double));
    w.stats_scratch = take(rows * STATS_BLOCKS * 5 * sizeof(double));
    w.coef = take(rows * 3 * sizeof(float));
    w.loss_rows = take(rows * sizeof(double));
    w.l1_rows = take(rows * sizeof(double));
    w.spec_rows = take(rows * sizeof(double));
  } else if (T > 0) {
    w.dspec = take(N * 2 * sizeof(float));
    w.adj_frames = take((size_t)B * Tf * c.n_fft * sizeof(float));
  }
  w.enc_sums = take((size_t)B * 2 * sizeof(double));
  w.l_frames = (l_fft > 0 && T > 0) ? 1 + T / l_hop : 0;
  w.l_freq = l_fft / 2 + 1;
  if (l_fft > 0 && T > 0) {
    w.ltab_tw = take((size_t)l_fft * sizeof(float)); w.ltab_win = take((size_t)l_fft * sizeof(float));
    w.lspec_e = take(rows * w.l_frames * w.l_freq * sizeof(float2));
    w.lspec_t = take(rows * w.l_frames * w.l_freq * sizeof(float2));
    w.lframes = take(rows * w.l_frames * (size_t)l_fft * sizeof(float));
  }
  w.det = tfl_option(TFL_OPT_DETERMINISTIC) ? take(det_scratch_bytes(pl, B, Tf, F, saved ? 0 : (int)rows)) : 0;
  w.total = off;
  return w;
}

// The three launchers below add into `out` / `dgamma` with atomics, or -- with `det` (the partials buffer of the
// deterministic mode) -- store per-split / per-block partials there and add them in index order.
static int wgrad_launch(TapWgrad g, int sm_count, cudaStream_t st, float* det = nullptr) {
  TFL_CHECK(g.Kc % 4 == 0 && g.N % 4 == 0, "weight-gradient GEMM needs Kc %% 4 == 0 and N %% 4 == 0 (Kc %d N %d)", g.Kc, g.N);
  const int tiles = g.taps * ((g.Kc + GBM - 1) / GBM) * ((g.N + GBN - 1) / GBN);
  const long long splits = wgrad_splits(g, det != nullptr ? DET_SMS : sm_count);
  const dim3 grid((unsigned)tiles, (unsigned)splits);
  if (det != nullptr) {
    float* out = g.out;
    g.out = det;
    if (g_gemm_mode == 2) tap_wgrad_bf16_kernel<true><<<grid, 256, 0, st>>>(g);
    else if (g_gemm_mode == 1) tap_wgrad_mma_kernel<true><<<grid, 256, 0, st>>>(g);
    else tap_wgrad_kernel<true><<<grid, 256, 0, st>>>(g);
    TFL_LAUNCH_CHECK();
    const long long slab = (long long)g.taps * g.Kc * g.N;
    return ordered_sum(det, (int)splits, slab, slab, out, st);
  }
  if (g_gemm_mode == 2) tap_wgrad_bf16_kernel<false><<<grid, 256, 0, st>>>(g);
  else if (g_gemm_mode == 1) tap_wgrad_mma_kernel<false><<<grid, 256, 0, st>>>(g);
  else tap_wgrad_kernel<false><<<grid, 256, 0, st>>>(g);
  TFL_LAUNCH_CHECK();
  return 0;
}

static int colsum_launch(const float* Bm, SeqMap bmap, int Sout, int N, long long R, float* out, int sm_count, cudaStream_t st,
                         float* det = nullptr) {
  TFL_CHECK(N % 4 == 0, "column sum needs N %% 4 == 0");
  const long long blocks = colsum_blocks(R, det != nullptr ? DET_SMS : sm_count);
  if (det != nullptr) {
    const int lanes = N / 4 < 256 ? N / 4 : 256;
    colsum_kernel<true><<<(unsigned)blocks, 256, (size_t)(256 / lanes) * N * sizeof(float), st>>>(Bm, bmap, Sout, N, R, det);
    TFL_LAUNCH_CHECK();
    return ordered_sum(det, (int)blocks, N, N, out, st);
  }
  colsum_kernel<false><<<(unsigned)blocks, 256, (size_t)N * sizeof(float), st>>>(Bm, bmap, Sout, N, R, out);
  TFL_LAUNCH_CHECK();
  return 0;
}

static int norm_bwd_launch(const float* x, const float* dy, float* dx_total, long long rows, int C, int G, const float* gamma,
                           float eps, float* dgamma, int sm_count, cudaStream_t st, float* det = nullptr) {
  int W;
  const long long blocks = norm_bwd_blocks(rows, C, G, det != nullptr ? DET_SMS : sm_count, det != nullptr, &W);
  TFL_CHECK(W <= 32, "emb_dim/num_groups > 128 is not supported");
  if (det != nullptr) {
    const size_t slots_d = (size_t)(256 / W) * (C / G);
    const size_t sm = (slots_d > (size_t)C ? slots_d : (size_t)C) * sizeof(float);
#define NB_CASE(w) case w: rms_group_norm_bwd_kernel<w, true><<<(int)blocks, 256, sm, st>>>(x, dy, dx_total, rows, C, G, gamma, eps, det); break;
    switch (W) { NB_CASE(1) NB_CASE(2) NB_CASE(4) NB_CASE(8) NB_CASE(16) NB_CASE(32) }
#undef NB_CASE
    TFL_LAUNCH_CHECK();
    return ordered_sum(det, (int)blocks, C, C, dgamma, st);
  }
  const size_t sm = (size_t)C * sizeof(float);
#define NB_CASE(w) case w: rms_group_norm_bwd_kernel<w, false><<<(int)blocks, 256, sm, st>>>(x, dy, dx_total, rows, C, G, gamma, eps, dgamma); break;
  switch (W) { NB_CASE(1) NB_CASE(2) NB_CASE(4) NB_CASE(8) NB_CASE(16) NB_CASE(32) }
#undef NB_CASE
  TFL_LAUNCH_CHECK();
  return 0;
}

struct GradPtrs {   // where the gradients of one path's tensors go (slices of the flat buffer)
  float* ffn_gamma[2]; float* w1[2]; float* b1[2]; float* w2[2]; float* b2[2];
  float* attn_gamma; float* wqkv; float* wo;
};
struct RawPtrs {    // the reference-layout parameter tensors of one path (device pointers)
  const float* w1[2]; const float* w2[2]; const float* wqkv; const float* wo;
};

static void path_ptrs(const tfl_plan* pl, const GradLayout& gl, float* grads, const float* const* w, int layer, int axis,
                      GradPtrs& gp, RawPtrs& rp) {
  int i = path_weight_index(pl, layer, axis);
  for (int j = 0; j < pl->n_ffn; ++j) gp.ffn_gamma[j] = grads + gl.off[i++];
  for (int j = 0; j < pl->n_ffn; ++j) {
    rp.w1[j] = w[i]; gp.w1[j] = grads + gl.off[i++];
    gp.b1[j] = grads + gl.off[i++];
    rp.w2[j] = w[i]; gp.w2[j] = grads + gl.off[i++];
    gp.b2[j] = grads + gl.off[i++];
  }
  gp.attn_gamma = grads + gl.off[i++];
  if (pl->cfg.rope) ++i;
  rp.wqkv = w[i]; gp.wqkv = grads + gl.off[i++];
  rp.wo = w[i]; gp.wo = grads + gl.off[i++];
}

// Backward of x_out = x_in + ConvSwiGLU(norm(x_in)) (models/mss_tflocoformer.py:443-447, :459-462, :626-655).
// dx holds dL/dx_out on entry and dL/dx_in on exit.
static int ffn_backward(const tfl_plan* pl, const char* packed, int layer, int axis, int j, const float* x_in, float* dx,
                        Dims d, const TrainWs& tw, char* wsp, const GradPtrs& gp, const RawPtrs& rp, cudaStream_t st) {
  NvtxRange nvtx_range("tfl::conv_swiglu_ffn_bwd");
  const tfl_config& c = pl->cfg;
  const FfnPack& f = pl->lay.paths[(size_t)layer * 2 + axis].ffn[j];
  const int C = c.emb_dim, K = c.conv_kernel, H = f.hidden;
  const int S = axis == TFL_AXIS_FREQ ? d.F : d.Tf;
  const int nseq = axis == TFL_AXIS_FREQ ? d.B * d.Tf : d.B * d.F;
  const long long rows = (long long)d.B * d.Tf * d.F, rows1 = (long long)nseq * (S + K - 1);
  float* xn = (float*)(wsp + tw.fwd.xn);
  float* dxn = (float*)(wsp + tw.dxn);
  float* dg = (float*)(wsp + tw.dg);
  float* hid = (float*)(wsp + tw.hid2);
  float* dh = (float*)(wsp + tw.dh);
  float* nat = (float*)(wsp + tw.nat);
  float* det = det_ptr(tw, wsp);
  float* nat_w1 = nat, *nat_b1 = nat_w1 + (size_t)K * C * 2 * H, *nat_w2 = nat_b1 + 2 * H;
  float* w2t = (float*)(wsp + tw.wt);                 // [K][C][H]:   w2t[t][c][h]  = deconv1d.weight[h][c][t]
  float* w1t = w2t + (size_t)K * C * H;               // [K][2H][C]:  w1t[t][2h+q][c] = conv1d.weight[q*H+h][c][K-1-t]
  const SeqMap xmap = make_seq_map(axis, d.Tf, d.F, C);
  const SeqMap hmap = make_dense_map((long long)(S + K - 1) * H, H);
  const SeqMap h2map = make_dense_map((long long)(S + K - 1) * 2 * H, 2 * H);
  permute(rp.w2[j], w2t, 1, K, C, H, 0, 1, K, (long long)C * K, 0, -1, st);
  permute(rp.w1[j], w1t, K, H, 2, C, -1, (long long)C * K, (long long)H * C * K, K, K - 1, -1, st);
  TFL_CUDA(cudaMemsetAsync(nat, 0, ((size_t)K * C * 2 * H + 2 * H + (size_t)K * H * C) * sizeof(float), st));
  // xn = norm(x_in)
  if (norm_launch(x_in, xn, rows, C, c.num_groups, (const float*)(packed + f.gamma), c.eps, pl->sm_count, st)) return -1;
  // dG[s, j'] = sum_t dY[s, j' + t - (K-1)] . w2t[t]
  TapGemm gd{dx, xmap, S, S + K - 1, K - 1, K, C, w2t, nullptr, H, rows1};
  if (gemm_launch(gd, EpiStoreDense{dg}, st)) return -1;
  // h = conv1d(xn) recomputed; hid = value * silu(gate); dH from dG
  TapGemm g1{xn, xmap, S, S + K - 1, K - 1, K, C, (const float*)(packed + f.w1), (const float*)(packed + f.b1), 2 * H, rows1};
  if (gemm_launch(g1, EpiSwiGLUBwd{dg, hid, dh, H}, st)) return -1;
  // transposed-conv weights: nat_w2[k'][h][c] = sum hid[s, i + k'][h] * dY[s, i][c];  bias: sum dY
  TapWgrad gw2{hid, hmap, S + K - 1, 0, K, H, dx, xmap, S, C, (long long)nseq * S, nat_w2, 0};
  if (wgrad_launch(gw2, pl->sm_count, st, det)) return -1;
  if (colsum_launch(dx, xmap, S, C, (long long)nseq * S, gp.b2[j], pl->sm_count, st, det)) return -1;
  // conv1d weights: nat_w1[k][c][n] = sum xn[s, j' + k - (K-1)][c] * dH[s, j'][n];  bias: sum dH
  TapWgrad gw1{xn, xmap, S, K - 1, K, C, dh, h2map, S + K - 1, 2 * H, rows1, nat_w1, 0};
  if (wgrad_launch(gw1, pl->sm_count, st, det)) return -1;
  if (colsum_launch(dh, h2map, S + K - 1, 2 * H, rows1, nat_b1, pl->sm_count, st, det)) return -1;
  // dxn[s, i] = sum_t dH[s, i + t] . w1t[t]
  TapGemm gx{dh, h2map, S + K - 1, S, 0, K, 2 * H, w1t, nullptr, C, (long long)nseq * S};
  if (gemm_launch(gx, EpiStoreMap{dxn, xmap}, st)) return -1;
  // through the norm, into the residual gradient
  if (norm_bwd_launch(x_in, dxn, dx, rows, C, c.num_groups, (const float*)(packed + f.gamma), c.eps, gp.ffn_gamma[j],
                      pl->sm_count, st, det)) return -1;
  // natural -> reference layouts
  permute(nat_w1, gp.w1[j], 2, H, C, K, 1, 2, 2 * H, (long long)C * 2 * H, 0, -1, st);       // conv1d.weight [2H, C, K]
  permute(nat_b1, gp.b1[j], 1, 1, 2, H, 0, 0, 1, 2, 0, -1, st);                              // conv1d.bias [2H]
  permute(nat_w2, gp.w2[j], 1, H, C, K, 0, C, 1, -(long long)H * C, (long long)(K - 1) * H * C, -1, st);   // deconv1d.weight [H, C, K]
  TFL_LAUNCH_CHECK();
  return 0;
}

// Backward of x_out = x_in + Wo . MHSA(RoPE(qkv(norm(x_in)))) (:452-456, :523-559).  Recomputes q|k|v, o and the
// log-sum-exp from x_in.
static int attn_backward(const tfl_plan* pl, const char* packed, int layer, int axis, const float* x_in, float* dx, Dims d,
                         const TrainWs& tw, char* wsp, const GradPtrs& gp, const RawPtrs& rp, cudaStream_t st) {
  NvtxRange nvtx_range("tfl::rope_attn_bwd");
  const tfl_config& c = pl->cfg;
  const PathPack& p = pl->lay.paths[(size_t)layer * 2 + axis];
  const int C = c.emb_dim, A = c.attention_dim, hd = pl->head_dim, heads = c.n_heads;
  const int L = axis == TFL_AXIS_FREQ ? d.F : d.Tf;
  const int nseq = axis == TFL_AXIS_FREQ ? d.B * d.Tf : d.B * d.F;
  const long long rows = (long long)d.B * d.Tf * d.F;
  float* xn = (float*)(wsp + tw.fwd.xn);
  float* qkv = (float*)(wsp + tw.fwd.qkv);
  float* o = (float*)(wsp + tw.fwd.o);
  float* lse = (float*)(wsp + tw.lse);
  float* Dbuf = (float*)(wsp + tw.dbuf);
  float* dO = (float*)(wsp + tw.dO);
  float* dqkv_h = (float*)(wsp + tw.dqkv_h);
  float* dqkv = (float*)(wsp + tw.dqkv);
  float* dxn = (float*)(wsp + tw.dxn);
  float* det = det_ptr(tw, wsp);
  const SeqMap xmap = make_seq_map(axis, d.Tf, d.F, C);
  const SeqMap omap = make_dense_map((long long)L * A, A);
  const SeqMap qmap = make_dense_map((long long)L * 3 * A, 3 * A);
  // forward recompute up to o (xn, q|k|v, o, lse); x_in is only read on this path
  if (attn_f32(pl, packed, layer, axis, const_cast<float*>(x_in), d, tw.fwd, wsp, st, lse, /*forward_only_to_o=*/true)) return -1;
  // dO = dY . Wo   (aggregate_heads.0.weight is [C, A]: exactly [Kc = C][N = A])
  TapGemm g_do{dx, xmap, L, L, 0, 1, C, rp.wo, nullptr, A, (long long)nseq * L};
  if (gemm_launch(g_do, EpiStoreDense{dO}, st)) return -1;
  // dWo[c][a] = sum_r dY[r][c] * o[r][a]
  TapWgrad gwo{dx, xmap, L, 0, 1, C, o, omap, L, A, (long long)nseq * L, gp.wo, 0};
  if (wgrad_launch(gwo, pl->sm_count, st, det)) return -1;
  const size_t per = (size_t)nseq * heads * L * hd;
  const float scale = 1.0f / sqrtf((float)hd);
  if (g_gemm_tf32 && hd % 2 == 0 && hd > 8 && hd <= 32) {   // tensor-core form (tf32 mma.sync), 64 rows per block
    dim3 grid64((L + 63) / 64, heads, nseq);
    if (g_gemm_mode == 2 && hd <= 16) {
      attn_bwd_dq_bf16_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, dO, lse, dqkv_h, Dbuf, L, hd, heads, scale);
      TFL_LAUNCH_CHECK();
      attn_bwd_dkv_bf16_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, dO, lse, Dbuf, dqkv_h + per, dqkv_h + 2 * per, L, hd, heads, scale);
    } else if (g_gemm_mode == 2) {
      attn_bwd_dq_bf16_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, dO, lse, dqkv_h, Dbuf, L, hd, heads, scale);
      TFL_LAUNCH_CHECK();
      attn_bwd_dkv_bf16_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, dO, lse, Dbuf, dqkv_h + per, dqkv_h + 2 * per, L, hd, heads, scale);
    } else if (hd <= 16) {
      attn_bwd_dq_mma_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, dO, lse, dqkv_h, Dbuf, L, hd, heads, scale);
      TFL_LAUNCH_CHECK();
      attn_bwd_dkv_mma_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, dO, lse, Dbuf, dqkv_h + per, dqkv_h + 2 * per, L, hd, heads, scale);
    } else {
      attn_bwd_dq_mma_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, dO, lse, dqkv_h, Dbuf, L, hd, heads, scale);
      TFL_LAUNCH_CHECK();
      attn_bwd_dkv_mma_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, dO, lse, Dbuf, dqkv_h + per, dqkv_h + 2 * per, L, hd, heads, scale);
    }
    TFL_LAUNCH_CHECK();
  } else {
  dim3 grid((L + 127) / 128, heads, nseq);
#define DQ_CASE(HD) attn_bwd_dq_kernel<HD><<<grid, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, dO, lse, dqkv_h, Dbuf, L, hd, heads, scale)
  if (hd <= 8) DQ_CASE(8); else if (hd <= 16) DQ_CASE(16); else if (hd <= 32) DQ_CASE(32); else DQ_CASE(64);
#undef DQ_CASE
  TFL_LAUNCH_CHECK();
#define DKV_CASE(HD) attn_bwd_dkv_kernel<HD><<<grid, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, dO, lse, Dbuf, dqkv_h + per, dqkv_h + 2 * per, L, hd, heads, scale)
  if (hd <= 8) DKV_CASE(8); else if (hd <= 16) DKV_CASE(16); else if (hd <= 32) DKV_CASE(32); else DKV_CASE(64);
#undef DKV_CASE
  TFL_LAUNCH_CHECK();
  }
  {
    const long long total = (long long)3 * nseq * heads * L * (hd / 2);
    long long blocks = (total + 255) / 256;
    if (blocks > (long long)pl->sm_count * 16) blocks = (long long)pl->sm_count * 16;
    qkv_unrope_kernel<<<(unsigned)blocks, 256, 0, st>>>(dqkv_h, dqkv, nseq, heads, L, hd, c.rope ? (const float*)(packed + p.rope) : nullptr);
    TFL_LAUNCH_CHECK();
  }
  // dWqkv[n][c] = sum_r dQKV[r][n] * xn[r][c]   (qkv.weight is [3A, C])
  TapWgrad gwq{dqkv, qmap, L, 0, 1, 3 * A, xn, xmap, L, C, (long long)nseq * L, gp.wqkv, 0};
  if (wgrad_launch(gwq, pl->sm_count, st, det)) return -1;
  // dxn = dQKV . Wqkv   (qkv.weight [3A, C] is exactly [Kc = 3A][N = C])
  TapGemm g_dx{dqkv, qmap, L, L, 0, 1, 3 * A, rp.wqkv, nullptr, C, (long long)nseq * L};
  if (gemm_launch(g_dx, EpiStoreMap{dxn, xmap}, st)) return -1;
  return norm_bwd_launch(x_in, dxn, dx, rows, C, c.num_groups, (const float*)(packed + p.attn_gamma), c.eps, gp.attn_gamma,
                         pl->sm_count, st, det);
}

// sub-blocks of the network in forward order: (layer, axis, kind) with kind 0 / 1 = ffn index, 2 = attention
struct SubBlock { int layer, axis, kind; };
static std::vector<SubBlock> sub_blocks(const tfl_plan* pl) {
  std::vector<SubBlock> v;
  for (int layer = 0; layer < pl->cfg.n_layers; ++layer) {
    const int first = pl->cfg.tf_order == 0 ? TFL_AXIS_FREQ : TFL_AXIS_TIME;
    for (int a = 0; a < 2; ++a) {
      const int axis = a == 0 ? first : 1 - first;
      if (pl->cfg.macaron) v.push_back({layer, axis, 1});
      v.push_back({layer, axis, 2});
      v.push_back({layer, axis, 0});
    }
  }
  return v;
}

struct Tf32Scope {   // GEMM arithmetic of one training call = TFL_OPT_TRAIN_MODE (0 fp32, 1 tf32, 2 bf16 MMAs); restored on exit
  int prev;
  Tf32Scope() : prev(g_gemm_mode) { const int m = tfl_option(TFL_OPT_TRAIN_MODE); g_gemm_mode = m < 0 ? 0 : (m > 2 ? 2 : m); }
  ~Tf32Scope() { g_gemm_mode = prev; }
};

static int check_train(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights) {
  TFL_CHECK(pl && packed && w, "null argument");
  TFL_CHECK(n_weights == tfl_num_weight_tensors(pl), "expected %d weight tensors, got %d", tfl_num_weight_tensors(pl), n_weights);
  TFL_CHECK(pl->cfg.emb_dim <= 256, "training kernels support emb_dim <= 256");
  if (ensure_device_ready()) return -1;
  return timeout_pending();
}

// ---- pieces of a training step, shared by the MSS step and the separator / blocks autograd entry points ----------------
static float* ckpt_slot(const TrainWs& tw, char* wsp, Dims d, int C, size_t k) {
  return (float*)(wsp + tw.ckpt + k * (size_t)d.B * d.Tf * d.F * C * sizeof(float));
}

// The sub-blocks with the residual stream kept: x_k = input of sub-block k lives in checkpoint slot k (slot 0 must hold
// the blocks' input; slot n_sub receives their output).  Mixed mode (TFL_OPT_TRAIN_MODE 2, the reference's bf16-autocast
// forward): sub-blocks the tcgen05 kernels cover run on them -- the fused FFN kernel writes slot k + 1 straight from
// slot k --, the rest stays on the fp32 path.
static int saved_blocks_forward(const tfl_plan* pl, const char* pk, Dims d, const TrainWs& tw, char* wsp, bool mixed,
                                cudaStream_t st) {
  const tfl_config& c = pl->cfg;
  const size_t act_bytes = (size_t)d.B * d.Tf * d.F * c.emb_dim * sizeof(float);
  const std::vector<SubBlock> subs = sub_blocks(pl);
  for (size_t k = 0; k < subs.size(); ++k) {
    const SubBlock& sb = subs[k];
    float* x_in = ckpt_slot(tw, wsp, d, c.emb_dim, k);
    float* x_out = ckpt_slot(tw, wsp, d, c.emb_dim, k + 1);
    if (sb.kind == 2) {
      TFL_CUDA(cudaMemcpyAsync(x_out, x_in, act_bytes, cudaMemcpyDeviceToDevice, st));
      if (mixed && tw.fwd16_base != 0) {
        if (attn_bf16(pl, pk, sb.layer, sb.axis, x_out, d, tw.fwd16, wsp + tw.fwd16_base, st)) return -1;
      } else if (attn_f32(pl, pk, sb.layer, sb.axis, x_out, d, tw.fwd, wsp, st)) return -1;
    } else {
      const FfnPack& f = pl->lay.paths[(size_t)sb.layer * 2 + sb.axis].ffn[sb.kind];
      FfnTcGeom geom;
      if (mixed && ffn_tc_geometry(c.emb_dim, f.hidden, c.conv_kernel, c.num_groups, &geom)) {
        if (tc_ffn(pl, pk, sb.layer, sb.axis, sb.kind, x_in, x_out, d.B, d.Tf, d.F, st)) return -1;
      } else {
        TFL_CUDA(cudaMemcpyAsync(x_out, x_in, act_bytes, cudaMemcpyDeviceToDevice, st));
        if (ffn_f32(pl, pk, sb.layer, sb.axis, sb.kind, x_out, d, tw.fwd, wsp, st)) return -1;
      }
    }
  }
  return 0;
}

// Backward of the sub-blocks: tw.dx holds dL/d(blocks output) on entry and dL/d(blocks input) on exit; the parameter
// gradients land in their slices of `grads` (accumulated: the caller zeroes the buffer).
static int blocks_backward(const tfl_plan* pl, const char* pk, const float* const* w, const GradLayout& gl, float* grads,
                           Dims d, const TrainWs& tw, char* wsp, cudaStream_t st) {
  float* dx = (float*)(wsp + tw.dx);
  const std::vector<SubBlock> subs = sub_blocks(pl);
  for (int k = (int)subs.size() - 1; k >= 0; --k) {
    const SubBlock& sb = subs[k];
    const float* x_in = ckpt_slot(tw, wsp, d, pl->cfg.emb_dim, (size_t)k);
    GradPtrs gp; RawPtrs rp;
    path_ptrs(pl, gl, grads, w, sb.layer, sb.axis, gp, rp);
    if (sb.kind == 2) { if (attn_backward(pl, pk, sb.layer, sb.axis, x_in, dx, d, tw, wsp, gp, rp, st)) return -1; }
    else if (ffn_backward(pl, pk, sb.layer, sb.axis, sb.kind, x_in, dx, d, tw, wsp, gp, rp, st)) return -1;
  }
  return 0;
}

// Decoder backward from dEst [B, S, Tf, F, 2]: deconv.weight / deconv.bias gradients, and dL/dx (decoder input x) into
// tw.dx.
static int dec_backward(const tfl_plan* pl, const char* pk, const GradLayout& gl, float* grads, int n_w, const float* x,
                        const float* dest, Dims d, const TrainWs& tw, char* wsp, cudaStream_t st) {
  const int C = pl->cfg.emb_dim, S = pl->cfg.n_src;
  const size_t N = (size_t)d.B * d.Tf * d.F;
  const int cthreads = (C + 31) / 32 * 32;
  float* nat = (float*)(wsp + tw.nat);
  float* dx = (float*)(wsp + tw.dx);
  // weights: natural layout [9][8][C] -> deconv.weight [C, 2S, 3, 3]
  TFL_CUDA(cudaMemsetAsync(nat, 0, ((size_t)9 * 8 * C + 8) * sizeof(float), st));
  if (float* det = det_ptr(tw, wsp)) {
    dec_wgrad_kernel<true><<<DET_DEC_BLOCKS, cthreads, 0, st>>>(x, dest, d.Tf, d.F, C, 2 * S, (long long)N, det);
    TFL_LAUNCH_CHECK();
    if (ordered_sum(det, DET_DEC_BLOCKS, (long long)72 * C, (long long)72 * C, nat, st)) return -1;
  } else {
    dec_wgrad_kernel<false><<<pl->sm_count * 4, cthreads, 0, st>>>(x, dest, d.Tf, d.F, C, 2 * S, (long long)N, nat);
    TFL_LAUNCH_CHECK();
  }
  permute(nat, grads + gl.off[n_w - 2], C, 2 * S, 3, 3, 1, C, (long long)3 * 8 * C, (long long)8 * C, 0, -1, st);
  dec_bias_grad_kernel<<<2 * S, 256, 0, st>>>(dest, d.B, S, (long long)d.Tf * d.F, grads + gl.off[n_w - 1]);
  TFL_LAUNCH_CHECK();
  const size_t smem = (size_t)9 * C * 8 * sizeof(float);
  TFL_CUDA(opt_in_smem(dec_dgrad_kernel, smem));
  dec_dgrad_kernel<<<pl->sm_count * 8, 256, smem, st>>>(dest, d.Tf, d.F, C, 2 * S, (const float*)(pk + pl->lay.dec_w), dx,
                                                       (long long)N);
  TFL_LAUNCH_CHECK();
  return 0;
}

// Encoder backward from tw.dx = dL/d(encoder output): v = conv(spec) recomputed into xn, then GroupNorm(1, C) backward
// and the conv weight gradient; with d_spec, also dL/d spec [B, Tf, F, 2] (overwritten).
static int enc_backward(const tfl_plan* pl, const char* pk, const GradLayout& gl, float* grads, const float* spec, Dims d,
                        const TrainWs& tw, char* wsp, cudaStream_t st, float* d_spec = nullptr) {
  const tfl_config& c = pl->cfg;
  const int C = c.emb_dim, B = d.B, Tf = d.Tf, F = d.F;
  const int cthreads = (C + 31) / 32 * 32;
  float* nat = (float*)(wsp + tw.nat);
  float* dx = (float*)(wsp + tw.dx);
  float* v = (float*)(wsp + tw.fwd.xn);
  double* part = (double*)(wsp + tw.fwd.gln_part);
  float* stats = (float*)(wsp + tw.fwd.gln_stats);
  double* sums = (double*)(wsp + tw.enc_sums);
  const size_t smem = ((size_t)9 * 2 * C + C) * sizeof(float);
  enc_conv_kernel<2><<<dim3(tw.fwd.gln_blocks, B), 256, smem, st>>>(spec, Tf, F, C, (const float*)(pk + pl->lay.enc_w),
                                                                   (const float*)(pk + pl->lay.enc_b), v, part);
  TFL_LAUNCH_CHECK();
  gln_finalize_kernel<<<B, 256, 0, st>>>(part, tw.fwd.gln_blocks, (double)Tf * F * C, c.eps, stats);
  TFL_LAUNCH_CHECK();
  TFL_CUDA(cudaMemsetAsync(sums, 0, (size_t)B * 2 * sizeof(double), st));
  TFL_CUDA(cudaMemsetAsync(nat, 0, ((size_t)18 * C + C) * sizeof(float), st));
  if (float* det = det_ptr(tw, wsp)) {
    // (dgw, dgb) partials [B][blocks][2C], then the statistics partials [B][blocks][2] in double
    const long long parts = (long long)B * DET_ENC_BLOCKS;
    double* sums_part = (double*)((char*)det + align_up((size_t)parts * 2 * C * sizeof(float)));
    const dim3 grid(DET_ENC_BLOCKS, B);
    enc_gln_bwd_stats_kernel<true><<<grid, cthreads, 0, st>>>(v, dx, (long long)Tf * F, C, stats, (const float*)(pk + pl->lay.gln_w),
                                                              det, nullptr, sums_part);
    TFL_LAUNCH_CHECK();
    if (ordered_sum(det, (int)parts, 2LL * C, (long long)C, grads + gl.off[2], st)) return -1;
    if (ordered_sum(det + C, (int)parts, 2LL * C, (long long)C, grads + gl.off[3], st)) return -1;
    if (ordered_sum(sums_part, DET_ENC_BLOCKS, 2LL, 2LL, sums, st, B, 2LL * DET_ENC_BLOCKS, 2LL)) return -1;
    enc_wgrad_kernel<2, true><<<grid, cthreads, 0, st>>>(v, dx, spec, Tf, F, C, stats, sums, (const float*)(pk + pl->lay.gln_w),
                                                         det, nullptr);
    TFL_LAUNCH_CHECK();
    if (ordered_sum(det, (int)parts, 19LL * C, 19LL * C, nat, st)) return -1;   // [18 C] weights, then [C] bias, as in nat
  } else {
    enc_gln_bwd_stats_kernel<false><<<dim3(pl->sm_count * 2, B), cthreads, 0, st>>>(v, dx, (long long)Tf * F, C, stats, (const float*)(pk + pl->lay.gln_w),
                                                                                    grads + gl.off[2], grads + gl.off[3], sums);
    TFL_LAUNCH_CHECK();
    enc_wgrad_kernel<2, false><<<dim3(pl->sm_count * 2, B), cthreads, 0, st>>>(v, dx, spec, Tf, F, C, stats, sums, (const float*)(pk + pl->lay.gln_w),
                                                                               nat, nat + (size_t)18 * C);
    TFL_LAUNCH_CHECK();
  }
  // natural [9][ci][C] -> conv.0.weight [C, ci, 3, 3]
  permute(nat, grads + gl.off[0], 1, C, 2, 9, 0, 1, C, (long long)2 * C, 0, -1, st);
  permute(nat + (size_t)18 * C, grads + gl.off[1], 1, 1, 1, C, 0, 0, 0, 1, 0, -1, st);
  TFL_LAUNCH_CHECK();
  if (d_spec != nullptr) {
    const size_t ism = ((size_t)18 * C + (size_t)(ENC_IG_TT + 2) * (ENC_IG_FT + 2) * 18) * sizeof(float);
    TFL_CUDA(opt_in_smem(enc_input_grad_kernel<2>, ism));
    const dim3 grid((F + ENC_IG_FT - 1) / ENC_IG_FT, (Tf + ENC_IG_TT - 1) / ENC_IG_TT, B);
    enc_input_grad_kernel<2><<<grid, 256, ism, st>>>(v, dx, Tf, F, C, stats, sums, (const float*)(pk + pl->lay.gln_w),
                                                     (const float*)(pk + pl->lay.enc_w), d_spec);
    TFL_LAUNCH_CHECK();
  }
  return 0;
}

// Shared argument checks of the saved-forward / backward pairs; fills the workspace plan.
static int check_saved(const tfl_plan* pl, const void* packed, int B, int Tf, int F, bool conv, size_t ws_bytes, TrainWs* tw,
                       int T = 0) {
  TFL_CHECK(pl && packed, "null argument");
  TFL_CHECK(B >= 1 && Tf >= 1 && F >= 1, "empty input (batch %d, frames %d, bins %d)", B, Tf, F);
  TFL_CHECK(pl->cfg.emb_dim <= 256, "training kernels support emb_dim <= 256");
  if (conv) {
    TFL_CHECK(pl->cfg.enc_in_ch == 2, "this entry point needs a plan with the conv encoder / decoder (enc_in_ch == 2)");
    TFL_CHECK(pl->cfg.n_src * 2 <= 8, "the decoder backward supports at most 4 sources");
  } else {
    TFL_CHECK(pl->cfg.enc_in_ch == 0, "this entry point needs a blocks-only plan (enc_in_ch == 0)");
  }
  *tw = plan_train_ws(pl, B, Tf, F, T, 0, 0, /*saved=*/true);
  TFL_CHECK(ws_bytes >= tw->total, "workspace too small (%zu < %zu)", ws_bytes, tw->total);
  if (ensure_device_ready()) return -1;
  return timeout_pending();
}

// The TFLocoformerMSS pair: plan with STFT and conv encoder, T past the reflect padding; (Tf, F) from T.
static int check_mss(const tfl_plan* pl, const void* packed, int B, int T, size_t ws_bytes, TrainWs* tw, Dims* d) {
  TFL_CHECK(pl && packed, "null argument");
  const tfl_config& c = pl->cfg;
  TFL_CHECK(c.n_fft > 0 && c.enc_in_ch == 2, "this entry point needs the full TFLocoformerMSS plan (STFT + conv encoder)");
  TFL_CHECK(B >= 1 && T > c.n_fft / 2, "reflect padding needs more than n_fft/2 = %d samples (got %d)", c.n_fft / 2, T);
  *d = Dims{B, 1 + T / c.hop, c.n_fft / 2 + 1};
  return check_saved(pl, packed, B, d->Tf, d->F, true, ws_bytes, tw, T);
}

// tfl_sep_train_backward, with dL/d spec into d_spec when it is not NULL.
static int sep_backward(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights, const float* d_est,
                        const float* spec, int B, int Tf, int F, float* grads, void* workspace, size_t ws_bytes,
                        float* d_spec, cudaStream_t st) {
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TrainWs tw;
  if (check_saved(pl, packed, B, Tf, F, true, ws_bytes, &tw)) return -1;
  TFL_CHECK(d_est && spec && grads && workspace, "null argument");
  const Dims d{B, Tf, F};
  const char* pk = (const char*)packed;
  char* wsp = (char*)workspace;
  const GradLayout gl = grad_layout(pl);
  TFL_CUDA(cudaMemsetAsync(grads, 0, (size_t)gl.total * sizeof(float), st));
  const float* x = ckpt_slot(tw, wsp, d, pl->cfg.emb_dim, (size_t)tw.n_sub);
  if (dec_backward(pl, pk, gl, grads, n_weights, x, d_est, d, tw, wsp, st)) return -1;
  if (blocks_backward(pl, pk, w, gl, grads, d, tw, wsp, st)) return -1;
  return enc_backward(pl, pk, gl, grads, spec, d, tw, wsp, st, d_spec);
}

}  // namespace tfl

extern "C" {

int64_t tfl_train_grad_layout(const tfl_plan* pl, int64_t* offsets, int64_t* sizes, int n_weights) {
  if (pl == nullptr) return -1;
  const GradLayout g = grad_layout(pl);
  if (offsets != nullptr || sizes != nullptr) {
    if (n_weights != (int)g.off.size()) { set_error("expected %d weight tensors, got %d", (int)g.off.size(), n_weights); return -1; }
    for (size_t i = 0; i < g.off.size(); ++i) {
      if (offsets) offsets[i] = g.off[i];
      if (sizes) sizes[i] = g.size[i];
    }
  }
  return g.total;
}

size_t tfl_train_workspace_bytes(const tfl_plan* pl, int B, int T, int spec_n_fft, int spec_hop) {
  if (pl == nullptr || pl->cfg.n_fft <= 0) return 0;
  return plan_train_ws(pl, B, 1 + T / pl->cfg.hop, pl->cfg.n_fft / 2 + 1, T, spec_n_fft, spec_hop).total;
}

size_t tfl_train_stage_workspace_bytes(const tfl_plan* pl, int B, int Tf, int F) {
  return pl == nullptr ? 0 : plan_train_ws(pl, B, Tf, F, 0, 0, 0).total;
}

// Stage-level backward entry points (parity tests against autograd of the reference modules): dx holds dL/dx_out on entry
// and dL/dx_in on exit; the parameter gradients of the sub-block are ACCUMULATED into their slices of `grads`.
int tfl_conv_swiglu_ffn_bwd(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights, int layer, int axis,
                            int ffn_index, const float* x_in, float* dx, int B, int Tf, int F, float* grads,
                            void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TFL_CHECK(x_in && dx && grads && workspace, "null argument");
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1) && ffn_index >= 0 && ffn_index < pl->n_ffn,
            "bad layer / axis / ffn index");
  const TrainWs tw = plan_train_ws(pl, B, Tf, F, 0, 0, 0);
  TFL_CHECK(ws_bytes >= tw.total, "workspace too small (%zu < %zu)", ws_bytes, tw.total);
  const GradLayout gl = grad_layout(pl);
  GradPtrs gp; RawPtrs rp;
  path_ptrs(pl, gl, grads, w, layer, axis, gp, rp);
  return ffn_backward(pl, (const char*)packed, layer, axis, ffn_index, x_in, dx, Dims{B, Tf, F}, tw, (char*)workspace, gp, rp,
                      (cudaStream_t)stream);
}

int tfl_rope_attn_bwd(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights, int layer, int axis,
                      const float* x_in, float* dx, int B, int Tf, int F, float* grads, void* workspace, size_t ws_bytes,
                      tfl_stream_t stream) {
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TFL_CHECK(x_in && dx && grads && workspace, "null argument");
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1), "bad layer / axis");
  const TrainWs tw = plan_train_ws(pl, B, Tf, F, 0, 0, 0);
  TFL_CHECK(ws_bytes >= tw.total, "workspace too small (%zu < %zu)", ws_bytes, tw.total);
  const GradLayout gl = grad_layout(pl);
  GradPtrs gp; RawPtrs rp;
  path_ptrs(pl, gl, grads, w, layer, axis, gp, rp);
  return attn_backward(pl, (const char*)packed, layer, axis, x_in, dx, Dims{B, Tf, F}, tw, (char*)workspace, gp, rp,
                       (cudaStream_t)stream);
}

// One training step up to the gradients: forward (fp32, sub-block inputs saved) -> MSSLoss -> backward.
//   mixture [B][T], targets [n_src][B][T] (mono, as train.py:103-110 down-mixes them);  grads: flat buffer of
//   tfl_train_grad_layout (overwritten);  loss_out[0] = total_loss, then {si_sdr, l1, spectral} per source;
//   est_audio (optional) [n_src][B][T] = the forward's separated audio.
// Dropout is not applied (parity is defined for p = 0, SURVEY section 8(d) config 5).
int tfl_train_forward_backward(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights,
                               const float* mixture, const float* targets, int B, int T, const tfl_loss_config* loss,
                               float* grads, float* loss_out, float* est_audio, void* workspace, size_t ws_bytes,
                               tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::train_forward_backward");
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TFL_CHECK(mixture && targets && loss && grads && loss_out && workspace, "null argument");
  const tfl_config& c = pl->cfg;
  TFL_CHECK(c.n_fft > 0 && c.enc_in_ch == 2, "training needs the full TFLocoformerMSS plan (STFT + conv encoder)");
  TFL_CHECK(B >= 1 && T > c.n_fft / 2, "reflect padding needs more than n_fft/2 = %d samples (got %d)", c.n_fft / 2, T);
  const bool spec_on = loss->spectral_weight > 0.f;
  const int l_fft = spec_on ? loss->spec_n_fft : 0, l_hop = spec_on ? loss->spec_hop : 0;
  if (spec_on) {
    TFL_CHECK(l_fft >= 16 && l_fft <= 8192 && (l_fft & (l_fft - 1)) == 0 && l_hop > 0 && l_hop <= l_fft, "bad spectral-loss STFT size");
    TFL_CHECK(T > l_fft / 2, "spectral loss: reflect padding needs more than %d samples", l_fft / 2);
  }
  const int Tf = 1 + T / c.hop, F = c.n_fft / 2 + 1, C = c.emb_dim, S = c.n_src;
  const Dims d{B, Tf, F};
  const TrainWs tw = plan_train_ws(pl, B, Tf, F, T, l_fft, l_hop);
  TFL_CHECK(ws_bytes >= tw.total, "workspace too small (%zu < %zu)", ws_bytes, tw.total);
  cudaStream_t st = (cudaStream_t)stream;
  char* wsp = (char*)workspace;
  const char* pk = (const char*)packed;
  const GradLayout gl = grad_layout(pl);
  float* spec = (float*)(wsp + tw.fwd.spec);
  float* est = (float*)(wsp + tw.fwd.est);
  float* audio = (float*)(wsp + tw.audio);
  float* daudio = (float*)(wsp + tw.daudio);
  float* dest = (float*)(wsp + tw.dest);
  float* det = det_ptr(tw, wsp);
  TFL_CUDA(cudaMemsetAsync(grads, 0, (size_t)gl.total * sizeof(float), st));

  // ---------------- forward ----------------
  // The residual stream is kept (saved_blocks_forward): x_0 = encoder output, x_n_sub = decoder input.  Mixed mode runs
  // the encoder / decoder in the tf32 arithmetic of the bf16 inference path; the whole backward pass stays on the tf32 /
  // fp32 GEMM path.
  const bool mixed = tfl_option(TFL_OPT_TRAIN_MODE) >= 2;
  const int enc_prec = mixed ? TFL_PRECISION_BF16 : TFL_PRECISION_FP32;
  if (tfl_stft(pl, packed, mixture, B, T, spec, stream)) return -1;
  if (enc_conv_gln_any(pl, packed, spec, B, Tf, F, ckpt_slot(tw, wsp, d, C, 0), workspace, ws_bytes, enc_prec, stream)) return -1;
  if (saved_blocks_forward(pl, pk, d, tw, wsp, mixed, st)) return -1;
  const float* x = ckpt_slot(tw, wsp, d, C, (size_t)tw.n_sub);   // decoder input
  if (dec_conv_any(pl, packed, x, B, Tf, F, est, enc_prec, stream)) return -1;
  if (tfl_istft_ola(pl, packed, est, B, Tf, T, audio, stream)) return -1;
  if (est_audio != nullptr)
    TFL_CUDA(cudaMemcpyAsync(est_audio, audio, (size_t)S * B * T * sizeof(float), cudaMemcpyDeviceToDevice, st));

  // ---------------- loss and its gradient w.r.t. the separated audio ----------------
  const int rows = S * B;
  LossCfg lc{loss->si_sdr_weight, loss->l1_weight, loss->spectral_weight, loss->eps, S, B, T, l_fft, l_fft > 0 ? ilog2(l_fft) : 0,
             l_hop, tw.l_frames};
  double* s5 = (double*)(wsp + tw.s5);
  if (tfl_pair_stats(audio, targets, rows, T, s5, (double*)(wsp + tw.stats_scratch), (size_t)rows * STATS_BLOCKS * 5 * sizeof(double), stream)) return -1;
  float* coef = (float*)(wsp + tw.coef);
  double* loss_rows = (double*)(wsp + tw.loss_rows);
  double* l1_rows = (double*)(wsp + tw.l1_rows);
  double* spec_rows = (double*)(wsp + tw.spec_rows);
  TFL_CUDA(cudaMemsetAsync(l1_rows, 0, rows * sizeof(double), st));
  TFL_CUDA(cudaMemsetAsync(spec_rows, 0, rows * sizeof(double), st));
  sisdr_coef_kernel<<<(rows + 63) / 64, 64, 0, st>>>(s5, lc, coef, loss_rows);
  TFL_LAUNCH_CHECK();
  const float* frames = nullptr;
  long long spec_count = 1;
  if (spec_on) {
    float2* ltw = (float2*)(wsp + tw.ltab_tw);
    float* lwin = (float*)(wsp + tw.ltab_win);
    fft_tables_kernel<<<(l_fft + 255) / 256, 256, 0, st>>>(ltw, lwin, l_fft);
    TFL_LAUNCH_CHECK();
    float2* se = (float2*)(wsp + tw.lspec_e);
    float2* stt = (float2*)(wsp + tw.lspec_t);
    const size_t fsm = (size_t)l_fft * sizeof(float2);
    TFL_CUDA(opt_in_smem(stft_kernel, fsm));
    stft_kernel<<<dim3(tw.l_frames, rows), 256, fsm, st>>>(audio, T, l_fft, lc.l_log, l_hop, tw.l_frames, ltw, lwin, (float*)se);
    TFL_LAUNCH_CHECK();
    stft_kernel<<<dim3(tw.l_frames, rows), 256, fsm, st>>>(targets, T, l_fft, lc.l_log, l_hop, tw.l_frames, ltw, lwin, (float*)stt);
    TFL_LAUNCH_CHECK();
    const long long per_row = (long long)tw.l_frames * tw.l_freq;
    spec_count = (long long)B * per_row;
    if (det != nullptr) {
      double* part = (double*)det;
      spec_loss_kernel<true><<<dim3(DET_LOSS_BLOCKS, rows), 256, 0, st>>>(se, stt, per_row, loss->spectral_weight / (float)spec_count, part);
      TFL_LAUNCH_CHECK();
      if (ordered_sum(part, DET_LOSS_BLOCKS, 1LL, 1LL, spec_rows, st, rows, (long long)DET_LOSS_BLOCKS, 1LL)) return -1;
    } else {
      spec_loss_kernel<false><<<dim3(pl->sm_count, rows), 256, 0, st>>>(se, stt, per_row, loss->spectral_weight / (float)spec_count, spec_rows);
      TFL_LAUNCH_CHECK();
    }
    TFL_CUDA(opt_in_smem(stft_adj_frames_kernel, fsm));
    stft_adj_frames_kernel<<<dim3(tw.l_frames, rows), 256, fsm, st>>>(se, l_fft, lc.l_log, tw.l_frames, ltw, lwin, (float*)(wsp + tw.lframes));
    TFL_LAUNCH_CHECK();
    frames = (const float*)(wsp + tw.lframes);
  }
  if (det != nullptr) {
    double* part = (double*)det;
    loss_grad_kernel<true><<<dim3(DET_LOSS_BLOCKS * 2, rows), 256, 0, st>>>(audio, targets, coef, frames, lc, daudio, part);
    TFL_LAUNCH_CHECK();
    if (ordered_sum(part, DET_LOSS_BLOCKS * 2, 1LL, 1LL, l1_rows, st, rows, (long long)DET_LOSS_BLOCKS * 2, 1LL)) return -1;
  } else {
    loss_grad_kernel<false><<<dim3(pl->sm_count * 2, rows), 256, 0, st>>>(audio, targets, coef, frames, lc, daudio, l1_rows);
    TFL_LAUNCH_CHECK();
  }
  loss_finish_kernel<<<1, 32, 0, st>>>(loss_rows, l1_rows, spec_on ? spec_rows : nullptr, lc, spec_count, loss_out);
  TFL_LAUNCH_CHECK();

  // ---------------- backward ----------------
  {   // iSTFT + overlap-add
    const size_t fsm = (size_t)c.n_fft * sizeof(float2);
    TFL_CUDA(opt_in_smem(istft_bwd_kernel, fsm));
    istft_bwd_kernel<<<dim3(Tf, S, B), 256, fsm, st>>>(daudio, S, B, T, c.n_fft, ilog2(c.n_fft), c.hop, Tf,
                                                       (const float2*)(pk + pl->lay.twiddle), (const float*)(pk + pl->lay.window), dest);
    TFL_LAUNCH_CHECK();
  }
  if (dec_backward(pl, pk, gl, grads, n_weights, x, dest, d, tw, wsp, st)) return -1;
  if (blocks_backward(pl, pk, w, gl, grads, d, tw, wsp, st)) return -1;
  return enc_backward(pl, pk, gl, grads, spec, d, tw, wsp, st);
}

size_t tfl_sep_train_workspace_bytes(const tfl_plan* pl, int B, int Tf, int F) {
  return pl == nullptr ? 0 : plan_train_ws(pl, B, Tf, F, 0, 0, 0, /*saved=*/true).total;
}

// TFLocoformerSeparator forward with the sub-block inputs saved in `workspace` for tfl_sep_train_backward: the stages of
// tfl_separator_forward in the arithmetic the MSS training step uses for TFL_OPT_TRAIN_MODE.
int tfl_sep_train_forward(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* est,
                          void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::sep_train_forward");
  Tf32Scope tf32_scope;
  TrainWs tw;
  if (check_saved(pl, packed, B, Tf, F, true, ws_bytes, &tw)) return -1;
  TFL_CHECK(spec && est && workspace, "null argument");
  const Dims d{B, Tf, F};
  const bool mixed = tfl_option(TFL_OPT_TRAIN_MODE) >= 2;
  const int prec = mixed ? TFL_PRECISION_BF16 : TFL_PRECISION_FP32;
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  if (enc_conv_gln_any(pl, packed, spec, B, Tf, F, ckpt_slot(tw, wsp, d, pl->cfg.emb_dim, 0), workspace, ws_bytes, prec,
                       stream)) return -1;
  if (saved_blocks_forward(pl, (const char*)packed, d, tw, wsp, mixed, st)) return -1;
  return dec_conv_any(pl, packed, ckpt_slot(tw, wsp, d, pl->cfg.emb_dim, (size_t)tw.n_sub), B, Tf, F, est, prec, stream);
}

// Backward of tfl_sep_train_forward from dEst [B, S, Tf, F, 2] (same spec, packed image and workspace as the forward):
// every parameter gradient into `grads` (tfl_train_grad_layout, overwritten).  No gradient for spec.
int tfl_sep_train_backward(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights, const float* d_est,
                           const float* spec, int B, int Tf, int F, float* grads, void* workspace, size_t ws_bytes,
                           tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::sep_train_backward");
  return sep_backward(pl, packed, w, n_weights, d_est, spec, B, Tf, F, grads, workspace, ws_bytes, nullptr,
                      (cudaStream_t)stream);
}

// tfl_sep_train_backward plus the input gradient d_spec [B, Tf, F, 2] (overwritten).
int tfl_sep_train_backward_input(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights,
                                 const float* d_est, const float* spec, int B, int Tf, int F, float* grads, void* workspace,
                                 size_t ws_bytes, tfl_stream_t stream, float* d_spec) {
  NvtxRange nvtx_range("tfl::sep_train_backward_input");
  TFL_CHECK(d_spec, "null argument");
  return sep_backward(pl, packed, w, n_weights, d_est, spec, B, Tf, F, grads, workspace, ws_bytes, d_spec,
                      (cudaStream_t)stream);
}

size_t tfl_mss_train_workspace_bytes(const tfl_plan* pl, int B, int T) {
  if (pl == nullptr || pl->cfg.n_fft <= 0 || B < 1 || T < 1) return 0;
  return plan_train_ws(pl, B, 1 + T / pl->cfg.hop, pl->cfg.n_fft / 2 + 1, T, 0, 0, /*saved=*/true).total;
}

// TFLocoformerMSS forward with the sub-block inputs and the spectrogram saved in `workspace` for tfl_mss_train_backward:
// the forward of tfl_train_forward_backward (STFT, encoder, saved blocks, decoder, iSTFT) without the loss.
int tfl_mss_train_forward(const tfl_plan* pl, const void* packed, const float* mixture, int B, int T, float* audio,
                          float* est, void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::mss_train_forward");
  Tf32Scope tf32_scope;
  TrainWs tw;
  Dims d;
  if (check_mss(pl, packed, B, T, ws_bytes, &tw, &d)) return -1;
  TFL_CHECK(mixture && workspace, "null argument");
  const int C = pl->cfg.emb_dim;
  const bool mixed = tfl_option(TFL_OPT_TRAIN_MODE) >= 2;
  const int prec = mixed ? TFL_PRECISION_BF16 : TFL_PRECISION_FP32;
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  float* spec = (float*)(wsp + tw.fwd.spec);
  float* e = est != nullptr ? est : (float*)(wsp + tw.fwd.est);
  if (tfl_stft(pl, packed, mixture, B, T, spec, stream)) return -1;
  if (enc_conv_gln_any(pl, packed, spec, B, d.Tf, d.F, ckpt_slot(tw, wsp, d, C, 0), workspace, ws_bytes, prec, stream)) return -1;
  if (saved_blocks_forward(pl, (const char*)packed, d, tw, wsp, mixed, st)) return -1;
  if (dec_conv_any(pl, packed, ckpt_slot(tw, wsp, d, C, (size_t)tw.n_sub), B, d.Tf, d.F, e, prec, stream)) return -1;
  if (audio != nullptr) return tfl_istft_ola(pl, packed, e, B, d.Tf, T, audio, stream);
  return 0;
}

// Backward of tfl_mss_train_forward from d_audio [S][B][T] or d_est [B][S][Tf][F][2] (exactly one): every parameter
// gradient into `grads` (tfl_train_grad_layout, overwritten) and, when d_mixture is not NULL, dL/d mixture [B][T].
int tfl_mss_train_backward(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights, const float* d_audio,
                           const float* d_est, int B, int T, float* grads, float* d_mixture, void* workspace,
                           size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::mss_train_backward");
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TrainWs tw;
  Dims d;
  if (check_mss(pl, packed, B, T, ws_bytes, &tw, &d)) return -1;
  TFL_CHECK((d_audio == nullptr) != (d_est == nullptr), "exactly one of d_audio / d_est must be given");
  TFL_CHECK(grads && workspace, "null argument");
  const tfl_config& c = pl->cfg;
  const char* pk = (const char*)packed;
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const GradLayout gl = grad_layout(pl);
  const float2* twid = (const float2*)(pk + pl->lay.twiddle);
  const float* win = (const float*)(pk + pl->lay.window);
  const size_t fsm = (size_t)c.n_fft * sizeof(float2);
  TFL_CUDA(cudaMemsetAsync(grads, 0, (size_t)gl.total * sizeof(float), st));
  const float* dest = d_est;
  if (d_audio != nullptr) {
    TFL_CUDA(opt_in_smem(istft_bwd_kernel, fsm));
    istft_bwd_kernel<<<dim3(d.Tf, c.n_src, B), 256, fsm, st>>>(d_audio, c.n_src, B, T, c.n_fft, ilog2(c.n_fft), c.hop, d.Tf,
                                                               twid, win, (float*)(wsp + tw.dest));
    TFL_LAUNCH_CHECK();
    dest = (const float*)(wsp + tw.dest);
  }
  const float* x = ckpt_slot(tw, wsp, d, c.emb_dim, (size_t)tw.n_sub);
  if (dec_backward(pl, pk, gl, grads, n_weights, x, dest, d, tw, wsp, st)) return -1;
  if (blocks_backward(pl, pk, w, gl, grads, d, tw, wsp, st)) return -1;
  float* dspec = d_mixture != nullptr ? (float*)(wsp + tw.dspec) : nullptr;
  if (enc_backward(pl, pk, gl, grads, (const float*)(wsp + tw.fwd.spec), d, tw, wsp, st, dspec)) return -1;
  if (d_mixture == nullptr) return 0;
  float* frames = (float*)(wsp + tw.adj_frames);
  TFL_CUDA(opt_in_smem(stft_adj_frames_kernel, fsm));
  stft_adj_frames_kernel<<<dim3(d.Tf, B), 256, fsm, st>>>((const float2*)dspec, c.n_fft, ilog2(c.n_fft), d.Tf, twid, win, frames);
  TFL_LAUNCH_CHECK();
  long long blocks = ((long long)T + 255) / 256;
  if (blocks > (long long)pl->sm_count * 4) blocks = (long long)pl->sm_count * 4;
  stft_fold_kernel<<<dim3((unsigned)blocks, B), 256, 0, st>>>(frames, T, c.n_fft, c.hop, d.Tf, d_mixture);
  TFL_LAUNCH_CHECK();
  return 0;
}

// The same pair for a blocks-only plan (enc_in_ch == 0): x_in [B, Tf, F, C] -> x_out, and from dL/dx_out the block
// parameter gradients and dL/dx_in.  Tf / F are the two sequence axes (BS-Locoformer: frames and bands).
int tfl_blocks_train_forward(const tfl_plan* pl, const void* packed, const float* x_in, int B, int Tf, int F, float* x_out,
                             void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::blocks_train_forward");
  Tf32Scope tf32_scope;
  TrainWs tw;
  if (check_saved(pl, packed, B, Tf, F, false, ws_bytes, &tw)) return -1;
  TFL_CHECK(x_in && x_out && workspace, "null argument");
  const Dims d{B, Tf, F};
  const int C = pl->cfg.emb_dim;
  const size_t act_bytes = (size_t)B * Tf * F * C * sizeof(float);
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  TFL_CUDA(cudaMemcpyAsync(ckpt_slot(tw, wsp, d, C, 0), x_in, act_bytes, cudaMemcpyDeviceToDevice, st));
  if (saved_blocks_forward(pl, (const char*)packed, d, tw, wsp, tfl_option(TFL_OPT_TRAIN_MODE) >= 2, st)) return -1;
  TFL_CUDA(cudaMemcpyAsync(x_out, ckpt_slot(tw, wsp, d, C, (size_t)tw.n_sub), act_bytes, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int tfl_blocks_train_backward(const tfl_plan* pl, const void* packed, const float* const* w, int n_weights,
                              const float* dx_out, int B, int Tf, int F, float* dx_in, float* grads, void* workspace,
                              size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::blocks_train_backward");
  Tf32Scope tf32_scope;
  if (check_train(pl, packed, w, n_weights)) return -1;
  TrainWs tw;
  if (check_saved(pl, packed, B, Tf, F, false, ws_bytes, &tw)) return -1;
  TFL_CHECK(dx_out && dx_in && grads && workspace, "null argument");
  const Dims d{B, Tf, F};
  const size_t act_bytes = (size_t)B * Tf * F * pl->cfg.emb_dim * sizeof(float);
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const GradLayout gl = grad_layout(pl);
  TFL_CUDA(cudaMemsetAsync(grads, 0, (size_t)gl.total * sizeof(float), st));
  TFL_CUDA(cudaMemcpyAsync(wsp + tw.dx, dx_out, act_bytes, cudaMemcpyDeviceToDevice, st));
  if (blocks_backward(pl, (const char*)packed, w, gl, grads, d, tw, wsp, st)) return -1;
  TFL_CUDA(cudaMemcpyAsync(dx_in, wsp + tw.dx, act_bytes, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// torch.nn.utils.clip_grad_norm_(max_norm): norm_out[0] = total L2 norm, norm_out[1] = the coefficient AdamW applies.
int tfl_grad_clip_norm(const float* grads, int64_t n, float max_norm, float* norm_out, double* scratch, size_t scratch_bytes,
                       tfl_stream_t stream) {
  TFL_CHECK(grads && norm_out && scratch && n >= 1, "null / empty argument");
  const int blocks = 592;
  TFL_CHECK(scratch_bytes >= blocks * sizeof(double), "scratch too small (need %zu bytes)", blocks * sizeof(double));
  sqnorm_partial_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(grads, (long long)n, scratch);
  TFL_LAUNCH_CHECK();
  sqnorm_finish_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(scratch, blocks, max_norm, norm_out);
  TFL_LAUNCH_CHECK();
  return 0;
}

// acc = (overwrite ? 0 : acc) + scale * grads: micro-batch gradient accumulation (train.py:117-146).
int tfl_grad_accumulate(float* acc, const float* grads, int64_t n, float scale, int overwrite, tfl_stream_t stream) {
  TFL_CHECK(acc && grads && n >= 1, "null / empty argument");
  long long blocks = (n + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  grad_accumulate_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(acc, grads, (long long)n, scale, overwrite);
  TFL_LAUNCH_CHECK();
  return 0;
}

// torch.optim.AdamW step t (1-based) over flat buffers; `clip` = norm_out of tfl_grad_clip_norm (device) or NULL.
int tfl_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* clip, float lr,
                   float beta1, float beta2, float eps, float weight_decay, int step, tfl_stream_t stream) {
  TFL_CHECK(params && grads && exp_avg && exp_avg_sq && n >= 1 && step >= 1, "null / empty argument");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  long long blocks = (n + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  adamw_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, (long long)n, clip, lr, beta1, beta2, eps,
                                                                  weight_decay, bc1, sqrtf(bc2));
  TFL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
