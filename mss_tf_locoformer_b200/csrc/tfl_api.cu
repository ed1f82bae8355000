// C ABI (include/tfl.h) of the B200-native TF-Locoformer forward path: plan / weight
// packing / workspace planning and the launch sequences.  Host side only; kernels live in
// kernels_f32.cuh (CUDA-core fp32 + bandwidth-bound stages) and kernels_tc.cuh (tcgen05).
#include <math.h>
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <mutex>
#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges cost nothing unless a profiler is attached

#include "common.cuh"
#include "kernels_f32.cuh"
#include "kernels_tc.cuh"
#include "kernels_tc2.cuh"
#include "kernels_attn.cuh"
#include "kernels_attn2.cuh"
#include "kernels_bs.cuh"
#include "kernels_bwd.cuh"
#include "kernels_mma.cuh"
#include "kernels_tf32.cuh"

namespace tfl {

static thread_local char g_err[1024] = "";
static std::atomic<int> g_options[TFL_OPT_COUNT] = {{2}, {2}, {0}, {2}, {0}, {2}, {2}, {0}};   // tfl_debug_set_option
int tfl_option(int key) { return g_options[key].load(std::memory_order_relaxed); }
std::atomic<unsigned long long> g_launches{0};

// ---- per-device one-time setup: the host-mapped record of an expired bounded wait (tc_common.cuh) -------------------
static std::mutex g_init_mu;
static unsigned int* g_timeout_rec = nullptr;      // pinned, mapped, portable; 5 words (flag, block, thread, barrier, parity)
static bool g_dev_ready[64] = {false};
static int ensure_device_ready() {
  int dev = 0;
  TFL_CUDA(cudaGetDevice(&dev));
  TFL_CHECK(dev >= 0 && dev < 64, "device index %d out of range", dev);
  std::lock_guard<std::mutex> lock(g_init_mu);
  if (g_dev_ready[dev]) return 0;
  if (g_timeout_rec == nullptr) {
    void* h = nullptr;
    TFL_CUDA(cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable));
    memset(h, 0, 64);
    g_timeout_rec = (unsigned int*)h;
  }
  unsigned int* dptr = nullptr;
  TFL_CUDA(cudaHostGetDevicePointer((void**)&dptr, g_timeout_rec, 0));
  TFL_CUDA(cudaMemcpyToSymbol(tc::g_timeout_host, &dptr, sizeof(dptr)));
  g_dev_ready[dev] = true;
  return 0;
}
// An mbarrier wait of an EARLIER launch expired (the kernel trapped): refuse to go on, say where.
static int timeout_pending() {
  const volatile unsigned int* r = g_timeout_rec;
  TFL_CHECK(r == nullptr || r[0] == 0,
            "a bounded mbarrier wait expired in an earlier launch (block %u, thread %u, barrier smem address 0x%x, parity %u): "
            "pipeline protocol error, results are invalid", r[1], r[2], r[3], r[4]);
  return 0;
}
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }
struct NvtxRange {   // one range per stage / sub-block (nsys and ncu --nvtx group the launches under these names)
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};
static inline int ilog2(int n) { int l = 0; while ((1 << l) < n) ++l; return l; }

// ---- generic strided-permute copy used by the weight packer ---------------------------
struct Permute {
  int n[4]; long long s[4]; long long offset; int last_valid; int dim2_valid;
};
__global__ void permute_kernel(const float* __restrict__ src, float* __restrict__ dst, Permute p) {
  const long long total = (long long)p.n[0] * p.n[1] * p.n[2] * p.n[3];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int i3 = (int)(r % p.n[3]); r /= p.n[3];
    const int i2 = (int)(r % p.n[2]); r /= p.n[2];
    const int i1 = (int)(r % p.n[1]); r /= p.n[1];
    const int i0 = (int)r;
    dst[i] = (i3 < p.last_valid && i2 < p.dim2_valid) ? src[p.offset + i0 * p.s[0] + i1 * p.s[1] + i2 * p.s[2] + i3 * p.s[3]] : 0.f;
  }
}
static void permute(const float* src, float* dst, int n0, int n1, int n2, int n3, long long s0, long long s1,
                    long long s2, long long s3, long long offset, int last_valid, cudaStream_t st, int dim2_valid = -1) {
  Permute p{{n0, n1, n2, n3}, {s0, s1, s2, s3}, offset, last_valid < 0 ? n3 : last_valid, dim2_valid < 0 ? n2 : dim2_valid};
  const long long total = (long long)n0 * n1 * n2 * n3;
  const int blocks = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
  permute_kernel<<<blocks, 256, 0, st>>>(src, dst, p);
}

__global__ void fft_tables_kernel(float2* tw, float* win, int n_fft) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_fft / 2) {
    double s, c;
    sincospi(-2.0 * (double)i / (double)n_fft, &s, &c);
    tw[i] = make_float2((float)c, (float)s);
  }
  if (i < n_fft) win[i] = (float)(0.5 - 0.5 * cospi(2.0 * (double)i / (double)n_fft));
}

// ---- packed layout --------------------------------------------------------------------
static void build_layout(tfl_plan* pl) {
  const tfl_config& c = pl->cfg;
  PackLayout& L = pl->lay;
  size_t off = 0;
  auto take = [&](size_t n_float) { size_t o = off; off = align_up(off + n_float * sizeof(float)); return o; };
  const int C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel;
  L.enc_w = L.enc_b = L.gln_w = L.gln_b = L.dec_w = L.dec_b = 0;
  if (c.enc_in_ch > 0) {
    L.enc_w = take((size_t)9 * c.enc_in_ch * C); L.enc_b = take(C); L.gln_w = take(C); L.gln_b = take(C);
    L.dec_w = take((size_t)9 * C * 8); L.dec_b = take(8);
  }
  L.twiddle = L.window = 0;
  if (c.n_fft > 0) { L.twiddle = take(c.n_fft); L.window = take(c.n_fft); }
  L.paths.resize((size_t)c.n_layers * 2);
  for (auto& p : L.paths) {
    for (int j = 0; j < pl->n_ffn; ++j) {
      FfnPack& f = p.ffn[j];
      f.hidden = j == 0 ? c.ffn_hidden0 : c.ffn_hidden1;
      f.gamma = take(C);
      f.w1 = take((size_t)K * C * 2 * f.hidden); f.b1 = take(2 * f.hidden); f.b1raw = take(2 * f.hidden);
      f.w2 = take((size_t)K * f.hidden * C); f.b2 = take(C);
      f.tc = take(tc_ffn_image_bytes(C, f.hidden, K) / sizeof(float));
      f.tc2_ok = tc_ffn2_image_bytes(C, f.hidden, K, c.num_groups) > 0;   // else the FFN runs on ffn_tc_kernel
      f.tc2 = take(tc_ffn2_image_bytes(C, f.hidden, K, c.num_groups) / sizeof(float));
    }
    p.attn_gamma = take(C);
    p.rope = take(pl->head_dim / 2 + 1);
    p.wqkv = take((size_t)C * 3 * A);
    p.wo = take((size_t)A * C);
    p.tc_qkv = take(tc_qkv_image_bytes(C, c.n_heads, pl->head_dim) / sizeof(float));
    p.tc_wo = take(tc_wo_image_bytes(C, c.n_heads, pl->head_dim) / sizeof(float));
    p.rope_tab = (c.rope && attn_tc_supported(C, c.n_heads, pl->head_dim))
                     ? take((size_t)ROPE_TAB_LEN * ((pl->head_dim + 15) / 16 * 16 / 2) * 2) : 0;
  }
  L.total = off;
}

}  // namespace tfl

using namespace tfl;

extern "C" {

int tfl_version(void) { return 200; }
const char* tfl_last_error(void) { return g_err; }
uint64_t tfl_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int tfl_plan_create(const tfl_config* cfg, tfl_plan** out) {
  TFL_CHECK(cfg != nullptr && out != nullptr, "null argument");
  const tfl_config& c = *cfg;
  TFL_CHECK(c.emb_dim > 0 && c.emb_dim % 8 == 0, "emb_dim must be a positive multiple of 8 (got %d)", c.emb_dim);
  TFL_CHECK(c.num_groups > 0 && c.emb_dim % c.num_groups == 0 && (c.emb_dim / c.num_groups) % 4 == 0,
            "emb_dim/num_groups must be a multiple of 4 (emb_dim %d, groups %d)", c.emb_dim, c.num_groups);
  TFL_CHECK(c.n_heads > 0 && c.attention_dim % c.n_heads == 0, "attention_dim %% n_heads != 0");
  TFL_CHECK(c.attention_dim % 8 == 0, "attention_dim must be a multiple of 8");
  const int hd = c.attention_dim / c.n_heads;
  TFL_CHECK(hd % 2 == 0 && hd <= 64, "head_dim must be even and <= 64 (got %d)", hd);
  TFL_CHECK(c.conv_kernel >= 1 && c.conv_kernel <= 16, "conv1d_kernel out of range");
  TFL_CHECK(c.ffn_hidden0 > 0 && c.ffn_hidden0 % 8 == 0, "ffn_hidden_dim must be a multiple of 8");
  TFL_CHECK(!c.macaron || (c.ffn_hidden1 > 0 && c.ffn_hidden1 % 8 == 0), "ffn_hidden_dim must be a multiple of 8");
  TFL_CHECK(c.n_layers >= 1 && c.n_src >= 1, "n_layers / n_src must be >= 1");
  TFL_CHECK(c.enc_in_ch == 0 || c.enc_in_ch == 2, "encoder conv supports 2 input channels (re, im)");
  TFL_CHECK(c.enc_in_ch == 0 || c.n_src * 2 <= 8, "decoder supports up to 4 sources");
  if (c.n_fft > 0) {
    TFL_CHECK((c.n_fft & (c.n_fft - 1)) == 0 && c.n_fft >= 16 && c.n_fft <= 8192, "n_fft must be a power of two in [16, 8192]");
    TFL_CHECK(c.hop > 0 && c.hop <= c.n_fft, "hop_length must be in (0, n_fft]");
  }
  tfl_plan* pl = new tfl_plan();
  pl->cfg = c;
  pl->head_dim = hd;
  pl->n_ffn = c.macaron ? 2 : 1;
  int dev = 0;
  pl->sm_count = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) pl->sm_count = n;
  }
  (void)cudaGetLastError();
  build_layout(pl);
  *out = pl;
  return 0;
}

void tfl_plan_destroy(tfl_plan* plan) { delete plan; }

int tfl_num_weight_tensors(const tfl_plan* pl) {
  const tfl_config& c = pl->cfg;
  const int per_path = pl->n_ffn + 4 * pl->n_ffn + 1 + (c.rope ? 1 : 0) + 2;
  return (c.enc_in_ch > 0 ? 6 : 0) + c.n_layers * 2 * per_path;
}

size_t tfl_packed_bytes(const tfl_plan* pl) { return pl->lay.total; }

int tfl_pack_weights(const tfl_plan* pl, const float* const* w, int n_weights, void* packed, size_t packed_bytes,
                     tfl_stream_t stream) {
  TFL_CHECK(pl && w && packed, "null argument");
  TFL_CHECK(n_weights == tfl_num_weight_tensors(pl), "expected %d weight tensors, got %d", tfl_num_weight_tensors(pl), n_weights);
  TFL_CHECK(packed_bytes >= pl->lay.total, "packed buffer too small");
  const tfl_config& c = pl->cfg;
  const PackLayout& L = pl->lay;
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)packed;
  auto dst = [&](size_t off) { return (float*)(base + off); };
  auto copy = [&](const float* src, size_t off, int n) { permute(src, dst(off), 1, 1, 1, n, 0, 0, 0, 1, 0, -1, st); };
  const int C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel, S2 = c.n_src * 2;
  TFL_CUDA(cudaMemsetAsync(packed, 0, pl->lay.total, st));
  int i = 0;
  if (c.enc_in_ch > 0) {
    const int ci = c.enc_in_ch;
    // conv.0.weight [C, ci, 3, 3] -> [9][ci][C]
    permute(w[i++], dst(L.enc_w), 1, 9, ci, C, 0, 1, 9, (long long)ci * 9, 0, -1, st);
    copy(w[i++], L.enc_b, C); copy(w[i++], L.gln_w, C); copy(w[i++], L.gln_b, C);
  }
  for (int layer = 0; layer < c.n_layers; ++layer)
    for (int axis = 0; axis < 2; ++axis) {
      const PathPack& p = L.paths[(size_t)layer * 2 + axis];
      for (int j = 0; j < pl->n_ffn; ++j) copy(w[i++], p.ffn[j].gamma, C);
      for (int j = 0; j < pl->n_ffn; ++j) {
        const FfnPack& f = p.ffn[j];
        const int H = f.hidden;
        const float* w1 = w[i++]; const float* b1 = w[i++]; const float* w2 = w[i++]; const float* b2 = w[i++];
        // conv1d.weight [2H, C, K] -> [K][C][H][2] (value, gate interleaved)
        permute(w1, dst(f.w1), K, C, H, 2, 1, K, (long long)C * K, (long long)H * C * K, 0, -1, st);
        permute(b1, dst(f.b1), 1, 1, H, 2, 0, 0, 1, H, 0, -1, st);
        copy(b1, f.b1raw, 2 * H);
        // deconv1d.weight [H, C, K] -> [K'][H][C] with k = K-1-k'
        permute(w2, dst(f.w2), 1, K, H, C, 0, -1, (long long)C * K, K, K - 1, -1, st);
        copy(b2, f.b2, C);
        TFL_CHECK(tc_pack_ffn(w1, b1, w2, b2, (char*)packed + f.tc, C, H, K, st) == 0, "tc_pack_ffn failed");
        if (f.tc2_ok) TFL_CHECK(tc_pack_ffn2(w1, w2, (char*)packed + f.tc2, C, H, K, c.num_groups, st) == 0, "tc_pack_ffn2 failed");
      }
      const float* attn_gamma_raw = w[i];
      copy(w[i++], p.attn_gamma, C);
      if (c.rope) copy(w[i++], p.rope, pl->head_dim / 2);
      const float* wqkv_raw = w[i++];
      const float* wo_raw = w[i++];
      permute(wqkv_raw, dst(p.wqkv), 1, 1, C, 3 * A, 0, 0, 1, C, 0, -1, st);  // [3A, C] -> [C][3A]
      permute(wo_raw, dst(p.wo), 1, 1, A, C, 0, 0, 1, A, 0, -1, st);          // [C, A] -> [A][C]
      if (attn_tc_supported(C, c.n_heads, pl->head_dim))
        tc_pack_qkv_kernel<<<296, 256, 0, st>>>(wqkv_raw, wo_raw, attn_gamma_raw, (__nv_bfloat16*)(base + p.tc_qkv),
                                                (__nv_bfloat16*)(base + p.tc_wo), C, A, c.n_heads, pl->head_dim,
                                                (pl->head_dim + 15) / 16 * 16,
                                                1.4426950408889634f / sqrtf((float)pl->head_dim));
      if (p.rope_tab != 0) {   // RoPE (cos, sin) table, once per weight pack instead of once per attention call
        const int HDP = (pl->head_dim + 15) / 16 * 16;
        rope_table_kernel<<<(ROPE_TAB_LEN * (HDP / 2) + 255) / 256, 256, 0, st>>>((float2*)(base + p.rope_tab), dst(p.rope), ROPE_TAB_LEN,
                                                                                 pl->head_dim / 2, HDP / 2);
      }
    }
  if (c.enc_in_ch > 0) {
    // deconv.weight [C, 2S, 3, 3] -> [9][8][C] (outputs >= 2S stay zero from the memset)
    permute(w[i++], dst(L.dec_w), 1, 9, 8, C, 0, 1, 9, (long long)S2 * 9, 0, -1, st, S2);
    copy(w[i++], L.dec_b, S2);
  }
  if (c.n_fft > 0)
    fft_tables_kernel<<<(c.n_fft + 255) / 256, 256, 0, st>>>((float2*)(base + L.twiddle), dst(L.window), c.n_fft);
  TFL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"

// ---- workspace ------------------------------------------------------------------------
namespace tfl {
struct Workspace {
  size_t spec, x, xn, hid, qkv, o, est, gln_part, gln_stats, prefix, tc, qkv_img, o_img, rope, total;
  int gln_blocks;
};
static Workspace plan_workspace(const tfl_plan* pl, int B, int Tf, int F, int precision) {
  const tfl_config& c = pl->cfg;
  Workspace w{};
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  const size_t N = (size_t)B * Tf * F;
  const int C = c.emb_dim, A = c.attention_dim, K = c.conv_kernel;
  const int Hmax = c.ffn_hidden0 > c.ffn_hidden1 ? c.ffn_hidden0 : c.ffn_hidden1;
  w.spec = take(N * 2 * sizeof(float));
  w.x = take(N * C * sizeof(float));
  w.est = take(N * 2 * c.n_src * sizeof(float));
  w.gln_blocks = pl->sm_count * 2;
  w.gln_part = take((size_t)B * w.gln_blocks * 2 * sizeof(double));
  w.gln_stats = take((size_t)B * 2 * sizeof(float));
  w.prefix = off;   // everything above is precision-independent (tfl_enc_conv_gln uses only this part)
  if (precision == TFL_PRECISION_FP32 || precision == TFL_PRECISION_TF32) {   // normalised copy, hidden, q|k|v, attention output
    const size_t hid_rows_f = (size_t)B * Tf * (F + K - 1), hid_rows_t = (size_t)B * F * (Tf + K - 1);
    const size_t hid_rows = hid_rows_f > hid_rows_t ? hid_rows_f : hid_rows_t;
    w.xn = take(N * C * sizeof(float));
    w.hid = take(hid_rows * Hmax * sizeof(float));
    w.qkv = take(N * 3 * A * sizeof(float));
    w.o = take(N * A * sizeof(float));
  }
  w.tc = take(tc_workspace_bytes(pl, B, Tf, F));
  if (precision == TFL_PRECISION_BF16) {  // 128-row bf16 tile images of q|k|v and of the attention output
    const size_t HDP = (size_t)(pl->head_dim + 15) / 16 * 16;
    const size_t tiles_f = (size_t)B * Tf * ((F + 127) / 128), tiles_t = (size_t)B * F * ((Tf + 127) / 128);
    const size_t tiles = tiles_f > tiles_t ? tiles_f : tiles_t;
    w.o_img = take(tiles * 128 * c.n_heads * HDP * 2);
    w.qkv_img = take(3 * tiles * 128 * c.n_heads * HDP * 2);
    w.rope = take((size_t)(F > Tf ? F : Tf) * (HDP / 2) * sizeof(float2));
  }
  w.total = off;
  return w;
}

static int norm_launch(const float* x, float* y, long long rows, int C, int G, const float* gamma, float eps,
                       int sm_count, cudaStream_t st) {
  const int lanes = (C / G) / 4;
  int W = 1;
  while (W < lanes) W <<= 1;
  TFL_CHECK(W <= 32, "emb_dim/num_groups > 128 is not supported");
  const long long pairs = rows * G;
  const long long per_block = 256 / W;
  long long blocks = (pairs + per_block - 1) / per_block;
  const long long cap = (long long)sm_count * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
#define NORM_CASE(w) case w: rms_group_norm_kernel<w, float><<<(int)blocks, 256, 0, st>>>(x, y, rows, C, G, gamma, eps); break;
  switch (W) { NORM_CASE(1) NORM_CASE(2) NORM_CASE(4) NORM_CASE(8) NORM_CASE(16) NORM_CASE(32) }
#undef NORM_CASE
  TFL_LAUNCH_CHECK();
  return 0;
}

// Set (per thread, for the duration of a call) by the training entry points when tf32 tensor-core GEMMs are selected
// (tfl_train.cuh); the inference / parity path never sets it: TFL_PRECISION_FP32 stays exact fp32 on CUDA cores.
static thread_local int g_gemm_mode = 0;   // 0 = fp32 CUDA cores, 1 = tf32 mma.sync, 2 = bf16 mma.sync (fp32 accumulation)
#define g_gemm_tf32 (g_gemm_mode != 0)

template <class Epi>
static int gemm_launch(const TapGemm& g, const Epi& epi, cudaStream_t st) {
  TFL_CHECK(g.Kc % GBK == 0 && g.N % 4 == 0, "tap-GEMM needs Kc %% 8 == 0 and N %% 4 == 0 (Kc %d N %d)", g.Kc, g.N);
  dim3 grid((unsigned)((g.M + GBM - 1) / GBM), (unsigned)((g.N + GBN - 1) / GBN));
  if (g_gemm_mode == 2 && g.Kc % 32 == 0) tap_gemm_bf16_kernel<Epi><<<grid, 256, 0, st>>>(g, epi);
  else if (g_gemm_mode != 0 && g.Kc % MMA_BK == 0) tap_gemm_mma_kernel<Epi><<<grid, 256, 0, st>>>(g, epi);
  else tap_gemm_kernel<Epi><<<grid, 256, 0, st>>>(g, epi);
  TFL_LAUNCH_CHECK();
  return 0;
}

struct Dims { int B, Tf, F; };

// tf32 = the same dataflow with both GEMMs on the tcgen05 kind::tf32 tap-GEMM (kernels_tf32.cuh)
static int ffn_f32(const tfl_plan* pl, const char* packed, int layer, int axis, int j, float* x, Dims d,
                   const Workspace& ws, char* wsp, cudaStream_t st, bool tf32 = false) {
  NvtxRange nvtx_range(tf32 ? "tfl::conv_swiglu_ffn[tf32]" : "tfl::conv_swiglu_ffn[fp32]");
  const tfl_config& c = pl->cfg;
  const FfnPack& f = pl->lay.paths[(size_t)layer * 2 + axis].ffn[j];
  const int C = c.emb_dim, K = c.conv_kernel, H = f.hidden;
  const int S = axis == TFL_AXIS_FREQ ? d.F : d.Tf;
  const int nseq = axis == TFL_AXIS_FREQ ? d.B * d.Tf : d.B * d.F;
  const long long rows = (long long)d.B * d.Tf * d.F;
  float* xn = (float*)(wsp + ws.xn);
  float* hid = (float*)(wsp + ws.hid);
  if (norm_launch(x, xn, rows, C, c.num_groups, (const float*)(packed + f.gamma), c.eps, pl->sm_count, st)) return -1;
  const SeqMap xmap = make_seq_map(axis, d.Tf, d.F, C);
  TapGemm g1{xn, xmap, S, S + K - 1, K - 1, K, C, (const float*)(packed + f.w1), (const float*)(packed + f.b1),
             2 * H, (long long)nseq * (S + K - 1)};
  TapGemm g2{hid, make_dense_map((long long)(S + K - 1) * H, H), S + K - 1, S, 0, K, H,
             (const float*)(packed + f.w2), (const float*)(packed + f.b2), C, (long long)nseq * S};
  if (tf32) {
    if (tap_gemm_tf32_launch(g1, EpiSwiGLU{hid, H}, st)) return -1;
    return tap_gemm_tf32_launch(g2, EpiResidual{x, xmap}, st);
  }
  if (gemm_launch(g1, EpiSwiGLU{hid, H}, st)) return -1;
  return gemm_launch(g2, EpiResidual{x, xmap}, st);
}

// lse != nullptr (training): the log-sum-exp of every (sequence, head, query) is kept and the head-merge projection +
// residual are skipped when `forward_only_to_o` (the backward pass recomputes q|k|v and o from the saved input).
static int attn_f32(const tfl_plan* pl, const char* packed, int layer, int axis, float* x, Dims d,
                    const Workspace& ws, char* wsp, cudaStream_t st, float* lse = nullptr, bool forward_only_to_o = false) {
  NvtxRange nvtx_range("tfl::rope_attn[fp32]");
  const tfl_config& c = pl->cfg;
  const PathPack& p = pl->lay.paths[(size_t)layer * 2 + axis];
  const int C = c.emb_dim, A = c.attention_dim, hd = pl->head_dim, heads = c.n_heads;
  const int L = axis == TFL_AXIS_FREQ ? d.F : d.Tf;
  const int nseq = axis == TFL_AXIS_FREQ ? d.B * d.Tf : d.B * d.F;
  const long long rows = (long long)d.B * d.Tf * d.F;
  float* xn = (float*)(wsp + ws.xn);
  float* qkv = (float*)(wsp + ws.qkv);
  float* o = (float*)(wsp + ws.o);
  if (norm_launch(x, xn, rows, C, c.num_groups, (const float*)(packed + p.attn_gamma), c.eps, pl->sm_count, st)) return -1;
  const SeqMap xmap = make_seq_map(axis, d.Tf, d.F, C);
  TapGemm g1{xn, xmap, L, L, 0, 1, C, (const float*)(packed + p.wqkv), nullptr, 3 * A, (long long)nseq * L};
  EpiQkvRope e1{qkv, A, hd, heads, L, nseq, c.rope ? (const float*)(packed + p.rope) : nullptr};
  if (gemm_launch(g1, e1, st)) return -1;
  const size_t per = (size_t)nseq * heads * L * hd;
  const float scale = 1.0f / sqrtf((float)hd);
  if (g_gemm_tf32 && hd % 2 == 0 && hd > 8 && hd <= 32) {   // training modes >= 1: tf32 mma.sync form (kernels_mma.cuh)
    dim3 grid64((L + 63) / 64, heads, nseq);
    if (g_gemm_mode == 2 && hd <= 16) attn_fwd_bf16_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, L, hd, heads, scale, lse);
    else if (g_gemm_mode == 2) attn_fwd_bf16_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, L, hd, heads, scale, lse);
    else if (hd <= 16) attn_fwd_mma_kernel<16><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, L, hd, heads, scale, lse);
    else attn_fwd_mma_kernel<32><<<grid64, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, L, hd, heads, scale, lse);
  } else {
  dim3 grid((L + 127) / 128, heads, nseq);
#define ATT_CASE(HD) attn_f32_kernel<HD><<<grid, 128, 0, st>>>(qkv, qkv + per, qkv + 2 * per, o, L, hd, heads, scale, lse)
  if (hd <= 8) ATT_CASE(8); else if (hd <= 16) ATT_CASE(16); else if (hd <= 32) ATT_CASE(32); else ATT_CASE(64);
#undef ATT_CASE
  }
  TFL_LAUNCH_CHECK();
  if (forward_only_to_o) return 0;
  TapGemm g2{o, make_dense_map((long long)L * A, A), L, L, 0, 1, A, (const float*)(packed + p.wo), nullptr, C,
             (long long)nseq * L};
  return gemm_launch(g2, EpiResidual{x, xmap}, st);
}

// bf16 attention sub-block (models/mss_tflocoformer.py:452-456): three tcgen05 kernels,
//   qkv_tc   RMSGroupNorm -> q|k|v projection -> RoPE -> bf16 tile images
//   attn_tc  softmax(q k^T) v per (sequence, head)
//   proj_tc  head merge projection + residual, in place on x
static int attn_bf16(const tfl_plan* pl, const char* packed, int layer, int axis, float* x, Dims d,
                     const Workspace& ws, char* wsp, cudaStream_t st) {
  NvtxRange nvtx_range("tfl::rope_attn[bf16]");
  const tfl_config& c = pl->cfg;
  const PathPack& p = pl->lay.paths[(size_t)layer * 2 + axis];
  const int C = c.emb_dim, hd = pl->head_dim, heads = c.n_heads;
  TFL_CHECK(attn_tc_supported(C, heads, hd),
            "bf16 tcgen05 attention needs an even head_dim <= 32, emb_dim %% 16 == 0 and n_heads * head_dim(padded to 16) "
            "in {32,64,96,128} (got emb_dim %d, n_heads %d, head_dim %d); use precision fp32", C, heads, hd);
  const int HDP = (hd + 15) / 16 * 16, NPART = heads * HDP;
  const int L = axis == TFL_AXIS_FREQ ? d.F : d.Tf;
  const int nseq = axis == TFL_AXIS_FREQ ? d.B * d.Tf : d.B * d.F;
  const int NTL = (L + 127) / 128;
  __nv_bfloat16* qkv = (__nv_bfloat16*)(wsp + ws.qkv_img);
  __nv_bfloat16* oimg = (__nv_bfloat16*)(wsp + ws.o_img);
  const float2* rope = (const float2*)(wsp + ws.rope);
  const SeqMap xmap = make_seq_map(axis, d.Tf, d.F, C);
  int rope_stride = L;
  if (c.rope && L <= ROPE_TAB_LEN && p.rope_tab != 0) {        // the pack-time table covers this length
    rope = (const float2*)(packed + p.rope_tab);
    rope_stride = ROPE_TAB_LEN;
  } else if (c.rope) {
    rope_table_kernel<<<(L * (HDP / 2) + 255) / 256, 256, 0, st>>>((float2*)(wsp + ws.rope), (const float*)(packed + p.rope), L, hd / 2, HDP / 2);
    TFL_LAUNCH_CHECK();
  }
  {
    QkvTcParams q;
    q.x = x; q.map = xmap; q.gamma = (const float*)(packed + p.attn_gamma); q.eps = c.eps;
    q.wimg = packed + p.tc_qkv; q.rope = c.rope ? rope : nullptr; q.rope_stride = rope_stride; q.qkv = qkv;
    q.C = C; q.G = c.num_groups; q.L = L; q.NTL = NTL; q.nseq = nseq; q.heads = heads; q.hd = hd; q.HDP = HDP;
    q.NPART = NPART; q.n_tiles = nseq * NTL; q.pad_to = tfl_option(TFL_OPT_ATTN_KERNEL) == 1 ? 64 : 16; q.qscale = 1.4426950408889634f / sqrtf((float)hd);
    const uint32_t smem = 3u * C * NPART * 2 + 3u * C * 256 + C * 4 + 256;
    TFL_CUDA(opt_in_smem(qkv_tc_kernel, smem));
    const int grid = q.n_tiles < pl->sm_count ? q.n_tiles : pl->sm_count;
    TFL_CUDA(launch_pdl(qkv_tc_kernel, dim3(grid), dim3(QKV_THREADS), smem, st, q));
    TFL_LAUNCH_CHECK();
  }
  {
    // query rows that do not fill a tile run on CUDA cores when there are only a few of them (1025 = 8*128 + 1,
    // 259 = 2*128 + 3): a mostly empty tensor-core tile costs as much as a full one
    const int Lpad = (L + 31) & ~31;
    const size_t tsm = (size_t)8 * Lpad * sizeof(float);      // score rows of the 8 warps of a tail-row block
    const int tail_q = (L > 128 && L % 128 != 0 && L % 128 <= 8 && tsm <= 160 * 1024) ? L % 128 : 0;
    AttnTcParams ap;
    ap.qkv = qkv; ap.o = oimg; ap.nseq = nseq; ap.heads = heads; ap.L = L; ap.NTL = NTL; ap.HDP = HDP;
    ap.NQT = tail_q ? L / 128 : NTL;
    ap.NU = (L + 63) / 64;
    ap.NP = (ap.NQT + 1) / 2; ap.n_items = nseq * heads * ap.NP;
    if (tfl_option(TFL_OPT_ATTN_KERNEL) == 1) {
      const uint32_t smem = attn_tc_smem(HDP);
      TFL_CUDA(opt_in_smem(attn_tc_kernel, smem));
      const int grid = ap.n_items < pl->sm_count ? ap.n_items : pl->sm_count;
      attn_tc_kernel<<<grid, 352, smem, st>>>(ap);
    } else {
      Attn2Params a2;
      a2.qkv = qkv; a2.o = oimg; a2.nseq = nseq; a2.heads = heads; a2.L = L; a2.NTL = NTL; a2.HDP = HDP;
      a2.NQT = ap.NQT;
      a2.QG = a2.NQT >= 3 ? 4 : (a2.NQT == 2 ? 2 : 1);         // 4 groups = QG query tiles x HG heads
      a2.HG = ATT2_G / a2.QG;
      a2.NQG = (a2.NQT + a2.QG - 1) / a2.QG; a2.NHG = (heads + a2.HG - 1) / a2.HG;
      a2.n_items = nseq * a2.NHG * a2.NQG;
      const uint32_t smem = attn2_smem(HDP, a2.HG, &a2.NS);
      TFL_CHECK(a2.NS >= 2, "attention K/V ring does not fit in shared memory");
      auto kern = HDP == 16 ? attn_tc2_kernel<1> : attn_tc2_kernel<2>;
      TFL_CUDA(opt_in_smem(kern, smem));
      const int grid = a2.n_items < pl->sm_count ? a2.n_items : pl->sm_count;
      TFL_CUDA(launch_pdl(kern, dim3(grid), dim3(ATT2_THREADS), smem, st, a2));
    }
    TFL_LAUNCH_CHECK();
    // one tail row (frequency axis of n_fft 2048: 1025 = 8 * 128 + 1) has nothing to share between rows and long key
    // ranges: the CUDA-core kernel is at its K / V traffic floor there (0.20 ms vs 0.25 ms, r02); several rows: mma.sync
    if (tail_q >= 2 && tfl_option(TFL_OPT_TAIL_KERNEL) != 1) {
      // warp-level tensor-core path: one warp per (sequence, head), all tail rows at once
      long long blocks = ((long long)nseq * heads + 7) / 8;
      if (blocks > (long long)pl->sm_count * 8) blocks = (long long)pl->sm_count * 8;
      if (HDP == 16) TFL_CUDA(launch_pdl(attn_tail_mma_kernel<1>, dim3((unsigned)blocks), dim3(256), 0, st, ap, ap.NQT * 128));
      else TFL_CUDA(launch_pdl(attn_tail_mma_kernel<2>, dim3((unsigned)blocks), dim3(256), 0, st, ap, ap.NQT * 128));
      TFL_LAUNCH_CHECK();
    } else if (tail_q) {
      const long long warps = (long long)nseq * heads * tail_q;
      long long blocks = (warps + 7) / 8;
      if (blocks > (long long)pl->sm_count * 8) blocks = (long long)pl->sm_count * 8;
      TFL_CUDA(opt_in_smem(attn_tail_rows_kernel<1>, tsm));
      TFL_CUDA(launch_pdl(attn_tail_rows_kernel<1>, dim3((unsigned)blocks), dim3(256), tsm, st, ap, ap.NQT * 128));
      TFL_LAUNCH_CHECK();
    }
  }
  {
    ProjTcParams pp;
    pp.oimg = oimg; pp.wimg = packed + p.tc_wo; pp.x = x; pp.map = xmap;
    pp.C = C; pp.AP = NPART; pp.L = L; pp.NTL = NTL; pp.n_tiles = nseq * NTL;
    const uint32_t smem = (uint32_t)NPART * C * 2 + PROJ_STAGES * (uint32_t)NPART * 256 + 2 * PROJ_STG_BYTES + 256;
    TFL_CUDA(opt_in_smem(proj_tc_kernel, smem));
    const int grid = pp.n_tiles < pl->sm_count ? pp.n_tiles : pl->sm_count;
    TFL_CUDA(launch_pdl(proj_tc_kernel, dim3(grid), dim3(320), smem, st, pp));
    TFL_LAUNCH_CHECK();
  }
  return 0;
}

// LocoformerBlock.forward, models/mss_tflocoformer.py:430-464.  fp32: in place on *cur.  bf16: every fused
// FFN kernel reads *cur and writes *alt (tile halos forbid in-place), after which the two swap.
static int path_forward(const tfl_plan* pl, const char* packed, int layer, int axis, float** cur, float** alt, Dims d,
                        const Workspace& ws, char* wsp, int precision, cudaStream_t st) {
  auto ffn = [&](int j) -> int {
    if (precision == TFL_PRECISION_BF16) {
      if (tc_ffn(pl, packed, layer, axis, j, *cur, *alt, d.B, d.Tf, d.F, st)) return -1;
      float* t = *cur; *cur = *alt; *alt = t;
      return 0;
    }
    return ffn_f32(pl, packed, layer, axis, j, *cur, d, ws, wsp, st, precision == TFL_PRECISION_TF32);
  };
  if (pl->cfg.macaron && ffn(1)) return -1;
  if (precision == TFL_PRECISION_BF16) {
    if (attn_bf16(pl, packed, layer, axis, *cur, d, ws, wsp, st)) return -1;
  } else if (attn_f32(pl, packed, layer, axis, *cur, d, ws, wsp, st)) return -1;
  return ffn(0);
}

static int blocks_forward(const tfl_plan* pl, const char* packed, float* x, Dims d, const Workspace& ws, char* wsp,
                          int precision, cudaStream_t st) {
  NvtxRange nvtx_range("tfl::blocks");
  float* cur = x;
  float* alt = (float*)(wsp + ws.tc);
  for (int layer = 0; layer < pl->cfg.n_layers; ++layer) {
    const int first = pl->cfg.tf_order == 0 ? TFL_AXIS_FREQ : TFL_AXIS_TIME;  // :332-353
    if (path_forward(pl, packed, layer, first, &cur, &alt, d, ws, wsp, precision, st)) return -1;
    if (path_forward(pl, packed, layer, 1 - first, &cur, &alt, d, ws, wsp, precision, st)) return -1;
  }
  TFL_CHECK(cur == x, "internal: residual ping-pong did not end in the caller's buffer");
  return 0;
}

static int check_common(const tfl_plan* pl, const void* packed, int B, int Tf, int F, int precision) {
  TFL_CHECK(pl != nullptr && packed != nullptr, "null plan / packed weights");
  TFL_CHECK(B >= 1 && Tf >= 1 && F >= 1, "empty input (batch %d, frames %d, bins %d)", B, Tf, F);
  TFL_CHECK(precision == TFL_PRECISION_FP32 || precision == TFL_PRECISION_BF16 || precision == TFL_PRECISION_TF32,
            "unknown precision %d", precision);
  if (ensure_device_ready()) return -1;
  return timeout_pending();
}
}  // namespace tfl

extern "C" {

size_t tfl_workspace_bytes(const tfl_plan* pl, int B, int Tf, int F, int precision) {
  return plan_workspace(pl, B, Tf, F, precision).total;
}

int tfl_stft(const tfl_plan* pl, const void* packed, const float* audio, int B, int T, float* spec, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::stft");
  TFL_CHECK(pl && packed && audio && spec, "null argument");
  const tfl_config& c = pl->cfg;
  TFL_CHECK(c.n_fft > 0, "plan has no STFT (n_fft == 0)");
  TFL_CHECK(B >= 1, "empty batch");
  TFL_CHECK(T > c.n_fft / 2, "reflect padding needs more than n_fft/2 = %d samples (got %d)", c.n_fft / 2, T);
  const int Tf = 1 + T / c.hop;
  const char* base = (const char*)packed;
  TFL_CUDA(opt_in_smem(stft_kernel, c.n_fft * sizeof(float2)));
  stft_kernel<<<dim3(Tf, B), 256, c.n_fft * sizeof(float2), (cudaStream_t)stream>>>(
      audio, T, c.n_fft, ilog2(c.n_fft), c.hop, Tf, (const float2*)(base + pl->lay.twiddle),
      (const float*)(base + pl->lay.window), spec);
  TFL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
namespace tfl {
static int enc_conv_gln_any(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* x,
                            void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream);
}
extern "C" {
int tfl_enc_conv_gln(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* x,
                     void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  return enc_conv_gln_any(pl, packed, spec, B, Tf, F, x, workspace, ws_bytes, TFL_PRECISION_FP32, stream);
}
int tfl_enc_conv_gln_mode(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* x,
                          void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  TFL_CHECK(precision == TFL_PRECISION_FP32 || precision == TFL_PRECISION_BF16 || precision == TFL_PRECISION_TF32,
            "unknown precision %d", precision);
  return enc_conv_gln_any(pl, packed, spec, B, Tf, F, x, workspace, ws_bytes, precision, stream);
}
}  // extern "C"
namespace tfl {
static int enc_conv_gln_any(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* x,
                            void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::enc_conv_gln");
  if (check_common(pl, packed, B, Tf, F, 0)) return -1;
  TFL_CHECK(pl->cfg.enc_in_ch == 2, "plan has no conv encoder");
  const Workspace ws = plan_workspace(pl, B, Tf, F, 0);  // only the precision-independent prefix is used here
  TFL_CHECK(workspace && ws_bytes >= ws.prefix, "workspace too small (%zu < %zu)", ws_bytes, ws.prefix);
  const tfl_config& c = pl->cfg;
  const char* base = (const char*)packed;
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = c.emb_dim;
  double* part = (double*)(wsp + ws.gln_part);
  float* stats = (float*)(wsp + ws.gln_stats);
  const size_t smem = ((size_t)9 * 2 * C + C) * sizeof(float);
  if (precision != TFL_PRECISION_FP32 && C % 8 == 0) {   // bf16 and tf32 modes: tf32 mma.sync, two passes (enc_conv_mma_kernel)
    const size_t msm = ((size_t)24 * (C + 8) + 3 * C) * sizeof(float);
    TFL_CUDA(opt_in_smem(enc_conv_mma_kernel<2, 0>, msm));
    TFL_CUDA(opt_in_smem(enc_conv_mma_kernel<2, 1>, msm));
    const float* ew = (const float*)(base + pl->lay.enc_w);
    const float* eb = (const float*)(base + pl->lay.enc_b);
    const float* gw = (const float*)(base + pl->lay.gln_w);
    const float* gb = (const float*)(base + pl->lay.gln_b);
    enc_conv_mma_kernel<2, 0><<<dim3(ws.gln_blocks, B), 256, msm, st>>>(spec, Tf, F, C, ew, eb, x, part, nullptr, gw, gb);
    TFL_LAUNCH_CHECK();
    gln_finalize_kernel<<<B, 256, 0, st>>>(part, ws.gln_blocks, (double)Tf * F * C, c.eps, stats);
    TFL_LAUNCH_CHECK();
    enc_conv_mma_kernel<2, 1><<<dim3(ws.gln_blocks, B), 256, msm, st>>>(spec, Tf, F, C, ew, eb, x, part, stats, gw, gb);
    TFL_LAUNCH_CHECK();
    return 0;
  }
  enc_conv_kernel<2><<<dim3(ws.gln_blocks, B), 256, smem, st>>>(spec, Tf, F, C, (const float*)(base + pl->lay.enc_w),
                                                              (const float*)(base + pl->lay.enc_b), x, part);
  TFL_LAUNCH_CHECK();
  gln_finalize_kernel<<<B, 256, 0, st>>>(part, ws.gln_blocks, (double)Tf * F * C, c.eps, stats);
  TFL_LAUNCH_CHECK();
  gln_apply_kernel<<<dim3(pl->sm_count * 4, B), 256, 0, st>>>(x, (long long)Tf * F * C / 4, C, stats,
                                                            (const float*)(base + pl->lay.gln_w),
                                                            (const float*)(base + pl->lay.gln_b));
  TFL_LAUNCH_CHECK();
  return 0;
}

}  // namespace tfl
extern "C" {

int tfl_rms_group_norm(const tfl_plan* pl, const void* packed, int layer, int axis, int which, const float* x,
                       float* y, int64_t rows, tfl_stream_t stream) {
  TFL_CHECK(pl && packed && x && y, "null argument");
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1), "bad layer/axis");
  TFL_CHECK(which == 2 || (which >= 0 && which < pl->n_ffn), "bad norm selector %d", which);
  if (rows == 0) return 0;
  const PathPack& p = pl->lay.paths[(size_t)layer * 2 + axis];
  const size_t goff = which == 2 ? p.attn_gamma : p.ffn[which].gamma;
  return norm_launch(x, y, rows, pl->cfg.emb_dim, pl->cfg.num_groups, (const float*)((const char*)packed + goff),
                     pl->cfg.eps, pl->sm_count, (cudaStream_t)stream);
}

int tfl_conv_swiglu_ffn(const tfl_plan* pl, const void* packed, int layer, int axis, int ffn_index, float* x, int B,
                        int Tf, int F, void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1), "bad layer/axis");
  TFL_CHECK(ffn_index >= 0 && ffn_index < pl->n_ffn, "bad ffn index %d", ffn_index);
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  if (precision == TFL_PRECISION_BF16) {
    float* y = (float*)((char*)workspace + ws.tc);
    if (tc_ffn(pl, (const char*)packed, layer, axis, ffn_index, x, y, B, Tf, F, (cudaStream_t)stream)) return -1;
    TFL_CUDA(cudaMemcpyAsync(x, y, (size_t)B * Tf * F * pl->cfg.emb_dim * sizeof(float), cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
    return 0;
  }
  return ffn_f32(pl, (const char*)packed, layer, axis, ffn_index, x, Dims{B, Tf, F}, ws, (char*)workspace,
                 (cudaStream_t)stream, precision == TFL_PRECISION_TF32);
}

int tfl_conv_swiglu_ffn_out(const tfl_plan* pl, const void* packed, int layer, int axis, int ffn_index, const float* x,
                            float* y, int B, int Tf, int F, void* workspace, size_t ws_bytes, int precision,
                            tfl_stream_t stream) {
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  TFL_CHECK(x != nullptr && y != nullptr && x != y, "x and y must be distinct buffers");
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1), "bad layer/axis");
  TFL_CHECK(ffn_index >= 0 && ffn_index < pl->n_ffn, "bad ffn index %d", ffn_index);
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  if (precision == TFL_PRECISION_BF16)
    return tc_ffn(pl, (const char*)packed, layer, axis, ffn_index, const_cast<float*>(x), y, B, Tf, F, (cudaStream_t)stream);
  TFL_CUDA(cudaMemcpyAsync(y, x, (size_t)B * Tf * F * pl->cfg.emb_dim * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return ffn_f32(pl, (const char*)packed, layer, axis, ffn_index, y, Dims{B, Tf, F}, ws, (char*)workspace,
                 (cudaStream_t)stream, precision == TFL_PRECISION_TF32);
}

int tfl_rope_attn(const tfl_plan* pl, const void* packed, int layer, int axis, float* x, int B, int Tf, int F,
                  void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  TFL_CHECK(layer >= 0 && layer < pl->cfg.n_layers && (axis == 0 || axis == 1), "bad layer/axis");
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  if (precision == TFL_PRECISION_BF16)
    return attn_bf16(pl, (const char*)packed, layer, axis, x, Dims{B, Tf, F}, ws, (char*)workspace, (cudaStream_t)stream);
  return attn_f32(pl, (const char*)packed, layer, axis, x, Dims{B, Tf, F}, ws, (char*)workspace, (cudaStream_t)stream);
}

}  // extern "C"
namespace tfl {
// bf16 and tf32 modes: tf32 mma.sync decoder (C % 16 == 0); fp32 mode and odd widths: the CUDA-core kernel (tfl_dec_conv)
static int dec_conv_any(const tfl_plan* pl, const void* packed, const float* x, int B, int Tf, int F, float* est,
                        int precision, tfl_stream_t stream) {
  const int C = pl->cfg.emb_dim;
  if (precision == TFL_PRECISION_FP32 || C % 16 != 0 || pl->cfg.n_src * 2 > 8) return tfl_dec_conv(pl, packed, x, B, Tf, F, est, stream);
  NvtxRange nvtx_range("tfl::dec_conv[tf32]");
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  if (C % 32 == 0 && C <= 128 && tfl_option(TFL_OPT_DEC_KERNEL) != 1) {
    // scatter form: every x row read once; strips of equal width, frame runs sized so that the items fill whole waves
    const int NS = (F + DEC_WOUT - 1) / DEC_WOUT, WOUT = (F + NS - 1) / NS;
    const int slots = 2 * pl->sm_count;
    int NR = 1;
    for (int w = 1; w <= 16; ++w) {
      long long nr = (long long)slots * w / ((long long)B * NS);
      if (nr < 1) continue;
      if (nr > (Tf + 3) / 4) nr = (Tf + 3) / 4;
      NR = (int)nr;
      if ((Tf + NR - 1) / NR <= 80) break;
    }
    const int R = (Tf + NR - 1) / NR;
    NR = (Tf + R - 1) / R;
    const long long items = (long long)B * NS * NR;
    const int grid = (int)(items < slots ? items : slots);
    const size_t smem = ((size_t)72 * (C + 16) + (size_t)3 * 4 * DEC_WB * 2) * sizeof(float);
    const char* base = (const char*)packed;
    const float* wd = (const float*)(base + pl->lay.dec_w);
    const float* bd = (const float*)(base + pl->lay.dec_b);
    const int n_out = pl->cfg.n_src * 2;
    cudaStream_t st = (cudaStream_t)stream;
#define TFL_DEC_SCATTER(NCH)                                                                                    \
    {                                                                                                           \
      TFL_CUDA(opt_in_smem(dec_conv_scatter_kernel<NCH>, smem));                                                \
      dec_conv_scatter_kernel<NCH><<<grid, 256, smem, st>>>(x, B, Tf, F, n_out, wd, bd, est, NS, WOUT, NR, R);  \
    }
    switch (C / 32) {
      case 1: TFL_DEC_SCATTER(1) break;
      case 2: TFL_DEC_SCATTER(2) break;
      case 3: TFL_DEC_SCATTER(3) break;
      default: TFL_DEC_SCATTER(4) break;
    }
#undef TFL_DEC_SCATTER
    TFL_LAUNCH_CHECK();
    return 0;
  }
  const size_t smem = (size_t)9 * C * 8 * sizeof(float);
  TFL_CUDA(opt_in_smem(dec_conv_mma_kernel, smem));
  const char* base = (const char*)packed;
  long long blocks = (long long)B * ((Tf + 7) / 8) * ((F + 15) / 16);   // patches of 8 frames x 16 bins
  const long long cap = (long long)pl->sm_count * (smem > 56 * 1024 ? 2 : 4);
  if (blocks > cap) blocks = cap;
  dec_conv_mma_kernel<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(x, Tf, F, C, pl->cfg.n_src * 2,
                                                                       (const float*)(base + pl->lay.dec_w),
                                                                       (const float*)(base + pl->lay.dec_b), est,
                                                                       (long long)B * Tf);
  TFL_LAUNCH_CHECK();
  return 0;
}
}  // namespace tfl
extern "C" {

int tfl_dec_conv_mode(const tfl_plan* pl, const void* packed, const float* x, int B, int Tf, int F, float* est,
                      int precision, tfl_stream_t stream) {
  TFL_CHECK(pl && packed && x && est, "null argument");
  TFL_CHECK(pl->cfg.enc_in_ch == 2, "plan has no conv decoder");
  return dec_conv_any(pl, packed, x, B, Tf, F, est, precision, stream);
}

int tfl_dec_conv(const tfl_plan* pl, const void* packed, const float* x, int B, int Tf, int F, float* est,
                 tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::dec_conv");
  if (check_common(pl, packed, B, Tf, F, 0)) return -1;
  TFL_CHECK(pl->cfg.enc_in_ch == 2, "plan has no conv decoder");
  const int C = pl->cfg.emb_dim;
  const size_t smem = (size_t)9 * C * 8 * sizeof(float);
  TFL_CUDA(opt_in_smem(dec_conv_kernel, smem));
  const long long n_pos = (long long)B * Tf * F;
  const char* base = (const char*)packed;
  long long blocks = ((long long)B * Tf * ((F + DEC_P - 1) / DEC_P) + 7) / 8;   // one warp per group of DEC_P bins
  if (blocks > (long long)pl->sm_count * 2) blocks = (long long)pl->sm_count * 2;   // two resident blocks per SM, grid-stride
  dec_conv_kernel<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(x, Tf, F, C, pl->cfg.n_src * 2,
                                                                   (const float*)(base + pl->lay.dec_w),
                                                                   (const float*)(base + pl->lay.dec_b), est, n_pos);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_istft_ola(const tfl_plan* pl, const void* packed, const float* est, int B, int Tf, int T, float* audio,
                  tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::istft_ola");
  TFL_CHECK(pl && packed && est && audio, "null argument");
  const tfl_config& c = pl->cfg;
  TFL_CHECK(c.n_fft > 0, "plan has no STFT (n_fft == 0)");
  TFL_CHECK(B >= 1 && Tf >= 1 && T >= 1, "empty input");
  const char* base = (const char*)packed;
  const size_t fixed = (size_t)c.n_fft * sizeof(float2) + (size_t)(c.n_fft / 2) * sizeof(float2);
  int run = ISTFT_RUN;
  while (run > 1 && fixed + (size_t)2 * run * c.hop * sizeof(float) > (size_t)160 * 1024) --run;
  const size_t smem = fixed + (size_t)2 * run * c.hop * sizeof(float);
  TFL_CHECK(smem <= (size_t)TC_SMEM_MAX, "n_fft / hop_length too large for the iSTFT kernel's shared memory");
  TFL_CUDA(opt_in_smem(istft_ola_kernel, smem));
  const int n_blocks = (T + c.hop - 1) / c.hop;
  dim3 grid((n_blocks + run - 1) / run, c.n_src, B);
  istft_ola_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(est, c.n_src, Tf, c.n_fft, ilog2(c.n_fft), c.hop, T,
                                                              (const float2*)(base + pl->lay.twiddle),
                                                              (const float*)(base + pl->lay.window), audio, B, run);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_blocks(const tfl_plan* pl, const void* packed, float* x, int B, int Tf, int F, void* workspace,
               size_t ws_bytes, int precision, tfl_stream_t stream) {
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  return blocks_forward(pl, (const char*)packed, x, Dims{B, Tf, F}, ws, (char*)workspace, precision,
                        (cudaStream_t)stream);
}

int tfl_separator_forward(const tfl_plan* pl, const void* packed, const float* spec, int B, int Tf, int F, float* est,
                          void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  if (check_common(pl, packed, B, Tf, F, precision)) return -1;
  TFL_CHECK(spec && est, "null argument");
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  char* wsp = (char*)workspace;
  float* x = (float*)(wsp + ws.x);
  if (enc_conv_gln_any(pl, packed, spec, B, Tf, F, x, workspace, ws_bytes, precision, stream)) return -1;
  if (blocks_forward(pl, (const char*)packed, x, Dims{B, Tf, F}, ws, wsp, precision, (cudaStream_t)stream)) return -1;
  return dec_conv_any(pl, packed, x, B, Tf, F, est, precision, stream);
}

int tfl_forward(const tfl_plan* pl, const void* packed, const float* mixture, int B, int T, float* audio,
                float* est_spec, void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::forward");
  TFL_CHECK(pl && packed && mixture, "null argument");
  const tfl_config& c = pl->cfg;
  TFL_CHECK(c.n_fft > 0, "plan has no STFT (n_fft == 0)");
  TFL_CHECK(B >= 1, "empty batch");
  TFL_CHECK(T > c.n_fft / 2, "reflect padding needs more than n_fft/2 = %d samples (got %d)", c.n_fft / 2, T);
  const int Tf = 1 + T / c.hop, F = c.n_fft / 2 + 1;
  const Workspace ws = plan_workspace(pl, B, Tf, F, precision);
  TFL_CHECK(workspace && ws_bytes >= ws.total, "workspace too small (%zu < %zu)", ws_bytes, ws.total);
  char* wsp = (char*)workspace;
  float* spec = (float*)(wsp + ws.spec);
  float* est = est_spec != nullptr ? est_spec : (float*)(wsp + ws.est);
  if (tfl_stft(pl, packed, mixture, B, T, spec, stream)) return -1;
  if (tfl_separator_forward(pl, packed, spec, B, Tf, F, est, workspace, ws_bytes, precision, stream)) return -1;
  if (audio != nullptr) return tfl_istft_ola(pl, packed, est, B, Tf, T, audio, stream);
  return 0;
}

int tfl_segment_ola(const float* seg_audio, int n_src, int B, int seg_len, int seg_index0, int n_seg_total,
                    float* track, int64_t n_track, int64_t track_origin, tfl_stream_t stream) {
  TFL_CHECK(seg_audio && track, "null argument");
  TFL_CHECK(n_src >= 1 && B >= 1 && seg_len >= 2 && seg_len % 2 == 0, "bad segment shape");
  TFL_CHECK(seg_index0 >= 0 && seg_index0 + B <= n_seg_total, "segment index out of range");
  dim3 grid((seg_len + 255) / 256 < 296 ? (seg_len + 255) / 256 : 296, B, n_src);
  segment_ola_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seg_audio, n_src, B, seg_len, seg_index0, n_seg_total,
                                                             track, n_track, track_origin);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_segment_ola_hop(const float* seg_audio, int rows, int channels, int B, int seg_len, int hop, int seg_index0,
                        int n_seg_total, float* track, int64_t n_track, int64_t track_origin, tfl_stream_t stream) {
  TFL_CHECK(seg_audio && track, "null argument");
  TFL_CHECK(rows >= 1 && channels >= 1 && rows * (int64_t)channels <= 65535 && B >= 1 && seg_len >= 2,
            "bad segment shape");
  TFL_CHECK(hop >= 1 && hop < seg_len, "hop must be in [1, seg_len) (got %d for seg_len %d)", hop, seg_len);
  TFL_CHECK(seg_index0 >= 0 && seg_index0 + B <= n_seg_total, "segment index out of range");
  TFL_CHECK(n_track >= 0 && track_origin >= 0, "bad track range");
  // Output samples this call touches: the span of its segments, clipped to the local buffer.
  const int64_t lo = (int64_t)seg_index0 * hop - track_origin;
  const int64_t hi = (int64_t)(seg_index0 + B - 1) * hop + seg_len - track_origin;
  const int64_t j0 = lo > 0 ? lo : 0, j1 = hi < n_track ? hi : n_track;
  if (j1 <= j0) return 0;
  dim3 grid((unsigned)((j1 - j0 + 255) / 256), rows * channels);
  segment_ola_hop_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seg_audio, channels, B, seg_len, hop, seg_index0,
                                                                 n_seg_total, track, n_track, track_origin, j0, j1);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_bs_band_split(const float* spec, int B, int M, int T, int F, int C, int nb, int max_width,
                      const int64_t* table, const float* weights, float* x, tfl_stream_t stream) {
  TFL_CHECK(spec && table && weights && x, "null argument");
  TFL_CHECK(B >= 1 && (M == 1 || M == 2) && T >= 1 && F >= 1 && C >= 1 && nb >= 1 && max_width >= 1, "bad band-split shape");
  const size_t smem = ((size_t)max_width * 2 * M * BS_TT + 64) * sizeof(float);
  TFL_CUDA(opt_in_smem(bs_split_kernel, smem));
  dim3 grid(nb, (T + BS_TT - 1) / BS_TT, B);
  bs_split_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(spec, M, T, F, C, nb, (const long long*)table, weights, x, 1e-5f);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_bs_band_decode(const float* x, const float* spec, int B, int M, int T, int F, int C, int nb, int n_src,
                       const int64_t* table, const float* weights, float* est, int masking, tfl_stream_t stream) {
  TFL_CHECK(x && spec && table && weights && est, "null argument");
  TFL_CHECK(B >= 1 && (M == 1 || M == 2) && T >= 1 && F >= 1 && C >= 1 && nb >= 1 && n_src >= 1, "bad band-decode shape");
  const size_t smem = ((size_t)9 * C * BS_TT + 64) * sizeof(float);
  TFL_CHECK(smem <= (size_t)TC_SMEM_MAX, "emb_dim too large for the band decoder");
  TFL_CUDA(opt_in_smem(bs_decode_kernel, smem));
  dim3 grid(nb, (T + BS_TT - 1) / BS_TT, B);
  bs_decode_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(x, spec, M, T, F, C, nb, n_src, (const long long*)table, weights,
                                                              est, masking, 1e-5f);
  TFL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
namespace tfl {
struct BsBwdWs { size_t xn, h1, h2, dh1, dh2, dxn, dz, xs, xsn, dyin, stats, sums, total; };
static BsBwdWs bs_bwd_ws(int B, int M, int T, int F, int C, int nb, int S) {
  BsBwdWs w{};
  size_t off = 0;
  auto take = [&](size_t floats) { size_t o = off; off = align_up(off + floats * sizeof(float)); return o; };
  const size_t R = (size_t)B * T, rc = (size_t)nb * R * C;
  w.xn = take(rc); w.h1 = take(4 * rc); w.h2 = take(4 * rc); w.dh1 = take(4 * rc); w.dh2 = take(4 * rc); w.dxn = take(rc);
  w.dz = take(R * F * S * 4 * M);
  w.xs = take(R * F * 2 * M); w.xsn = take(R * F * 2 * M); w.dyin = take(R * F * 2 * M);
  w.stats = take((size_t)B * nb * 2);
  w.sums = take((size_t)B * nb * 4);   // doubles
  w.total = off;
  return w;
}
static inline BandMat band_mat(const void* p, long long per_band, long long per_bin, int ld0, int ldw) {
  return BandMat{(const float*)p, per_band, per_bin, ld0, ldw};
}
static int bs_bwd_check(int B, int M, int T, int F, int C, int nb, int S, int max_width, size_t ws_bytes) {
  TFL_CHECK(B >= 1 && (M == 1 || M == 2) && T >= 1 && F >= 1 && C >= 1 && nb >= 1 && S >= 1 && max_width >= 1,
            "bad band backward shape");
  TFL_CHECK(ws_bytes >= bs_bwd_ws(B, M, T, F, C, nb, S).total, "workspace too small (%zu < %zu)", ws_bytes,
            bs_bwd_ws(B, M, T, F, C, nb, S).total);
  return 0;
}
}  // namespace tfl
extern "C" {

size_t tfl_bs_band_bwd_workspace_bytes(int B, int M, int T, int F, int C, int nb, int n_src, int max_width) {
  (void)max_width;
  return bs_bwd_ws(B, M, T, F, C, nb, n_src).total;
}

int tfl_bs_band_decode_bwd(const float* x, const float* spec, const float* d_est, int B, int M, int T, int F, int C, int nb,
                           int n_src, int max_width, const int64_t* table, const float* weights, int masking, float* dx,
                           float* d_weights, void* workspace, size_t ws_bytes, tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::bs_band_decode_bwd");
  TFL_CHECK(x && spec && d_est && table && weights && dx && d_weights && workspace, "null argument");
  if (bs_bwd_check(B, M, T, F, C, nb, n_src, max_width, ws_bytes)) return -1;
  const BsBwdWs ws = bs_bwd_ws(B, M, T, F, C, nb, n_src);
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const long long* tab = (const long long*)table;
  const long long R = (long long)B * T;
  const int C4 = 4 * C, S4M = n_src * 4 * M;
  const size_t smem = ((size_t)9 * C * BS_TT + 64) * sizeof(float);
  TFL_CHECK(smem <= (size_t)TC_SMEM_MAX, "emb_dim too large for the band decoder");
  TFL_CUDA(opt_in_smem(bs_decode_bwd_rows_kernel, smem));
  bs_decode_bwd_rows_kernel<<<dim3(nb, (T + BS_TT - 1) / BS_TT, B), 256, smem, st>>>(
      x, spec, d_est, M, T, F, C, nb, n_src, tab, weights, masking, 1e-5f, (float*)(wsp + ws.xn), (float*)(wsp + ws.h1),
      (float*)(wsp + ws.h2), (float*)(wsp + ws.dz));
  TFL_LAUNCH_CHECK();
  const BandMat xn = band_mat(wsp + ws.xn, R * C, 0, C, 0), dxn = band_mat(wsp + ws.dxn, R * C, 0, C, 0);
  const BandMat h1 = band_mat(wsp + ws.h1, R * C4, 0, C4, 0), h2 = band_mat(wsp + ws.h2, R * C4, 0, C4, 0);
  const BandMat dh1 = band_mat(wsp + ws.dh1, R * C4, 0, C4, 0), dh2 = band_mat(wsp + ws.dh2, R * C4, 0, C4, 0);
  const BandMat dz = band_mat(wsp + ws.dz, 0, R * S4M, 0, S4M), none = band_mat(nullptr, 0, 0, 0, 0);
  const unsigned rt = (unsigned)((R + 63) / 64), omax_t = (unsigned)((max_width * S4M + 63) / 64);
  const unsigned c4_t = (unsigned)((C4 + 63) / 64), c_t = (unsigned)((C + 63) / 64);
  // data gradients: dh2 = dz . W4, dh1 = (dh2 . W3) * tanh', dxn = dh1 . W1
  bs_gemm_nt_kernel<<<dim3(rt, c4_t, nb), 256, 0, st>>>(BsGemm{dz, dh2, none, C4, 0, 0, S4M, 12, R}, tab, weights);
  TFL_LAUNCH_CHECK();
  bs_gemm_nt_kernel<<<dim3(rt, c4_t, nb), 256, 0, st>>>(BsGemm{dh2, dh1, h1, C4, 0, C4, 0, 10, R}, tab, weights);
  TFL_LAUNCH_CHECK();
  bs_gemm_nt_kernel<<<dim3(rt, c_t, nb), 256, 0, st>>>(BsGemm{dh1, dxn, none, C, 0, C4, 0, 8, R}, tab, weights);
  TFL_LAUNCH_CHECK();
  // weight and bias gradients of the three 1x1 convs
  bs_wgrad_kernel<<<dim3(omax_t, c4_t, nb), 256, 0, st>>>(BsWgrad{h2, dz, C4, 0, 0, S4M, 12, 13, R}, tab, d_weights);
  TFL_LAUNCH_CHECK();
  bs_wgrad_kernel<<<dim3(c4_t, c4_t, nb), 256, 0, st>>>(BsWgrad{h1, dh2, C4, 0, C4, 0, 10, 11, R}, tab, d_weights);
  TFL_LAUNCH_CHECK();
  bs_wgrad_kernel<<<dim3(c4_t, c_t, nb), 256, 0, st>>>(BsWgrad{xn, dh1, C, 0, C4, 0, 8, 9, R}, tab, d_weights);
  TFL_LAUNCH_CHECK();
  // GroupNorm(1, C) over (C, T): statistics and the two sums, then its parameter gradients and dx
  const BsNorm nrm{band_mat(x, C, 0, nb * C, 0), dxn, C, 0, 6, T};
  float* stats = (float*)(wsp + ws.stats);
  double* sums = (double*)(wsp + ws.sums);
  bs_gn_sums_kernel<<<dim3(nb, B), 256, 0, st>>>(nrm, tab, weights, 1e-5f, stats, sums);
  TFL_LAUNCH_CHECK();
  bs_gn_bwd_kernel<<<dim3(nb, (C + 31) / 32), dim3(32, 8), 0, st>>>(nrm, band_mat(dx, C, 0, nb * C, 0), B, tab, weights,
                                                                    stats, sums, d_weights);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_bs_band_split_bwd(const float* spec, const float* dx, int B, int M, int T, int F, int C, int nb, int max_width,
                          const int64_t* table, const float* weights, float* d_weights, void* workspace, size_t ws_bytes,
                          tfl_stream_t stream) {
  NvtxRange nvtx_range("tfl::bs_band_split_bwd");
  TFL_CHECK(spec && dx && table && weights && d_weights && workspace, "null argument");
  if (bs_bwd_check(B, M, T, F, C, nb, 1, max_width, ws_bytes)) return -1;
  const BsBwdWs ws = bs_bwd_ws(B, M, T, F, C, nb, 1);
  char* wsp = (char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const long long* tab = (const long long*)table;
  const long long R = (long long)B * T;
  const int M2 = 2 * M;
  float* stats = (float*)(wsp + ws.stats);
  const BandMat xs = band_mat(wsp + ws.xs, 0, R * M2, 0, M2), xsn = band_mat(wsp + ws.xsn, 0, R * M2, 0, M2);
  const BandMat dyin = band_mat(wsp + ws.dyin, 0, R * M2, 0, M2), dxm = band_mat(dx, C, 0, nb * C, 0);
  const BandMat none = band_mat(nullptr, 0, 0, 0, 0);
  // input features, their GroupNorm(1, K_b) statistics over (K_b, T), and the normalised features
  bs_split_rows_kernel<<<dim3(nb, B), 256, 0, st>>>(spec, M, T, F, tab, weights, nullptr, (float*)(wsp + ws.xs), nullptr);
  TFL_LAUNCH_CHECK();
  const BsNorm nrm{xs, dyin, 0, M2, 2, T};
  bs_gn_sums_kernel<<<dim3(nb, B), 256, 0, st>>>(BsNorm{xs, none, 0, M2, 2, T}, tab, weights, 1e-5f, stats, nullptr);
  TFL_LAUNCH_CHECK();
  bs_split_rows_kernel<<<dim3(nb, B), 256, 0, st>>>(spec, M, T, F, tab, weights, stats, (float*)(wsp + ws.xs),
                                                    (float*)(wsp + ws.xsn));
  TFL_LAUNCH_CHECK();
  // conv weight / bias gradients, then the gradient of the GroupNorm output and its parameter gradients
  const unsigned rt = (unsigned)((R + 63) / 64), kt = (unsigned)((max_width * M2 + 63) / 64), ct = (unsigned)((C + 63) / 64);
  bs_wgrad_kernel<<<dim3(ct, kt, nb), 256, 0, st>>>(BsWgrad{xsn, dxm, 0, M2, C, 0, 4, 5, R}, tab, d_weights);
  TFL_LAUNCH_CHECK();
  bs_gemm_nt_kernel<<<dim3(rt, kt, nb), 256, 0, st>>>(BsGemm{dxm, dyin, none, 0, M2, C, 0, 4, R}, tab, weights);
  TFL_LAUNCH_CHECK();
  bs_gn_bwd_kernel<<<dim3(nb, (max_width * M2 + 31) / 32), dim3(32, 8), 0, st>>>(nrm, none, B, tab, weights, stats, nullptr,
                                                                                 d_weights);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_pair_stats(const float* est, const float* tgt, int rows, int64_t n, double* out5, double* scratch,
                   size_t scratch_bytes, tfl_stream_t stream) {
  TFL_CHECK(est && tgt && out5 && scratch, "null argument");
  TFL_CHECK(rows >= 1 && n >= 1, "empty input");
  TFL_CHECK(scratch_bytes >= (size_t)rows * STATS_BLOCKS * 5 * sizeof(double), "scratch too small");
  pair_stats_partial_kernel<<<dim3(STATS_BLOCKS, rows), 256, 0, (cudaStream_t)stream>>>(est, tgt, (long long)n, scratch);
  TFL_LAUNCH_CHECK();
  pair_stats_finish_kernel<<<rows, 32, 0, (cudaStream_t)stream>>>(scratch, STATS_BLOCKS, out5);
  TFL_LAUNCH_CHECK();
  return 0;
}

int tfl_debug_set_option(int key, int value) {
  TFL_CHECK(key >= 0 && key < TFL_OPT_COUNT, "unknown option %d", key);
  g_options[key].store(value, std::memory_order_relaxed);
  if (key == TFL_OPT_TRACE_BASE) TFL_CUDA(cudaMemcpyToSymbol(tc::g_trace_base, &value, sizeof(int)));
  return 0;
}

int tfl_debug_set_trace(void* device_buffer) {
  unsigned long long* ptr = (unsigned long long*)device_buffer;
  TFL_CUDA(cudaMemcpyToSymbol(tc::g_trace, &ptr, sizeof(ptr)));
  return 0;
}

int tfl_debug_timeout(uint32_t* out5, int reset) {
  TFL_CHECK(out5 != nullptr, "null argument");
  std::lock_guard<std::mutex> lock(g_init_mu);
  for (int i = 0; i < 5; ++i) out5[i] = g_timeout_rec != nullptr ? g_timeout_rec[i] : 0u;
  if (reset && g_timeout_rec != nullptr) {
    for (int i = 0; i < 5; ++i) g_timeout_rec[i] = 0u;
    const uint32_t zero[5] = {0, 0, 0, 0, 0};
    (void)cudaMemcpyToSymbol(tc::g_wait_timeout, zero, sizeof(zero));   // fails after a trap (dead context): ignored
    (void)cudaGetLastError();
  }
  return 0;
}

int tfl_tc_selftest(const float* A, const float* B, float* D, void* scratch, int N, int Kd, int taps, int mode,
                    tfl_stream_t stream) {
  TFL_CHECK(A && B && D && scratch, "null argument");
  if (mode == 3) {
    TFL_CHECK(N % 16 == 0 && N <= 256 && Kd % 8 == 0 && taps >= 1 && taps <= 8, "selftest shape");
    return tf32_selftest(A, B, D, scratch, N, Kd, taps, (cudaStream_t)stream);
  }
  return tc_selftest(A, B, D, scratch, N, Kd, taps, mode, (cudaStream_t)stream);
}

}  // extern "C"

#include "tfl_train.cuh"
