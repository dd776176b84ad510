// C ABI of linetr_b200 (see include/linetr_b200.h): checkpoint folding/packing, workspace
// carving and the launch sequence of the line-descriptor forward and the matcher.
#include "../../include/linetr_b200.h"
#include "../../include/linetr_b200_debug.h"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <unordered_map>

#include "common.cuh"
#include "encoder_kernels.cuh"
#include "linear_f32.cuh"
#include "tc_weight.cuh"
#include "gemm_img.cuh"
#include "token_fused.cuh"
#include "sig_attention_tc.cuh"
#include "tokenizer_kernels.cuh"
#include "match_kernels.cuh"
#include "match_tc.cuh"

namespace ltr {

thread_local std::string g_last_error;
std::atomic<int64_t> g_launches{0};
Profiler g_prof;
std::mutex g_state_mutex;
std::vector<std::pair<const void*, int>> g_smem_configured;

int set_error(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

const char* kernel_class_name(int kc) {
  static const char* names[KC_COUNT] = {"small_mlp", "linear", "img_convert", "sig_attention", "final_norm",
                                         "dist", "segmean", "argmin", "mutual", "token_fused",
                                         "tokenize", "desc_tiles", "match_tc", "match_tail"};
  return (kc >= 0 && kc < KC_COUNT) ? names[kc] : "?";
}

cudaEvent_t Profiler::get() {
  if (!pool.empty()) {
    cudaEvent_t e = pool.back();
    pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

// ------------------------------------------------------------------ packed model
// One wide linear layer: fp32 bias and the packed split-bf16 tile image of the folded matrix.
struct Lin {
  const float* b = nullptr;
  TcWeight tw;
};

// Positional encoders: 3 (token) or 5 (line) inputs -> 32 -> 64 -> 128 -> 256 -> 256, ReLU after all but the last
// layer.  Each holds exactly what its kernels read.
struct TokenPosWeights {  // token stage (token_fused_kernel)
  const float *w1, *b1;   // 3 -> 32 in fp32
  Lin l2;                 // 32 -> 64 with K zero-padded to one 64-wide k-block
  Lin l3, l4, l5;
};

struct LinePosWeights {   // line stage: narrow head (small_mlp_kernel), then the two wide layers
  SmallMlpWeights head;   // 5 -> 32 -> 64 -> 128 in fp32
  Lin l4, l5;
};

struct SigLayer {
  Lin qkv;    // [768,256] head-major rows, q rows pre-scaled by 1/8
  Lin mlp1;   // [512,512] BN folded, attention output projection (`merge`) folded into the o-half
  Lin mlp2;   // [256,512]
};

}  // namespace ltr

struct LtrModel {
  int device = 0;
  LtrConfig cfg{};
  float* arena = nullptr;
  uint16_t* tc_arena = nullptr;
  size_t arena_floats = 0;
  ltr::TokenPosWeights wpe{};
  ltr::LinePosWeights lpe{};
  float *U = nullptr, *s_cls = nullptr, *cls = nullptr;
  ltr::Lin wv, wfc, w1, w2, wf;  // wv: 4 heads of [64,256]; wfc bias includes the CLS residual
  float *ln1g = nullptr, *ln1b = nullptr, *ln2g = nullptr, *ln2b = nullptr;
  std::vector<ltr::SigLayer> sig;
};

namespace ltr {

using TensorMap = std::unordered_map<std::string, std::pair<const float*, int64_t>>;

struct LinOff { size_t b, tc; int N, K; };

struct HostPack {
  std::vector<float> buf;
  std::vector<uint16_t> tc;  // packed split-bf16 images: hi at off, lo at off + N*K
  size_t add(const std::vector<double>& v) {
    size_t off = (buf.size() + 63) / 64 * 64;  // 256-byte alignment of every tensor
    buf.resize(off + v.size());
    for (size_t i = 0; i < v.size(); ++i) buf[off + i] = (float)v[i];
    return off;
  }
  // wide layer [N,K]: bias + tensor-core image
  LinOff add_lin(const std::vector<double>& W, const std::vector<double>& b, int N, int K) {
    LinOff o{add(b), 0, N, K};
    size_t off = (tc.size() + 511) / 512 * 512;  // 1024-byte alignment
    tc.resize(off + 2 * (size_t)N * K);
    pack_tc_weight(W.data(), N, K, tc.data() + off, tc.data() + off + (size_t)N * K);
    o.tc = off;
    return o;
  }
};

static Lin bind_lin(const LinOff& o, float* fbase, uint16_t* tbase) {
  Lin l;
  l.b = fbase + o.b;
  l.tw.hi = reinterpret_cast<const __nv_bfloat16*>(tbase + o.tc);
  l.tw.lo = reinterpret_cast<const __nv_bfloat16*>(tbase + o.tc + (size_t)o.N * o.K);
  l.tw.N = o.N;
  l.tw.K = o.K;
  return l;
}

static bool fetch(const TensorMap& tm, const std::string& name, int64_t numel, const float** out, std::string& err) {
  auto it = tm.find(name);
  if (it == tm.end()) { err = "missing checkpoint tensor '" + name + "'"; return false; }
  if (it->second.second != numel) {
    err = "checkpoint tensor '" + name + "' has " + std::to_string(it->second.second) + " elements, expected " +
          std::to_string(numel);
    return false;
  }
  *out = it->second.first;
  return true;
}

// Conv1d(k=1)/Linear [out,in] (+ eval BatchNorm1d at bn_prefix, eps 1e-5) -> folded W, b in fp64.
static bool fold_layer(const TensorMap& tm, const std::string& conv, const std::string& bn, int out, int in,
                       std::vector<double>& W, std::vector<double>& b, std::string& err) {
  const float *w, *bias;
  if (!fetch(tm, conv + ".weight", (int64_t)out * in, &w, err) || !fetch(tm, conv + ".bias", out, &bias, err)) return false;
  W.assign((size_t)out * in, 0.0);
  b.assign(out, 0.0);
  for (int o = 0; o < out; ++o) {
    double s = 1.0, shift = 0.0;
    if (!bn.empty()) {
      const float *g, *be, *mu, *var;
      if (!fetch(tm, bn + ".weight", out, &g, err) || !fetch(tm, bn + ".bias", out, &be, err) ||
          !fetch(tm, bn + ".running_mean", out, &mu, err) || !fetch(tm, bn + ".running_var", out, &var, err))
        return false;
      s = (double)g[o] / std::sqrt((double)var[o] + 1e-5);
      shift = (double)be[o] - (double)mu[o] * s;
    }
    for (int i = 0; i < in; ++i) W[(size_t)o * in + i] = (double)w[(size_t)o * in + i] * s;
    b[o] = (double)bias[o] * s + shift;
  }
  return true;
}

// The five layers of a positional encoder (models/line_transformer.py:9-20), eval-BatchNorm folded into the first four.
static bool fold_pos_encoder(const TensorMap& tm, const std::string& prefix, int in, std::vector<double> (&W)[5],
                             std::vector<double> (&b)[5], std::string& err) {
  const int ch[6] = {in, 32, 64, 128, 256, 256};
  for (int l = 0; l < 5; ++l) {
    const std::string conv = prefix + "." + std::to_string(3 * l);
    const std::string bn = (l < 4) ? prefix + "." + std::to_string(3 * l + 1) : std::string();
    if (!fold_layer(tm, conv, bn, ch[l + 1], ch[l], W[l], b[l], err)) return false;
  }
  return true;
}

struct TokenPosOff { size_t w1, b1; LinOff l2, l3, l4, l5; };

static bool pack_token_pos(const TensorMap& tm, HostPack& hp, TokenPosOff& off, std::string& err) {
  std::vector<double> W[5], b[5];
  if (!fold_pos_encoder(tm, "klenc.word_position_enc.encoder", 3, W, b, err)) return false;
  off.w1 = hp.add(W[0]);
  off.b1 = hp.add(b[0]);
  std::vector<double> W2((size_t)64 * 64, 0.0);
  for (int o = 0; o < 64; ++o)
    for (int i = 0; i < 32; ++i) W2[(size_t)o * 64 + i] = W[1][(size_t)o * 32 + i];
  off.l2 = hp.add_lin(W2, b[1], 64, 64);
  off.l3 = hp.add_lin(W[2], b[2], 128, 64);
  off.l4 = hp.add_lin(W[3], b[3], 256, 128);
  off.l5 = hp.add_lin(W[4], b[4], 256, 256);
  return true;
}

struct LinePosOff { size_t w[3], b[3]; LinOff l4, l5; };

static bool pack_line_pos(const TensorMap& tm, HostPack& hp, LinePosOff& off, std::string& err) {
  std::vector<double> W[5], b[5];
  if (!fold_pos_encoder(tm, "klenc.line_position_enc.encoder", 5, W, b, err)) return false;
  for (int l = 0; l < 3; ++l) {
    off.w[l] = hp.add(W[l]);
    off.b[l] = hp.add(b[l]);
  }
  off.l4 = hp.add_lin(W[3], b[3], 256, 128);
  off.l5 = hp.add_lin(W[4], b[4], 256, 256);
  return true;
}

static cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ------------------------------------------------------------------ workspace
struct EncodeWs {
  // line stage
  ActImg z, ctx, y1i, g, l128, l256, lpos;  // images [R, 1024 / 256 / 256 / 1024 / 128 / 256 / 256]
  // signature stage
  ActImg xm, hm;       // images [R, 512] = [x | attention output], [R, 512]
  ActImg qkv;          // image [R, 768]: k-block h = q of head h, 4 + h = k, 8 + h = v
  float* yf;           // fp32 [R, 256] (final projection when the channel-first layout is requested)
  int64_t bytes;
};

static EncodeWs carve(const LtrModel* m, int n_lines, char* base) {
  EncodeWs w{};
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* p = base + off;
    off = align_up(off + bytes, 1024);
    return p;
  };
  auto takef = [&](int64_t floats) { return reinterpret_cast<float*>(take(floats * 4)); };
  auto takei = [&](int64_t rows, int K) {
    const int64_t mpad = align_up(rows, 256);
    ActImg a;
    a.hi = reinterpret_cast<__nv_bfloat16*>(take(mpad * K * 2));
    a.lo = reinterpret_cast<__nv_bfloat16*>(take(mpad * K * 2));
    a.kblocks = K / 64;
    return a;
  };
  const int64_t R = n_lines;
  w.z = takei(R, 1024);
  w.ctx = takei(R, 256);
  w.y1i = takei(R, 256);
  w.g = takei(R, m->cfg.d_inner);   // FFN hidden activation [R, d_inner]
  w.l128 = takei(R, 128);
  w.l256 = takei(R, 256);
  w.lpos = takei(R, 256);
  w.xm = takei(R, 512);
  w.hm = takei(R, 512);
  w.qkv = takei(R, 768);
  w.yf = takef(R * 256);
  w.bytes = off;
  return w;
}

static LinearArgs lin(const float* A, int lda, const float* W, const float* b, float* C, int ldc, int M, int N, int K,
                      int act, const float* R = nullptr, int ldr = 0) {
  LinearArgs a{};
  a.A = A; a.lda = lda; a.W = W; a.bias = b; a.R = R; a.ldr = ldr; a.C = C; a.ldc = ldc;
  a.M = M; a.N = N; a.K = K; a.act = act; a.nz = 1;
  return a;
}

// One wide layer on the tensor-core engine: A image k-blocks [a_kb0, a_kb0 + K/64) -> fp32 rows C
// (optional) and/or image O k-blocks from o_kb0 (optional); R = fp32 residual.
static GemmImgArgs gemm_args(const Lin& L, const ActImg& A, int a_kb0, int M, int act, float* C, int ldc,
                             const ActImg* O = nullptr, int o_kb0 = 0, const float* R = nullptr, int ldr = 0,
                             const ActImg* Rimg = nullptr, int r_kb0 = 0, int a_kb_nb = 0) {
  GemmImgArgs a{};
  a.A = A; a.a_kb0 = a_kb0; a.W = L.tw; a.bias = L.b; a.R = R; a.ldr = ldr; a.C = C; a.ldc = ldc;
  if (O) { a.O = *O; a.o_kb0 = o_kb0; }
  if (Rimg) { a.Rimg = *Rimg; a.r_kb0 = r_kb0; }
  a.M = M; a.act = act; a.a_kb_nb = a_kb_nb;
  return a;
}

static int gemm(const Lin& L, const ActImg& A, int a_kb0, int M, int act, cudaStream_t s, float* C, int ldc,
                const ActImg* O = nullptr, int o_kb0 = 0, const float* R = nullptr, int ldr = 0,
                const ActImg* Rimg = nullptr, int r_kb0 = 0, int bn_hint = 0, int a_kb_nb = 0) {
  return launch_gemm_img(gemm_args(L, A, a_kb0, M, act, C, ldc, O, o_kb0, R, ldr, Rimg, r_kb0, a_kb_nb), s, bn_hint);
}

// Batches with at least this many 128-row tiles run the row-local GEMMs of a signature layer as ONE chained
// launch (gemm_chain2_kernel); smaller ones keep one launch per layer, which spreads the n-blocks of the few
// m-tiles over more SMs.  LTR_CHAIN_MIN_TILES overrides (0 = never chain).
static int chain_min_tiles() {
  static const int v = [] {
    const char* e = std::getenv("LTR_CHAIN_MIN_TILES");
    return e ? std::atoi(e) : 96;
  }();
  return v;
}

static int launch_small_mlp(const SmallMlpWeights& w, const float* in0, const float* in1, const float* in2, ActImg out,
                            int rows, float width, float height, cudaStream_t s) {
  if (rows <= 0) return 0;
  const int smem = (int)sizeof(SmallMlpSmem);
  LTR_CUDA_TRY(ensure_dynamic_smem(small_mlp_kernel, smem));
  const int groups = cdiv(rows, SM_ROWS);
  int grid = cdiv(groups, SM_WARPS);
  if (grid > 148 * 3) grid = 148 * 3;
  const float scale = fmaxf(width, height) * 0.7f;
  LaunchScope ls(KC_SMALL_MLP, s);
  LTR_CUDA_TRY(launch_pdl(small_mlp_kernel, dim3(grid), dim3(SM_WARPS * 32), (size_t)smem, s, w, in0, in1, in2, out, rows,
                          width / 2.f, height / 2.f, scale));
  return 0;
}

#define LTR_TRY(expr)        \
  do {                       \
    int _rc = (expr);        \
    if (_rc != 0) return _rc; \
  } while (0)

static ActImg tiles_image(void* tiles, int64_t n_lines) {
  ActImg a;
  const int64_t plane = align_up(n_lines, 128) * MT_D;   // bf16 elements per plane
  a.hi = reinterpret_cast<__nv_bfloat16*>(tiles);
  a.lo = a.hi + plane;
  a.kblocks = MT_KB;
  return a;
}

static int encode_impl(LtrModel* m, const LtrEncodeInput& in, float* out_cf, float* out_rows, void* out_tiles,
                       const EncodeWs& w, cudaStream_t s) {
  const int R = in.n_lines, T = in.n_tokens;
  const int* cu = in.cu_lines_dev;
  // ---- token stage: one fused persistent kernel (narrow MLP, 3 tensor-core layers, + desc, CLS pooling) ----
  {
    TokenFusedArgs a{};
    a.pnt = in.pnt; a.score = in.score; a.desc = in.desc;
    a.w1 = m->wpe.w1; a.b1 = m->wpe.b1; a.b2 = m->wpe.l2.b;
    a.W2 = m->wpe.l2.tw; a.W3 = m->wpe.l3.tw; a.W4 = m->wpe.l4.tw; a.W5 = m->wpe.l5.tw;
    a.b3 = m->wpe.l3.b; a.b4 = m->wpe.l4.b; a.b5 = m->wpe.l5.b;
    a.U = m->U; a.s_cls = m->s_cls; a.cls = m->cls;
    a.z = w.z; a.R = R; a.T = T;
    a.cx = in.image_width / 2.f; a.cy = in.image_height / 2.f;
    a.scale = fmaxf(in.image_width, in.image_height) * 0.7f;
    LTR_TRY(launch_token_fused(a, s));
  }
  // ---- line stage: V projection (block diagonal over heads), fc + CLS residual, LN, FFN, LN, + line pos ----
  LTR_TRY(gemm(m->wv, w.z, 0, R, ACT_NONE, s, nullptr, 0, &w.ctx, 0, nullptr, 0, nullptr, 0, 64, 4));
  const bool chain = chain_min_tiles() > 0 && cdiv(R, 128) >= chain_min_tiles() && !out_cf && !m->sig.empty();
  const bool chain_line = chain && m->cfg.d_inner % 256 == 0;
  // line positional encoder first (its output is added in the w_2 epilogue)
  LTR_TRY(launch_small_mlp(m->lpe.head, in.sublines, in.resp, in.angle, w.l128, R, in.image_width, in.image_height, s));
  LTR_TRY(gemm(m->lpe.l4, w.l128, 0, R, ACT_RELU, s, nullptr, 0, &w.l256, 0));
  LTR_TRY(gemm(m->lpe.l5, w.l256, 0, R, ACT_NONE, s, nullptr, 0, &w.lpos, 0));
  {
    // fc (+ CLS residual folded into the bias) -> LayerNorm in the epilogue -> y1.  y1 and the line position code live
    // only as split-bf16 images (hi + lo: ~2^-17 relative): the FFN residual and the post-norm addend are read back
    // from them, row by row, straight into registers
    GemmImgArgs fc = gemm_args(m->wfc, w.ctx, 0, R, ACT_NONE, nullptr, 0, &w.y1i, 0);
    fc.norm = NORM_LAYER; fc.eps = 1e-6f; fc.ng = m->ln1g; fc.nbeta = m->ln1b;
    GemmImgArgs w1 = gemm_args(m->w1, w.y1i, 0, R, ACT_GELU, nullptr, 0, &w.g, 0);
    // sentence = klines_pos + LN(y1 + ffn)  -> image xm[:, :256] (the running descriptor), all in the w_2 epilogue
    GemmImgArgs w2 = gemm_args(m->w2, w.g, 0, R, ACT_NONE, nullptr, 0, &w.xm, 0, nullptr, 0, &w.y1i, 0);
    w2.norm = NORM_LAYER; w2.eps = 1e-6f; w2.ng = m->ln2g; w2.nbeta = m->ln2b; w2.NaddImg = w.lpos; w2.nadd_kb0 = 0;
    if (chain_line) {   // row-local: fc -> w_1 -> w_2 -> qkv of signature layer 0 in one launch
      GemmImgArgs ops[4] = {fc, w1, w2, gemm_args(m->sig[0].qkv, w.xm, 0, R, ACT_NONE, nullptr, 0, &w.qkv, 0)};
      LTR_TRY(launch_gemm_chain(ops, 4, s));
    } else {
      LTR_TRY(launch_gemm_img(fc, s, 256));
      LTR_TRY(launch_gemm_img(w1, s));
      LTR_TRY(launch_gemm_img(w2, s, 256));
    }
  }
  // ---- line signature layers ----
  int max_l = in.lines_per_image;
  if (in.cu_lines_host) {
    max_l = 0;
    for (int i = 0; i < in.n_images; ++i) max_l = std::max(max_l, in.cu_lines_host[i + 1] - in.cu_lines_host[i]);
  }
  ActImg tiles{};
  if (out_tiles) tiles = tiles_image(out_tiles, R);
  GemmImgArgs fin = gemm_args(m->wf, w.xm, 0, R, ACT_NONE, out_rows, 256, out_tiles ? &tiles : nullptr, 0);
  fin.norm = NORM_L2; fin.eps = 1e-6f;   // final_proj + F.normalize in one epilogue (rows-only output)
  for (size_t li = 0; li < m->sig.size(); ++li) {
    const SigLayer& L = m->sig[li];
    if (!chain || (li == 0 && !chain_line)) LTR_TRY(gemm(L.qkv, w.xm, 0, R, ACT_NONE, s, nullptr, 0, &w.qkv, 0));
    // o -> xm[:, 256:]
    LTR_TRY(launch_sig_attention_tc(w.qkv, w.xm, 256, cu, in.lines_per_image, max_l, in.n_images, s));
    // x += delta: the running descriptor lives ONLY as the split-bf16 image xm[:, :256] (hi + lo carries
    // ~2^-17 relative precision; an fp32 copy would double the store traffic of this epilogue)
    if (chain) {
      // mlp1 -> mlp2 (+ residual, in place) -> qkv of the next layer / final projection: row-local, one launch
      const bool last = li + 1 == m->sig.size();
      GemmImgArgs ops[3] = {gemm_args(L.mlp1, w.xm, 0, R, ACT_RELU, nullptr, 0, &w.hm, 0),
                            gemm_args(L.mlp2, w.hm, 0, R, ACT_NONE, nullptr, 0, &w.xm, 0, nullptr, 0, &w.xm, 0),
                            last ? fin : gemm_args(m->sig[li + 1].qkv, w.xm, 0, R, ACT_NONE, nullptr, 0, &w.qkv, 0)};
      LTR_TRY(launch_gemm_chain(ops, 3, s));
    } else {
      LTR_TRY(gemm(L.mlp1, w.xm, 0, R, ACT_RELU, s, nullptr, 0, &w.hm, 0));
      LTR_TRY(gemm(L.mlp2, w.hm, 0, R, ACT_NONE, s, nullptr, 0, &w.xm, 0, nullptr, 0, &w.xm, 0));
    }
  }
  if (chain) return 0;
  if (!out_cf) {   // rows (+ matcher tile image): projection + L2 normalisation in one launch
    LTR_TRY(launch_gemm_img(fin, s, 256));
    return 0;
  }
  LTR_TRY(gemm(m->wf, w.xm, 0, R, ACT_NONE, s, w.yf, 256));
  if (max_l > 0) {
    LaunchScope ls(KC_FINAL_NORM, s);
    dim3 grid(cdiv(max_l, 32), in.n_images);
    LTR_CUDA_TRY(launch_pdl(final_norm_kernel, grid, dim3(256), 0, s, (const float*)w.yf, out_rows, out_cf, cu, in.lines_per_image));
  }
  return 0;
}

static int run_nn(const NNArgs& a, int n_pairs, int max_k0, int max_k1, cudaStream_t s) {
  if (max_k0 <= 0) {
    LTR_CUDA_TRY(cudaMemsetAsync(a.counts, 0, sizeof(int) * n_pairs, s));
    return 0;
  }
  {
    LaunchScope ls(KC_ARGMIN, s);   // also zeroes counts[pair]
    LTR_CUDA_TRY(launch_pdl(row_argmin_kernel, dim3(cdiv(max_k0, 8), n_pairs), dim3(256), 0, s, a));
  }
  if (a.mutual && max_k1 > 0) {
    LaunchScope ls(KC_ARGMIN, s);
    LTR_CUDA_TRY(launch_pdl(col_argmin_kernel, dim3(cdiv(max_k1, 32), n_pairs), dim3(256), 0, s, a));
  }
  {
    LaunchScope ls(KC_MUTUAL, s);
    LTR_CUDA_TRY(launch_pdl(mutual_kernel, dim3(cdiv(max_k0, 256), n_pairs), dim3(256), 0, s, a));
  }
  return 0;
}

}  // namespace ltr

using namespace ltr;

extern "C" {

int ltr_abi_version(void) { return LTR_ABI_VERSION; }
const char* ltr_last_error(void) { return g_last_error.c_str(); }
int64_t ltr_launch_count(void) { return g_launches.load(); }
void ltr_reset_launch_count(void) { g_launches.store(0); }

void ltr_profile_begin(void) {
  for (auto& r : g_prof.recs) { g_prof.pool.push_back(r.a); g_prof.pool.push_back(r.b); }
  g_prof.recs.clear();
  g_prof.on = true;
}

int ltr_profile_end(const char** names, float* ms, int32_t* launches, int32_t max_classes) {
  g_prof.on = false;
  cudaDeviceSynchronize();
  float tot[KC_COUNT] = {0};
  int cnt[KC_COUNT] = {0};
  for (auto& r : g_prof.recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { tot[r.kc] += t; cnt[r.kc]++; }
    g_prof.pool.push_back(r.a);
    g_prof.pool.push_back(r.b);
  }
  g_prof.recs.clear();
  int n = 0;
  for (int k = 0; k < KC_COUNT && n < max_classes; ++k) {
    if (!cnt[k]) continue;
    names[n] = kernel_class_name(k);
    ms[n] = tot[k];
    launches[n] = cnt[k];
    ++n;
  }
  return n;
}

int ltr_create(const LtrTensor* tensors, int32_t n_tensors, const LtrConfig* cfg, int32_t device, LtrModel** out) {
  if (!tensors || !cfg || !out) return set_error(LTR_E_INVALID, "ltr_create: null argument");
  if (cfg->d_model != 256 || cfg->n_heads != 4)
    return set_error(LTR_E_UNSUPPORTED, "ltr_create: kernels are specialised for d_model=256, n_heads=4");
  if (cfg->d_inner <= 0 || cfg->d_inner % 128 || cfg->n_desc_layers < 1 || cfg->n_sig_layers < 0)
    return set_error(LTR_E_INVALID, "ltr_create: bad d_inner / layer counts");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_error(LTR_E_CUDA, "ltr_create: no CUDA device (there is no CPU fallback)");
  if (device < 0 || device >= ndev) return set_error(LTR_E_INVALID, "ltr_create: bad device index");
  LTR_CUDA_TRY(cudaSetDevice(device));

  TensorMap tm;
  for (int i = 0; i < n_tensors; ++i) tm[tensors[i].name] = {tensors[i].data, tensors[i].numel};
  std::string err;
  HostPack hp;
  const int D = 256, DI = cfg->d_inner;
  TokenPosOff wpe_o{};
  LinePosOff lpe_o{};
  if (!pack_token_pos(tm, hp, wpe_o, err) || !pack_line_pos(tm, hp, lpe_o, err)) return set_error(LTR_E_INVALID, err);

  // ---- descriptive layer (only the last one is live) ----
  const std::string dl = "klenc.desc_layers." + std::to_string(cfg->n_desc_layers - 1);
  const float *cls, *wq, *bq, *wk, *bk, *wv, *bv, *wfc, *bfc, *ln1g, *ln1b, *w1, *b1, *w2, *b2, *ln2g, *ln2b;
  if (!fetch(tm, "klenc.cls_token", D, &cls, err) ||
      !fetch(tm, dl + ".slf_attn.w_qs.weight", D * D, &wq, err) || !fetch(tm, dl + ".slf_attn.w_qs.bias", D, &bq, err) ||
      !fetch(tm, dl + ".slf_attn.w_ks.weight", D * D, &wk, err) || !fetch(tm, dl + ".slf_attn.w_ks.bias", D, &bk, err) ||
      !fetch(tm, dl + ".slf_attn.w_vs.weight", D * D, &wv, err) || !fetch(tm, dl + ".slf_attn.w_vs.bias", D, &bv, err) ||
      !fetch(tm, dl + ".slf_attn.fc.weight", D * D, &wfc, err) || !fetch(tm, dl + ".slf_attn.fc.bias", D, &bfc, err) ||
      !fetch(tm, dl + ".slf_attn.layer_norm.weight", D, &ln1g, err) ||
      !fetch(tm, dl + ".slf_attn.layer_norm.bias", D, &ln1b, err) ||
      !fetch(tm, dl + ".pos_ffn.w_1.weight", (int64_t)DI * D, &w1, err) || !fetch(tm, dl + ".pos_ffn.w_1.bias", DI, &b1, err) ||
      !fetch(tm, dl + ".pos_ffn.w_2.weight", (int64_t)D * DI, &w2, err) || !fetch(tm, dl + ".pos_ffn.w_2.bias", D, &b2, err) ||
      !fetch(tm, dl + ".pos_ffn.layer_norm.weight", D, &ln2g, err) ||
      !fetch(tm, dl + ".pos_ffn.layer_norm.bias", D, &ln2b, err))
    return set_error(LTR_E_INVALID, err);
  (void)bk;  // the key bias shifts all scores of a head equally: cancels in the softmax
  auto vec = [](const float* p, size_t n) { return std::vector<double>(p, p + n); };
  // q_cls = W_q cls + b_q ;  u_h = W_k,h^T q_h / sqrt(64) ;  s_cls,h = cls . u_h
  std::vector<double> q(D), U(4 * D, 0.0), scls(4, 0.0);
  for (int o = 0; o < D; ++o) {
    double a = bq[o];
    for (int i = 0; i < D; ++i) a += (double)wq[o * D + i] * cls[i];
    q[o] = a;
  }
  for (int h = 0; h < 4; ++h) {
    for (int c = 0; c < D; ++c) {
      double a = 0;
      for (int d = 0; d < 64; ++d) a += (double)wk[(h * 64 + d) * D + c] * q[h * 64 + d];
      U[h * D + c] = a / 8.0;
    }
    for (int c = 0; c < D; ++c) scls[h] += (double)cls[c] * U[h * D + c];
  }
  std::vector<double> bfc_cls(D);
  for (int i = 0; i < D; ++i) bfc_cls[i] = (double)bfc[i] + cls[i];  // fc bias + CLS residual (line_attention.py:72)
  size_t oU = hp.add(U), oS = hp.add(scls), oC = hp.add(vec(cls, D));
  // V projection of the pooled per-head inputs z = [z_0 | z_1 | z_2 | z_3]: output channels h*64..h*64+63
  // only see z_h, i.e. a block-diagonal GEMM - run as N = 256, K = 256 with 64-wide n-blocks whose A
  // k-blocks start at 4*h (GemmImgArgs::a_kb_nb).
  LinOff oWv = hp.add_lin(vec(wv, D * D), vec(bv, D), D, D);
  LinOff oWfc = hp.add_lin(vec(wfc, D * D), bfc_cls, D, D);
  size_t oL1g = hp.add(vec(ln1g, D)), oL1b = hp.add(vec(ln1b, D));
  LinOff oW1 = hp.add_lin(vec(w1, (size_t)DI * D), vec(b1, DI), DI, D);
  LinOff oW2 = hp.add_lin(vec(w2, (size_t)D * DI), vec(b2, D), D, DI);
  size_t oL2g = hp.add(vec(ln2g, D)), oL2b = hp.add(vec(ln2b, D));

  // ---- signature layers ----
  struct SigOff { LinOff qkv, mlp1, mlp2; };
  std::vector<SigOff> so(cfg->n_sig_layers);
  for (int li = 0; li < cfg->n_sig_layers; ++li) {
    const std::string p = "selfattn.layers." + std::to_string(li);
    std::vector<double> Wqkv((size_t)768 * D), bqkv(768);
    for (int t = 0; t < 3; ++t) {
      const float *w, *b;
      if (!fetch(tm, p + ".attn.proj." + std::to_string(t) + ".weight", D * D, &w, err) ||
          !fetch(tm, p + ".attn.proj." + std::to_string(t) + ".bias", D, &b, err))
        return set_error(LTR_E_INVALID, err);
      const double sc = (t == 0) ? 0.125 : 1.0;  // scores / sqrt(64), line_transformer.py:134
      for (int h = 0; h < 4; ++h)
        for (int d = 0; d < 64; ++d) {
          const int oldr = d * 4 + h, newr = t * 256 + h * 64 + d;  // view(b, dim, heads, n), :151
          for (int i = 0; i < D; ++i) Wqkv[(size_t)newr * D + i] = (double)w[oldr * D + i] * sc;
          bqkv[newr] = (double)b[oldr] * sc;
        }
    }
    const float *wm, *bm;
    if (!fetch(tm, p + ".attn.merge.weight", D * D, &wm, err) || !fetch(tm, p + ".attn.merge.bias", D, &bm, err))
      return set_error(LTR_E_INVALID, err);
    std::vector<double> Wm((size_t)D * D);
    for (int o = 0; o < D; ++o)
      for (int h = 0; h < 4; ++h)
        for (int d = 0; d < 64; ++d) Wm[(size_t)o * D + h * 64 + d] = wm[o * D + d * 4 + h];
    std::vector<double> W1, B1, W2, B2;
    if (!fold_layer(tm, p + ".mlp.0", p + ".mlp.1", 2 * D, 2 * D, W1, B1, err) ||
        !fold_layer(tm, p + ".mlp.3", "", D, 2 * D, W2, B2, err))
      return set_error(LTR_E_INVALID, err);
    // Fold the attention output projection (`merge`) into the first MLP layer:
    //   mlp1([x | merge(o)]) = W1a x + W1b (Wm o + bm) + b1 = [W1a | W1b Wm] [x | o] + (b1 + W1b bm)
    // so the attention kernel writes o straight into the second half of the MLP input and the
    // merge GEMM (one launch + one activation round trip per layer) disappears.
    std::vector<double> W1f((size_t)2 * D * 2 * D), B1f(2 * D);
    for (int o = 0; o < 2 * D; ++o) {
      double bacc = B1[o];
      for (int i = 0; i < D; ++i) W1f[(size_t)o * 2 * D + i] = W1[(size_t)o * 2 * D + i];
      for (int j = 0; j < D; ++j) {
        double a = 0.0;
        for (int i = 0; i < D; ++i) a += W1[(size_t)o * 2 * D + D + i] * Wm[(size_t)i * D + j];
        W1f[(size_t)o * 2 * D + D + j] = a;
      }
      for (int i = 0; i < D; ++i) bacc += W1[(size_t)o * 2 * D + D + i] * (double)bm[i];
      B1f[o] = bacc;
    }
    so[li] = {hp.add_lin(Wqkv, bqkv, 768, D), hp.add_lin(W1f, B1f, 2 * D, 2 * D), hp.add_lin(W2, B2, D, 2 * D)};
  }
  std::vector<double> Wf, Bf;
  if (!fold_layer(tm, "final_proj", "", D, D, Wf, Bf, err)) return set_error(LTR_E_INVALID, err);
  LinOff oWf = hp.add_lin(Wf, Bf, D, D);

  LtrModel* m = new LtrModel();
  m->device = device;
  m->cfg = *cfg;
  m->arena_floats = hp.buf.size();
  cudaError_t ce = cudaMalloc(&m->arena, hp.buf.size() * sizeof(float));
  if (ce == cudaSuccess) ce = cudaMemcpy(m->arena, hp.buf.data(), hp.buf.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMalloc(&m->tc_arena, hp.tc.size() * sizeof(uint16_t));
  if (ce == cudaSuccess) ce = cudaMemcpy(m->tc_arena, hp.tc.data(), hp.tc.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) {
    if (m->arena) cudaFree(m->arena);
    if (m->tc_arena) cudaFree(m->tc_arena);
    delete m;
    return set_error(LTR_E_CUDA, std::string("ltr_create: ") + cudaGetErrorString(ce));
  }
  float* B = m->arena;
  uint16_t* TB = m->tc_arena;
  m->wpe = {B + wpe_o.w1, B + wpe_o.b1, bind_lin(wpe_o.l2, B, TB), bind_lin(wpe_o.l3, B, TB), bind_lin(wpe_o.l4, B, TB),
            bind_lin(wpe_o.l5, B, TB)};
  m->lpe = {{B + lpe_o.w[0], B + lpe_o.b[0], B + lpe_o.w[1], B + lpe_o.b[1], B + lpe_o.w[2], B + lpe_o.b[2]},
            bind_lin(lpe_o.l4, B, TB), bind_lin(lpe_o.l5, B, TB)};
  m->U = B + oU; m->s_cls = B + oS; m->cls = B + oC;
  m->wv = bind_lin(oWv, B, TB);
  m->wfc = bind_lin(oWfc, B, TB);
  m->ln1g = B + oL1g; m->ln1b = B + oL1b;
  m->w1 = bind_lin(oW1, B, TB);
  m->w2 = bind_lin(oW2, B, TB);
  m->ln2g = B + oL2g; m->ln2b = B + oL2b;
  for (auto& o : so)
    m->sig.push_back({bind_lin(o.qkv, B, TB), bind_lin(o.mlp1, B, TB), bind_lin(o.mlp2, B, TB)});
  m->wf = bind_lin(oWf, B, TB);
  *out = m;
  return LTR_OK;
}

void ltr_destroy(LtrModel* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  if (m->arena) cudaFree(m->arena);
  if (m->tc_arena) cudaFree(m->tc_arena);
  delete m;
}

int64_t ltr_encode_workspace_bytes(const LtrModel* m, int32_t n_images, int32_t n_lines, int32_t n_tokens) {
  (void)n_images;
  if (!m || n_lines < 0 || n_tokens < 1) return set_error(LTR_E_INVALID, "ltr_encode_workspace_bytes: bad argument");
  return carve(m, n_lines, nullptr).bytes + 256;
}

int64_t ltr_desc_tiles_bytes(int32_t n_lines) {
  if (n_lines < 0) return set_error(LTR_E_INVALID, "ltr_desc_tiles_bytes: bad argument");
  return align_up(n_lines, 128) * MT_D * 2 * 2;   // hi + lo plane, bf16
}

int ltr_encode(LtrModel* m, const LtrEncodeInput* in, const LtrEncodeOutput* out, void* workspace, int64_t workspace_bytes,
               void* stream) {
  if (!m || !in || !out) return set_error(LTR_E_INVALID, "ltr_encode: null argument");
  if (in->n_lines == 0 || in->n_images == 0) return LTR_OK;
  if (in->n_tokens < 1 || in->n_tokens > 128) return set_error(LTR_E_UNSUPPORTED, "ltr_encode: n_tokens must be in 1..128");
  if (!in->sublines || !in->resp || !in->angle || !in->pnt || !in->desc || !in->score)
    return set_error(LTR_E_INVALID, "ltr_encode: null input tensor");
  if ((in->cu_lines_host == nullptr) != (in->cu_lines_dev == nullptr))
    return set_error(LTR_E_INVALID, "ltr_encode: cu_lines_host and cu_lines_dev must be given together");
  if (!in->cu_lines_host && (int64_t)in->lines_per_image * in->n_images != in->n_lines)
    return set_error(LTR_E_INVALID, "ltr_encode: uniform batch needs n_lines == n_images * lines_per_image");
  if (in->cu_lines_host && (in->cu_lines_host[0] != 0 || in->cu_lines_host[in->n_images] != in->n_lines))
    return set_error(LTR_E_INVALID, "ltr_encode: cu_lines must start at 0 and end at n_lines");
  if (!(in->image_width > 0.f) || !(in->image_height > 0.f)) return set_error(LTR_E_INVALID, "ltr_encode: bad image shape");
  if (out->desc_tiles && (out->desc_cf || !out->desc_rows))
    return set_error(LTR_E_UNSUPPORTED, "ltr_encode: desc_tiles needs desc_rows and no desc_cf");
  if (out->desc_tiles && (reinterpret_cast<uintptr_t>(out->desc_tiles) & 15))
    return set_error(LTR_E_INVALID, "ltr_encode: desc_tiles must be 16-byte aligned");
  LTR_CUDA_TRY(cudaSetDevice(m->device));
  char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<int64_t>(workspace), 256));
  EncodeWs w = carve(m, in->n_lines, base);
  if (!workspace || (base - (char*)workspace) + w.bytes > workspace_bytes)
    return set_error(LTR_E_WORKSPACE, "ltr_encode: workspace too small, need " + std::to_string(w.bytes + 256));
  return encode_impl(m, *in, out->desc_cf, out->desc_rows, out->desc_tiles, w, as_stream(stream));
}

// ---- tensor-core matcher plumbing (d == 256) ----
struct MatchPlan {
  int mx[2], tmax[2], total[2];
  bool direct[2];       // side uses the caller's tile image (written by ltr_encode)
  ActImg img[2];
  uint2* slot[2];
  float* sq[2];
  int* done;
  int64_t bytes;
};

static MatchPlan plan_match(const LtrMatchInput& in, char* base) {
  MatchPlan pl{};
  const int P = in.n_pairs;
  const int n[2] = {in.n0, in.n1};
  const int mxn[2] = {in.max_n0, in.max_n1};
  const int tot[2] = {in.total_n0, in.total_n1};
  const void* tiles[2] = {in.tiles0, in.tiles1};
  const int tl[2] = {in.tiles_lines0, in.tiles_lines1};
  const int tr0[2] = {in.tiles_row0_0, in.tiles_row0_1};
  const bool varlen = in.cu0 != nullptr;
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* p = base + off;
    off = align_up(off + bytes, 1024);
    return p;
  };
  for (int s = 0; s < 2; ++s) {
    pl.mx[s] = varlen ? mxn[s] : n[s];
    pl.tmax[s] = cdiv(pl.mx[s], 128);
    pl.total[s] = varlen ? tot[s] : P * n[s];
    pl.direct[s] = tiles[s] && !varlen && in.dist_mode == 0 && n[s] % 128 == 0 && tr0[s] % 128 == 0 && tr0[s] >= 0 &&
                   (int64_t)tr0[s] + (int64_t)P * n[s] <= align_up(tl[s], 128);
    if (pl.direct[s]) {
      pl.img[s] = tiles_image(const_cast<void*>(tiles[s]), tl[s]);
    } else {
      const int64_t plane = (int64_t)P * pl.tmax[s] * 128 * MT_D;   // bf16 elements
      pl.img[s].hi = reinterpret_cast<__nv_bfloat16*>(take(plane * 2));
      pl.img[s].lo = reinterpret_cast<__nv_bfloat16*>(take(plane * 2));
      pl.img[s].kblocks = MT_KB;
    }
    pl.slot[s] = reinterpret_cast<uint2*>(take((int64_t)std::max(pl.total[s], 1) * 8));
    pl.sq[s] = in.dist_mode == 1 ? reinterpret_cast<float*>(take((int64_t)std::max(pl.total[s], 1) * 4)) : nullptr;
  }
  pl.done = reinterpret_cast<int*>(take(256));
  pl.bytes = off;
  return pl;
}

static const char* check_match_input(const LtrMatchInput* in) {
  if (in->d <= 0 || in->d % 16) return "ltr_match: descriptor dim must be a multiple of 16";
  const bool seg = in->sub_off0 != nullptr || in->sub_off1 != nullptr;
  if (seg && (!in->sub_off0 || !in->sub_off1 || !in->cuk0 || !in->cuk1 || !in->cu0 || !in->cu1))
    return "ltr_match: keyline merging needs sub_off0/1, cuk0/1 and cu0/1";
  if ((in->cu0 == nullptr) != (in->cu1 == nullptr)) return "ltr_match: cu0/cu1 must be given together";
  if (in->dist_mode != 0 && in->dist_mode != 1) return "ltr_match: dist_mode must be 0 or 1";
  if (in->dist_mode == 1 && (in->d != MT_D || seg)) return "ltr_match: dist_mode 1 needs d == 256 and no keyline merging";
  if (in->d == MT_D && in->cu0 && (in->total_n0 < 0 || in->total_n1 < 0)) return "ltr_match: total_n0/total_n1 required with cu0/cu1";
  return nullptr;
}

}  // extern "C"

// launch sequence of the tensor-core matcher; returns 0 or an error code
static int run_match_tc(const LtrMatchInput& in, const LtrMatchOutput& out, const MatchPlan& pl, bool seg, long long stride_key,
                        cudaStream_t s) {
  const int P = in.n_pairs;
  const bool want_nn = out.matches0 != nullptr && !seg;
  const bool both = want_nn && in.mutual;
  if (pl.mx[0] > 0 && pl.mx[1] > 0) {
    if (!pl.direct[0] || !pl.direct[1]) {
      DescTilesArgs da{};
      da.layout = in.layout;
      const float* d[2] = {in.desc0, in.desc1};
      const int* cu[2] = {in.cu0, in.cu1};
      const int n[2] = {in.n0, in.n1};
      int tm = 0;
      for (int sd = 0; sd < 2; ++sd) {
        da.d[sd] = d[sd]; da.cu[sd] = cu[sd]; da.n[sd] = n[sd]; da.img[sd] = pl.img[sd];
        da.tmax[sd] = pl.direct[sd] ? 0 : pl.tmax[sd];
        da.sq[sd] = pl.sq[sd];
        tm = std::max(tm, da.tmax[sd]);
      }
      LaunchScope ls(KC_DESC_TILES, s);
      LTR_CUDA_TRY(launch_pdl(desc_tiles_kernel, dim3(tm * 4, P, 2), dim3(256), 0, s, da));
    }
    MatchTcArgs ma{};
    const int* cu[2] = {in.cu0, in.cu1};
    const int n[2] = {in.n0, in.n1};
    const int tr0[2] = {in.tiles_row0_0, in.tiles_row0_1};
    for (int sd = 0; sd < 2; ++sd) {
      ma.s[sd].img = pl.img[sd]; ma.s[sd].cu = cu[sd]; ma.s[sd].n = n[sd];
      ma.s[sd].tile_mode = pl.direct[sd] ? 1 : 0; ma.s[sd].tile_row0 = pl.direct[sd] ? tr0[sd] : 0;
      ma.s[sd].tmax = pl.tmax[sd]; ma.s[sd].sq = pl.sq[sd]; ma.s[sd].slot = pl.slot[sd];
    }
    ma.dist_mode = in.dist_mode;
    ma.dist = seg ? out.dist_sub : out.dist_key;
    ma.dist_stride = seg ? (long long)pl.mx[0] * pl.mx[1] : stride_key;
    ma.counts = want_nn ? out.counts : nullptr;
    ma.done = want_nn ? pl.done : nullptr;
    ma.n_pairs = P;
    LTR_CUDA_TRY(ensure_dynamic_smem(match_tc_kernel, MT_SMEM));
    LaunchScope ls(KC_MATCH_TC, s);
    LTR_CUDA_TRY(launch_pdl(match_tc_kernel, dim3(pl.tmax[0] + (both ? pl.tmax[1] : 0), P), dim3(MT_THREADS), (size_t)MT_SMEM, s, ma));
  } else if (want_nn) {
    LTR_CUDA_TRY(cudaMemsetAsync(out.counts, 0, sizeof(int) * P, s));
    LTR_CUDA_TRY(cudaMemsetAsync(pl.done, 0, sizeof(int), s));
  }
  if (want_nn && pl.mx[0] > 0) {
    MatchTailArgs ta{};
    ta.d[0] = in.desc0; ta.d[1] = in.desc1; ta.layout = in.layout;
    ta.cu[0] = in.cu0; ta.cu[1] = in.cu1; ta.n[0] = in.n0; ta.n[1] = in.n1;
    ta.sq[0] = pl.sq[0]; ta.sq[1] = pl.sq[1]; ta.dist_mode = in.dist_mode;
    ta.slot[0] = pl.slot[0]; ta.slot[1] = pl.slot[1];
    ta.thr = in.nn_thresh; ta.mutual = in.mutual;
    ta.matches0 = out.matches0; ta.scores0 = out.scores0; ta.nn1 = out.nn1; ta.counts = out.counts;
    ta.max0 = pl.mx[0];
    ta.done = pl.done; ta.n_pairs = P; ta.world = 1;
    if (out.gather && out.gather->world > 1) {
      const LtrPeerGather& g = *out.gather;
      ta.mc_base = reinterpret_cast<int*>(g.mc_base);
      ta.peer_bases = reinterpret_cast<int* const*>(g.peer_bases);
      ta.rank = g.rank; ta.world = g.world; ta.gslot = g.slot; ta.epoch = g.epoch;
    }
    LaunchScope ls(KC_MATCH_TAIL, s);
    LTR_CUDA_TRY(launch_pdl(match_tail_kernel, dim3(cdiv(pl.mx[0] + (in.mutual ? pl.mx[1] : 0), 256), P), dim3(256), 0, s, ta));
  }
  return 0;
}

extern "C" {

int64_t ltr_match_workspace_bytes(const LtrMatchInput* in) {
  if (!in) return set_error(LTR_E_INVALID, "ltr_match_workspace_bytes: null argument");
  if (const char* e = check_match_input(in)) return set_error(LTR_E_INVALID, e);
  if (in->n_pairs <= 0 || in->d != MT_D) return 0;
  return plan_match(*in, nullptr).bytes + 1024;
}

int ltr_match(const LtrMatchInput* in, const LtrMatchOutput* out, int32_t device, void* stream) {
  if (!in || !out) return set_error(LTR_E_INVALID, "ltr_match: null argument");
  if (in->n_pairs <= 0) return LTR_OK;
  if (const char* e = check_match_input(in)) return set_error(in->d % 16 ? LTR_E_UNSUPPORTED : LTR_E_INVALID, e);
  const bool seg = in->sub_off0 != nullptr;
  const bool tc = in->d == MT_D;
  const bool want_nn = out->matches0 != nullptr;
  if (want_nn && (!out->scores0 || !out->nn1 || !out->counts))
    return set_error(LTR_E_INVALID, "ltr_match: matches0 needs scores0, nn1 and counts");
  if (!want_nn && !out->dist_key) return set_error(LTR_E_INVALID, "ltr_match: nothing to compute (matches0 and dist_key are NULL)");
  if (seg && (!out->dist_sub || !out->dist_key)) return set_error(LTR_E_INVALID, "ltr_match: keyline merging needs dist_sub and dist_key");
  if (out->gather && out->gather->world > 1) {
    const LtrPeerGather& g = *out->gather;
    if (seg || !tc || !want_nn) return set_error(LTR_E_UNSUPPORTED, "ltr_match: gather needs d == 256, no keyline merging, matches0");
    if ((!g.mc_base && !g.peer_bases) || g.rank < 0 || g.rank >= g.world || g.slot < 0 || g.slot >= LTR_GATHER_SLOTS || g.epoch <= 0)
      return set_error(LTR_E_INVALID, "ltr_match: bad LtrPeerGather");
    if ((in->cu0 ? in->max_n0 : in->n0) <= 0) return set_error(LTR_E_UNSUPPORTED, "ltr_match: gather needs a non-empty side 0");
  }
  if (!tc && !out->dist_key) return set_error(LTR_E_INVALID, "ltr_match: dist_key is required when d != 256");
  LTR_CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = as_stream(stream);
  const int mx0 = in->cu0 ? in->max_n0 : in->n0, mx1 = in->cu1 ? in->max_n1 : in->n1;
  const int mk0 = seg ? in->max_k0 : mx0, mk1 = seg ? in->max_k1 : mx1;
  const long long stride_key = in->dist_pair_stride > 0 ? in->dist_pair_stride : (long long)mk0 * mk1;
  if (mx0 > 0 && mx1 > 0 && (!in->desc0 || !in->desc1)) return set_error(LTR_E_INVALID, "ltr_match: null descriptors");
  if (tc) {
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<int64_t>(out->workspace), 1024));
    MatchPlan pl = plan_match(*in, base);
    if (pl.bytes > 0 && (!out->workspace || (base - (char*)out->workspace) + pl.bytes > out->workspace_bytes))
      return set_error(LTR_E_WORKSPACE, "ltr_match: workspace too small, need " + std::to_string(pl.bytes + 1024));
    LTR_TRY(run_match_tc(*in, *out, pl, seg, stride_key, s));
    if (!seg) return LTR_OK;
  } else if (mx0 > 0 && mx1 > 0) {
    // generic descriptor dimension: fp32 FMA distance tiles
    DistArgs da{};
    da.d0 = in->desc0; da.d1 = in->desc1; da.layout = in->layout; da.d = in->d;
    da.cu0 = in->cu0; da.cu1 = in->cu1; da.n0 = in->n0; da.n1 = in->n1;
    da.out = seg ? out->dist_sub : out->dist_key;
    da.stride = seg ? (long long)mx0 * mx1 : stride_key;
    dim3 grid(cdiv(mx0, DK_BM), cdiv(mx1, DK_BN), in->n_pairs);
    LaunchScope ls(KC_DIST, s);
    if (in->layout == LTR_LAYOUT_CHANNEL_FIRST) LTR_CUDA_TRY(launch_pdl(dist_kernel<true>, grid, dim3(DK_THREADS), 0, s, da));
    else LTR_CUDA_TRY(launch_pdl(dist_kernel<false>, grid, dim3(DK_THREADS), 0, s, da));
  }
  if (seg && mx0 > 0 && mx1 > 0 && mk0 > 0 && mk1 > 0) {
    SegMeanArgs sa{out->dist_sub, (long long)mx0 * mx1, out->dist_key, stride_key, in->cuk0, in->cuk1, in->sub_off0, in->sub_off1};
    LaunchScope ls(KC_SEGMEAN, s);
    segmean_kernel<<<dim3(cdiv(mk1, 32), cdiv(mk0, 8), in->n_pairs), 256, 0, s>>>(sa);
    LTR_CUDA_TRY(cudaGetLastError());
  }
  if (!want_nn) return LTR_OK;
  NNArgs na{};
  na.dist = out->dist_key; na.stride = stride_key;
  na.cuk0 = seg ? in->cuk0 : in->cu0; na.cuk1 = seg ? in->cuk1 : in->cu1;
  na.n0 = in->n0; na.n1 = in->n1; na.thr = in->nn_thresh; na.mutual = in->mutual;
  na.matches0 = out->matches0; na.scores0 = out->scores0; na.nn1 = out->nn1; na.counts = out->counts;
  return run_nn(na, in->n_pairs, mk0, mk1, s);
}

int ltr_gather_wait(const void* local_base, int32_t world, int32_t n_pairs, int32_t slot, int32_t epoch, int32_t* out,
                    int32_t device, void* stream) {
  if (!local_base || !out || world < 1 || world > 256 || n_pairs < 1 || slot < 0 || slot >= LTR_GATHER_SLOTS)
    return set_error(LTR_E_INVALID, "ltr_gather_wait: bad argument");
  LTR_CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = as_stream(stream);
  LaunchScope ls(KC_MUTUAL, s);
  LTR_CUDA_TRY(launch_pdl(gather_wait_kernel, dim3(1), dim3(256), 0, s, reinterpret_cast<const int*>(local_base), world, n_pairs, slot,
                          epoch, out));
  return LTR_OK;
}

int ltr_match_distmat(const float* dist, int32_t n_pairs, int32_t n0, int32_t n1, int64_t dist_pair_stride, float nn_thresh,
                      int32_t mutual, int32_t* matches0, float* scores0, int32_t* nn1, int32_t* counts, int32_t device,
                      void* stream) {
  if (n_pairs <= 0) return LTR_OK;
  if (!matches0 || !scores0 || !nn1 || !counts) return set_error(LTR_E_INVALID, "ltr_match_distmat: null output");
  if (n0 > 0 && n1 > 0 && !dist) return set_error(LTR_E_INVALID, "ltr_match_distmat: null distance matrix");
  LTR_CUDA_TRY(cudaSetDevice(device));
  NNArgs na{};
  na.dist = dist; na.stride = dist_pair_stride > 0 ? dist_pair_stride : (long long)n0 * n1;
  na.n0 = n0; na.n1 = n1; na.thr = nn_thresh; na.mutual = mutual;
  na.matches0 = matches0; na.scores0 = scores0; na.nn1 = nn1; na.counts = counts;
  return run_nn(na, n_pairs, n0, n1, as_stream(stream));
}

int ltr_merge_sublines(const float* dist_sub, int64_t stride_sub, int32_t n_pairs, const int32_t* cuk0,
                       const int32_t* cuk1, const int32_t* sub_off0, const int32_t* sub_off1, int32_t max_k0,
                       int32_t max_k1, float* dist_key, int64_t stride_key, int32_t device, void* stream) {
  if (n_pairs <= 0 || max_k0 <= 0 || max_k1 <= 0) return LTR_OK;
  if (!dist_sub || !cuk0 || !cuk1 || !sub_off0 || !sub_off1 || !dist_key)
    return set_error(LTR_E_INVALID, "ltr_merge_sublines: null argument");
  LTR_CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = as_stream(stream);
  SegMeanArgs sa{dist_sub, stride_sub, dist_key, stride_key, cuk0, cuk1, sub_off0, sub_off1};
  LaunchScope ls(KC_SEGMEAN, s);
  segmean_kernel<<<dim3(cdiv(max_k1, 32), cdiv(max_k0, 8), n_pairs), 256, 0, s>>>(sa);
  LTR_CUDA_TRY(cudaGetLastError());
  return LTR_OK;
}

int ltr_tokenize(const LtrTokenizeInput* in, float* sublines, float* pnt, float* mask, float* resp, float* angle,
                 float* desc, float* score, int32_t device, void* stream) {
  if (!in || !sublines || !pnt || !mask || !resp || !angle || !desc || !score)
    return set_error(LTR_E_INVALID, "ltr_tokenize: null argument");
  if (in->n_sublines <= 0 || in->n_keylines <= 0) return LTR_OK;
  if (in->n_tokens < 1 || in->desc_channels != 256)
    return set_error(LTR_E_UNSUPPORTED, "ltr_tokenize: n_tokens >= 1 and 256 descriptor channels required");
  if (!in->sp || !in->ep || !in->ep_clipped || !in->length || !in->angle || !in->n_tok || !in->sub0 || !in->sub2line ||
      !in->dense_desc || !in->dense_score)
    return set_error(LTR_E_INVALID, "ltr_tokenize: null input array");
  LTR_CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = as_stream(stream);
  TokLines L{in->sp, in->ep, in->ep_clipped, in->length, in->angle, in->n_tok, in->sub0, in->sub2line,
             in->n_keylines, in->n_sublines, in->n_tokens, in->token_distance};
  const long long n_tok = (long long)in->n_sublines * in->n_tokens;
  {
    LaunchScope ls(KC_TOKENIZE, s);
    tok_points_kernel<<<cdiv(n_tok, 256), 256, 0, s>>>(L, pnt, mask, sublines, resp, angle);
    LTR_CUDA_TRY(cudaGetLastError());
  }
  {
    LaunchScope ls(KC_TOKENIZE, s);
    tok_sample_kernel<<<cdiv(n_tok, 8), 256, 0, s>>>(pnt, (int)n_tok, in->dense_desc, in->desc_h, in->desc_w, in->dense_score,
                                                      in->score_h, in->score_w, in->align_corners, desc, score);
    LTR_CUDA_TRY(cudaGetLastError());
  }
  return LTR_OK;
}

int ltr_linear(const float* x, int32_t ldx, const float* w, const float* bias, const float* res, int32_t ldr, float* y,
               int32_t ldy, int32_t m, int32_t n, int32_t k, int32_t act, int32_t device, void* stream) {
  if (!x || !w || !y) return set_error(LTR_E_INVALID, "ltr_linear: null argument");
  LTR_CUDA_TRY(cudaSetDevice(device));
  return launch_linear_f32(lin(x, ldx, w, bias, y, ldy, m, n, k, act, res, ldr), as_stream(stream));
}

struct NormSpec { int norm; float eps; const float* g; const float* beta; const float* add; int ldadd; };

static int linear_img_impl(const float* x, int32_t ldx, const float* w_host, const float* bias, const float* res, int32_t ldr,
                           float* y, int32_t ldy, float* y_from_image, int32_t m, int32_t n, int32_t k, int32_t act,
                           int32_t bn_hint, int32_t device, void* stream, const NormSpec& ns) {
  if (!x || !w_host || (!y && !y_from_image)) return set_error(LTR_E_INVALID, "ltr_linear_img: null argument");
  if (n % 64 || k % 64) return set_error(LTR_E_UNSUPPORTED, "ltr_linear_img: n and k must be multiples of 64");
  LTR_CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = as_stream(stream);
  std::vector<double> W((size_t)n * k);
  for (size_t i = 0; i < W.size(); ++i) W[i] = w_host[i];
  std::vector<uint16_t> img(2 * (size_t)n * k);
  pack_tc_weight(W.data(), n, k, img.data(), img.data() + (size_t)n * k);
  const size_t mpad = (size_t)cdiv(m, 256) * 256;
  uint16_t *dw = nullptr, *da = nullptr, *dout = nullptr;
  cudaError_t ce = cudaMalloc(&dw, img.size() * 2);
  if (ce == cudaSuccess) ce = cudaMalloc(&da, 2 * mpad * k * 2);
  if (ce == cudaSuccess) ce = cudaMalloc(&dout, 2 * mpad * n * 2);
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(dw, img.data(), img.size() * 2, cudaMemcpyHostToDevice, s);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(da, 0, 2 * mpad * k * 2, s);
  int rc = 0;
  if (ce == cudaSuccess) {
    ActImg A{reinterpret_cast<__nv_bfloat16*>(da), reinterpret_cast<__nv_bfloat16*>(da + mpad * k), k / 64};
    ActImg O{reinterpret_cast<__nv_bfloat16*>(dout), reinterpret_cast<__nv_bfloat16*>(dout + mpad * n), n / 64};
    {
      LaunchScope ls(KC_IMG_CONVERT, s);
      to_image_kernel<<<cdiv((long long)m * (k / 8), 256), 256, 0, s>>>(x, ldx, m, k, A, 0);
    }
    GemmImgArgs a{};
    a.A = A; a.a_kb0 = 0; a.bias = bias; a.R = res; a.ldr = ldr; a.C = y; a.ldc = ldy; a.M = m; a.act = act;
    a.W.hi = reinterpret_cast<const __nv_bfloat16*>(dw);
    a.W.lo = reinterpret_cast<const __nv_bfloat16*>(dw + (size_t)n * k);
    a.W.N = n; a.W.K = k;
    if (y_from_image) { a.O = O; a.o_kb0 = 0; }
    a.norm = ns.norm; a.eps = ns.eps; a.ng = ns.g; a.nbeta = ns.beta; a.nadd = ns.add; a.ldadd = ns.ldadd;
    rc = launch_gemm_img(a, s, bn_hint);
    if (rc == 0 && y_from_image) {
      LaunchScope ls(KC_IMG_CONVERT, s);
      from_image_kernel<<<cdiv((long long)m * n, 256), 256, 0, s>>>(O, 0, y_from_image, n, m, n);
    }
    ce = cudaStreamSynchronize(s);
  }
  cudaFree(dw); cudaFree(da); cudaFree(dout);
  if (rc != 0) return rc;
  if (ce != cudaSuccess) return set_error(LTR_E_CUDA, std::string("ltr_linear_img: ") + cudaGetErrorString(ce));
  return LTR_OK;
}

int ltr_linear_img(const float* x, int32_t ldx, const float* w_host, const float* bias, const float* res, int32_t ldr,
                   float* y, int32_t ldy, float* y_from_image, int32_t m, int32_t n, int32_t k, int32_t act,
                   int32_t bn_hint, int32_t device, void* stream) {
  return linear_img_impl(x, ldx, w_host, bias, res, ldr, y, ldy, y_from_image, m, n, k, act, bn_hint, device, stream,
                         NormSpec{NORM_NONE, 0.f, nullptr, nullptr, nullptr, 0});
}

int ltr_linear_img_norm(const float* x, int32_t ldx, const float* w_host, const float* bias, const float* res, int32_t ldr,
                        int32_t norm, float eps, const float* gamma, const float* beta, const float* add, int32_t ldadd,
                        float* y, int32_t ldy, float* y_from_image, int32_t m, int32_t k, int32_t device, void* stream) {
  if (norm != NORM_LAYER && norm != NORM_L2) return set_error(LTR_E_INVALID, "ltr_linear_img_norm: norm must be 1 (LayerNorm) or 2 (L2)");
  if (norm == NORM_LAYER && (!gamma || !beta)) return set_error(LTR_E_INVALID, "ltr_linear_img_norm: LayerNorm needs gamma and beta");
  return linear_img_impl(x, ldx, w_host, bias, res, ldr, y, ldy, y_from_image, m, 256, k, ACT_NONE, 256, device, stream,
                         NormSpec{norm, eps, gamma, beta, add, ldadd});
}

// Micro-benchmark of the image GEMM engine: average device ms per launch of an [m,k]x[n,k]^T
// problem with zero-filled operands (timing only).  out_mode: 0 fp32 rows, 1 image, 2 both.
// debug: arm / read the clock64 stamps kernels of CTA 0 leave in g_dbg_trace (see LTR_DBG_STAMP)
void ltr_debug_trace_arm(int32_t on) {
  int v = on;
  dbg_chain_sel() = -1;
  if (on >= 100) {   // trace only chained-GEMM launch number (on - 100) from now on
    dbg_chain_sel() = on - 100;
    dbg_chain_cnt() = 0;
    v = 0;
  }
  cudaMemcpyToSymbol(g_dbg_on, &v, sizeof(int));
  if (on) {
    static unsigned long long zeros[128] = {0};
    cudaMemcpyToSymbol(g_dbg_trace, zeros, sizeof(zeros));
  }
}
int ltr_debug_trace_read(unsigned long long* out128) {
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out128, g_dbg_trace, 128 * sizeof(unsigned long long)) == cudaSuccess ? 0 : -2;
}

static unsigned long long g_trace_host[64];
const unsigned long long* ltr_gemm_trace(void) { return g_trace_host; }

float ltr_gemm_bench(int32_t m, int32_t n, int32_t k, int32_t bn_hint, int32_t out_mode, int32_t iters, int32_t device) {
  if (cudaSetDevice(device) != cudaSuccess) return -1.f;
  const size_t mpad = (size_t)cdiv(m, 256) * 256;
  uint16_t *dw = nullptr, *da = nullptr, *dout = nullptr;
  float* dc = nullptr;
  cudaMalloc(&dw, 2 * (size_t)n * k * 2);
  cudaMalloc(&da, 2 * mpad * k * 2);
  cudaMalloc(&dout, 2 * mpad * n * 2);
  cudaMalloc(&dc, mpad * n * 4);
  cudaMemset(dw, 0, 2 * (size_t)n * k * 2);
  cudaMemset(da, 0, 2 * mpad * k * 2);
  GemmImgArgs a{};
  a.A = ActImg{reinterpret_cast<__nv_bfloat16*>(da), reinterpret_cast<__nv_bfloat16*>(da + mpad * k), k / 64};
  a.W.hi = reinterpret_cast<const __nv_bfloat16*>(dw);
  a.W.lo = reinterpret_cast<const __nv_bfloat16*>(dw + (size_t)n * k);
  a.W.N = n; a.W.K = k; a.M = m; a.act = 1;
  if (out_mode == 0 || out_mode == 2) { a.C = dc; a.ldc = n; }
  if (out_mode == 1 || out_mode == 2) a.O = ActImg{reinterpret_cast<__nv_bfloat16*>(dout), reinterpret_cast<__nv_bfloat16*>(dout + mpad * n), n / 64};
  unsigned long long* dtrace = nullptr;
  cudaMalloc(&dtrace, 64 * 8);
  cudaMemset(dtrace, 0, 64 * 8);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int i = 0; i < 3; ++i) launch_gemm_img(a, 0, bn_hint);
  a.trace = dtrace;
  launch_gemm_img(a, 0, bn_hint);
  a.trace = nullptr;
  cudaMemcpy(g_trace_host, dtrace, 64 * 8, cudaMemcpyDeviceToHost);
  cudaFree(dtrace);
  cudaEventRecord(e0, 0);
  for (int i = 0; i < iters; ++i) launch_gemm_img(a, 0, bn_hint);
  cudaEventRecord(e1, 0);
  cudaEventSynchronize(e1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(dw); cudaFree(da); cudaFree(dout); cudaFree(dc);
  return cudaGetLastError() == cudaSuccess ? ms / iters : -1.f;
}

}  // extern "C"
