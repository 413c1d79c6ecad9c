// weights_device.cu — spb_load_weights_device / spb_chess_load_weights_device: the network from a learner's device tensors.
//
// The table is resolved by the resolver of the safetensors path (weights.cu), so names, census and shapes are checked the
// same way and give the same messages.  Then, on the engine's stream:
//   k_fold_bn  one thread per output channel of a conv: the BatchNorm scale s = g / sqrt(var + eps) and folded bias
//              (b - mean) s + beta in f64, rounded like the host fold (this file is built with --fmad=false, and the
//              intrinsics fix every rounding anyway)
//   k_pack     the weight image in gather form: one thread per 4-byte word of the image works out which source element
//              (if any) lands there, so every byte is written exactly once and every pad is zero.  Weights are
//              (float)((double)w * s) rounded to bf16 by f2bf, as Evaluator::upload / umma::pack_weights / net_upload do.
// The source pointers travel in the kernels' parameters (Sources), the per-channel scales in the engine's stage: a load
// allocates nothing once the engine holds an image.
#include <string>
#include <vector>

#include "bf16.cuh"
#include "chess_engine.hpp"
#include "chess_net.cuh"
#include "engine.hpp"
#include "evaluator_umma.cuh"
#include "weights.cuh"

namespace spb {
namespace {

constexpr int FOLD_STRIDE = 256;   // per-conv stride of the fold scratch (the widest conv)
constexpr int MAX_SEGS = 48;

struct Sources {
  const void* p[CH_ROLES];
  int32_t dtype[CH_ROLES];         // SPB_DTYPE_F32 / BF16 / F64
};

// element i of a role's tensor as f32, converted as load_f32 (weights.cu) converts it
__device__ __forceinline__ float src_f32(const Sources& S, int role, size_t i) {
  const void* p = S.p[role];
  switch (S.dtype[role]) {
    case SPB_DTYPE_BF16: return __uint_as_float((uint32_t)static_cast<const uint16_t*>(p)[i] << 16);
    case SPB_DTYPE_F64: return __double2float_rn(static_cast<const double*>(p)[i]);
    default: return static_cast<const float*>(p)[i];
  }
}

struct FoldArgs {
  int convs;
  int oc[21];
  float eps;
};

__global__ void __launch_bounds__(256) k_fold_bn(const __grid_constant__ Sources S, const __grid_constant__ FoldArgs F, double* scale,
                                                 float* bias) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x, c = idx / FOLD_STRIDE, o = idx % FOLD_STRIDE;
  if (c >= F.convs || o >= F.oc[c]) return;
  const double g = src_f32(S, 6 * c + ROLE_G, o), var = src_f32(S, 6 * c + ROLE_VAR, o);
  const double b = src_f32(S, 6 * c + ROLE_B, o), mean = src_f32(S, 6 * c + ROLE_MEAN, o), beta = src_f32(S, 6 * c + ROLE_BETA, o);
  const double s = __ddiv_rn(g, __dsqrt_rn(__dadd_rn(var, (double)F.eps)));
  scale[idx] = s;
  bias[idx] = __double2float_rn(__dadd_rn(__dmul_rn(__dsub_rn(b, mean), s), beta));
}

// What a segment of the image holds.  bf16 kinds produce two elements per word, f32 kinds one; past a segment's real
// elements the words are zero (the alignment gaps).
enum SegKind : int32_t {
  SEG_SIMT_W,       // bf16 folded conv weights [oc][ic*9] (conv)
  SEG_BIAS,         // f32 folded biases [oc] (conv)
  SEG_RAW,          // f32 copy of `count` elements of a role
  SEG_UMMA_STEM,    // bf16: per tap [2 chunks][64 n][8 k] of conv 0
  SEG_UMMA_LAYER,   // bf16: per kernel row [KC chunks][3N (centre | right | left)][8 k] of layer `conv` (9: the fused head)
  SEG_UMMA_BIAS,    // f32 [10][64]: layer biases, the head's policy then value channels
  SEG_UMMA_WP,      // f32 [A][P][32]: the policy Linear, channel innermost
  SEG_UMMA_WV,      // f32 [P][8]: the value Linear, channels 3..7 zero
  SEG_UMMA_FCB,     // f32 [32]: policy biases at 0..A-1, the value bias at 16
  SEG_CHESS_CONV,   // bf16 stages [kc32][tap][4 chunks][N][8] of pack_conv (chess_net.cu); `conv` < 0: an unfolded 1x1 conv
  SEG_CHESS_F1W,    // f32 fc1 transposed to [64][256]
};

struct Seg {
  uint32_t begin, end;             // 4-byte words of the image
  int32_t kind, conv, role, oc, ic, count;
  int32_t n, kc, taps, halves;     // UMMA layer: n = N, kc = K chunks; chess conv: n = N, kc = kc32, taps, halves
};

struct Segs {
  Seg s[MAX_SEGS];
  int32_t P, A;                    // Connect4 / tic-tac-toe geometry
};

__device__ __forceinline__ uint16_t folded(const Sources& S, const double* scale, int conv, int o, size_t widx) {
  return f2bf(__double2float_rn(__dmul_rn((double)src_f32(S, 6 * conv + ROLE_W, widx), scale[conv * FOLD_STRIDE + o])));
}

__device__ uint16_t bf16_at(const Sources& S, const Seg& g, const double* scale, uint32_t e) {
  switch (g.kind) {
    case SEG_SIMT_W: {
      const uint32_t K = (uint32_t)g.ic * 9;
      return e < (uint32_t)g.oc * K ? folded(S, scale, g.conv, (int)(e / K), e) : 0;
    }
    case SEG_UMMA_STEM: {
      const uint32_t tap = e / 1024, j = e % 1024, k = (j / 512) * 8 + j % 8, n = (j / 8) % 64;
      return (int)k < g.ic ? folded(S, scale, 0, (int)n, ((size_t)n * g.ic + k) * 9 + tap) : 0;
    }
    case SEG_UMMA_LAYER: {
      const uint32_t N = (uint32_t)g.n, block = 3u * g.kc * N * 8;
      const uint32_t ky = e / block, j = e % block, q = j / 8, m = q % (3 * N), k = (q / (3 * N)) * 8 + j % 8;
      const uint32_t part = m / N, n = m % N, kx = part == 0 ? 1 : (part == 1 ? 2 : 0);
      const bool head = g.conv == 9;
      if (n >= (head ? 35u : 64u)) return 0;
      const int conv = head ? (n < 32 ? 9 : 10) : g.conv, oc = head && n >= 32 ? (int)n - 32 : (int)n;
      return folded(S, scale, conv, oc, ((size_t)oc * 64 + k) * 9 + ky * 3 + kx);
    }
    default: {  // SEG_CHESS_CONV
      const uint32_t N = (uint32_t)g.n, NH = g.halves ? N / 2 : N, st = e / (32 * N), j = e % (32 * N);
      const uint32_t kc = st / g.taps, tap = st % g.taps, h = j / (32 * NH), r = j % (32 * NH), q = r / 8;
      const uint32_t n = h * NH + q % NH, k = kc * 32 + (q / NH) * 8 + r % 8;
      if ((int)n >= g.oc || (int)k >= g.ic) return 0;
      const size_t widx = ((size_t)n * g.ic + k) * g.taps + tap;
      return g.conv >= 0 ? folded(S, scale, g.conv, (int)n, widx) : f2bf(src_f32(S, g.role, widx));
    }
  }
}

__device__ float f32_at(const Sources& S, const Seg& g, const Segs& G, const float* bias, uint32_t j) {
  switch (g.kind) {
    case SEG_BIAS: return (int)j < g.oc ? bias[g.conv * FOLD_STRIDE + j] : 0.0f;
    case SEG_RAW: return (int)j < g.count ? src_f32(S, g.role, j) : 0.0f;
    case SEG_UMMA_BIAS: {
      const uint32_t l = j / 64, n = j % 64;
      if (l < 9) return bias[l * FOLD_STRIDE + n];
      return n < 32 ? bias[9 * FOLD_STRIDE + n] : (n < 35 ? bias[10 * FOLD_STRIDE + n - 32] : 0.0f);
    }
    case SEG_UMMA_WP: {
      const uint32_t P = (uint32_t)G.P, ch = j % 32, pos = (j / 32) % P, a = j / (32 * P);
      return src_f32(S, NET_ROLE_PFC_W, (size_t)a * 32 * P + ch * P + pos);
    }
    case SEG_UMMA_WV: {
      const uint32_t pos = j / 8, ch = j % 8;
      return ch < 3 ? src_f32(S, NET_ROLE_VFC_W, (size_t)ch * G.P + pos) : 0.0f;
    }
    case SEG_UMMA_FCB: return (int)j < G.A ? src_f32(S, NET_ROLE_PFC_B, j) : (j == 16 ? src_f32(S, NET_ROLE_VFC_B, 0) : 0.0f);
    default: return src_f32(S, CH_ROLE_F1_W, (size_t)(j % 256) * 64 + j / 256);   // SEG_CHESS_F1W
  }
}

// grid.y: one segment each; grid.x blocks stride over the segment's words
__global__ void __launch_bounds__(256) k_pack(const __grid_constant__ Sources S, const __grid_constant__ Segs G, const double* scale,
                                              const float* bias, uint32_t* image) {
  const Seg& g = G.s[blockIdx.y];
  const bool bf16 = g.kind == SEG_SIMT_W || g.kind == SEG_UMMA_STEM || g.kind == SEG_UMMA_LAYER || g.kind == SEG_CHESS_CONV;
  for (uint32_t w = g.begin + blockIdx.x * blockDim.x + threadIdx.x; w < g.end; w += gridDim.x * blockDim.x) {
    const uint32_t j = w - g.begin;
    image[w] = bf16 ? (uint32_t)bf16_at(S, g, scale, 2 * j) | (uint32_t)bf16_at(S, g, scale, 2 * j + 1) << 16
                    : __float_as_uint(f32_at(S, g, G, bias, j));
  }
}

// Segment list builder: segments are appended in image order and must tile it.
struct SegList {
  Segs segs{};
  int n = 0;
  uint32_t max_words = 0;
  Seg& add(size_t begin_bytes, size_t end_bytes, int kind) {
    Seg& g = segs.s[n++];
    g = Seg{};
    g.begin = (uint32_t)(begin_bytes / 4);
    g.end = (uint32_t)(end_bytes / 4);
    g.kind = kind;
    g.conv = -1;
    max_words = std::max(max_words, g.end - g.begin);
    return g;
  }
};

cudaError_t launch_pack(const Sources& S, const SegList& L, const double* scale, const float* bias, void* image, cudaStream_t stream) {
  const uint32_t gx = std::min<uint32_t>(1024u, (L.max_words + 1023u) / 1024u);
  k_pack<<<dim3(std::max(gx, 1u), (unsigned)L.n), 256, 0, stream>>>(S, L.segs, scale, bias, static_cast<uint32_t*>(image));
  return cudaGetLastError();
}

const char* dtype_name(int32_t d) {
  switch (d) {
    case SPB_DTYPE_F32: return "F32";
    case SPB_DTYPE_BF16: return "BF16";
    case SPB_DTYPE_F64: return "F64";
    case SPB_DTYPE_F16: return "F16";
    default: return nullptr;
  }
}

// The table as the resolver's entries, then the resolver with the per-tensor checks of the blob path.  SPB_ERR_ARG for a
// malformed table, SPB_ERR_WEIGHTS for what a blob with these tensors would be refused for.
template <class Eng, class Resolve>
int32_t resolve_table(Eng* e, const char* api, const spb_tensor* t, uint32_t n, size_t* re, Resolve resolve) {
  SPB_ARG(e, t, std::string(api) + ": null tensor table");
  std::vector<WeightEntry> entries(n);
  for (uint32_t i = 0; i < n; ++i) {
    SPB_ARG(e, t[i].name, std::string(api) + ": tensor " + std::to_string(i) + " has a null name");
    WeightEntry& w = entries[i];
    w.name = t[i].name;
    SPB_ARG(e, t[i].ndim >= 0 && t[i].ndim <= 4, std::string(api) + ": " + w.name + ": ndim " + std::to_string(t[i].ndim) + " outside 0..4");
    const char* dn = dtype_name(t[i].dtype);
    w.dtype = dn ? dn : "code " + std::to_string(t[i].dtype);
    w.shape.assign(t[i].shape, t[i].shape + t[i].ndim);
  }
  std::string err;
  const TakeRole check = [&](int, size_t i, std::string* er) { size_t count = 0; return element_size(entries[i], &count, er) != 0; };
  if (!resolve(entries, re, check, &err)) { e->set_error(std::string(api) + ": " + err); return SPB_ERR_WEIGHTS; }
  return SPB_OK;
}

// Every role's pointer: non-null, device memory of the engine's GPU (or managed), aligned to its element size.
template <class Eng>
int32_t gather_sources(Eng* e, const spb_tensor* t, const size_t* re, int roles, Sources* S) {
  *S = Sources{};
  for (int r = 0; r < roles; ++r) {
    const spb_tensor& x = t[re[r]];
    SPB_ARG(e, x.data, std::string(x.name) + " has a null data pointer");
    const size_t esz = x.dtype == SPB_DTYPE_F64 ? 8 : (x.dtype == SPB_DTYPE_BF16 ? 2 : 4);
    if (int32_t rc = e->check_device_pointers({{x.data, x.name, esz}})) return rc;
    S->p[r] = x.data;
    S->dtype[r] = x.dtype;
  }
  return SPB_OK;
}

}  // namespace
}  // namespace spb

using namespace spb;

extern "C" {

int32_t spb_load_weights_device(spb_engine* e, const spb_tensor* tensors, uint32_t n) {
  SPB_GUARD(e);
  const int game = e->cfg.game;
  size_t re[NET_ROLES];
  if (int32_t rc = resolve_table(e, "spb_load_weights_device", tensors, n, re, [game](const std::vector<WeightEntry>& t, size_t* r, const TakeRole& k, std::string* er) {
        return resolve_net(t, game, r, k, er);
      }))
    return rc;
  Sources S;
  if (int32_t rc = gather_sources(e, tensors, re, NET_ROLES, &S)) return rc;
  const size_t scale_bytes = (size_t)NET_CONVS * FOLD_STRIDE * 8;
  if (int32_t rc = e->ensure_stage(scale_bytes + (size_t)NET_CONVS * FOLD_STRIDE * 4, 0)) return rc;
  std::string err;
  uint8_t* img = e->evaluator.image_for(game, &err);
  if (!img) { e->set_error("spb_load_weights_device: " + err); return SPB_ERR_NOMEM; }

  const int P = game == SPB_GAME_CONNECT4 ? 42 : 9, A = game == SPB_GAME_CONNECT4 ? 7 : 9;
  const Evaluator::Layout L = Evaluator::layout(game);
  const umma::ImageLayout U = umma::image_layout(game);
  SegList segs;
  segs.segs.P = P;
  segs.segs.A = A;
  for (int i = 0; i < NET_CONVS; ++i) {
    const int oc = i <= 8 ? NET_HIDDEN : (i == 9 ? NET_POLICY_CH : NET_VALUE_CH), ic = i == 0 ? 3 : NET_HIDDEN;
    Seg& w = segs.add(L.wsimt[i], L.bias[i], SEG_SIMT_W);
    w.conv = i; w.oc = oc; w.ic = ic;
    Seg& b = segs.add(L.bias[i], i + 1 < NET_CONVS ? L.wsimt[i + 1] : L.pw, SEG_BIAS);
    b.conv = i; b.oc = oc;
  }
  const struct { size_t begin, end; int role, count; } raw[4] = {{L.pw, L.pb, NET_ROLE_PFC_W, A * NET_POLICY_CH * P}, {L.pb, L.vw, NET_ROLE_PFC_B, A},
                                                                {L.vw, L.vb, NET_ROLE_VFC_W, NET_VALUE_CH * P}, {L.vb, L.umma, NET_ROLE_VFC_B, 1}};
  for (const auto& r : raw) {
    Seg& g = segs.add(r.begin, r.end, SEG_RAW);
    g.role = r.role; g.count = r.count;
  }
  segs.add(L.umma, L.umma + U.layer_offset[1], SEG_UMMA_STEM).ic = 3;
  for (int l = 1; l < 10; ++l) {
    Seg& g = segs.add(L.umma + U.layer_offset[l], L.umma + (l + 1 < 10 ? U.layer_offset[l + 1] : U.off_bias), SEG_UMMA_LAYER);
    g.conv = l; g.n = U.layer_n[l]; g.kc = U.layer_kchunks[l];
  }
  segs.add(L.umma + U.off_bias, L.umma + U.off_wp, SEG_UMMA_BIAS);
  segs.add(L.umma + U.off_wp, L.umma + U.off_wv, SEG_UMMA_WP);
  segs.add(L.umma + U.off_wv, L.umma + U.off_fcb, SEG_UMMA_WV);
  segs.add(L.umma + U.off_fcb, L.umma + U.bytes, SEG_UMMA_FCB);

  FoldArgs F{};
  F.convs = NET_CONVS;
  for (int i = 0; i < NET_CONVS; ++i) F.oc[i] = i <= 8 ? NET_HIDDEN : (i == 9 ? NET_POLICY_CH : NET_VALUE_CH);
  F.eps = BN_EPS;
  double* scale = e->d_at<double>(0);
  float* bias = e->d_at<float>(scale_bytes);
  e->evaluator.set_loaded(false);
  k_fold_bn<<<(NET_CONVS * FOLD_STRIDE + 255) / 256, 256, 0, e->stream>>>(S, F, scale, bias);
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, launch_pack(S, segs, scale, bias, img, e->stream));
  e->launches += 2;
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  e->evaluator.set_loaded(true);
  // as spb_load_weights: the next search captures its step graph anew
  e->drop_step_graph();
  e->last_eval_parity = -1;
  return SPB_OK;
}

int32_t spb_chess_load_weights_device(spb_chess_engine* e, const spb_tensor* tensors, uint32_t n) {
  namespace ch = spb::chess;
  SPB_GUARD(e);
  size_t re[CH_ROLES];
  if (int32_t rc = resolve_table(e, "spb_chess_load_weights_device", tensors, n, re, resolve_chess)) return rc;
  Sources S;
  if (int32_t rc = gather_sources(e, tensors, re, CH_ROLES, &S)) return rc;
  const size_t scale_bytes = (size_t)ch::NET_CONV3 * FOLD_STRIDE * 8;
  if (int32_t rc = e->ensure_stage(scale_bytes + (size_t)ch::NET_CONV3 * FOLD_STRIDE * 4, 0)) return rc;
  if (!e->net) {
    std::string err;
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
    e->net = ch::net_create(e->T.G, &err);
    if (!e->net) { e->set_error("spb_chess_load_weights_device: " + err); return SPB_ERR_NOMEM; }
  }
  const ch::NetImage m = ch::net_image(e->net);
  SegList w;                                                             // d_w: 21 3x3 convs, then policy_conv1 / 2
  for (int i = 0; i < ch::NET_CONV3; ++i) {
    const int kc32 = i == 0 ? 1 : 8;
    Seg& g = w.add(m.off_conv[i], m.off_conv[i] + (size_t)9 * kc32 * 32 * 256 * 2, SEG_CHESS_CONV);
    g.conv = i; g.oc = 256; g.ic = i == 0 ? ch::NET_IN : 256; g.n = 256; g.kc = kc32; g.taps = 9; g.halves = i > 0 && m.res_halves;
  }
  const struct { size_t off; int role, oc, n; } heads[2] = {{m.off_p1, CH_ROLE_P1_W, 256, 256}, {m.off_p2, CH_ROLE_P2_W, ch::NET_MOVE_PLANES, 80}};
  for (const auto& h : heads) {
    Seg& g = w.add(h.off, h.off + (size_t)8 * 32 * h.n * 2, SEG_CHESS_CONV);
    g.role = h.role; g.oc = h.oc; g.ic = 256; g.n = h.n; g.kc = 8; g.taps = 1;
  }
  SegList f;                                                             // d_f, offsets in floats
  for (int i = 0; i < ch::NET_CONV3; ++i) {
    Seg& g = f.add(m.off_bias[i] * 4, (m.off_bias[i] + 256) * 4, SEG_BIAS);
    g.conv = i; g.oc = 256;
  }
  auto raw = [&f](size_t begin, size_t end, int role, int count) {
    Seg& g = f.add(begin * 4, end * 4, SEG_RAW);
    g.role = role; g.count = count;
  };
  raw(m.off_bp1, m.off_bp2, CH_ROLE_P1_B, 256);
  raw(m.off_bp2, m.off_vw, CH_ROLE_P2_B, ch::NET_MOVE_PLANES);
  raw(m.off_vw, m.off_vb, CH_ROLE_V_W, 256);
  raw(m.off_vb, m.off_f1w, CH_ROLE_V_B, 1);
  f.add(m.off_f1w * 4, m.off_f1b * 4, SEG_CHESS_F1W);
  raw(m.off_f1b, m.off_f2w, CH_ROLE_F1_B, 256);
  raw(m.off_f2w, m.off_f2b, CH_ROLE_F2_W, 256);
  raw(m.off_f2b, m.f_count, CH_ROLE_F2_B, 1);

  FoldArgs F{};
  F.convs = ch::NET_CONV3;
  for (int i = 0; i < ch::NET_CONV3; ++i) F.oc[i] = 256;
  F.eps = ch::NET_BN_EPS;
  double* scale = e->d_at<double>(0);
  float* bias = e->d_at<float>(scale_bytes);
  ch::net_set_loaded(e->net, false);
  k_fold_bn<<<(ch::NET_CONV3 * FOLD_STRIDE + 255) / 256, 256, 0, e->stream>>>(S, F, scale, bias);
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, launch_pack(S, w, scale, bias, m.d_w, e->stream));
  SPB_CUDA(e, launch_pack(S, f, scale, bias, m.d_f, e->stream));
  e->launches += 3;
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  ch::net_set_loaded(e->net, true);
  return SPB_OK;
}

}  // extern "C"
