// Host side of the model C-ABI: tensor registry keyed by the reference's state_dict names,
// eval-mode BatchNorm folding, weight packing for the fused kernels, forward dispatch.
//
// Folding (SURVEY.md 8a "Folded per-block math"; mdtc.py:55-59,115-118; tcn.py:75-84,101-114):
// for each BatchNorm with s = gamma / sqrt(var + 1e-5), t = beta - mean * s,
//     BN(conv(x; W, b)) = conv(x; W * s[out], b * s + t)
// computed in double and rounded once to fp32.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "conv_backbone.h"
#include "gru.h"
#include "gru_tc.h"
#include "mdtc_tc.h"
#include "tcn_tc.h"
#include "dstcn_tc.h"
#include "fsmn.h"
#include "linear_tc.h"
#include "tc_pack.h"

namespace wekws {

static thread_local std::string tl_error;
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  tl_error = buf;
}

int device_sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

namespace {

__global__ void softmax_rows_kernel(float* x, long long rows, int n) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float* p = x + row * n;
  float m = -INFINITY;
  for (int i = lane; i < n; i += 32) m = fmaxf(m, p[i]);
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
  for (int i = lane; i < n; i += 32) s += expf(p[i] - m);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  for (int i = lane; i < n; i += 32) p[i] = expf(p[i] - m) / s;
}

struct Folded {           // BN as per-channel scale/shift
  std::vector<double> s, t;
};

// A tensor-core kernel: the one pack prepared for a model, or the one a forward call takes (none: the backbone's FP32
// kernel).
enum class TcKernel { none, mdtc, tcn, ds_tcn, gru };

}  // namespace
}  // namespace wekws

using namespace wekws;

struct wekws_model {
  wekws_model_config cfg;
  std::map<std::string, std::vector<float>> tensors;
  bool finalized = false;
  int device = 0;
  int padmax = 0;                           // widest per-block cache slice of a conv backbone
  bool has_cmvn = false;
  std::vector<float> h_stream, h_vec;
  std::vector<int> h_chunk_off;
  float* d_stream = nullptr;
  float* d_vec = nullptr;
  int* d_chunk_off = nullptr;
  ConvArgs conv{};
  GruArgs gru{};
  int conv_max_T = 0;
  std::vector<std::vector<float>> folded;   // folded GEMM weights W^T [K][C] in consumption order
  TcKernel tc = TcKernel::none;             // the tensor-core kernel pack prepared: its weight images live in h_wimg / d_wimg
  std::vector<uint8_t> h_wimg;
  uint8_t* d_wimg = nullptr;
  int precision = 0;                        // 0 auto (tensor cores where eligible), 1 fp32 FFMA only, 2 tensor cores
  TcArgs tcargs{};                          // mdtc, hidden 64 (mdtc_tc.cu)
  TcnTcArgs tcnargs{};                      // dense TCN, hidden 64 (tcn_tc.cu)
  DsTcArgs dsargs{};                        // depthwise-separable TCN, hidden 256 (dstcn_tc.cu)
  GruTcArgs grutc{};                        // GRU (gru_tc.cu)
  FsmnArgs fsmn{};                          // FSMN backbone (fsmn.cu): weights live in h_vec / d_vec
  bool cls_tc = false;                      // wide classifier head (odim > 4) as its own tcgen05 GEMM (linear_tc.cu)
  std::vector<uint8_t> h_cimg;              //   behind the tensor-core DS-TCN backbone
  std::vector<float> h_cbias;
  uint8_t* d_cimg = nullptr;
  float* d_cbias = nullptr;
  float* d_hidden = nullptr;                // (B, T, 256) scratch between the two kernels; grows monotonically
  size_t hidden_cap = 0;
};

namespace {

int get_tensor(const wekws_model* m, const std::string& name, size_t numel, const float** out) {
  auto it = m->tensors.find(name);
  if (it == m->tensors.end()) {
    set_error("finalize: tensor '%s' was never set", name.c_str());
    return WEKWS_ERR_STATE;
  }
  if (it->second.size() != numel) {
    set_error("finalize: tensor '%s' has %zu elements, expected %zu", name.c_str(), it->second.size(), numel);
    return WEKWS_ERR_INVALID;
  }
  *out = it->second.data();
  return WEKWS_OK;
}

#define GET(ptr, name, numel)                                            \
  const float* ptr = nullptr;                                            \
  do { int _rc = get_tensor(m, (name), (numel), &ptr); if (_rc) return _rc; } while (0)

int fold_bn(const wekws_model* m, const std::string& p, int C, Folded* f) {
  GET(g, p + ".weight", (size_t)C);
  GET(b, p + ".bias", (size_t)C);
  GET(mu, p + ".running_mean", (size_t)C);
  GET(var, p + ".running_var", (size_t)C);
  f->s.resize(C); f->t.resize(C);
  for (int c = 0; c < C; ++c) {
    const double s = (double)g[c] / sqrt((double)var[c] + 1e-5);
    f->s[c] = s;
    f->t[c] = (double)b[c] - (double)mu[c] * s;
  }
  return WEKWS_OK;
}

size_t pad4(size_t n) { return (n + 3) & ~(size_t)3; }

// Appends W^T (K x C, from W[o][c] * s[o] with arbitrary source strides) as row chunks.
void push_gemm(wekws_model* m, int K, int C, const float* W, size_t o_stride, size_t c_stride, const double* s) {
  const int KC = conv_chunk_rows(C);
  m->folded.emplace_back((size_t)K * C);
  for (int k = 0; k < K; ++k)
    for (int o = 0; o < C; ++o)
      m->folded.back()[(size_t)k * C + o] = (float)((double)W[o * o_stride + k * c_stride] * (s ? s[o] : 1.0));
  for (int k0 = 0; k0 < K; k0 += KC) {
    const int kk = K - k0 < KC ? K - k0 : KC;
    m->h_chunk_off.push_back((int)m->h_stream.size());
    for (int k = k0; k < k0 + kk; ++k)
      for (int o = 0; o < C; ++o)
        m->h_stream.push_back((float)((double)W[o * o_stride + k * c_stride] * (s ? s[o] : 1.0)));
  }
}

int pack_common_front(wekws_model* m, int* v_mean, int* v_istd) {
  const int idim = m->cfg.idim;
  m->has_cmvn = m->tensors.count("global_cmvn.mean") != 0;
  *v_mean = (int)m->h_vec.size();
  m->h_vec.resize(m->h_vec.size() + pad4(idim), 0.f);
  *v_istd = (int)m->h_vec.size();
  m->h_vec.resize(m->h_vec.size() + pad4(idim), 1.f);
  if (m->has_cmvn) {
    GET(mean, "global_cmvn.mean", (size_t)idim);
    GET(istd, "global_cmvn.istd", (size_t)idim);
    for (int k = 0; k < idim; ++k) {
      m->h_vec[*v_mean + k] = mean[k];
      m->h_vec[*v_istd + k] = m->cfg.norm_var ? istd[k] : 1.f;   // cmvn.py:46-47
    }
  }
  return WEKWS_OK;
}

int pack_classifier(wekws_model* m, int H, int* v_wc, int* v_bc) {
  const int odim = m->cfg.odim;
  GET(wc, "classifier.linear.weight", (size_t)odim * H);
  GET(bc, "classifier.linear.bias", (size_t)odim);
  *v_wc = (int)m->h_vec.size();
  m->h_vec.resize(m->h_vec.size() + pad4((size_t)H * odim), 0.f);
  for (int c = 0; c < H; ++c)
    for (int j = 0; j < odim; ++j) m->h_vec[*v_wc + c * odim + j] = wc[j * H + c];
  *v_bc = (int)m->h_vec.size();
  m->h_vec.resize(m->h_vec.size() + pad4(odim), 0.f);
  for (int j = 0; j < odim; ++j) m->h_vec[*v_bc + j] = bc[j];
  return WEKWS_OK;
}

// K-major SWIZZLE_128B image of W[n][k0 .. k0+64) (n < 64) from W^T [K][64]: hi at dst, lo at dst + 8192
void write_w_image(uint8_t* dst, const std::vector<float>& wt, int K, int k0) {
  write_sw128_image(dst, 8192, wt.data() + (size_t)k0 * 64, 64, 1, 64, K - k0 < 64 ? K - k0 : 64);
}

// Same layout for 128 output channels n0 .. n0+127 of a [K][ldn] matrix: hi at dst, lo at dst + 16384 (dstcn_tc.cu)
void write_w_image128(uint8_t* dst, const std::vector<float>& wt, int ldn, int K, int k0, int n0) {
  write_sw128_image(dst, 16384, wt.data() + (size_t)k0 * ldn + n0, 128, 1, (size_t)ldn, K - k0 < 64 ? K - k0 : 64);
}

// The model fields every tensor-core argument block repeats from ConvArgs, copied by name (the blocks' layouts differ)
template <typename Args>
void copy_model_fields(Args& t, const ConvArgs& a) {
  memset(&t, 0, sizeof(t));
  t.idim = a.idim; t.odim = a.odim; t.nblocks = a.nblocks; t.ktaps = a.ktaps; t.P = a.P;
  t.act = a.act; t.has_cmvn = a.has_cmvn;
  t.v_mean = a.v_mean; t.v_istd = a.v_istd; t.v_bp = a.v_bp; t.v_blocks = a.v_blocks;
  t.v_blk_stride = a.v_blk_stride; t.v_wc = a.v_wc; t.v_bc = a.v_bc;
  for (int b = 0; b < a.nblocks; ++b) { t.dil[b] = a.dil[b]; t.coff[b] = a.coff[b]; }
}

// Tensor-core eligibility + pre-swizzled bf16x3 weight images (mdtc_tc.cu, tcn_tc.cu, dstcn_tc.cu)
void pack_tc(wekws_model* m) {
  m->tc = TcKernel::none;
  m->cls_tc = false;
  m->h_wimg.clear();
  m->h_cimg.clear();
  const wekws_model_config& c = m->cfg;
  const ConvArgs& a = m->conv;
  if (c.backbone == WEKWS_BACKBONE_DSTCN) {
    DsTcArgs& t = m->dsargs;
    copy_model_fields(t, a);
    // output_dim > 4 (CTC vocabularies): the classifier becomes its own tensor-core GEMM fed from a hidden scratch
    const bool cls_tc = c.odim > 4 && linear_tc_eligible(c.odim, c.hdim);
    t.hidden = cls_tc ? reinterpret_cast<float*>(1) : nullptr;      // placeholder for the eligibility test only
    const bool ok = dstcn_tc_eligible(t, c.hdim);
    t.hidden = nullptr;
    if (!ok || m->folded.size() != (size_t)(1 + a.nblocks)) return;
    m->cls_tc = cls_tc;
    if (cls_tc) {        // W_c^T [256][odim] sits in h_vec at v_wc (pack_classifier), the bias at v_bc
      m->h_cimg.assign(linear_tc_image_bytes(c.odim, c.hdim), 0);
      linear_tc_pack(m->h_cimg.data(), m->h_vec.data() + a.v_wc, c.odim, c.odim, c.hdim);
      m->h_cbias.assign((size_t)((c.odim + 127) / 128) * 128, 0.f);
      for (int j = 0; j < c.odim; ++j) m->h_cbias[j] = m->h_vec[a.v_bc + j];
    }
    const int natoms = (a.idim + 63) / 64;
    m->h_wimg.assign((size_t)(2 * natoms + 8 * a.nblocks) * 32768, 0);
    uint8_t* dst = m->h_wimg.data();
    for (int at = 0; at < natoms; ++at)
      for (int h = 0; h < 2; ++h, dst += 32768) write_w_image128(dst, m->folded[0], 256, a.idim, 64 * at, 128 * h);
    for (int b = 0; b < a.nblocks; ++b)
      for (int ks = 0; ks < 4; ++ks)
        for (int h = 0; h < 2; ++h, dst += 32768) write_w_image128(dst, m->folded[1 + b], 256, 256, 64 * ks, 128 * h);
    m->tc = TcKernel::ds_tcn;
    return;
  }
  if (c.hdim != 64) return;
  if (c.backbone == WEKWS_BACKBONE_TCN) {
    TcnTcArgs& t = m->tcnargs;
    copy_model_fields(t, a);
    if (!tcn_tc_eligible(t, m->padmax) || m->folded.size() != (size_t)(1 + a.ktaps * a.nblocks)) return;
    m->tc = TcKernel::tcn;
  } else if (c.backbone == WEKWS_BACKBONE_MDTC) {
    TcArgs& t = m->tcargs;
    copy_model_fields(t, a);
    t.stack_size = a.stack_size;
    if (!tc_eligible(t, m->padmax) || m->folded.size() != (size_t)(1 + 2 * a.nblocks)) return;
    m->tc = TcKernel::mdtc;
  } else {
    return;
  }
  // mdtc / tcn: 16 KB images [Wp k 0..63][Wp k 64..127][every further folded GEMM in consumption order]
  const size_t ngemm = m->folded.size() - 1;
  m->h_wimg.assign((2 + ngemm) * 16384, 0);
  write_w_image(m->h_wimg.data(), m->folded[0], a.idim, 0);
  if (a.idim > 64) write_w_image(m->h_wimg.data() + 16384, m->folded[0], a.idim, 64);
  for (size_t g = 0; g < ngemm; ++g) write_w_image(m->h_wimg.data() + (2 + g) * 16384, m->folded[1 + g], 64, 0);
  if (m->tc != TcKernel::mdtc) return;
  // depthwise taps + the two GEMM biases of every block, passed by value with the launch (mdtc_tc.h TcArgs::cw)
  TcArgs& t = m->tcargs;
  for (int b = 0; b < a.nblocks; ++b) {
    const float* vb = m->h_vec.data() + a.v_blocks + (size_t)b * a.v_blk_stride;
    float* dst = reinterpret_cast<float*>(&t.cw[b][0]);
    for (int j = 0; j < 5; ++j)
      for (int ch = 0; ch < 64; ++ch) dst[j * 64 + ch] = j < a.ktaps ? vb[j * 64 + ch] : 0.f;
    // the folded depthwise bias goes through the pointwise-1 matrix into b1 (h = relu(W1 (dw + b_dw) + b1)), so the
    // depthwise loop of the kernel starts from zero instead of loading a per-channel bias
    const float* w1t = m->folded[1 + 2 * b].data();     // W1^T [k][n]
    const float* bdw = vb + a.ktaps * 64;
    for (int ch = 0; ch < 64; ++ch) {
      double acc = vb[(a.ktaps + 1) * 64 + ch];
      for (int k = 0; k < 64; ++k) acc += (double)w1t[(size_t)k * 64 + ch] * (double)bdw[k];
      dst[5 * 64 + ch] = (float)acc;
      dst[6 * 64 + ch] = vb[(a.ktaps + 2) * 64 + ch];
    }
  }
}

// Block schedule of the conv backbones: mdtc = preprocessor (dilation 1), then num_stack x stack_size res blocks with
// dilations 2^l; tcn / ds_tcn = num_layers blocks with dilations 2^i.  Block b (state_dict prefix[b]) keeps
// dil[b] * (kernel_size - 1) cache columns starting at coff[b]; padding is their total (backbone.padding), padmax the
// widest slice.
struct ConvLayout {
  std::vector<std::string> prefix;
  std::vector<int> dil, coff;
  int padding = 0, padmax = 0;
};

ConvLayout conv_layout(const wekws_model_config& c) {
  ConvLayout L;
  auto block = [&](std::string prefix, int dil) {
    const int pad = dil * (c.kernel_size - 1);
    L.prefix.push_back(std::move(prefix));
    L.dil.push_back(dil);
    L.coff.push_back(L.padding);
    L.padding += pad;
    if (pad > L.padmax) L.padmax = pad;
  };
  if (c.backbone == WEKWS_BACKBONE_MDTC) {
    block("backbone.preprocessor", 1);
    for (int s = 0; s < c.num_stack; ++s)
      for (int l = 0; l < c.stack_size; ++l)
        block("backbone.blocks." + std::to_string(s) + ".res_blocks." + std::to_string(l), 1 << l);
  } else {
    for (int i = 0; i < c.num_layers; ++i) block("backbone.network." + std::to_string(i) + ".cnn", 1 << i);
  }
  return L;
}

int pack_conv(wekws_model* m) {
  const wekws_model_config& c = m->cfg;
  const int C = c.hdim, K = c.kernel_size, idim = c.idim;
  WEKWS_REQUIRE(C == 32 || C == 64 || C == 128 || C == 256, "hidden_dim %d unsupported (32/64/128/256)", C);
  WEKWS_REQUIRE(K >= 2 && K <= 8, "kernel_size %d unsupported (2..8)", K);
  WEKWS_REQUIRE(idim >= 1 && idim <= 128, "input_dim %d unsupported (1..128)", idim);
  if (c.backbone == WEKWS_BACKBONE_MDTC)
    WEKWS_REQUIRE(c.num_stack >= 1 && c.stack_size >= 1, "mdtc: num_stack/stack_size must be >= 1");
  else
    WEKWS_REQUIRE(c.num_layers >= 1, "tcn: num_layers must be >= 1");
  const ConvLayout layout = conv_layout(c);
  const int nblocks = (int)layout.dil.size();
  WEKWS_REQUIRE(nblocks <= kMaxBlocks, "%d blocks exceed the supported %d", nblocks, kMaxBlocks);
  m->padmax = layout.padmax;
  m->h_stream.clear(); m->h_vec.clear(); m->h_chunk_off.clear(); m->folded.clear();
  ConvArgs& a = m->conv;
  memset(&a, 0, sizeof(a));
  int rc = pack_common_front(m, &a.v_mean, &a.v_istd);
  if (rc) return rc;
  // preprocessing Linear (subsampling.py:45-48): W (C, idim)
  {
    GET(w, "preprocessing.out.0.weight", (size_t)C * idim);
    GET(b, "preprocessing.out.0.bias", (size_t)C);
    push_gemm(m, idim, C, w, idim, 1, nullptr);
    a.v_bp = (int)m->h_vec.size();
    m->h_vec.insert(m->h_vec.end(), b, b + C);
  }
  a.v_blocks = (int)m->h_vec.size();
  a.v_blk_stride = c.backbone == WEKWS_BACKBONE_MDTC ? (K + 3) * C
                 : c.backbone == WEKWS_BACKBONE_DSTCN ? (K + 2) * C : C;
  for (int bi = 0; bi < nblocks; ++bi) {
    const std::string& p = layout.prefix[bi];
    const size_t v0 = m->h_vec.size();
    if (c.backbone == WEKWS_BACKBONE_MDTC || c.backbone == WEKWS_BACKBONE_DSTCN) {
      const bool md = c.backbone == WEKWS_BACKBONE_MDTC;
      const std::string dw = md ? p + ".conv1.conv" : p + ".0";
      const std::string dwbn = md ? p + ".conv1.bn" : p + ".1";
      const std::string pw = md ? p + ".conv1.pointwise" : p + ".3";
      const std::string pwbn = md ? p + ".bn1" : p + ".4";
      GET(wd, dw + ".weight", (size_t)C * K);
      GET(bd, dw + ".bias", (size_t)C);
      Folded f0, f1;
      if ((rc = fold_bn(m, dwbn, C, &f0))) return rc;
      if ((rc = fold_bn(m, pwbn, C, &f1))) return rc;
      for (int j = 0; j < K; ++j)
        for (int ch = 0; ch < C; ++ch) m->h_vec.push_back((float)((double)wd[ch * K + j] * f0.s[ch]));
      for (int ch = 0; ch < C; ++ch) m->h_vec.push_back((float)((double)bd[ch] * f0.s[ch] + f0.t[ch]));
      GET(w1, pw + ".weight", (size_t)C * C);
      GET(b1, pw + ".bias", (size_t)C);
      push_gemm(m, C, C, w1, C, 1, f1.s.data());
      for (int o = 0; o < C; ++o) m->h_vec.push_back((float)((double)b1[o] * f1.s[o] + f1.t[o]));
      if (md) {
        Folded f2;
        if ((rc = fold_bn(m, p + ".bn2", C, &f2))) return rc;
        GET(w2, p + ".conv2.weight", (size_t)C * C);
        GET(b2, p + ".conv2.bias", (size_t)C);
        push_gemm(m, C, C, w2, C, 1, f2.s.data());
        for (int o = 0; o < C; ++o) m->h_vec.push_back((float)((double)b2[o] * f2.s[o] + f2.t[o]));
      }
    } else {  // dense TCN: weight (C, C, K) -> K tap matrices
      GET(w, p + ".0.weight", (size_t)C * C * K);
      GET(b, p + ".0.bias", (size_t)C);
      Folded f;
      if ((rc = fold_bn(m, p + ".1", C, &f))) return rc;
      for (int j = 0; j < K; ++j) push_gemm(m, C, C, w + j, (size_t)C * K, K, f.s.data());
      for (int o = 0; o < C; ++o) m->h_vec.push_back((float)((double)b[o] * f.s[o] + f.t[o]));
    }
    if (m->h_vec.size() - v0 != (size_t)a.v_blk_stride) {
      set_error("internal: block vector stride mismatch");
      return WEKWS_ERR_INVALID;
    }
  }
  if ((rc = pack_classifier(m, C, &a.v_wc, &a.v_bc))) return rc;
  m->h_chunk_off.push_back((int)m->h_stream.size());
  a.kind = c.backbone; a.C = C; a.idim = idim; a.odim = c.odim; a.nblocks = nblocks; a.ktaps = K;
  a.P = layout.padding; a.stack_size = c.stack_size > 0 ? c.stack_size : 1; a.act = c.activation;
  a.has_cmvn = m->has_cmvn ? 1 : 0;
  a.n_chunks = (int)m->h_chunk_off.size() - 1;
  for (int b = 0; b < nblocks; ++b) { a.dil[b] = layout.dil[b]; a.coff[b] = layout.coff[b]; }
  pack_tc(m);
  return WEKWS_OK;
}

int pack_gru(wekws_model* m) {
  const wekws_model_config& c = m->cfg;
  const int H = c.hdim, G = 3 * H, idim = c.idim, L = c.num_layers;
  WEKWS_REQUIRE(H == 128, "GRU hidden_dim %d unsupported (128 only)", H);
  WEKWS_REQUIRE(L >= 1 && L <= 4, "GRU num_layers %d unsupported (1..4)", L);
  WEKWS_REQUIRE(idim >= 1 && idim <= 128, "input_dim %d unsupported (1..128)", idim);
  m->h_stream.clear(); m->h_vec.clear(); m->h_chunk_off.clear();
  GruArgs& a = m->gru;
  memset(&a, 0, sizeof(a));
  int rc = pack_common_front(m, &a.v_mean, &a.v_istd);
  if (rc) return rc;
  GET(wp, "preprocessing.out.0.weight", (size_t)H * idim);
  GET(bp, "preprocessing.out.0.bias", (size_t)H);
  a.v_wp = (int)m->h_vec.size();
  for (int k = 0; k < idim; ++k)
    for (int j = 0; j < H; ++j) m->h_vec.push_back(wp[j * idim + k]);
  a.v_bp = (int)m->h_vec.size();
  m->h_vec.insert(m->h_vec.end(), bp, bp + H);
  a.v_layers = (int)m->h_vec.size();
  a.v_layer_stride = 2 * H * G + 2 * G;
  for (int l = 0; l < L; ++l) {
    const std::string sfx = "_l" + std::to_string(l);
    GET(wih, "backbone.weight_ih" + sfx, (size_t)G * H);
    GET(whh, "backbone.weight_hh" + sfx, (size_t)G * H);
    GET(bih, "backbone.bias_ih" + sfx, (size_t)G);
    GET(bhh, "backbone.bias_hh" + sfx, (size_t)G);
    for (int k = 0; k < H; ++k) {            // row k: [W_ih[:, k] | W_hh[:, k]]  (768 floats, streamed by TMA)
      for (int g = 0; g < G; ++g) m->h_vec.push_back(wih[g * H + k]);
      for (int g = 0; g < G; ++g) m->h_vec.push_back(whh[g * H + k]);
    }
    m->h_vec.insert(m->h_vec.end(), bih, bih + G);
    m->h_vec.insert(m->h_vec.end(), bhh, bhh + G);
  }
  if ((rc = pack_classifier(m, H, &a.v_wc, &a.v_bc))) return rc;
  a.L = L; a.H = H; a.idim = idim; a.odim = c.odim; a.act = c.activation; a.has_cmvn = m->has_cmvn ? 1 : 0;
  // tensor-core variant: the per-step weight stream as pre-swizzled bf16 hi|lo operand chunks
  m->tc = TcKernel::none;
  m->h_wimg.clear();
  if (gru_tc_eligible(L, H, idim)) {
    const float* wih[4];
    const float* whh[4];
    for (int l = 0; l < L; ++l) {
      const std::string sfx = "_l" + std::to_string(l);
      if ((rc = get_tensor(m, "backbone.weight_ih" + sfx, (size_t)G * H, &wih[l]))) return rc;
      if ((rc = get_tensor(m, "backbone.weight_hh" + sfx, (size_t)G * H, &whh[l]))) return rc;
    }
    m->h_wimg.assign(gru_tc_image_bytes(L, idim), 0);
    gru_tc_pack(m->h_wimg.data(), wp, idim, wih, whh, L);
    GruTcArgs& t = m->grutc;
    memset(&t, 0, sizeof(t));
    t.L = L; t.idim = idim; t.odim = c.odim; t.act = c.activation; t.has_cmvn = a.has_cmvn;
    t.v_mean = a.v_mean; t.v_istd = a.v_istd; t.v_bp = a.v_bp; t.v_layers = a.v_layers;
    t.v_layer_stride = a.v_layer_stride; t.v_wc = a.v_wc; t.v_bc = a.v_bc;
    m->tc = TcKernel::gru;
  }
  return WEKWS_OK;
}


// FSMN (wekws/model/fsmn.py:401-495): every matrix transposed to [K][Npad] (Npad = N rounded up to the GEMM pass width,
// zero filled) so the kernel streams K-chunks with 16-byte cp.async; biases padded the same way; memory taps as
// [lorder + rorder][proj] (left taps, then right taps).
int pack_fsmn(wekws_model* m) {
  const wekws_model_config& c = m->cfg;
  const int idim = c.idim, A1 = c.fsmn_input_affine_dim, D = c.fsmn_linear_dim, P = c.fsmn_proj_dim;
  const int A2 = c.fsmn_output_affine_dim, O = c.odim, L = c.num_layers, lo = c.fsmn_left_order, ro = c.fsmn_right_order;
  WEKWS_REQUIRE(idim >= 1 && A1 >= 1 && D >= 1 && P >= 1 && A2 >= 1 && L >= 1 && L <= 16, "fsmn: bad layer dimensions");
  WEKWS_REQUIRE(lo >= 1 && ro >= 1, "fsmn: left_order %d / right_order %d unsupported (the reference's FSMNBlock itself "
                "breaks for right_order = 0: fsmn.py:235 slices x_pad[:, :, :-0])", lo, ro);
  m->h_stream.clear(); m->h_vec.clear(); m->h_chunk_off.clear();
  FsmnArgs& a = m->fsmn;
  memset(&a, 0, sizeof(a));
  int rc = pack_common_front(m, &a.o_mean, &a.o_istd);
  if (rc) return rc;
  const int NP = fsmn_pass_cols();
  auto npad = [&](int n) { return (n + NP - 1) / NP * NP; };
  auto push_wt = [&](const float* W, int N, int K, int* off) {      // W[n][k] -> W^T [K][npad(N)]
    *off = (int)m->h_vec.size();
    const int np = npad(N);
    m->h_vec.resize(m->h_vec.size() + (size_t)K * np, 0.f);
    for (int k = 0; k < K; ++k)
      for (int n = 0; n < N; ++n) m->h_vec[*off + (size_t)k * np + n] = W[(size_t)n * K + k];
  };
  auto push_b = [&](const float* b, int N, int* off) {
    *off = (int)m->h_vec.size();
    m->h_vec.resize(m->h_vec.size() + npad(N), 0.f);
    for (int n = 0; n < N; ++n) m->h_vec[*off + n] = b[n];
  };
  GET(w1, "backbone.in_linear1.linear.weight", (size_t)A1 * idim);
  GET(b1, "backbone.in_linear1.linear.bias", (size_t)A1);
  GET(w2, "backbone.in_linear2.linear.weight", (size_t)D * A1);
  GET(b2, "backbone.in_linear2.linear.bias", (size_t)D);
  push_wt(w1, A1, idim, &a.o_w_in1); push_b(b1, A1, &a.o_b_in1);
  push_wt(w2, D, A1, &a.o_w_in2); push_b(b2, D, &a.o_b_in2);
  a.o_layers = (int)m->h_vec.size();
  for (int l = 0; l < L; ++l) {
    const std::string p = "backbone.fsmn." + std::to_string(l) + ".";
    GET(wp, p + "0.linear.weight", (size_t)P * D);
    GET(wl, p + "1.conv_left.weight", (size_t)P * lo);
    GET(wr, p + "1.conv_right.weight", (size_t)P * ro);
    GET(wa, p + "2.linear.weight", (size_t)D * P);
    GET(ba, p + "2.linear.bias", (size_t)D);
    const int base = (int)m->h_vec.size();
    int off;
    push_wt(wp, P, D, &off);
    if (l == 0) a.lo_wp = off - base;
    off = (int)m->h_vec.size();
    if (l == 0) a.lo_taps = off - base;
    m->h_vec.resize(m->h_vec.size() + pad4((size_t)(lo + ro) * P), 0.f);
    for (int i = 0; i < lo; ++i)
      for (int ch = 0; ch < P; ++ch) m->h_vec[off + (size_t)i * P + ch] = wl[(size_t)ch * lo + i];
    for (int j = 0; j < ro; ++j)
      for (int ch = 0; ch < P; ++ch) m->h_vec[off + (size_t)(lo + j) * P + ch] = wr[(size_t)ch * ro + j];
    push_wt(wa, D, P, &off);
    if (l == 0) a.lo_wa = off - base;
    push_b(ba, D, &off);
    if (l == 0) a.lo_ba = off - base;
    if (l == 0) a.layer_stride = (int)m->h_vec.size() - base;
  }
  GET(wo1, "backbone.out_linear1.linear.weight", (size_t)A2 * D);
  GET(bo1, "backbone.out_linear1.linear.bias", (size_t)A2);
  GET(wo2, "backbone.out_linear2.linear.weight", (size_t)O * A2);
  GET(bo2, "backbone.out_linear2.linear.bias", (size_t)O);
  push_wt(wo1, A2, D, &a.o_w_out1); push_b(bo1, A2, &a.o_b_out1);
  push_wt(wo2, O, A2, &a.o_w_out2); push_b(bo2, O, &a.o_b_out2);
  a.idim = idim; a.aff_in = A1; a.lin = D; a.proj = P; a.aff_out = A2; a.odim = O; a.L = L; a.lorder = lo; a.rorder = ro;
  a.act = c.activation; a.has_cmvn = m->has_cmvn ? 1 : 0; a.norm_var = 1;      // istd already 1 when norm_var is off
  a.np_aff_in = npad(A1); a.np_lin = npad(D); a.np_proj = npad(P); a.np_aff_out = npad(A2); a.np_odim = npad(O);
  const int m0 = idim > D ? idim : D;
  int m1 = A1 > P ? A1 : P;
  if (A2 > m1) m1 = A2;
  a.sp0 = (int)pad4(m0) + 4; a.sp1 = (int)pad4(m1) + 4; a.spm = (int)pad4(P) + 4;   // +4: rows start in different banks
  WEKWS_REQUIRE(fsmn_smem_bytes(a) <= 226 * 1024, "fsmn: layer widths (%d, %d, %d) exceed the fused kernel's shared memory", m0, m1, P);
  return WEKWS_OK;
}

void free_device(wekws_model* m) {
  cudaFree(m->d_stream); cudaFree(m->d_vec); cudaFree(m->d_chunk_off); cudaFree(m->d_wimg);
  cudaFree(m->d_cimg); cudaFree(m->d_cbias); cudaFree(m->d_hidden);
  m->d_stream = nullptr; m->d_vec = nullptr; m->d_chunk_off = nullptr; m->d_wimg = nullptr;
  m->d_cimg = nullptr; m->d_cbias = nullptr; m->d_hidden = nullptr; m->hidden_cap = 0;
}

}  // namespace

// ------------------------------------------------------------------------------- C ABI
extern "C" const char* wekws_last_error(void) { return tl_error.c_str(); }
extern "C" int wekws_abi_version(void) { return WEKWS_B200_ABI_VERSION; }
extern "C" uint64_t wekws_launch_count(void) { return g_launches.load(); }

extern "C" int wekws_model_create(const wekws_model_config* cfg, wekws_model** out) {
  WEKWS_REQUIRE(cfg && out, "wekws_model_create: null argument");
  WEKWS_REQUIRE(cfg->backbone >= WEKWS_BACKBONE_MDTC && cfg->backbone <= WEKWS_BACKBONE_FSMN,
                "unknown backbone id %d", cfg->backbone);
  WEKWS_REQUIRE(cfg->odim >= 1, "output_dim must be >= 1");
  WEKWS_REQUIRE(cfg->activation == WEKWS_ACT_IDENTITY || cfg->activation == WEKWS_ACT_SIGMOID,
                "unknown activation id %d", cfg->activation);
  wekws_model* m = new (std::nothrow) wekws_model();
  if (!m) { set_error("out of host memory"); return WEKWS_ERR_NOMEM; }
  m->cfg = *cfg;
  *out = m;
  return WEKWS_OK;
}

extern "C" void wekws_model_destroy(wekws_model* m) {
  if (!m) return;
  free_device(m);
  delete m;
}

extern "C" int wekws_model_padding(const wekws_model* m) {
  if (!m) return 0;
  if (m->cfg.backbone == WEKWS_BACKBONE_GRU) return 0;
  if (m->cfg.backbone == WEKWS_BACKBONE_FSMN) return m->cfg.fsmn_left_order - 1 + m->cfg.fsmn_right_order;
  return conv_layout(m->cfg).padding;
}

extern "C" int wekws_model_set_tensor(wekws_model* m, const char* name, const float* h_data, int64_t numel) {
  WEKWS_REQUIRE(m && name && (h_data || numel == 0) && numel >= 0, "wekws_model_set_tensor: bad argument");
  m->tensors[name].assign(h_data, h_data + numel);
  m->finalized = false;
  return WEKWS_OK;
}

extern "C" int wekws_model_pack(wekws_model* m) {
  WEKWS_REQUIRE(m, "wekws_model_pack: null handle");
  if (m->cfg.backbone == WEKWS_BACKBONE_FSMN) return pack_fsmn(m);
  return m->cfg.backbone == WEKWS_BACKBONE_GRU ? pack_gru(m) : pack_conv(m);
}

extern "C" int wekws_model_finalize(wekws_model* m) {
  WEKWS_REQUIRE(m, "wekws_model_finalize: null handle");
  int rc = wekws_model_pack(m);
  if (rc) return rc;
  free_device(m);
  WEKWS_CUDA_OK(cudaGetDevice(&m->device));
  WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_vec, m->h_vec.size() * sizeof(float)));
  WEKWS_CUDA_OK(cudaMemcpy(m->d_vec, m->h_vec.data(), m->h_vec.size() * sizeof(float), cudaMemcpyHostToDevice));
  if (m->tc != TcKernel::none) {
    WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_wimg, m->h_wimg.size()));
    WEKWS_CUDA_OK(cudaMemcpy(m->d_wimg, m->h_wimg.data(), m->h_wimg.size(), cudaMemcpyHostToDevice));
  }
  if (m->cfg.backbone == WEKWS_BACKBONE_FSMN) {
    m->fsmn.w = m->d_vec;
  } else if (m->cfg.backbone == WEKWS_BACKBONE_GRU) {
    m->gru.vec = m->d_vec;
    m->grutc.vec = m->d_vec; m->grutc.wimg = m->d_wimg;
  } else {
    WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_stream, m->h_stream.size() * sizeof(float)));
    WEKWS_CUDA_OK(cudaMemcpy(m->d_stream, m->h_stream.data(), m->h_stream.size() * sizeof(float), cudaMemcpyHostToDevice));
    WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_chunk_off, m->h_chunk_off.size() * sizeof(int)));
    WEKWS_CUDA_OK(cudaMemcpy(m->d_chunk_off, m->h_chunk_off.data(), m->h_chunk_off.size() * sizeof(int), cudaMemcpyHostToDevice));
    m->conv.wstream = m->d_stream; m->conv.chunk_off = m->d_chunk_off; m->conv.vec = m->d_vec;
    m->tcargs.wimg = m->d_wimg; m->tcargs.vec = m->d_vec;
    m->tcnargs.wimg = m->d_wimg; m->tcnargs.vec = m->d_vec;
    m->dsargs.wimg = m->d_wimg; m->dsargs.vec = m->d_vec;
    if (m->cls_tc) {
      WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_cimg, m->h_cimg.size()));
      WEKWS_CUDA_OK(cudaMemcpy(m->d_cimg, m->h_cimg.data(), m->h_cimg.size(), cudaMemcpyHostToDevice));
      WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_cbias, m->h_cbias.size() * sizeof(float)));
      WEKWS_CUDA_OK(cudaMemcpy(m->d_cbias, m->h_cbias.data(), m->h_cbias.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    m->conv_max_T = conv_backbone_max_T(m->conv, m->padmax);
    WEKWS_REQUIRE(m->conv_max_T >= 1, "model does not fit the fused kernel's shared memory");
  }
  m->finalized = true;
  return WEKWS_OK;
}

extern "C" int wekws_model_set_precision(wekws_model* m, int mode) {
  WEKWS_REQUIRE(m && mode >= 0 && mode <= 2, "wekws_model_set_precision: mode must be 0 (auto), 1 (fp32) or 2 (tensor cores wherever a kernel exists)");
  m->precision = mode;
  return WEKWS_OK;
}

// GRU: which kernel is faster depends on the batch as well (measured on B200, scripts/gru_sweep.py): the weight-streaming
// tensor-core kernel takes ~9-10 us per step whatever the batch (up to 148 x 64 streams), the FP32 kernel scales with
// the streams per SM and has the shorter single-step latency at small batches.
static bool gru_takes_tc(const wekws_model* m, int64_t B, int64_t T) {
  if (m->tc != TcKernel::gru || m->precision == 1 || T < 1) return false;
  if (m->precision == 2) return true;
  return B >= (T == 1 ? 640 : T < 8 ? 400 : 256);
}

// The kernel a forward call takes: the tensor-core kernel pack prepared, or none (the backbone's FP32 kernel).  The
// conv kernels need precision != 1, >= 8 frames per call and 16-byte aligned features; mdtc's also 16-byte aligned
// cache rows (null counts as aligned).
static TcKernel forward_kernel(const wekws_model* m, int64_t B, int64_t T, const float* feats, const float* in_cache,
                               const float* out_cache) {
  auto aligned = [](const float* p) { return ((uintptr_t)p & 15) == 0; };
  if (m->tc == TcKernel::gru) return gru_takes_tc(m, B, T) ? TcKernel::gru : TcKernel::none;
  if (m->tc == TcKernel::none || m->precision == 1 || T < 8 || !aligned(feats)) return TcKernel::none;
  if (m->tc == TcKernel::mdtc && !(aligned(in_cache) && aligned(out_cache))) return TcKernel::none;
  return m->tc;
}

extern "C" int wekws_model_uses_tensor_cores_bt(const wekws_model* m, int64_t B, int64_t T) {
  if (!m || !m->finalized) return 0;
  return forward_kernel(m, B, T, nullptr, nullptr, nullptr) != TcKernel::none ? 1 : 0;     // as for aligned tensors
}

extern "C" int wekws_model_uses_tensor_cores(const wekws_model* m, int64_t T) {
  return wekws_model_uses_tensor_cores_bt(m, 1 << 20, T);     // "for a large batch"
}

extern "C" int64_t wekws_model_packed_floats(const wekws_model* m, int which) {
  if (!m) return 0;
  if (which == 2) return (int64_t)(m->h_wimg.size() / sizeof(float));     // tensor-core weight images, raw bytes
  if (which == 3) return (int64_t)(m->h_cimg.size() / sizeof(float));     // tensor-core classifier images, raw bytes
  return which == 0 ? (int64_t)m->h_stream.size() : (int64_t)m->h_vec.size();
}

extern "C" int wekws_model_packed_copy(const wekws_model* m, int which, float* h_dst, int64_t capacity) {
  WEKWS_REQUIRE(m && h_dst, "wekws_model_packed_copy: null argument");
  if (which == 2 || which == 3) {
    const std::vector<uint8_t>& img = which == 2 ? m->h_wimg : m->h_cimg;
    WEKWS_REQUIRE((int64_t)(img.size() / sizeof(float)) <= capacity, "wekws_model_packed_copy: capacity too small");
    memcpy(h_dst, img.data(), img.size());
    return WEKWS_OK;
  }
  const std::vector<float>& v = which == 0 ? m->h_stream : m->h_vec;
  WEKWS_REQUIRE((int64_t)v.size() <= capacity, "wekws_model_packed_copy: capacity too small");
  memcpy(h_dst, v.data(), v.size() * sizeof(float));
  return WEKWS_OK;
}

extern "C" int wekws_model_forward(wekws_model* m, const float* d_feats, const float* d_in_cache,
                                   float* d_out, float* d_out_cache, int64_t B, int64_t T,
                                   uint32_t flags, void* stream) {
  WEKWS_REQUIRE(m, "wekws_model_forward: null handle");
  if (!m->finalized) { set_error("wekws_model_forward called before wekws_model_finalize"); return WEKWS_ERR_STATE; }
  WEKWS_REQUIRE(B >= 0 && T >= 0 && B < (1 << 30) && T < (1 << 30), "wekws_model_forward: bad B/T");
  if (B == 0 || T == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_feats && d_out && d_out_cache, "wekws_model_forward: null tensor");
  int dev = 0;
  WEKWS_CUDA_OK(cudaGetDevice(&dev));
  WEKWS_REQUIRE(dev == m->device, "model was finalized on device %d but current device is %d", m->device, dev);
  cudaStream_t st = (cudaStream_t)stream;
  const TcKernel k = forward_kernel(m, B, T, d_feats, d_in_cache, d_out_cache);
  const bool cls_tc = k == TcKernel::ds_tcn && m->cls_tc;
  const bool fsmn = m->cfg.backbone == WEKWS_BACKBONE_FSMN;
  if (m->cfg.backbone == WEKWS_BACKBONE_GRU) {
    auto call = [&](const auto& model_args) {
      auto a = model_args;
      a.feats = d_feats; a.in_cache = d_in_cache; a.out = d_out; a.out_cache = d_out_cache;
      a.B = (int)B; a.T = (int)T;
      return a;
    };
    int rc = k == TcKernel::gru ? gru_tc_launch(call(m->grutc), st) : gru_launch(call(m->gru), st);
    if (rc) return rc;
  } else {
    // time-chunk long inputs; the cache carries the state between chunks exactly as in
    // streaming use (chunked == full utterance, SURVEY.md 8a "Numerical facts")
    const int maxT = k == TcKernel::mdtc ? tc_max_T() : k == TcKernel::tcn ? tcn_tc_max_T()
                   : k == TcKernel::ds_tcn ? dstcn_tc_max_T() : fsmn ? fsmn_tile_rows() : m->conv_max_T;
    if (cls_tc) {      // hidden scratch between the backbone kernel and the classifier GEMM
      const size_t need = (size_t)B * (size_t)T * (size_t)m->cfg.hdim;
      if (need > m->hidden_cap) {
        WEKWS_CUDA_OK(cudaStreamSynchronize(st));          // the old scratch may still be in use on this stream
        cudaFree(m->d_hidden);
        m->d_hidden = nullptr; m->hidden_cap = 0;
        WEKWS_CUDA_OK(cudaMalloc((void**)&m->d_hidden, need * sizeof(float)));
        m->hidden_cap = need;
      }
    }
    const int nchunk = (int)((T + maxT - 1) / maxT);
    const int Tc = (int)((T + nchunk - 1) / nchunk);
    for (int64_t t0 = 0; t0 < T; t0 += Tc) {
      // the per-chunk fields of every chunked kernel's argument block, set by name (the blocks' layouts differ)
      auto chunk = [&](const auto& model_args) {
        auto a = model_args;
        a.feats = d_feats + t0 * m->cfg.idim;
        a.out = d_out + t0 * m->cfg.odim;
        a.in_cache = t0 == 0 ? d_in_cache : d_out_cache;
        a.out_cache = d_out_cache;
        a.B = (int)B;
        a.T = (int)(T - t0 < Tc ? T - t0 : Tc);
        a.feat_bstride = T * m->cfg.idim;
        a.out_bstride = T * m->cfg.odim;
        return a;
      };
      int rc;
      switch (k) {
        case TcKernel::mdtc: rc = mdtc_tc_launch(chunk(m->tcargs), m->padmax, st); break;
        case TcKernel::tcn: rc = tcn_tc_launch(chunk(m->tcnargs), m->padmax, st); break;
        case TcKernel::ds_tcn: {
          DsTcArgs a = chunk(m->dsargs);
          if (cls_tc) { a.hidden = m->d_hidden + t0 * m->cfg.hdim; a.hidden_bstride = T * m->cfg.hdim; }
          rc = dstcn_tc_launch(a, st);
          break;
        }
        default: rc = fsmn ? fsmn_launch(chunk(m->fsmn), st) : conv_backbone_launch(chunk(m->conv), m->padmax, st);
      }
      if (rc) return rc;
    }
  }
  if (cls_tc) {
    // classifier (+ activation) of all B*T frames in one tensor-core GEMM over the hidden scratch (classifier.py:63-67)
    LinearTcArgs a;
    a.x = m->d_hidden; a.out = d_out; a.wimg = m->d_cimg; a.bias = m->d_cbias;
    a.rows = B * T; a.x_stride = m->cfg.hdim; a.out_stride = m->cfg.odim;
    a.N = m->cfg.odim; a.K = m->cfg.hdim; a.act = m->cfg.activation; a.n_mtiles = 0;
    int rc = linear_tc_launch(a, st);
    if (rc) return rc;
  }
  if (flags & WEKWS_FWD_SOFTMAX) {
    const long long rows = B * T;
    const int wpb = 8;
    softmax_rows_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, st>>>(d_out, rows, m->cfg.odim);
    int rc = check_launch("softmax_rows_kernel");
    if (rc) return rc;
  }
  return WEKWS_OK;
}

extern "C" int wekws_pipeline_forward(wekws_fbank* fb, wekws_model* m, const void* d_pcm, int pcm_dtype,
                                      int64_t B, int64_t num_samples, int64_t pcm_stride,
                                      float* d_feat_scratch, const float* d_in_cache, float* d_out,
                                      float* d_out_cache, uint32_t flags, void* stream) {
  WEKWS_REQUIRE(fb && m && d_feat_scratch, "wekws_pipeline_forward: null argument");
  WEKWS_REQUIRE(wekws_fbank_feature_dim(fb) == m->cfg.idim, "pipeline: the front-end produces %d features but the model expects input_dim %d",
                wekws_fbank_feature_dim(fb), m->cfg.idim);
  const int64_t frames = wekws_fbank_num_frames(fb, num_samples);
  // The feature tensor only lives between the two launches.  Pin it in L2 for their duration (persisting access-policy
  // window on this stream): the front-end's writes stay in the cache, the model kernel's first-Linear reads hit there,
  // and the lines are released (not written back as "persisting") afterwards -- the 320 B/frame never has to make the
  // HBM round trip as long as B * frames * idim * 4 fits the device's persisting-L2 carve-out.
  cudaStream_t st = (cudaStream_t)stream;
  const size_t feat_bytes = (size_t)B * (size_t)frames * (size_t)m->cfg.idim * sizeof(float);
  bool windowed = false;
  if (feat_bytes > 0) {
    int dev = 0, max_persist = 0, max_window = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev) == cudaSuccess && max_persist > 0) {
      static bool limit_set[64] = {false};
      if (dev >= 0 && dev < 64 && !limit_set[dev]) {
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)max_persist);
        limit_set[dev] = true;
      }
      cudaStreamAttrValue attr;
      memset(&attr, 0, sizeof(attr));
      attr.accessPolicyWindow.base_ptr = d_feat_scratch;
      attr.accessPolicyWindow.num_bytes = feat_bytes < (size_t)max_window ? feat_bytes : (size_t)max_window;
      attr.accessPolicyWindow.hitRatio = feat_bytes <= (size_t)max_persist ? 1.0f : (float)max_persist / (float)feat_bytes;
      attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
      windowed = cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
    }
    cudaGetLastError();      // the window is an optimisation: never fatal
  }
  int rc = wekws_fbank_forward(fb, d_pcm, pcm_dtype, B, num_samples, pcm_stride, nullptr, nullptr, nullptr,
                               d_feat_scratch, frames, stream);
  if (rc == 0) rc = wekws_model_forward(m, d_feat_scratch, d_in_cache, d_out, d_out_cache, B, frames, flags, stream);
  if (windowed) {
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    attr.accessPolicyWindow.num_bytes = 0;                       // window off for whatever the caller runs next
    cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr);
    cudaGetLastError();
  }
  return rc;
}
