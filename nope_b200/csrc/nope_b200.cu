// nope_b200 -- engine + C ABI (include/nope_b200.h).
//
// The engine owns the repacked UNet weights, a per-chunk activation workspace and the
// layer schedule of UNet.forward (reference:
// src/model/u_net/denoising_diffusion_pytorch/u_net.py:160-198), batched over all pose
// hypotheses of a chunk.  Host code is plain C++; kernels live in conv_tc.cuh / kernels.cuh.
#include "../../include/nope_b200.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "conv_tc.cuh"
#include "conv_tc2.cuh"
#include "kernels.cuh"
#include "linattn_tc.cuh"
#include "encoder.cuh"
#include "ldm.cuh"
#include "vsd.cuh"

using namespace nope;

namespace {

constexpr int kAbiVersion = 2;
constexpr int kHeadsHidden = 128;  // 4 heads x 32 (model_utils.py:368,394)

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> data;
};

struct ConvLayer {
  int mode = 0;  // 0: 3x3 pad1, 1: 1x1, 2: unshuffle+1x1, 3: nearest-x2 upsample + 3x3 (folded)
  int cin = 0, cout = 0, K = 0, bn = 0;
  int Kp = 0;             // packed row length: K (fp16 weights) or 2K (W_hi | W_lo, precision >= 1)
  __half* w = nullptr;    // [rows][Kp] fp16
  float* bias = nullptr;  // [cout] fp32 or nullptr
  CUtensorMap wmap;
  CUtensorMap wmap_half;  // BN/2-row box for the 2-CTA kernel
  bool has_map = false;
  // pre-norm folded into this (bias-free 1x1) layer: weights hold W diag(gamma); see GnFuse::pre_*
  float* pre_w1 = nullptr;
  float* pre_wb = nullptr;
};

struct NormLayer {
  float* gamma = nullptr;
  float* beta = nullptr;
  int C = 0, G = 1;
};

// NHWC fp16 activation [n_img, S, S, C]; `lo` carries the fp16 remainder x - fp16(x) in the
// split-precision mode (nullptr otherwise)
struct Act {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int C = 0;
  Act() {}
  Act(__half* h, int c, __half* l = nullptr) : hi(h), lo(l), C(c) {}
};

// what the fused epilogue applies after the convolution (ResnetBlock / Block / to_out)
struct GnSpec {
  const NormLayer* norm = nullptr;   // nullptr: no normalisation
  bool silu = false;
  int pb_offset = -1;                // pose-projection columns of this block, -1: none
  Act res;                           // residual (hi == nullptr: none)
  int res_div = 0, res_base = 0;     // residual image = (res_base + img) / res_div (hoisted prefix)
  float2* emit = nullptr;            // GroupNorm(1) partial sums of the output for a following pre-norm
  const float2* pre_stats = nullptr; // folded pre-norm: partial sums of the INPUT images ([img][pre_parts])
  int pre_parts = 0;
};

// bump allocator over one device slab (base == nullptr: size computation only)
struct Bump {
  uint8_t* base = nullptr;
  size_t off = 0;
  template <typename T> void take(T** out, size_t n) {
    off = (off + 255) & ~static_cast<size_t>(255);
    if (base) *out = reinterpret_cast<T*>(base + off);     // size-only passes leave the engine untouched
    off += n * sizeof(T);
  }
};

}  // namespace

struct nope_unet {
  int dim = 0, Cl = 0, S0 = 0, rot_dim = 6, cemb = 0, device = 0, num_sms = 148;
  int dims[5] = {0, 0, 0, 0, 0};
  bool finalized = false;
  int conv_impl = 2;   // 0: tcgen05 1-CTA tiles, 1: SIMT debug twin, 2: tcgen05 CTA pairs (default)
  bool fuse_gn = true; // GroupNorm / SiLU / pose bias / residual in the conv epilogue (conv_impl 2 only)
  // 0: fp16 operands; 1: exact weights (W_hi + W_lo K-segments, 2x the MMA work); 2: split precision
  // (exact weights + activations carried as hi + lo: A_hi W_hi + A_hi W_lo + A_lo W_hi, 3x);
  // 3: bf16 operands and activations (8-bit mantissa: its own, looser tolerance)
  int precision = 0;
  int attn_impl = 0;         // LinearAttention core: 0 tcgen05 (token counts >= 128), 1 CUDA cores
  int metric = 0;            // NOPE_METRIC_* of the fused scoring
  float occ_threshold = 0.2f;
  int chunk = 642;
  int64_t launches = 0;

  std::map<std::string, HostTensor> host;
  std::map<std::string, std::vector<int64_t>> expected;  // key -> shape

  std::map<std::string, ConvLayer> convs;
  std::map<std::string, NormLayer> norms;
  std::map<std::string, int> pb_off;
  int P = 0;  // total pose-projection width
  ConvLayer poseproj;
  float *pose_w = nullptr, *pose_b = nullptr, *init_w = nullptr, *init_b = nullptr,
        *final_w = nullptr, *final_b = nullptr;
  std::vector<void*> owned;  // every cudaMalloc'd weight pointer

  // workspace: one slab, either caller-provided (nope_unet_set_workspace) or owned
  int cap = 0, cap_ref = 0;
  uint8_t* ws_base = nullptr;
  size_t ws_bytes = 0;
  bool ws_external = false;
  bool ws_fresh = false;            // counters not zeroed yet
  Act sk[4][2];
  Act TA, TB, TC, TD, XA, XB, RB;
  __half *cs = nullptr, *pb = nullptr;
  Act x0, g1;                       // per-reference pre-stage
  __half* pt = nullptr;
  float2* gn_partial = nullptr;   // gn_stats_kernel output (per-op test path only)
  float2 *SA = nullptr, *SB = nullptr;   // unfused statistics: conv epilogue / gn_apply emit; SB also fused emit
  uint2* xpart = nullptr;         // fused GroupNorm: cross-tile partial sums, {value, epoch} words
  size_t xpart_words = 0;
  unsigned gn_epoch = 0;          // tag of the last fused launch that exchanged partial sums
  int* ref_of = nullptr;
  float* score_partial = nullptr;
  float* sim_buf = nullptr;

  std::map<std::tuple<const void*, int, int, int, int>, CUtensorMap> tmaps;

  // per-launch CUDA-event profile of the convolution kernel (bench.py roofline)
  bool profile = false;
  std::vector<cudaEvent_t> prof_ev;      // pairs
  std::vector<double> prof_flops;

  // debug tap
  std::string tap_name;
  float* tap_out = nullptr;
  int64_t tap_cap = 0;
  int tap_C = 0, tap_S = 0;
  bool tap_hit = false;

  ~nope_unet() {
    for (void* p : owned) cudaFree(p);
    if (ws_base && !ws_external) cudaFree(ws_base);
    for (cudaEvent_t e : prof_ev) cudaEventDestroy(e);
  }
  bool fused() const { return fuse_gn && conv_impl == 2; }
  bool split() const { return (precision == 2 || precision == 4) && fused(); }
  // precision 4: the residual stream, skip tensors and resampled maps keep their (hi, lo) pair, the tensor INSIDE a
  // ResnetBlock (block1's output h, consumed only by block2's convolution) is a single fp16 value -- block2 runs two
  // products per tap instead of three.  CPU budget (tools/precision_sim.py): h alone costs 4.3e-4 on the embeddings.
  bool h_lo() const { return precision == 2 && fused(); }
  bool bf() const { return precision == 3; }     // bf16 storage (BASELINE configs[2]); fp16 otherwise

  // ------------------------------------------------------------------ schema
  void expect(const std::string& k, std::vector<int64_t> s) { expected[k] = std::move(s); }
  void expect_resblock(const std::string& p, int cin, int cout, bool mlp = true) {
    if (mlp) {
      expect(p + ".mlp.1.weight", {cout, cemb});
      expect(p + ".mlp.1.bias", {cout});
    }
    expect(p + ".block1.proj.weight", {cout, cin, 3, 3});
    expect(p + ".block1.proj.bias", {cout});
    expect(p + ".block1.norm.weight", {cout});
    expect(p + ".block1.norm.bias", {cout});
    expect(p + ".block2.proj.weight", {cout, cout, 3, 3});
    expect(p + ".block2.proj.bias", {cout});
    expect(p + ".block2.norm.weight", {cout});
    expect(p + ".block2.norm.bias", {cout});
    if (cin != cout) {
      expect(p + ".res_conv.weight", {cout, cin, 1, 1});
      expect(p + ".res_conv.bias", {cout});
    }
  }
  void expect_linattn(const std::string& p, int d) {
    expect(p + ".fn.fn.to_qkv.weight", {3 * kHeadsHidden, d, 1, 1});
    expect(p + ".fn.fn.to_out.0.weight", {d, kHeadsHidden, 1, 1});
    expect(p + ".fn.fn.to_out.0.bias", {d});
    expect(p + ".fn.fn.to_out.1.weight", {d});
    expect(p + ".fn.fn.to_out.1.bias", {d});
    expect(p + ".fn.norm.weight", {d});
    expect(p + ".fn.norm.bias", {d});
  }
  // state_dict schema of the reference UNet (u_net.py:27-158), encoder excluded.
  void build_schema() {
    expect("pose_mlp.0.weight", {cemb, rot_dim});
    expect("pose_mlp.0.bias", {cemb});
    expect("init_conv.weight", {dim, Cl, 3, 3});
    expect("init_conv.bias", {dim});
    for (int i = 0; i < 4; ++i) {
      const int din = dims[i], dout = dims[i + 1];
      const std::string p = "downs." + std::to_string(i);
      expect_resblock(p + ".0", din, din);
      expect_resblock(p + ".1", din, din);
      expect_linattn(p + ".2", din);
      if (i < 3) {
        expect(p + ".3.1.weight", {dout, din * 4, 1, 1});
        expect(p + ".3.1.bias", {dout});
      } else {
        expect(p + ".3.weight", {dout, din, 3, 3});
        expect(p + ".3.bias", {dout});
      }
    }
    const int mid = dims[4];
    expect("mid_attn.fn.fn.to_qkv.weight", {3 * kHeadsHidden, mid, 1, 1});
    expect("mid_attn.fn.fn.to_out.weight", {mid, kHeadsHidden, 1, 1});
    expect("mid_attn.fn.fn.to_out.bias", {mid});
    expect("mid_attn.fn.norm.weight", {mid});
    expect("mid_attn.fn.norm.bias", {mid});
    expect_resblock("mid_block1", mid, mid);
    expect_resblock("mid_block2", mid, mid);
    for (int j = 0; j < 4; ++j) {
      const int din = dims[3 - j], dout = dims[4 - j];
      const std::string p = "ups." + std::to_string(j);
      expect_resblock(p + ".0", dout + din, dout);
      expect_resblock(p + ".1", dout + din, dout);
      expect_linattn(p + ".2", dout);
      if (j < 3) {
        expect(p + ".3.1.weight", {din, dout, 3, 3});
        expect(p + ".3.1.bias", {din});
      } else {
        expect(p + ".3.weight", {din, dout, 3, 3});
        expect(p + ".3.bias", {din});
      }
    }
    expect_resblock("final_res_block", 2 * dim, dim);
    expect_resblock("final_conv.0", dim, dim);  // owns an unused mlp.1 (u_net.py:154-157)
    expect("final_conv.1.weight", {Cl, dim, 1, 1});
    expect("final_conv.1.bias", {Cl});
  }

  // ------------------------------------------------------------------ weights
  int upload_f32(const std::string& key, float** out) {
    auto it = host.find(key);
    NOPE_CHECK(it != host.end(), "missing tensor " + key);
    NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(out), it->second.data.size() * sizeof(float)));
    owned.push_back(*out);
    NOPE_CUDA(cudaMemcpy(*out, it->second.data.data(), it->second.data.size() * sizeof(float),
                         cudaMemcpyHostToDevice));
    return 0;
  }
  // pack one conv weight (+ bias) into a ConvLayer.  mode 3 (nearest-x2 upsample + conv3x3,
  // HardUpsample) first folds the 3x3 kernel into four 2x2 parity kernels (fold_upconv_kernel).
  // precision >= 1 appends the fp16 remainders as a second K-block: rows are [W_hi (K) | W_lo (K)].
  int make_conv(const std::string& name, const std::string& wkey, const std::string& bkey, int mode) {
    auto it = host.find(wkey);
    NOPE_CHECK(it != host.end(), "missing tensor " + wkey);
    const auto& sh = it->second.shape;
    ConvLayer L;
    L.mode = mode;
    L.cout = (int)sh[0];
    const int rows = mode == 3 ? 4 * L.cout : L.cout;   // weight-matrix rows
    const int taps = mode == 0 ? 9 : (mode == 1 ? 1 : 4);
    L.cin = mode == 2 ? (int)sh[1] / 4 : (int)sh[1];
    L.K = L.cin * taps;
    const bool wlo = precision == 1 || precision == 2 || precision == 4;
    L.Kp = wlo ? 2 * L.K : L.K;
    NOPE_CHECK(L.cin % 64 == 0, wkey + ": input channels must be a multiple of 64");
    L.bn = pick_bn(L.cout);
    NOPE_CHECK(L.bn != 0, wkey + ": output channels must be a multiple of 64");
    float *tmp = nullptr, *folded = nullptr;
    const size_t n = it->second.data.size();
    NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&tmp), n * sizeof(float)));
    NOPE_CUDA(cudaMemcpy(tmp, it->second.data.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    const size_t npack = (size_t)rows * L.Kp;
    const float* src = tmp;
    if (mode == 3) {
      NOPE_CHECK(sh.size() == 4 && sh[2] == 3 && sh[3] == 3, wkey + ": expected a 3x3 kernel");
      NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&folded), (size_t)rows * L.K * sizeof(float)));
      fold_upconv_kernel<<<ew_grid((long long)4 * L.cout * L.cin), 256>>>(tmp, folded, L.cout, L.cin);
      NOPE_CUDA(cudaGetLastError());
      src = folded;
    }
    NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&L.w), npack * sizeof(__half)));
    owned.push_back(L.w);
    pack_weight_kernel<<<ew_grid((long long)rows * L.K), 256>>>(src, L.w, rows, L.cin, taps, L.Kp, 0,
                                                                wlo ? L.K : 0, bf() ? 1 : 0);
    NOPE_CUDA(cudaGetLastError());
    NOPE_CUDA(cudaDeviceSynchronize());
    NOPE_CUDA(cudaFree(tmp));
    if (folded) NOPE_CUDA(cudaFree(folded));
    if (!bkey.empty()) {
      if (upload_f32(bkey, &L.bias)) return -1;
    }
    if (make_weight_map(&L.wmap, L.w, rows, L.Kp, L.bn)) return -1;
    if (make_weight_map(&L.wmap_half, L.w, rows, L.Kp, L.bn / 2)) return -1;
    L.has_map = true;
    convs[name] = L;
    return 0;
  }
  int make_norm(const std::string& name, const std::string& prefix, int G) {
    NormLayer n;
    auto it = host.find(prefix + ".weight");
    NOPE_CHECK(it != host.end(), "missing tensor " + prefix + ".weight");
    n.C = (int)it->second.shape[0];
    n.G = G;
    NOPE_CHECK(n.C % (8 * G) == 0, prefix + ": channels per group must be a multiple of 8");
    if (upload_f32(prefix + ".weight", &n.gamma)) return -1;
    if (upload_f32(prefix + ".bias", &n.beta)) return -1;
    norms[name] = n;
    return 0;
  }
  int make_resblock(const std::string& p) {
    if (make_conv(p + ".block1", p + ".block1.proj.weight", p + ".block1.proj.bias", 0)) return -1;
    if (make_conv(p + ".block2", p + ".block2.proj.weight", p + ".block2.proj.bias", 0)) return -1;
    if (make_norm(p + ".norm1", p + ".block1.norm", 8)) return -1;
    if (make_norm(p + ".norm2", p + ".block2.norm", 8)) return -1;
    if (host.count(p + ".res_conv.weight"))
      if (make_conv(p + ".res", p + ".res_conv.weight", p + ".res_conv.bias", 1)) return -1;
    return 0;
  }
  // to_qkv with the PreNorm GroupNorm(1) folded in (model_utils.py:226-234, 399): packed weights
  // W' = W diag(gamma); w1[c] = sum_k W'[c,k] over the values the tensor core actually multiplies
  // (fp16 hi, + lo in the exact-weight modes); wb[c] = sum_k W[c,k] beta[k].
  int make_qkv_folded(const std::string& name, const std::string& wkey, const std::string& nprefix) {
    const HostTensor& W = host.at(wkey);
    const std::vector<float>& gm = host.at(nprefix + ".weight").data;
    const std::vector<float>& bt = host.at(nprefix + ".bias").data;
    const int rows = (int)W.shape[0], cin = (int)W.shape[1];
    HostTensor Wf;
    Wf.shape = W.shape;
    Wf.data.resize(W.data.size());
    std::vector<float> w1(rows), wb(rows);
    for (int o = 0; o < rows; ++o) {
      double s1 = 0.0, sb = 0.0;
      for (int k = 0; k < cin; ++k) {
        const float w = W.data[(size_t)o * cin + k];
        const float wf = w * gm[k];
        Wf.data[(size_t)o * cin + k] = wf;
        if (precision == 3) {
          uint32_t u;
          std::memcpy(&u, &wf, 4);
          u = (u + 0x7fffu + ((u >> 16) & 1u)) & 0xffff0000u;        // round to nearest even bf16
          float r;
          std::memcpy(&r, &u, 4);
          s1 += (double)r;
        } else {
          const __half hi = __float2half_rn(wf);
          s1 += (double)__half2float(hi);
          if (precision >= 1) s1 += (double)__half2float(__float2half_rn(wf - __half2float(hi)));
        }
        sb += (double)w * (double)bt[k];
      }
      w1[o] = (float)s1;
      wb[o] = (float)sb;
    }
    const std::string tmpkey = "__folded." + name;
    host[tmpkey] = std::move(Wf);
    if (make_conv(name, tmpkey, "", 1)) return -1;
    host.erase(tmpkey);
    ConvLayer& L = convs[name];
    for (auto pr : {std::make_pair(&L.pre_w1, &w1), std::make_pair(&L.pre_wb, &wb)}) {
      NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(pr.first), rows * sizeof(float)));
      owned.push_back(*pr.first);
      NOPE_CUDA(cudaMemcpy(*pr.first, pr.second->data(), rows * sizeof(float), cudaMemcpyHostToDevice));
    }
    return 0;
  }
  int make_linattn(const std::string& p) {
    if (make_norm(p + ".prenorm", p + ".fn.norm", 1)) return -1;
    if (make_conv(p + ".qkv", p + ".fn.fn.to_qkv.weight", "", 1)) return -1;
    if (make_qkv_folded(p + ".qkvf", p + ".fn.fn.to_qkv.weight", p + ".fn.norm")) return -1;
    if (make_conv(p + ".out", p + ".fn.fn.to_out.0.weight", p + ".fn.fn.to_out.0.bias", 1)) return -1;
    if (make_norm(p + ".outnorm", p + ".fn.fn.to_out.1", 1)) return -1;
    return 0;
  }
  // concatenate the 19 pose projections (model_utils.py:261-263) into one [P, cemb] GEMM
  int make_poseproj() {
    std::vector<std::string> blocks;
    for (int i = 0; i < 4; ++i)
      for (int b = 0; b < 2; ++b) blocks.push_back("downs." + std::to_string(i) + "." + std::to_string(b));
    blocks.push_back("mid_block1");
    blocks.push_back("mid_block2");
    for (int j = 0; j < 4; ++j)
      for (int b = 0; b < 2; ++b) blocks.push_back("ups." + std::to_string(j) + "." + std::to_string(b));
    blocks.push_back("final_res_block");
    std::vector<float> w, bias;
    P = 0;
    for (const auto& b : blocks) {
      const HostTensor& hw = host.at(b + ".mlp.1.weight");
      const HostTensor& hb = host.at(b + ".mlp.1.bias");
      pb_off[b] = P;
      P += (int)hw.shape[0];
      w.insert(w.end(), hw.data.begin(), hw.data.end());
      bias.insert(bias.end(), hb.data.begin(), hb.data.end());
    }
    HostTensor tw;
    tw.shape = {P, cemb, 1, 1};
    tw.data = std::move(w);
    HostTensor tb;
    tb.shape = {P};
    tb.data = std::move(bias);
    host["__poseproj.weight"] = std::move(tw);
    host["__poseproj.bias"] = std::move(tb);
    if (make_conv("__poseproj", "__poseproj.weight", "__poseproj.bias", 1)) return -1;
    poseproj = convs["__poseproj"];
    return 0;
  }

  int finalize() {
    NOPE_CHECK(!finalized, "already finalized");
    for (const auto& kv : expected)
      NOPE_CHECK(host.count(kv.first), "state_dict is missing " + kv.first);
    NOPE_CHECK(precision == 0 || conv_impl != 1, "the SIMT debug convolution only runs fp16 weights");
    NOPE_CHECK(precision < 2 || fused(), "split precision / bf16 need the fused schedule on the CTA-pair kernel");
    NOPE_CUDA(cudaSetDevice(device));
    if (upload_f32("pose_mlp.0.weight", &pose_w) || upload_f32("pose_mlp.0.bias", &pose_b) ||
        upload_f32("init_conv.weight", &init_w) || upload_f32("init_conv.bias", &init_b) ||
        upload_f32("final_conv.1.weight", &final_w) || upload_f32("final_conv.1.bias", &final_b))
      return -1;
    for (int i = 0; i < 4; ++i) {
      const std::string p = "downs." + std::to_string(i);
      if (make_resblock(p + ".0") || make_resblock(p + ".1") || make_linattn(p + ".2")) return -1;
      if (i < 3) {
        if (make_conv(p + ".3", p + ".3.1.weight", p + ".3.1.bias", 2)) return -1;
      } else {
        if (make_conv(p + ".3", p + ".3.weight", p + ".3.bias", 0)) return -1;
      }
    }
    if (make_resblock("mid_block1") || make_resblock("mid_block2")) return -1;
    if (make_norm("mid_attn.prenorm", "mid_attn.fn.norm", 1)) return -1;
    if (make_conv("mid_attn.qkv", "mid_attn.fn.fn.to_qkv.weight", "", 1)) return -1;
    if (make_qkv_folded("mid_attn.qkvf", "mid_attn.fn.fn.to_qkv.weight", "mid_attn.fn.norm")) return -1;
    if (make_conv("mid_attn.out", "mid_attn.fn.fn.to_out.weight", "mid_attn.fn.fn.to_out.bias", 1))
      return -1;
    for (int j = 0; j < 4; ++j) {
      const std::string p = "ups." + std::to_string(j);
      if (make_resblock(p + ".0") || make_resblock(p + ".1") || make_linattn(p + ".2")) return -1;
      if (j < 3) {
        if (make_conv(p + ".3", p + ".3.1.weight", p + ".3.1.bias", 3)) return -1;
      } else {
        if (make_conv(p + ".3", p + ".3.weight", p + ".3.bias", 0)) return -1;
      }
    }
    if (make_resblock("final_res_block") || make_resblock("final_conv.0")) return -1;
    if (make_poseproj()) return -1;
    host.clear();
    finalized = true;
    return 0;
  }

  // ------------------------------------------------------------------ workspace
  // One slab carved by a bump allocator: ~6 MB per hypothesis (12 MB in the split-precision mode).
  // layout(b) assigns every buffer for capacities (c hypotheses, r references).
  void take_act(Bump& b, Act* a, size_t n, int C, bool with_lo) {
    if (b.base) {
      a->C = C;
      a->lo = nullptr;
    }
    b.take(&a->hi, n);
    if (with_lo) b.take(&a->lo, n);
  }
  size_t layout(Bump& b, int c_hyp, int c_ref, int n_total_scores) {
    const size_t c = (size_t)c_hyp, r = (size_t)c_ref;
    const bool lo = precision == 2 || precision == 4;
    // temporaries hold the widest full-resolution tensor: a concat-conv output (<= 2*dim
    // channels) or the attention qkv tensor (3 x 128 channels, independent of dim)
    const size_t big = (size_t)S0 * S0 * std::max(dim * 2, 3 * kHeadsHidden);
    const size_t xsz = (size_t)S0 * S0 * dim;      // one full-resolution feature map
    for (int i = 0; i < 4; ++i) {
      const int s = S0 >> i;
      for (int k = 0; k < 2; ++k) take_act(b, &sk[i][k], c * s * s * dims[i], dims[i], lo);
    }
    take_act(b, &TA, c * big, 0, false);
    take_act(b, &TB, c * big, 0, lo);
    take_act(b, &TC, c * big, 0, lo);
    take_act(b, &TD, c * big, 0, false);
    take_act(b, &XA, c * xsz, 0, lo);
    take_act(b, &XB, c * xsz, 0, lo);
    take_act(b, &RB, c * xsz, dim, lo);
    b.take(&cs, c * cemb);
    b.take(&pb, c * (size_t)P);
    take_act(b, &x0, r * xsz, dim, lo);
    take_act(b, &g1, r * xsz, dim, lo);
    b.take(&pt, r * xsz);
    const size_t m = std::max(c, r);
    b.take(&gn_partial, m * 8 * 8);
    b.take(&ref_of, m);
    b.take(&SA, m * ((size_t)S0 * S0 * dim / 256));   // (hw/32) x (C/8) at the top level
    b.take(&SB, m * 8);
    // <= 64 (slot, image, group) entries of two {value, epoch} words per image
    if (b.base) xpart_words = (m + 8) * 64 * 2;
    b.take(&xpart, (m + 8) * 64 * 2);
    const int nslab = (S0 * S0 + kFinalPix - 1) / kFinalPix;
    b.take(&score_partial, (size_t)n_total_scores * nslab * kScoreParts);
    b.take(&sim_buf, (size_t)n_total_scores);
    return b.off;
  }
  size_t workspace_bytes(int c_hyp, int c_ref, int n_scores) {
    Bump b;
    return layout(b, c_hyp, c_ref, n_scores) + 256;
  }
  int scores_cap = 0;
  int ensure_workspace(int need_cap, int need_ref, int need_scores = 0) {
    if (need_cap <= cap && need_ref <= cap_ref && need_scores <= scores_cap) return 0;
    NOPE_CHECK(!ws_external, "the caller-provided workspace is too small for this sweep "
                             "(nope_unet_workspace_bytes / nope_unet_set_workspace)");
    NOPE_CUDA(cudaDeviceSynchronize());
    if (ws_base) cudaFree(ws_base);
    ws_base = nullptr;
    const int c = std::max(cap, need_cap), r = std::max(cap_ref, need_ref), sc = std::max(scores_cap, need_scores);
    const size_t bytes = workspace_bytes(c, r, sc);
    NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&ws_base), bytes));
    ws_bytes = bytes;
    return adopt(c, r, sc);
  }
  int adopt(int c, int r, int sc) {
    tmaps.clear();
    cap = c; cap_ref = r; scores_cap = sc;
    Bump b;
    b.base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws_base) + 255) & ~static_cast<uintptr_t>(255));
    layout(b, c, r, sc);
    ws_fresh = true;
    return 0;
  }
  int set_workspace(void* ptr, size_t bytes, int c, int r, int sc) {
    NOPE_CHECK(ptr && c >= 1 && r >= 1, "bad workspace arguments");
    NOPE_CHECK(bytes >= workspace_bytes(c, r, sc), "workspace buffer smaller than nope_unet_workspace_bytes");
    if (ws_base && !ws_external) {
      NOPE_CUDA(cudaDeviceSynchronize());
      cudaFree(ws_base);
    }
    ws_base = static_cast<uint8_t*>(ptr);
    ws_bytes = bytes;
    ws_external = true;
    return adopt(c, r, sc);
  }
  // the tile-sync words of a fresh slab carry epoch 0, which no launch uses
  int prepare_stream(cudaStream_t st) {
    if (ws_fresh) {
      NOPE_CUDA(cudaMemsetAsync(xpart, 0, xpart_words * sizeof(uint2), st));
      ws_fresh = false;
    }
    return 0;
  }

  // ------------------------------------------------------------------ tensor maps
  int get_map(const CUtensorMap** out, const void* base, int cap_img, int C, const TileGeom& g,
              int kind /* -1: plain, 0..3: unshuffle (p1*2+p2) */) {
    auto key = std::make_tuple(base, cap_img * 8 + (kind + 1), C, g.H, g.W);
    auto it = tmaps.find(key);
    if (it == tmaps.end()) {
      CUtensorMap m;
      int rc = kind < 0 ? make_act_map(&m, base, cap_img, C, g)
                        : make_unshuffle_map(&m, base, cap_img, C, g, kind >> 1, kind & 1);
      if (rc) return -1;
      it = tmaps.emplace(key, m).first;
    }
    *out = &it->second;
    return 0;
  }

  // ------------------------------------------------------------------ op launchers
  // out[n_img, So, So, cout] = conv(L, in0 (++ in1)).  The K loop walks, per filter tap and source
  // tensor, up to three products: A_hi W_hi, A_hi W_lo (precision >= 1), A_lo W_hi (sources that
  // carry a remainder).  `gs` selects the fused GroupNorm epilogue; `stats` the unfused partial sums.
  int conv(const ConvLayer& L, const Act& in0, const Act& in1, const Act& out, int So, int n_img, int cap_img,
           cudaStream_t st, float2* stats = nullptr, const GnSpec* gs = nullptr) {
    const int c0 = in0.C, c1 = in1.hi ? in1.C : 0;
    NOPE_CHECK(c0 + c1 == L.cin, "conv: channel mismatch");
    ++launches;
    if (conv_impl == 1) {
      NOPE_CHECK(!gs && L.Kp == L.K, "the SIMT debug convolution has no fused epilogue / split weights");
      SimtConvArgs a;
      a.src0 = in0.hi; a.src1 = in1.hi; a.C0 = c0; a.C1 = c1; a.w = L.w; a.bias = L.bias; a.out = out.hi;
      a.n_img = n_img; a.H = So; a.W = So; a.Cout = L.cout; a.K = L.K; a.mode = L.mode;
      conv_simt_kernel<<<ew_grid((long long)n_img * So * So * L.cout, 256, 148 * 32), 256, 0, st>>>(a);
      NOPE_CUDA(cudaGetLastError());
      if (stats) {
        // the SIMT twin has no fused statistics: produce them in the conv-epilogue format
        // (parts = max(1, hw/32), noct = C/8) with a plain reduction kernel
        const int hw = So * So;
        stats_ref_kernel<<<dim3(hw < 32 ? 1 : hw / 32, n_img), 256, 0, st>>>(out.hi, stats, hw, L.cout);
        NOPE_CUDA(cudaGetLastError());
      }
      return 0;
    }
    TileGeom g;
    if (make_geom(So, So, &g)) return -1;
    ConvParams p;
    memset(&p, 0, sizeof p);
    const CUtensorMap* m = nullptr;
    p.n_par = 1;
    const bool wlo = L.Kp > L.K;                       // packed rows carry W_lo at column K + ...
    const bool alo0 = in0.lo != nullptr, alo1 = in1.hi && in1.lo != nullptr;
    // taps: (dy, dx, lattice) ; sources: (hi map, lo map, channels, weight column offset inside a tap)
    struct Tap { int dy, dx, lat; };
    std::vector<Tap> taps;
    int n_lat = 1;
    if (L.mode == 3) {
      // So is the OUTPUT side (2x the source side); tiles and input maps use the source geometry
      NOPE_CHECK(in1.hi == nullptr && So % 2 == 0, "upsample conv takes one source");
      if (make_geom(So / 2, So / 2, &g)) return -1;
      for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b) taps.push_back(Tap{a - 1, b - 1, 0});
      p.n_par = 4;
    } else if (L.mode == 2) {
      NOPE_CHECK(in1.hi == nullptr, "unshuffle conv takes one source");
      for (int t = 0; t < 4; ++t) taps.push_back(Tap{0, 0, t});
      n_lat = 4;
    } else if (L.mode == 0) {
      for (int t = 0; t < 9; ++t) taps.push_back(Tap{t / 3 - 1, t % 3 - 1, 0});
    } else {
      taps.push_back(Tap{0, 0, 0});
    }
    // activation maps: index = lattice + n_lat * (source + 2 * is_lo)
    auto map_index = [&](int lat, int src, int lo) { return lat + n_lat * (src + 2 * lo); };
    int max_map = 0;
    bool map_set[kMaxAMaps] = {false};
    for (int lat = 0; lat < n_lat; ++lat)
      for (int src = 0; src < (in1.hi ? 2 : 1); ++src)
        for (int lo = 0; lo < 2; ++lo) {
          const Act& a = src ? in1 : in0;
          const __half* base = lo ? a.lo : a.hi;
          if (!base) continue;
          // unshuffle with a remainder: 4 lattices x (hi, lo) of ONE source = maps 0..3, 4..7
          const int idx = (n_lat == 4) ? lat + 4 * lo : map_index(lat, src, lo);
          NOPE_CHECK(idx < kMaxAMaps, "conv: activation map table overflow");
          if (get_map(&m, base, cap_img, a.C, g, L.mode == 2 ? lat : -1)) return -1;
          p.amap[idx] = *m;
          map_set[idx] = true;
          max_map = std::max(max_map, idx);
        }
    p.n_amaps = max_map + 1;
    for (int i = 1; i < p.n_amaps; ++i)      // unused slots: any valid descriptor (they are only prefetched)
      if (!map_set[i]) p.amap[i] = p.amap[0];
    int nseg = 0, ksteps = 0;
    auto add_seg = [&](int map, const Tap& t, int nch, int wcol) {
      p.seg[nseg++] = ConvSeg{(int16_t)map, (int16_t)t.dy, (int16_t)t.dx, (int16_t)nch, wcol + 1};
      ksteps += nch;
    };
    const int n_products = 1 + (wlo ? 1 : 0) + ((alo0 || alo1) ? 1 : 0);
    NOPE_CHECK((int)taps.size() * (in1.hi ? 2 : 1) * n_products <= kMaxSeg, "conv: segment table overflow");
    for (size_t ti = 0; ti < taps.size(); ++ti) {
      const Tap& t = taps[ti];
      const int wbase = (int)ti * L.cin;
      const int mh0 = (n_lat == 4) ? t.lat : map_index(0, 0, 0);
      const int ml0 = (n_lat == 4) ? t.lat + 4 : map_index(0, 0, 1);
      // A_hi W_hi
      add_seg(mh0, t, c0 / 64, wbase);
      if (in1.hi) add_seg(map_index(0, 1, 0), t, c1 / 64, wbase + c0);
      // A_hi W_lo
      if (wlo) {
        add_seg(mh0, t, c0 / 64, L.K + wbase);
        if (in1.hi) add_seg(map_index(0, 1, 0), t, c1 / 64, L.K + wbase + c0);
      }
      // A_lo W_hi
      if (alo0) add_seg(ml0, t, c0 / 64, wbase);
      if (alo1) add_seg(map_index(0, 1, 1), t, c1 / 64, wbase + c0);
    }
    p.bmap = L.wmap;
    p.bmap_half = L.wmap_half;
    p.bf16 = bf() ? 1 : 0;
    static const int l2pf = std::getenv("NOPE_L2_PREFETCH") ? std::atoi(std::getenv("NOPE_L2_PREFETCH")) : 0;   // measured 3 % slower when on
    p.l2_prefetch = l2pf;
    if (L.mode == 3) {
      for (int t = 0; t < 4; ++t) {
        if (get_map(&m, out.hi, cap_img, L.cout, g, t)) return -1;   // stride-2 sub-lattice (py, px)
        p.omap[t] = *m;
      }
      p.src_w = g.W;
      p.src_hw = g.H * g.W;
    } else {
      if (get_map(&m, out.hi, cap_img, L.cout, g, -1)) return -1;
      for (int t = 0; t < 4; ++t) p.omap[t] = *m;
    }
    p.bias = L.bias;
    p.stats = stats;
    p.stats_hw = So * So;
    p.stats_noct = L.cout / 8;
    p.n_total = L.cout;
    p.m_valid = n_img * g.H * g.W;     // rows of the GEMM (source pixels for the folded upsample conv)
    p.nseg = nseg;
    p.ksteps = ksteps;
    p.m_tiles = geom_m_tiles(g, n_img);
    p.n_tiles_par = L.cout / L.bn;
    p.n_tiles = p.n_tiles_par * p.n_par;
    p.tiles_per_img = g.tiles_per_img;
    p.h_cnt = g.h_cnt;
    p.b_cnt = g.b_cnt;
    NOPE_CHECK(!(stats && L.mode == 3), "fused statistics are not available on the upsample conv");
    if (gs) {
      NOPE_CHECK(conv_impl == 2 && L.mode != 3 && !stats, "fused GroupNorm epilogue: CTA-pair kernel, no upsample");
      GnFuse& f = p.gn;
      const int hw = So * So;
      f.G = gs->norm ? gs->norm->G : 0;
      if (gs->norm) {
        NOPE_CHECK(gs->norm->C == L.cout, "fused GroupNorm: channel mismatch");
        f.gamma = gs->norm->gamma;
        f.beta = gs->norm->beta;
        f.cpg = L.cout / f.G;
        NOPE_CHECK(f.cpg % 8 == 0 && (f.cpg >= L.bn ? f.cpg % L.bn == 0 : L.bn % f.cpg == 0),
                   "fused GroupNorm: groups must tile the channel tiles");
      } else {
        f.cpg = L.cout;
      }
      f.gpt = std::max(1, L.bn / f.cpg);
      f.tpg = std::max(1, f.cpg / L.bn);
      f.mt = std::max(1, g.tiles_per_img);
      f.ipt = g.tiles_per_img > 0 ? 1 : g.b_cnt;
      f.expected = f.G > 0 ? f.mt * f.tpg : 1;
      int sh = 0;
      while ((1 << sh) < hw) ++sh;
      NOPE_CHECK((1 << sh) == hw, "fused GroupNorm: H*W must be a power of two");
      f.hw_shift = sh;
      f.inv_cnt = 1.0f / ((float)hw * (float)f.cpg);
      f.eps = 1e-5f;
      f.silu = gs->silu ? 1 : 0;
      f.pb = gs->pb_offset >= 0 ? pb : nullptr;
      f.pb_stride = P;
      f.pb_off = std::max(gs->pb_offset, 0);
      f.n_img = n_img;
      if (gs->res.hi) {
        NOPE_CHECK(gs->res.C == L.cout, "fused residual: channel mismatch");
        NOPE_CHECK(gs->res_div == 0 || g.tiles_per_img > 0, "residual image mapping needs >= 128-pixel images");
        if (get_map(&m, gs->res.hi, gs->res_div > 0 ? cap_ref : cap_img, L.cout, g, -1)) return -1;
        p.rmap = *m;
        f.has_res = 1;
        f.res_lo = gs->res.lo;
      } else {
        p.rmap = p.omap[0];
      }
      f.res_div = gs->res_div;
      f.res_base = gs->res_base;
      if (gs->pre_stats) {
        NOPE_CHECK(!gs->norm && L.pre_w1 && L.pre_wb && L.mode == 1 && !L.bias, "pre-norm fold: bias-free 1x1 layer with folded weights");
        f.pre_stats = gs->pre_stats;
        f.pre_parts = gs->pre_parts;
        f.pre_inv_cnt = 1.0f / ((float)hw * (float)L.cin);
        f.pre_w1 = L.pre_w1;
        f.pre_wb = L.pre_wb;
      }
      f.out_lo = out.lo;
      static const int dbg = std::getenv("NOPE_GN_DBG") ? std::atoi(std::getenv("NOPE_GN_DBG")) : 0;
      f.dbg = dbg;
      f.emit = gs->emit;
      f.emit_parts = f.mt * p.n_tiles;
      NOPE_CHECK(f.ipt * f.gpt <= 64 && f.ipt <= 8, "fused GroupNorm: tile holds too many (image, group) pairs");
      if (f.expected > 1) {
        const size_t n_sg = (size_t)(p.m_tiles / f.mt + 1) * (p.n_tiles / f.tpg);
        NOPE_CHECK(xpart && f.expected * f.ipt * f.gpt * 2 <= 256, "fused GroupNorm: sync group too large");
        NOPE_CHECK(n_sg * f.expected * f.ipt * f.gpt * 2 <= xpart_words, "fused GroupNorm: partial-sum buffer too small");
        f.xpart = xpart;
        if (++gn_epoch == 0) ++gn_epoch;     // 0 is the tag of a fresh buffer
        f.epoch = gn_epoch;
      }
    } else if (out.lo) {
      p.out_lo = out.lo;                // extras epilogue writes the remainder
    }
    // development: NOPE_GN_TS=<k> records phase timestamps of the k-th fused launch into NOPE_GN_TS_FILE
    unsigned long long* ts_dev = nullptr;
    if (gs) {
      static const int ts_k = std::getenv("NOPE_GN_TS") ? std::atoi(std::getenv("NOPE_GN_TS")) : -1;
      static int ts_count = 0;
      if (ts_k >= 0 && ts_count++ == ts_k) {
        cudaMalloc(reinterpret_cast<void**>(&ts_dev), (size_t)num_sms * 64 * 16 * sizeof(unsigned long long));
        cudaMemset(ts_dev, 0, (size_t)num_sms * 64 * 16 * sizeof(unsigned long long));
        p.gn.ts = ts_dev;
      }
    }
    auto launch = [&]() {
      if (gs) return launch_conv_gn(p, L.bn, num_sms, st);
      return conv_impl == 2 ? launch_conv_tc2(p, L.bn, num_sms, st) : launch_conv_tc(p, L.bn, num_sms, st);
    };
    if (ts_dev) {
      const int rc = launch();
      cudaDeviceSynchronize();
      std::vector<unsigned long long> h((size_t)num_sms * 64 * 16);
      cudaMemcpy(h.data(), ts_dev, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
      cudaFree(ts_dev);
      if (FILE* f = std::fopen(std::getenv("NOPE_GN_TS_FILE") ? std::getenv("NOPE_GN_TS_FILE") : "gn_ts.csv", "w")) {
        std::fprintf(f, "# So=%d n_img=%d cout=%d K=%d expected=%d m_tiles=%d n_tiles=%d\n", So, n_img, L.cout, L.K,
                     p.gn.expected, p.m_tiles, p.n_tiles);
        for (int c = 0; c < num_sms; ++c)
          for (int it = 0; it < 64; ++it) {
            const unsigned long long* r = &h[((size_t)c * 64 + it) * 16];
            if (r[0] == 0) continue;
            {
              std::fprintf(f, "%d,%d", c, it);
              for (int k = 0; k < 16; ++k) std::fprintf(f, ",%llu", r[k]);
              std::fprintf(f, "\n");
            }
          }
        std::fclose(f);
      }
      return rc;
    }
    if (!profile) return launch();
    cudaEvent_t e0, e1;
    NOPE_CUDA(cudaEventCreate(&e0));
    NOPE_CUDA(cudaEventCreate(&e1));
    NOPE_CUDA(cudaEventRecord(e0, st));
    const int rc = launch();
    NOPE_CUDA(cudaEventRecord(e1, st));
    prof_ev.push_back(e0);
    prof_ev.push_back(e1);
    // executed FLOPs: mode 3 runs 4 parity GEMMs of K = 4 Cin over the source-resolution pixels;
    // the split-precision modes execute 2x / 3x the K-steps of the fp16 mode
    prof_flops.push_back(2.0 * (double)n_img * So * So * (double)L.cout * (double)ksteps * 64.0);
    prof_alg.push_back(2.0 * (double)n_img * So * So * (double)L.cout * (double)L.K);
    return rc;
  }
  std::vector<double> prof_alg;     // algorithmic (fp16-mode) FLOPs of the same launches

  // pixel slabs per image for the GroupNorm kernels: as few as keep >= ~4 CTAs per SM in
  // flight (every CTA pays a fixed statistics prologue), at most 8, and >= 32 pixels each
  static int gn_nslab(int hw, int n_img) {
    int ns = 1;
    while (ns < 8 && hw / (ns * 2) >= 32 && (long long)n_img * ns < 600) ns *= 2;
    return ns;
  }

  // y = [silu](GN(x)) + pb[:, off:off+C] + res.  Statistics come from `stats`
  // ([img][st_parts][st_noct], see GnApplyArgs); stats == nullptr with N != nullptr runs the
  // stand-alone gn_stats_kernel first (per-op test path).  `emit` (optional) receives the
  // per-(img, slab) sums of y for a following GroupNorm(1, C).
  int gn(const NormLayer* N, const __half* x, __half* y, int S, int C, int n_img, bool silu,
         int pb_offset, const __half* res, const int* res_map, cudaStream_t st,
         const float2* stats = nullptr, int st_parts = 0, int st_noct = 0, float2* emit = nullptr) {
    const int hw = S * S;
    const int nslab = gn_nslab(hw, n_img);
    const int threads = (C / 8) * gn_rows(C);
    NOPE_CHECK(threads <= 1024 && threads % 32 == 0 && threads >= 256 && C % 8 == 0,
               "gn: unsupported channel count");
    if (N) {
      NOPE_CHECK(N->C == C, "gn: channel mismatch");
      if (!stats) {
        gn_stats_kernel<<<dim3(nslab, n_img), threads, threads * sizeof(float2), st>>>(
            x, gn_partial, hw, C, N->G, nslab);
        NOPE_CUDA(cudaGetLastError());
        ++launches;
        stats = gn_partial;
        st_parts = nslab;
        st_noct = N->G;
      }
      NOPE_CHECK(st_noct % N->G == 0, "gn: statistics granularity does not match the groups");
    }
    GnApplyArgs a;
    a.x = x; a.y = y; a.stats = N ? stats : nullptr; a.st_parts = st_parts; a.st_noct = st_noct;
    a.gamma = N ? N->gamma : nullptr; a.beta = N ? N->beta : nullptr;
    a.pb = pb_offset >= 0 ? pb : nullptr; a.pb_stride = P; a.pb_off = pb_offset >= 0 ? pb_offset : 0;
    a.res = res; a.res_of = res_map; a.emit = emit; a.emit_parts = emit_parts_of(hw);
    a.hw = hw; a.C = C; a.G = N ? N->G : 1; a.nslab = nslab;
    a.silu = silu ? 1 : 0; a.eps = 1e-5f; a.bf16 = bf() ? 1 : 0;
    NOPE_CUDA(launch_gn_apply(a, dim3(nslab, n_img), threads, st));
    ++launches;
    return 0;
  }
  static int st_parts_of(int S) { return S * S < 32 ? 1 : S * S / 32; }
  // fixed number of sub-slabs per image for statistics emitted by gn_apply (<= 8, >= 32 pixels
  // each): independent of the number of images, so results do not depend on chunk / shard size
  static int emit_parts_of(int hw) { return hw >= 256 ? 8 : (hw >= 32 ? hw / 32 : 1); }
  // partial sums per image emitted by the fused epilogue: one per (M-tile of the image, N-tile)
  static int fused_emit_parts(int S, int C) {
    return std::max(1, S * S / kBM) * (C / pick_bn(C));
  }

  int tap(const char* name, const Act& buf, int C, int S, int n, cudaStream_t st) {
    if (tap_out == nullptr || tap_name != name || tap_hit) return 0;
    NOPE_CHECK((int64_t)n * C * S * S <= tap_cap, "debug tap: output buffer too small");
    nhwc_f16_to_nchw_f32_kernel<<<ew_grid((long long)n * C * S * S), 256, 0, st>>>(buf.hi, tap_out, n, C, S * S,
                                                                                   buf.lo, bf());
    NOPE_CUDA(cudaGetLastError());
    tap_C = C; tap_S = S; tap_hit = true;
    return 0;
  }

  // ResnetBlock.forward (model_utils.py:271-279) on NHWC fp16.
  // Fused schedule: conv1 [GN8 + SiLU + pose bias] -> h ; (res_conv) ; conv2 [GN8 + SiLU + residual] -> out:
  // two or three launches, no tensor is written un-normalised.  `emit_g1` makes conv2's epilogue also
  // emit the GroupNorm(1, C) statistics of the block output into SB for a following attention pre-norm.
  // Unfused schedule (conv_impl 0 / 1 or fuse_gn off): GroupNorm statistics ride on the conv epilogues
  // (SA) and gn_apply_kernel normalises in a separate pass.
  int resblock(const std::string& p, const Act& in0, const Act& in1, const Act& out, int S, int n, bool pose,
               cudaStream_t st, bool emit_g1 = false, int res_div = 0, int res_base = 0, const Act* hoisted_h = nullptr) {
    const ConvLayer& b1 = convs.at(p + ".block1");
    const ConvLayer& b2 = convs.at(p + ".block2");
    const int co = b1.cout;
    const int parts = st_parts_of(S);
    auto it = convs.find(p + ".res");
    if (fused()) {
      Act h(TB.hi, co, h_lo() ? TB.lo : nullptr);
      if (hoisted_h) {
        h = *hoisted_h;
        if (!h_lo()) h.lo = nullptr;
      } else {
        GnSpec s1;
        s1.norm = &norms.at(p + ".norm1");
        s1.silu = true;
        s1.pb_offset = pose ? pb_off.at(p) : -1;
        if (conv(b1, in0, in1, h, S, n, cap, st, nullptr, &s1)) return -1;
      }
      GnSpec s2;
      s2.norm = &norms.at(p + ".norm2");
      s2.silu = true;
      if (it != convs.end()) {
        Act r(TC.hi, co, split() ? TC.lo : nullptr);
        // (routing this plain 1x1 through the EPI 4 role split measured 8 % slower than the plain epilogue:
        // NOPE_PLAIN_EPI4=1 is the A/B switch)
        static const bool plain_via_gn = std::getenv("NOPE_PLAIN_EPI4") && std::atoi(std::getenv("NOPE_PLAIN_EPI4"));
        GnSpec s0;
        if (conv(it->second, in0, in1, r, S, n, cap, st, nullptr, plain_via_gn ? &s0 : nullptr)) return -1;
        s2.res = r;
      } else {
        NOPE_CHECK(in1.hi == nullptr && in0.C == co, "resblock: identity residual needs Cin == Cout");
        s2.res = in0;
        s2.res_div = res_div;
        s2.res_base = res_base;
      }
      s2.emit = emit_g1 ? SB : nullptr;
      return conv(b2, h, Act(), out, S, n, cap, st, nullptr, &s2);
    }
    NOPE_CHECK(!hoisted_h && res_div == 0, "resblock: hoisting arguments belong to the fused schedule");
    if (conv(b1, in0, in1, Act(TA.hi, co), S, n, cap, st, SA)) return -1;
    if (gn(&norms.at(p + ".norm1"), TA.hi, TB.hi, S, co, n, true, pose ? pb_off.at(p) : -1, nullptr, nullptr, st,
           SA, parts, co / 8))
      return -1;
    if (conv(b2, Act(TB.hi, co), Act(), Act(TA.hi, co), S, n, cap, st, SA)) return -1;
    const __half* res = in0.hi;
    if (it != convs.end()) {
      if (conv(it->second, in0, in1, Act(TC.hi, co), S, n, cap, st)) return -1;
      res = TC.hi;
    } else {
      NOPE_CHECK(in1.hi == nullptr && in0.C == co, "resblock: identity residual needs Cin == Cout");
    }
    return gn(&norms.at(p + ".norm2"), TA.hi, out.hi, S, co, n, true, -1, res, nullptr, st, SA, parts, co / 8,
              emit_g1 ? SB : nullptr);
  }

  // Residual(PreNorm(LinearAttention)) (model_utils.py:393-418).  x's GroupNorm(1) statistics
  // were emitted into SB by the producer of x; to_out[1] (GroupNorm(1)) + the residual add run in the
  // to_out convolution's epilogue (fused) or come from its epilogue statistics (unfused).
  int linattn(const std::string& p, const Act& x, const Act& out, int C, int S, int n, cudaStream_t st) {
    const int eparts = fused() ? fused_emit_parts(S, C) : emit_parts_of(S * S);
    if (fused()) {
      // pre-norm folded into to_qkv: x is read once, un-normalised, by the 1x1 itself
      GnSpec s;
      s.pre_stats = SB;
      s.pre_parts = eparts;
      if (conv(convs.at(p + ".qkvf"), x, Act(), Act(TD.hi, 3 * kHeadsHidden), S, n, cap, st, nullptr, &s)) return -1;
    } else {
      if (gn(&norms.at(p + ".prenorm"), x.hi, TB.hi, S, C, n, false, -1, nullptr, nullptr, st, SB, eparts, 1))
        return -1;
      if (conv(convs.at(p + ".qkv"), Act(TB.hi, C), Act(), Act(TD.hi, 3 * kHeadsHidden), S, n, cap, st)) return -1;
    }
    if (attn_impl == 0 && S * S >= kBM) {
      if (launch_linattn_tc(TD.hi, TC.hi, n, S * S, num_sms, st, bf())) return -1;
    } else {
      NOPE_CUDA(launch_pdl(linattn_kernel, dim3(4, n), dim3(kLinAttnThreads), 0, st, TD.hi, TC.hi, S * S, bf()));
    }
    ++launches;
    // to_out (K = 128: two K-steps per tile) + GroupNorm(1) + residual in one kernel.  With the lock-step epilogue
    // this measured slower than the plain convolution plus one normalisation pass (319 vs 244 us at 32x32); with the
    // role-split epilogue the two forms take the same time (18.80 vs 18.71 ms over the step under ncu) and the fused
    // one never rounds the un-normalised output to 16 bits (full-size configs[2] scores: 0.99e-3 vs 1.06e-3), so it is
    // the default; NOPE_FUSE_TO_OUT=0 restores conv + gn_apply for A/B
    static const bool fuse_to_out = !(std::getenv("NOPE_FUSE_TO_OUT") && !std::atoi(std::getenv("NOPE_FUSE_TO_OUT")));
    if (fused() && (split() || fuse_to_out)) {
      GnSpec s;
      s.norm = &norms.at(p + ".outnorm");
      s.res = x;
      return conv(convs.at(p + ".out"), Act(TC.hi, kHeadsHidden), Act(), out, S, n, cap, st, nullptr, &s);
    }
    if (conv(convs.at(p + ".out"), Act(TC.hi, kHeadsHidden), Act(), Act(TA.hi, C), S, n, cap, st, SA)) return -1;
    return gn(&norms.at(p + ".outnorm"), TA.hi, out.hi, S, C, n, false, -1, x.hi, nullptr, st, SA, st_parts_of(S),
              C / 8);
  }

  // Residual(PreNorm(Attention)) (model_utils.py:367-390)
  int midattn(const Act& x, const Act& out, int C, int S, int n, cudaStream_t st) {
    NOPE_CHECK(S * S <= 32, "bottleneck attention supports at most 32 tokens");
    const int eparts = fused() ? fused_emit_parts(S, C) : emit_parts_of(S * S);
    if (fused()) {
      GnSpec s;
      s.pre_stats = SB;
      s.pre_parts = eparts;
      if (conv(convs.at("mid_attn.qkvf"), x, Act(), Act(TD.hi, 3 * kHeadsHidden), S, n, cap, st, nullptr, &s)) return -1;
    } else {
      if (gn(&norms.at("mid_attn.prenorm"), x.hi, TB.hi, S, C, n, false, -1, nullptr, nullptr, st, SB, eparts, 1))
        return -1;
      if (conv(convs.at("mid_attn.qkv"), Act(TB.hi, C), Act(), Act(TD.hi, 3 * kHeadsHidden), S, n, cap, st)) return -1;
    }
    NOPE_CUDA(launch_pdl(midattn_kernel, dim3(n), dim3(128), 0, st, TD.hi, TC.hi, S * S, bf()));
    ++launches;
    if (fused()) {
      GnSpec s;                // no normalisation: out = to_out(attn) + x
      s.res = x;
      return conv(convs.at("mid_attn.out"), Act(TC.hi, kHeadsHidden), Act(), out, S, n, cap, st, nullptr, &s);
    }
    if (conv(convs.at("mid_attn.out"), Act(TC.hi, kHeadsHidden), Act(), Act(TA.hi, C), S, n, cap, st)) return -1;
    return gn(nullptr, TA.hi, out.hi, S, C, n, false, -1, x.hi, nullptr, st);
  }

  // pose-independent prefix, once per reference image: x0 = init_conv(ref),
  // g1 = SiLU(GN(downs.0.0.block1.proj(x0)))   (u_net.py:161; model_utils.py:272)
  int prestage(const float* ref_feat, int B, cudaStream_t st) {
    init_conv_kernel<<<ew_grid((long long)B * S0 * S0 * dim), 256, 0, st>>>(ref_feat, init_w, init_b, x0.hi,
                                                                            B, Cl, S0, S0, dim, split() ? x0.lo : nullptr, bf());
    NOPE_CUDA(cudaGetLastError());
    ++launches;
    const Act xin(x0.hi, dim, split() ? x0.lo : nullptr);
    if (fused()) {
      GnSpec s;
      s.norm = &norms.at("downs.0.0.norm1");
      s.silu = true;
      return conv(convs.at("downs.0.0.block1"), xin, Act(), Act(g1.hi, dim, h_lo() ? g1.lo : nullptr), S0, B,
                  cap_ref, st, nullptr, &s);
    }
    if (conv(convs.at("downs.0.0.block1"), xin, Act(), Act(pt, dim), S0, B, cap_ref, st, SA)) return -1;
    return gn(&norms.at("downs.0.0.norm1"), pt, g1.hi, S0, dim, B, true, -1, nullptr, nullptr, st, SA,
              st_parts_of(S0), dim / 8);
  }

  // UNet.forward for hypotheses [hyp0, hyp0 + n) of the flattened (b, pose) list
  int forward_chunk(const float* poses, int hyp0, int n, int N, const float* query_feat,
                    float* out_emb, float* score_part, cudaStream_t st) {
    const bool sp = split();
    auto A = [&](const Act& buf, int C) { return Act(buf.hi, C, sp ? buf.lo : nullptr); };
    // hypothesis -> reference image
    iota_div(ref_of, hyp0, N, n, st);
    // pose embedding + all 19 pose projections in one GEMM
    NOPE_CUDA(launch_pdl(pose_embed_kernel, dim3(n), dim3(256), 0, st, poses + (size_t)hyp0 * rot_dim, pose_w, pose_b,
                         cs, n, rot_dim, cemb, bf()));
    ++launches;
    if (conv_pose(n, st)) return -1;

    // r (= init_conv output) and the hoisted block1 output, broadcast per hypothesis
    const int hw0 = S0 * S0;
    NOPE_CUDA(launch_pdl(bcast_add_kernel, dim3(ew_grid((long long)hw0 * dim / 8 / 4), n), dim3(256), 0, st, x0.hi, ref_of,
                         nullptr, 0, 0, RB.hi, n, hw0, dim, sp ? x0.lo : nullptr, sp ? RB.lo : nullptr, bf()));
    NOPE_CUDA(launch_pdl(bcast_add_kernel, dim3(ew_grid((long long)hw0 * dim / 8 / 4), n), dim3(256), 0, st, g1.hi, ref_of,
                         pb, P, pb_off.at("downs.0.0"), TB.hi, n, hw0, dim, h_lo() ? g1.lo : nullptr,
                         h_lo() ? TB.lo : nullptr, bf()));
    launches += 2;
    if (tap("init_conv", A(RB, dim), dim, S0, n, st)) return -1;

    // ---- downs
    Act cur;
    int S = S0;
    for (int i = 0; i < 4; ++i) {
      const int C = dims[i];
      const std::string p = "downs." + std::to_string(i);
      const Act s0 = A(sk[i][0], C), s1 = A(sk[i][1], C);
      if (i == 0) {
        // block 0 with its block1 half hoisted: TB already holds SiLU(GN(conv(x0))) + pose bias
        if (fused()) {
          const Act h = A(TB, C);
          if (resblock(p + ".0", A(x0, C), Act(), s0, S, n, true, st, false, N, hyp0, &h)) return -1;
        } else {
          if (conv(convs.at(p + ".0.block2"), Act(TB.hi, C), Act(), Act(TA.hi, C), S, n, cap, st, SA)) return -1;
          if (gn(&norms.at(p + ".0.norm2"), TA.hi, s0.hi, S, C, n, true, -1, x0.hi, ref_of, st, SA,
                 st_parts_of(S), C / 8))
            return -1;
        }
      } else {
        if (resblock(p + ".0", cur, Act(), s0, S, n, true, st)) return -1;
      }
      if (tap((p + ".0").c_str(), s0, C, S, n, st)) return -1;
      if (resblock(p + ".1", s0, Act(), A(XA, C), S, n, true, st, true)) return -1;
      if (tap((p + ".1").c_str(), A(XA, C), C, S, n, st)) return -1;
      if (linattn(p + ".2", A(XA, C), s1, C, S, n, st)) return -1;
      if (tap((p + ".2").c_str(), s1, C, S, n, st)) return -1;
      if (i < 3) S >>= 1;
      if (conv(convs.at(p + ".3"), s1, Act(), A(XB, dims[i + 1]), S, n, cap, st)) return -1;
      if (tap((p + ".3").c_str(), A(XB, dims[i + 1]), dims[i + 1], S, n, st)) return -1;
      cur = A(XB, dims[i + 1]);
    }
    // ---- mid, twice with shared weights (u_net.py:177-183)
    const int Cm = dims[4];
    Act xa = XA, xb = XB;
    for (int rep = 0; rep < 2; ++rep) {
      if (resblock("mid_block1", A(xb, Cm), Act(), A(xa, Cm), S, n, true, st, true)) return -1;
      if (midattn(A(xa, Cm), A(xb, Cm), Cm, S, n, st)) return -1;
      if (resblock("mid_block2", A(xb, Cm), Act(), A(xa, Cm), S, n, true, st)) return -1;
      if (tap(rep == 0 ? "mid.0" : "mid.1", A(xa, Cm), Cm, S, n, st)) return -1;
      std::swap(xa, xb);
    }
    Act curb = xb, othb = xa;     // buffers (channel counts vary per level)
    // ---- ups
    int ccur = Cm;
    for (int j = 0; j < 4; ++j) {
      const int din = dims[3 - j], dout = dims[4 - j];
      const std::string p = "ups." + std::to_string(j);
      if (resblock(p + ".0", A(curb, dout), A(sk[3 - j][1], din), A(othb, dout), S, n, true, st)) return -1;
      std::swap(curb, othb);
      if (tap((p + ".0").c_str(), A(curb, dout), dout, S, n, st)) return -1;
      if (resblock(p + ".1", A(curb, dout), A(sk[3 - j][0], din), A(othb, dout), S, n, true, st, true)) return -1;
      std::swap(curb, othb);
      if (linattn(p + ".2", A(curb, dout), A(othb, dout), dout, S, n, st)) return -1;
      std::swap(curb, othb);
      if (tap((p + ".2").c_str(), A(curb, dout), dout, S, n, st)) return -1;
      if (j < 3) S <<= 1;   // folded nearest-x2 + conv3x3: reads `cur` at S/2, writes `oth` at S
      if (conv(convs.at(p + ".3"), A(curb, dout), Act(), A(othb, din), S, n, cap, st)) return -1;
      std::swap(curb, othb);
      ccur = din;
      if (tap((p + ".3").c_str(), A(curb, din), din, S, n, st)) return -1;
    }
    // ---- head
    if (resblock("final_res_block", A(curb, ccur), A(RB, dim), A(othb, dim), S, n, true, st)) return -1;
    std::swap(curb, othb);
    if (tap("final_res_block", A(curb, dim), dim, S, n, st)) return -1;
    if (resblock("final_conv.0", A(curb, dim), Act(), A(othb, dim), S, n, false, st)) return -1;
    std::swap(curb, othb);
    if (tap("final_conv.0", A(curb, dim), dim, S, n, st)) return -1;
    const int hw = S * S;
    const int nslab = (hw + kFinalPix - 1) / kFinalPix;
    NOPE_CUDA(launch_pdl(final_conv_score_kernel, dim3(nslab, n), dim3(kFinalThreads), (size_t)kMaxLatent * dim * sizeof(float),
                         st, curb.hi, final_w, final_b, out_emb ? out_emb + (size_t)hyp0 * Cl * hw : nullptr, query_feat,
                         ref_of, score_part ? score_part + (size_t)hyp0 * nslab * kScoreParts : nullptr, hw, dim, Cl,
                         sp ? curb.lo : nullptr, metric, occ_threshold, bf()));
    ++launches;
    return 0;
  }

  int iota_div(int* r, int h0, int N, int n, cudaStream_t st);
  int conv_pose(int n, cudaStream_t st) {
    // pb[n, P] = cs[n, cemb] @ Wp^T + bp : the 1x1 "image" geometry of the conv kernel
    return conv(poseproj, Act(cs, cemb), Act(), Act(pb, P), 1, n, cap, st);
  }
};

namespace {
__global__ void iota_div_kernel(int* r, int h0, int N, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) r[i] = (h0 + i) / N;
}
}  // namespace

int nope_unet::iota_div(int* r, int h0, int N, int n, cudaStream_t st) {
  iota_div_kernel<<<(n + 255) / 256, 256, 0, st>>>(r, h0, N, n);
  ++launches;
  return 0;
}

namespace {
struct Scratch {
  std::vector<void*> p;
  ~Scratch() { for (void* q : p) cudaFree(q); }
  template <typename T> int get(T** out, size_t n) {
    NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(out), std::max<size_t>(n, 1) * sizeof(T)));
    p.push_back(*out);
    return 0;
  }
};
int to_nhwc(const float* x, __half** out, Scratch& s, int n, int C, int hw, cudaStream_t st,
            __half** out_lo = nullptr) {
  if (s.get(out, (size_t)n * C * hw)) return -1;
  if (out_lo && s.get(out_lo, (size_t)n * C * hw)) return -1;
  nchw_f32_to_nhwc_f16_kernel<<<ew_grid((long long)n * C * hw), 256, 0, st>>>(x, *out, n, C, hw,
                                                                              out_lo ? *out_lo : nullptr);
  NOPE_CUDA(cudaGetLastError());
  return 0;
}
int to_nchw(const __half* x, float* out, int n, int C, int hw, cudaStream_t st, const __half* x_lo = nullptr) {
  nhwc_f16_to_nchw_f32_kernel<<<ew_grid((long long)n * C * hw), 256, 0, st>>>(x, out, n, C, hw, x_lo);
  NOPE_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace

// =============================================================================
// C ABI
// =============================================================================
extern "C" {

const char* nope_last_error(void) { return last_error().c_str(); }
int nope_abi_version(void) { return kAbiVersion; }
const char* nope_build_arch(void) { return "sm_100a"; }

int nope_unet_create(nope_unet_t** out, int u_net_dim, int latent_ch, int latent_hw, int device) {
  NOPE_CHECK(out != nullptr, "null out pointer");
  NOPE_CHECK(u_net_dim > 0 && u_net_dim % 64 == 0, "u_net_dim must be a positive multiple of 64");
  NOPE_CHECK(latent_ch >= 1 && latent_ch <= kMaxLatent, "latent_ch must be in [1, 8]");
  NOPE_CHECK(latent_hw == 32, "latent_hw must be 32 (256x256 images) in this build");
  int ndev = 0;
  NOPE_CUDA(cudaGetDeviceCount(&ndev));
  NOPE_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  cudaDeviceProp prop;
  NOPE_CUDA(cudaGetDeviceProperties(&prop, device));
  NOPE_CHECK(prop.major == 10, "nope_b200 kernels are built for sm_100a only");
  auto u = std::make_unique<nope_unet>();
  u->dim = u_net_dim;
  u->Cl = latent_ch;
  u->S0 = latent_hw;
  u->cemb = 4 * u_net_dim;
  u->device = device;
  u->num_sms = prop.multiProcessorCount;
  const int mults[4] = {1, 2, 4, 8};
  u->dims[0] = u_net_dim;
  for (int i = 0; i < 4; ++i) u->dims[i + 1] = u_net_dim * mults[i];
  u->build_schema();
  *out = u.release();
  return 0;
}

void nope_unet_destroy(nope_unet_t* u) { delete u; }

int nope_unet_load_tensor(nope_unet_t* u, const char* key, const float* data, const int64_t* shape,
                          int ndim) {
  NOPE_CHECK(u && key && data && shape, "null argument");
  NOPE_CHECK(!u->finalized, "engine already finalized");
  auto it = u->expected.find(key);
  NOPE_CHECK(it != u->expected.end(), std::string("unexpected state_dict key: ") + key);
  NOPE_CHECK((int)it->second.size() == ndim, std::string("rank mismatch for ") + key);
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    NOPE_CHECK(it->second[i] == shape[i], std::string("shape mismatch for ") + key);
    n *= (size_t)shape[i];
  }
  HostTensor t;
  t.shape.assign(shape, shape + ndim);
  t.data.assign(data, data + n);
  u->host[key] = std::move(t);
  return 0;
}

int nope_unet_finalize(nope_unet_t* u) {
  NOPE_CHECK(u, "null engine");
  return u->finalize();
}

int nope_unet_set_chunk(nope_unet_t* u, int hyps) {
  NOPE_CHECK(u && hyps >= 1 && hyps <= 4096, "chunk must be in [1, 4096]");
  u->chunk = hyps;
  return 0;
}
int nope_unet_set_conv_impl(nope_unet_t* u, int impl) {
  NOPE_CHECK(u && impl >= 0 && impl <= 2, "impl must be 0 (tcgen05), 1 (simt) or 2 (tcgen05 2-CTA)");
  NOPE_CHECK(impl != 1 || u->precision == 0, "the SIMT debug convolution only runs fp16 weights");
  u->conv_impl = impl;
  return 0;
}
int nope_unet_set_option(nope_unet_t* u, const char* name, int value) {
  NOPE_CHECK(u && name, "null argument");
  if (std::strcmp(name, "fuse_gn") == 0) {
    NOPE_CHECK(value != 0 || u->precision < 2, "split precision / bf16 need the fused GroupNorm epilogue");
    u->fuse_gn = value != 0;
    return 0;
  }
  if (std::strcmp(name, "precision") == 0) {
    NOPE_CHECK(!u->finalized, "precision must be set before nope_unet_finalize");
    NOPE_CHECK(value == 0 || u->conv_impl != 1, "the SIMT debug convolution only runs fp16 weights");
    NOPE_CHECK(value >= 0 && value <= 4, "precision must be 0 (fp16), 1 (exact weights), 2 (split), 3 (bf16) or 4 (split, fp16 inside ResnetBlocks)");
    u->precision = value;
    return 0;
  }
  if (std::strcmp(name, "conv_impl") == 0) return nope_unet_set_conv_impl(u, value);
  if (std::strcmp(name, "attn_impl") == 0) {
    NOPE_CHECK(value == 0 || value == 1, "attn_impl must be 0 (tcgen05) or 1 (CUDA cores)");
    u->attn_impl = value;
    return 0;
  }
  return fail(std::string("unknown option: ") + name);
}
int nope_unet_get_option(const nope_unet_t* u, const char* name, int* value) {
  NOPE_CHECK(u && name && value, "null argument");
  if (std::strcmp(name, "fuse_gn") == 0) { *value = u->fuse_gn ? 1 : 0; return 0; }
  if (std::strcmp(name, "precision") == 0) { *value = u->precision; return 0; }
  if (std::strcmp(name, "conv_impl") == 0) { *value = u->conv_impl; return 0; }
  if (std::strcmp(name, "attn_impl") == 0) { *value = u->attn_impl; return 0; }
  return fail(std::string("unknown option: ") + name);
}
int64_t nope_unet_last_launch_count(const nope_unet_t* u) { return u ? u->launches : 0; }

int64_t nope_unet_workspace_bytes(nope_unet_t* u, int hyps, int refs, int scores) {
  if (!u || !u->finalized || hyps < 1 || refs < 1 || scores < 0) {
    fail("nope_unet_workspace_bytes: finalized engine, hyps >= 1, refs >= 1 required");
    return -1;
  }
  return (int64_t)u->workspace_bytes(hyps, refs, scores);
}
int nope_unet_set_workspace(nope_unet_t* u, void* ptr, int64_t bytes, int hyps, int refs, int scores) {
  NOPE_CHECK(u && u->finalized, "engine not finalized");
  NOPE_CUDA(cudaSetDevice(u->device));
  return u->set_workspace(ptr, (size_t)bytes, hyps, refs, scores);
}

int nope_unet_profile(nope_unet_t* u, int enable) {
  NOPE_CHECK(u, "null engine");
  for (cudaEvent_t e : u->prof_ev) cudaEventDestroy(e);
  u->prof_ev.clear();
  u->prof_flops.clear();
  u->prof_alg.clear();
  u->profile = enable != 0;
  return 0;
}

int nope_unet_profile_read(nope_unet_t* u, double* conv_ms, double* conv_flops, double* conv_alg_flops,
                           int64_t* conv_launches, double* max_launch_tflops) {
  NOPE_CHECK(u && conv_ms && conv_flops && conv_launches, "null argument");
  NOPE_CUDA(cudaDeviceSynchronize());
  double ms = 0.0, fl = 0.0, alg = 0.0, best = 0.0;
  for (size_t i = 0; i < u->prof_flops.size(); ++i) {
    float t = 0.f;
    NOPE_CUDA(cudaEventElapsedTime(&t, u->prof_ev[2 * i], u->prof_ev[2 * i + 1]));
    ms += t;
    fl += u->prof_flops[i];
    alg += u->prof_alg[i];
    if (t > 0.f) best = std::max(best, u->prof_flops[i] / (t * 1e-3) / 1e12);
  }
  if (const char* path = std::getenv("NOPE_PROF_DUMP")) {     // development aid: per-launch table
    if (FILE* f = std::fopen(path, "a")) {
      std::fprintf(f, "# launch,ms,executed_gflop,algorithmic_gflop\n");
      for (size_t i = 0; i < u->prof_flops.size(); ++i) {
        float t = 0.f;
        cudaEventElapsedTime(&t, u->prof_ev[2 * i], u->prof_ev[2 * i + 1]);
        std::fprintf(f, "%zu,%.4f,%.3f,%.3f\n", i, t, u->prof_flops[i] / 1e9, u->prof_alg[i] / 1e9);
      }
      std::fclose(f);
    }
  }
  *conv_ms = ms;
  *conv_flops = fl;
  if (conv_alg_flops) *conv_alg_flops = alg;
  *conv_launches = (int64_t)u->prof_flops.size();
  if (max_launch_tflops) *max_launch_tflops = best;
  return 0;
}

int nope_unet_sweep(nope_unet_t* u, const float* ref_feat, const float* poses, int B, int N,
                    const float* query_feat, float* out_emb, float* out_sim, int k, float* out_topv,
                    int64_t* out_topi, int64_t idx_base, void* stream) {
  NOPE_CHECK(u && u->finalized, "engine not finalized");
  NOPE_CHECK(ref_feat && poses && B >= 1 && N >= 1, "bad arguments");
  NOPE_CHECK(!(out_sim || k > 0) || query_feat, "scores / top-k need query_feat");
  NOPE_CHECK(k >= 0 && k <= N && k <= 64, "k must be in [0, min(N, 64)]");
  NOPE_CHECK(k == 0 || (out_topv && out_topi), "top-k outputs missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CUDA(cudaSetDevice(u->device));
  u->launches = 0;
  const int total = B * N;
  const int cap = std::min(u->chunk, total);
  // no allocation here when the caller provided the workspace (nope_unet_set_workspace); otherwise the
  // engine grows its own slab (device synchronisation + cudaMalloc on growth only)
  if (u->ensure_workspace(cap, B, query_feat ? total : 0)) return -1;
  if (u->prepare_stream(st)) return -1;
  const int hw = u->S0 * u->S0;
  const int nslab = (hw + kFinalPix - 1) / kFinalPix;
  float* part = query_feat ? u->score_partial : nullptr;
  if (u->prestage(ref_feat, B, st)) return -1;
  for (int h0 = 0; h0 < total; h0 += cap) {
    const int n = std::min(cap, total - h0);
    if (u->forward_chunk(poses, h0, n, N, query_feat, out_emb, part, st)) return -1;
  }
  if (query_feat && (out_sim || k > 0)) {
    float* sim = out_sim ? out_sim : u->sim_buf;
    NOPE_CUDA(launch_pdl(sim_topk_kernel, dim3(B), dim3(256), 0, st, part, nslab, sim, N, k, out_topv,
                         reinterpret_cast<long long*>(out_topi), (long long)idx_base, kScoreParts, u->metric, hw));
    ++u->launches;
  }
  return 0;
}

int nope_unet_set_metric(nope_unet_t* u, int metric, float occlusion_threshold) {
  NOPE_CHECK(u, "null engine");
  NOPE_CHECK(metric == NOPE_METRIC_L2 || metric == NOPE_METRIC_COSINE || metric == NOPE_METRIC_COSINE_OCC,
             "unknown similarity metric (l2, cosine and cosine_occlusion exist)");
  u->metric = metric;
  u->occ_threshold = occlusion_threshold;
  return 0;
}

int nope_score_topk(const float* query_feat, const float* emb, int B, int N, int C, int HW, int metric,
                    float occlusion_threshold, int k, float* out_sim, float* out_topv, int64_t* out_topi,
                    int64_t idx_base, void* stream) {
  NOPE_CHECK(query_feat && emb && out_sim, "null argument");
  NOPE_CHECK(metric == NOPE_METRIC_L2 || metric == NOPE_METRIC_COSINE || metric == NOPE_METRIC_COSINE_OCC,
             "unknown similarity metric (l2, cosine and cosine_occlusion exist)");
  NOPE_CHECK(k >= 0 && k <= N && k <= 64, "k must be in [0, min(N, 64)]");
  NOPE_CHECK(k == 0 || (out_topv && out_topi), "top-k outputs missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  score_kernel<<<dim3(N, B), 256, 0, st>>>(query_feat, emb, out_sim, N, C, HW, metric, occlusion_threshold);
  NOPE_CUDA(cudaGetLastError());
  if (k > 0) {
    sim_topk_kernel<<<B, 256, 0, st>>>(nullptr, 0, out_sim, N, k, out_topv,
                                       reinterpret_cast<long long*>(out_topi), (long long)idx_base);
    NOPE_CUDA(cudaGetLastError());
  }
  return 0;
}

int nope_topk(float* sim, int B, int N, int k, float* out_topv, int64_t* out_topi, int64_t idx_base,
              void* stream) {
  NOPE_CHECK(sim && out_topv && out_topi, "null argument");
  NOPE_CHECK(k >= 1 && k <= N && k <= 64, "k must be in [1, min(N, 64)]");
  sim_topk_kernel<<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      nullptr, 0, sim, N, k, out_topv, reinterpret_cast<long long*>(out_topi), (long long)idx_base);
  NOPE_CUDA(cudaGetLastError());
  return 0;
}

int64_t nope_topk_pack_floats(int B, int k, int n_local_max, int want_sim) {
  if (B < 1 || k < 1 || n_local_max < 0) return -1;
  const int64_t kk = ((int64_t)B * k + 1) & ~(int64_t)1;
  // rounded up to 4 floats: records sit back to back in the gathered buffer and every record's int64 block must
  // stay 8-byte aligned (an odd length misaligned every second record: 10 248 poses on 8 GPUs = 16 + 1281 floats)
  return (kk + 2 * (int64_t)B * k + (want_sim ? (int64_t)B * n_local_max : 0) + 3) & ~(int64_t)3;
}

int nope_topk_merge(const float* gathered, int world, int64_t pack_floats, int B, int k, int N, int per,
                    int has_sim, float* out_sim, float* out_topv, int64_t* out_topi, void* stream) {
  NOPE_CHECK(gathered && out_topv && out_topi, "null argument");
  NOPE_CHECK(world >= 1 && B >= 1 && k >= 1 && k <= N && world * k <= 1024, "bad merge geometry (world * k <= 1024)");
  NOPE_CHECK(per >= 1 && (int64_t)per * world >= N, "per-rank pose count does not cover the grid");
  NOPE_CHECK(pack_floats >= nope_topk_pack_floats(B, k, has_sim ? per : 0, has_sim) - 3, "packed record too short");
  NOPE_CHECK(pack_floats % 2 == 0 && (reinterpret_cast<uintptr_t>(gathered) & 7) == 0,
             "packed records must be 8-byte aligned: use nope_topk_pack_floats for the record length");
  NOPE_CHECK(!has_sim || out_sim, "similarity output missing");
  topk_merge_kernel<<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      gathered, world, (long long)pack_floats, B, k, N, per, has_sim, out_sim, out_topv,
      reinterpret_cast<long long*>(out_topi));
  NOPE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------
// template encoder
// ---------------------------------------------------------------------------------
int nope_encoder_create(nope_encoder_t** out, int descriptor_size, int device) {
  NOPE_CHECK(out != nullptr, "null out pointer");
  NOPE_CHECK(descriptor_size >= 1 && descriptor_size <= 64, "descriptor_size must be in [1, 64]");
  int ndev = 0;
  NOPE_CUDA(cudaGetDeviceCount(&ndev));
  NOPE_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  cudaDeviceProp prop;
  NOPE_CUDA(cudaGetDeviceProperties(&prop, device));
  NOPE_CHECK(prop.major == 10, "nope_b200 kernels are built for sm_100a only");
  auto e = std::make_unique<nope_encoder>();
  e->D = descriptor_size;
  e->device = device;
  e->num_sms = prop.multiProcessorCount;
  e->build_schema();
  *out = e.release();
  return 0;
}

void nope_encoder_destroy(nope_encoder_t* e) { delete e; }

int nope_encoder_load_tensor(nope_encoder_t* e, const char* key, const float* data, const int64_t* shape,
                             int ndim) {
  NOPE_CHECK(e && key && data && shape, "null argument");
  NOPE_CHECK(!e->finalized, "encoder already finalized");
  auto it = e->expected.find(key);
  NOPE_CHECK(it != e->expected.end(), std::string("unexpected encoder state_dict key: ") + key);
  NOPE_CHECK((int)it->second.size() == ndim, std::string("rank mismatch for ") + key);
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    NOPE_CHECK(it->second[i] == shape[i], std::string("shape mismatch for ") + key);
    n *= (size_t)shape[i];
  }
  auto& slot = e->host[key];
  slot.first.assign(shape, shape + ndim);
  slot.second.assign(data, data + n);
  return 0;
}

int nope_encoder_finalize(nope_encoder_t* e) {
  NOPE_CHECK(e, "null encoder");
  return e->finalize();
}

int nope_encoder_encode(nope_encoder_t* e, const float* images, int B, float* out, void* stream) {
  NOPE_CHECK(e && e->finalized, "encoder not finalized");
  NOPE_CHECK(images && out, "null images / out pointer");
  NOPE_CHECK(B >= 1, "B must be >= 1");
  NOPE_CUDA(cudaSetDevice(e->device));
  // The workspace is sized by the largest chunk (~80 MB per image): any B goes through, 32 images at a time.
  constexpr int kChunk = 32;
  int64_t launches = 0;
  for (int lo = 0; lo < B; lo += kChunk) {
    const int n = B - lo < kChunk ? B - lo : kChunk;
    const int rc = e->encode(images + (size_t)lo * 3 * 256 * 256, n, out + (size_t)lo * e->D * 32 * 32,
                             static_cast<cudaStream_t>(stream));
    if (rc != 0) return rc;
    launches += e->launches;
  }
  e->launches = launches;
  return 0;
}

int64_t nope_encoder_last_launch_count(const nope_encoder_t* e) { return e ? e->launches : 0; }

// ---------------------------------------------------------------------------------
// per-op entry points
// ---------------------------------------------------------------------------------

int nope_op_conv(int impl, int mode, const float* x0, int C0, const float* x1, int C1,
                 const float* weight, const float* bias, float* out, int n_img, int H, int W,
                 int Cout, void* stream) {
  NOPE_CHECK(x0 && weight && out, "null argument");
  NOPE_CHECK(mode >= 0 && mode <= 3, "mode must be 0..3");
  NOPE_CHECK(H == W, "square images only");
  NOPE_CHECK(C0 % 64 == 0 && C1 % 64 == 0 && Cout % 64 == 0, "channels must be multiples of 64");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  const int taps = mode == 0 ? 9 : (mode == 1 ? 1 : 4);
  const int cin = C0 + (x1 ? C1 : 0);
  const int Hin = mode == 2 ? 2 * H : (mode == 3 ? H / 2 : H);
  const int rows = mode == 3 ? 4 * Cout : Cout;
  __half *a0 = nullptr, *a1 = nullptr, *wp = nullptr, *o = nullptr;
  if (to_nhwc(x0, &a0, s, n_img, C0, Hin * Hin, st)) return -1;
  if (x1 && to_nhwc(x1, &a1, s, n_img, C1, Hin * Hin, st)) return -1;
  if (s.get(&wp, (size_t)rows * cin * taps) || s.get(&o, (size_t)n_img * H * W * Cout)) return -1;
  const float* wsrc = weight;
  if (mode == 3) {
    float* folded = nullptr;
    if (s.get(&folded, (size_t)rows * cin * taps)) return -1;
    fold_upconv_kernel<<<ew_grid((long long)4 * Cout * cin), 256, 0, st>>>(weight, folded, Cout, cin);
    NOPE_CUDA(cudaGetLastError());
    wsrc = folded;
  }
  pack_weight_kernel<<<ew_grid((long long)rows * cin * taps), 256, 0, st>>>(wsrc, wp, rows, cin, taps,
                                                                           cin * taps, 0);
  NOPE_CUDA(cudaGetLastError());
  nope_unet eng;  // only used for its conv launcher / map cache
  eng.conv_impl = impl;
  cudaDeviceProp prop;
  int dev = 0;
  NOPE_CUDA(cudaGetDevice(&dev));
  NOPE_CUDA(cudaGetDeviceProperties(&prop, dev));
  eng.num_sms = prop.multiProcessorCount;
  ConvLayer L;
  L.mode = mode; L.cin = cin; L.cout = Cout; L.K = cin * taps; L.Kp = L.K; L.bn = pick_bn(Cout); L.w = wp;
  float* dbias = nullptr;
  if (bias) {
    if (s.get(&dbias, Cout)) return -1;
    NOPE_CUDA(cudaMemcpyAsync(dbias, bias, Cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  L.bias = dbias;
  if (impl != 1 && (make_weight_map(&L.wmap, wp, rows, L.K, L.bn) ||
                    make_weight_map(&L.wmap_half, wp, rows, L.K, L.bn / 2)))
    return -1;
  if (eng.conv(L, Act(a0, C0), x1 ? Act(a1, C1) : Act(), Act(o, Cout), H, n_img, n_img, st)) return -1;
  if (to_nchw(o, out, n_img, Cout, H * W, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_conv_gn(int impl, int mode, const float* x0, int C0, const float* x1, int C1,
                    const float* weight, const float* bias, const float* gamma, const float* beta,
                    int G, int silu, float* out, int n_img, int H, int W, int Cout, void* stream) {
  NOPE_CHECK(x0 && weight && gamma && beta && out, "null argument");
  NOPE_CHECK(mode >= 0 && mode <= 2 && H == W, "bad mode / non-square image");
  NOPE_CHECK(C0 % 64 == 0 && C1 % 64 == 0 && Cout % 64 == 0, "channels must be multiples of 64");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  const int taps = mode == 0 ? 9 : (mode == 1 ? 1 : 4);
  const int cin = C0 + (x1 ? C1 : 0);
  const int Hin = mode == 2 ? 2 * H : H;
  __half *a0 = nullptr, *a1 = nullptr, *wp = nullptr, *o = nullptr, *y = nullptr;
  if (to_nhwc(x0, &a0, s, n_img, C0, Hin * Hin, st)) return -1;
  if (x1 && to_nhwc(x1, &a1, s, n_img, C1, Hin * Hin, st)) return -1;
  if (s.get(&wp, (size_t)Cout * cin * taps) || s.get(&o, (size_t)n_img * H * W * Cout) ||
      s.get(&y, (size_t)n_img * H * W * Cout))
    return -1;
  pack_weight_kernel<<<ew_grid((long long)Cout * cin * taps), 256, 0, st>>>(weight, wp, Cout, cin, taps,
                                                                            cin * taps, 0);
  NOPE_CUDA(cudaGetLastError());
  nope_unet eng;
  eng.conv_impl = impl;
  cudaDeviceProp prop;
  int dev = 0;
  NOPE_CUDA(cudaGetDevice(&dev));
  NOPE_CUDA(cudaGetDeviceProperties(&prop, dev));
  eng.num_sms = prop.multiProcessorCount;
  ConvLayer L;
  L.mode = mode; L.cin = cin; L.cout = Cout; L.K = cin * taps; L.Kp = L.K; L.bn = pick_bn(Cout); L.w = wp;
  L.bias = const_cast<float*>(bias);
  if (impl != 1 && (make_weight_map(&L.wmap, wp, Cout, L.K, L.bn) ||
                    make_weight_map(&L.wmap_half, wp, Cout, L.K, L.bn / 2)))
    return -1;
  const int parts = nope_unet::st_parts_of(H);
  float2* stats = nullptr;
  if (s.get(&stats, (size_t)n_img * parts * (Cout / 8))) return -1;
  if (eng.conv(L, Act(a0, C0), x1 ? Act(a1, C1) : Act(), Act(o, Cout), H, n_img, n_img, st, stats)) return -1;
  NormLayer N;
  N.C = Cout; N.G = G;
  N.gamma = const_cast<float*>(gamma);
  N.beta = const_cast<float*>(beta);
  if (eng.gn(&N, o, y, H, Cout, n_img, silu != 0, -1, nullptr, nullptr, st, stats, parts, Cout / 8))
    return -1;
  if (to_nchw(y, out, n_img, Cout, H * W, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// The sweep's fused layer: out = [SiLU](GroupNorm_G(conv(x) + bias)) + chan_bias[n, c] + residual, all in the
// epilogue of the CTA-pair kernel (GnFuse).  precision 0 / 1 / 2 as nope_unet_set_option("precision"); with 2 the
// inputs and the residual are split into fp16 (hi, lo) pairs and the output is the sum of its pair.
int nope_op_conv_gn_fused(int mode, int precision, const float* x0, int C0, const float* x1, int C1,
                          const float* weight, const float* bias, const float* gamma, const float* beta, int G,
                          int silu, const float* chan_bias, const float* residual, int res_div, float* out,
                          float* emit_out, int n_img, int H, int W, int Cout, void* stream) {
  NOPE_CHECK(x0 && weight && out, "null argument");
  NOPE_CHECK(mode >= 0 && mode <= 2 && H == W, "bad mode / non-square image");
  NOPE_CHECK(precision >= 0 && precision <= 2, "precision must be 0..2");
  NOPE_CHECK(C0 % 64 == 0 && C1 % 64 == 0 && Cout % 64 == 0, "channels must be multiples of 64");
  NOPE_CHECK(G == 0 || (gamma && beta), "GroupNorm needs gamma / beta");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  const bool sp = precision == 2;
  const int taps = mode == 0 ? 9 : (mode == 1 ? 1 : 4);
  const int cin = C0 + (x1 ? C1 : 0);
  const int Hin = mode == 2 ? 2 * H : H;
  const int hw = H * W;
  __half *a0 = nullptr, *a0l = nullptr, *a1 = nullptr, *a1l = nullptr, *wp = nullptr, *o = nullptr, *ol = nullptr,
         *r = nullptr, *rl = nullptr, *pbh = nullptr;
  if (to_nhwc(x0, &a0, s, n_img, C0, Hin * Hin, st, sp ? &a0l : nullptr)) return -1;
  if (x1 && to_nhwc(x1, &a1, s, n_img, C1, Hin * Hin, st, sp ? &a1l : nullptr)) return -1;
  const int n_res = residual ? (res_div > 0 ? (n_img + res_div - 1) / res_div : n_img) : 0;
  if (residual && to_nhwc(residual, &r, s, n_res, Cout, hw, st, sp ? &rl : nullptr)) return -1;
  if (chan_bias && to_nhwc(chan_bias, &pbh, s, n_img, Cout, 1, st)) return -1;
  const int K = cin * taps, Kp = precision >= 1 ? 2 * K : K;
  if (s.get(&wp, (size_t)Cout * Kp) || s.get(&o, (size_t)n_img * hw * Cout)) return -1;
  if (sp && s.get(&ol, (size_t)n_img * hw * Cout)) return -1;
  pack_weight_kernel<<<ew_grid((long long)Cout * K), 256, 0, st>>>(weight, wp, Cout, cin, taps, Kp, 0,
                                                                    precision >= 1 ? K : 0);
  NOPE_CUDA(cudaGetLastError());
  nope_unet eng;
  eng.conv_impl = 2;
  eng.precision = precision;
  cudaDeviceProp prop;
  int dev = 0;
  NOPE_CUDA(cudaGetDevice(&dev));
  NOPE_CUDA(cudaGetDeviceProperties(&prop, dev));
  eng.num_sms = prop.multiProcessorCount;
  eng.device = dev;
  if (eng.ensure_workspace(n_img, std::max(n_res, 1))) return -1;
  if (eng.prepare_stream(st)) return -1;
  eng.pb = pbh;
  eng.P = Cout;
  ConvLayer L;
  L.mode = mode; L.cin = cin; L.cout = Cout; L.K = K; L.Kp = Kp; L.bn = pick_bn(Cout); L.w = wp;
  L.bias = const_cast<float*>(bias);
  if (make_weight_map(&L.wmap, wp, Cout, Kp, L.bn) || make_weight_map(&L.wmap_half, wp, Cout, Kp, L.bn / 2))
    return -1;
  NormLayer N;
  N.C = Cout; N.G = std::max(G, 1);
  N.gamma = const_cast<float*>(gamma);
  N.beta = const_cast<float*>(beta);
  GnSpec gs;
  gs.norm = G > 0 ? &N : nullptr;
  gs.silu = silu != 0;
  gs.pb_offset = chan_bias ? 0 : -1;
  if (residual) gs.res = Act(r, Cout, rl);
  gs.res_div = residual ? res_div : 0;
  float2* em = nullptr;
  const int eparts = nope_unet::fused_emit_parts(H, Cout);
  if (emit_out) {
    if (s.get(&em, (size_t)n_img * eparts)) return -1;
    gs.emit = em;
  }
  if (eng.conv(L, Act(a0, C0, a0l), x1 ? Act(a1, C1, a1l) : Act(), Act(o, Cout, ol), H, n_img,
               n_img, st, nullptr, &gs))
    return -1;
  if (to_nchw(o, out, n_img, Cout, hw, st, ol)) return -1;
  if (emit_out) {
    // fold the per-tile partials on the host side of the test: [n_img][eparts] -> [n_img][2]
    std::vector<float2> h((size_t)n_img * eparts);
    NOPE_CUDA(cudaStreamSynchronize(st));
    NOPE_CUDA(cudaMemcpy(h.data(), em, h.size() * sizeof(float2), cudaMemcpyDeviceToHost));
    std::vector<float> sums((size_t)n_img * 2, 0.f);
    for (int i = 0; i < n_img; ++i)
      for (int e2 = 0; e2 < eparts; ++e2) {
        sums[2 * i] += h[(size_t)i * eparts + e2].x;
        sums[2 * i + 1] += h[(size_t)i * eparts + e2].y;
      }
    NOPE_CUDA(cudaMemcpy(emit_out, sums.data(), sums.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_groupnorm(const float* x, const float* gamma, const float* beta, int G, int silu,
                      const float* chan_bias, const float* residual, float* out, int n_img, int C,
                      int H, int W, void* stream) {
  NOPE_CHECK(x && gamma && beta && out && H == W, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  const int hw = H * W;
  __half *a = nullptr, *r = nullptr, *o = nullptr, *pbh = nullptr;
  if (to_nhwc(x, &a, s, n_img, C, hw, st)) return -1;
  if (residual && to_nhwc(residual, &r, s, n_img, C, hw, st)) return -1;
  if (chan_bias && to_nhwc(chan_bias, &pbh, s, n_img, C, 1, st)) return -1;
  if (s.get(&o, (size_t)n_img * C * hw)) return -1;
  nope_unet eng;
  if (s.get(&eng.gn_partial, (size_t)n_img * 64)) return -1;
  NormLayer N;
  N.C = C; N.G = G;
  N.gamma = const_cast<float*>(gamma);
  N.beta = const_cast<float*>(beta);
  eng.pb = pbh;
  eng.P = C;
  if (eng.gn(&N, a, o, H, C, n_img, silu != 0, chan_bias ? 0 : -1, r, nullptr, st)) return -1;
  if (to_nchw(o, out, n_img, C, hw, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_linear_attention(int impl, const float* qkv, float* out, int n_img, int H, int W, void* stream) {
  NOPE_CHECK(qkv && out, "null argument");
  NOPE_CHECK(impl == 1 || (impl == 0 && (H * W) % kBM == 0), "impl 0 (tcgen05) needs H*W % 128 == 0; impl 1 = CUDA cores");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  __half *a = nullptr, *o = nullptr;
  if (to_nhwc(qkv, &a, s, n_img, 384, H * W, st) || s.get(&o, (size_t)n_img * 128 * H * W)) return -1;
  if (impl == 0) {
    cudaDeviceProp prop;
    int dev = 0;
    NOPE_CUDA(cudaGetDevice(&dev));
    NOPE_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (launch_linattn_tc(a, o, n_img, H * W, prop.multiProcessorCount, st)) return -1;
  } else {
    linattn_kernel<<<dim3(4, n_img), kLinAttnThreads, 0, st>>>(a, o, H * W);
  }
  NOPE_CUDA(cudaGetLastError());
  if (to_nchw(o, out, n_img, 128, H * W, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_attention(const float* qkv, float* out, int n_img, int H, int W, void* stream) {
  NOPE_CHECK(qkv && out && H * W <= 32, "bad argument (H*W must be <= 32)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  __half *a = nullptr, *o = nullptr;
  if (to_nhwc(qkv, &a, s, n_img, 384, H * W, st) || s.get(&o, (size_t)n_img * 128 * H * W)) return -1;
  midattn_kernel<<<n_img, 128, 0, st>>>(a, o, H * W);
  NOPE_CUDA(cudaGetLastError());
  if (to_nchw(o, out, n_img, 128, H * W, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_upsample2x(const float* x, float* out, int n_img, int C, int H, int W, void* stream) {
  NOPE_CHECK(x && out && C % 8 == 0 && H == W, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Scratch s;
  __half *a = nullptr, *o = nullptr;
  if (to_nhwc(x, &a, s, n_img, C, H * W, st) || s.get(&o, (size_t)n_img * C * H * W * 4)) return -1;
  upsample2x_kernel<<<ew_grid((long long)n_img * 4 * H * W * C / 8), 256, 0, st>>>(a, o, n_img, H, W, C);
  NOPE_CUDA(cudaGetLastError());
  if (to_nchw(o, out, n_img, C, 4 * H * W, st)) return -1;
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_unet_debug_tap(nope_unet_t* u, const float* ref_feat, const float* poses, int N, const char* tap,
                        float* out, int64_t out_capacity_floats, int* out_C, int* out_H, void* stream) {
  NOPE_CHECK(u && u->finalized && ref_feat && poses && tap && out, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CHECK(N <= u->chunk, "debug tap: N must fit one chunk");
  NOPE_CUDA(cudaSetDevice(u->device));
  if (u->ensure_workspace(N, 1)) return -1;
  if (u->prepare_stream(st)) return -1;
  u->tap_name = tap;
  u->tap_out = out;
  u->tap_cap = out_capacity_floats;
  u->tap_hit = false;
  int rc = u->prestage(ref_feat, 1, st);
  if (!rc) rc = u->forward_chunk(poses, 0, N, N, nullptr, nullptr, nullptr, st);
  u->tap_out = nullptr;
  if (rc) return rc;
  NOPE_CUDA(cudaStreamSynchronize(st));
  NOPE_CHECK(u->tap_hit, std::string("unknown tap name: ") + tap);
  if (out_C) *out_C = u->tap_C;
  if (out_H) *out_H = u->tap_S;
  return 0;
}

// ---------------------------------------------------------------------------------
// LDM variant
// ---------------------------------------------------------------------------------
int nope_ldm_create(nope_ldm_t** out, int model_channels, int context_dim, int latent_ch, int latent_hw,
                    int device) {
  NOPE_CHECK(out != nullptr, "null out pointer");
  NOPE_CHECK(model_channels > 0 && model_channels % 256 == 0 && model_channels <= 512,
             "model_channels must be 256 or 512 (GroupNorm(32) statistics ride on 8-channel octets)");
  NOPE_CHECK(context_dim >= 1, "context_dim must be positive");
  NOPE_CHECK(latent_ch >= 1 && latent_ch <= kMaxLatent, "latent_ch must be in [1, 8]");
  NOPE_CHECK(latent_hw == 32, "latent_hw must be 32 in this build");
  int ndev = 0;
  NOPE_CUDA(cudaGetDeviceCount(&ndev));
  NOPE_CHECK(device >= 0 && device < ndev, "no such CUDA device");
  cudaDeviceProp prop;
  NOPE_CUDA(cudaGetDeviceProperties(&prop, device));
  NOPE_CHECK(prop.major == 10, "nope_b200 kernels are built for sm_100a only");
  auto m = std::make_unique<nope_ldm>();
  m->mc = model_channels;
  m->ctx = context_dim;
  m->Cl = latent_ch;
  m->S0 = latent_hw;
  m->device = device;
  m->num_sms = prop.multiProcessorCount;
  m->build_plan();
  m->build_schema();
  *out = m.release();
  return 0;
}

void nope_ldm_destroy(nope_ldm_t* m) { delete m; }

int nope_ldm_load_tensor(nope_ldm_t* m, const char* key, const float* data, const int64_t* shape, int ndim) {
  NOPE_CHECK(m && key && data && shape, "null argument");
  NOPE_CHECK(!m->finalized, "engine already finalized");
  auto it = m->expected.find(key);
  NOPE_CHECK(it != m->expected.end(), std::string("unexpected state_dict key: ") + key);
  NOPE_CHECK((int)it->second.size() == ndim, std::string("rank mismatch for ") + key);
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    NOPE_CHECK(it->second[i] == shape[i], std::string("shape mismatch for ") + key);
    n *= (size_t)shape[i];
  }
  if (std::strncmp(key, "time_embed.", 11) == 0 || std::strstr(key, ".emb_layers.1.weight") ||
      std::strstr(key, ".attn2.to_q.") || std::strstr(key, ".attn2.to_k.") || std::strstr(key, ".norm2.")) {
    // accepted for schema compatibility, never read: emb = 0 (adapt_openaimodel.py:143-146) and
    // the one-token cross-attention does not depend on its queries / keys
    m->host[key] = nope_ldm::HostT{std::vector<int64_t>(shape, shape + ndim), {}};
    return 0;
  }
  auto& slot = m->host[key];
  slot.first.assign(shape, shape + ndim);
  slot.second.assign(data, data + n);
  return 0;
}

int nope_ldm_finalize(nope_ldm_t* m) {
  NOPE_CHECK(m, "null engine");
  return m->finalize();
}
int nope_ldm_set_chunk(nope_ldm_t* m, int hyps) {
  NOPE_CHECK(m && hyps >= 1 && hyps <= 2048, "chunk must be in [1, 2048]");
  m->chunk = hyps;
  return 0;
}
int nope_ldm_set_impl(nope_ldm_t* m, int conv_impl, int attn_impl) {
  NOPE_CHECK(m && (conv_impl == 0 || conv_impl == 2), "conv_impl must be 0 (tcgen05) or 2 (tcgen05 2-CTA)");
  NOPE_CHECK(attn_impl == 0 || attn_impl == 1, "attn_impl must be 0 (tcgen05) or 1 (CUDA cores)");
  m->conv_impl = conv_impl;
  m->attn_impl = attn_impl;
  return 0;
}
int nope_ldm_set_option(nope_ldm_t* m, const char* name, int value) {
  NOPE_CHECK(m && name, "null argument");
  if (std::strcmp(name, "fuse_geglu") == 0) { m->fuse_geglu = value != 0; return 0; }
  if (std::strcmp(name, "hoist") == 0) { m->hoist = value != 0; return 0; }
  if (std::strcmp(name, "fold_residual") == 0) {
    NOPE_CHECK(!m->finalized, "fold_residual must be set before finalize");
    m->fold_residual = value != 0;
    return 0;
  }
  if (std::strcmp(name, "precision") == 0) {
    NOPE_CHECK(!m->finalized, "precision must be set before finalize");
    NOPE_CHECK(value == 0 || value == 1, "LDM precision: 0 (fp16 weights) or 1 (exact weights, W_hi + W_lo)");
    m->precision = value;
    return 0;
  }
  if (std::strcmp(name, "wide_tiles") == 0) {
    NOPE_CHECK(!m->finalized, "wide_tiles must be set before finalize");
    m->wide_tiles = value != 0;
    return 0;
  }
  return fail(std::string("unknown option: ") + name);
}
int64_t nope_ldm_last_launch_count(const nope_ldm_t* m) { return m ? m->launches : 0; }

int nope_ldm_profile(nope_ldm_t* m, int enable) {
  NOPE_CHECK(m, "null engine");
  for (cudaEvent_t e : m->prof_ev) cudaEventDestroy(e);
  m->prof_ev.clear();
  m->prof_flops.clear();
  m->prof_kind.clear();
  m->profile = enable != 0;
  return 0;
}
int nope_ldm_profile_read(nope_ldm_t* m, double* ms, double* flops, int64_t* launches) {
  NOPE_CHECK(m && ms && flops && launches, "null argument");
  NOPE_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 2; ++k) { ms[k] = 0.0; flops[k] = 0.0; launches[k] = 0; }
  for (size_t i = 0; i < m->prof_flops.size(); ++i) {
    float t = 0.f;
    NOPE_CUDA(cudaEventElapsedTime(&t, m->prof_ev[2 * i], m->prof_ev[2 * i + 1]));
    const int k = m->prof_kind[i];
    ms[k] += t;
    flops[k] += m->prof_flops[i];
    launches[k] += 1;
  }
  return 0;
}

int nope_ldm_sweep(nope_ldm_t* m, const float* ref_latent, const float* poses, int B, int N,
                   const float* query_latent, float* out_emb, float* out_sim, int k, float* out_topv,
                   int64_t* out_topi, int64_t idx_base, void* stream) {
  NOPE_CHECK(m && m->finalized, "engine not finalized");
  NOPE_CHECK(ref_latent && poses && B >= 1 && N >= 1, "bad arguments");
  NOPE_CHECK(!(out_sim || k > 0) || query_latent, "scores / top-k need query_latent");
  NOPE_CHECK(k >= 0 && k <= N && k <= 64, "k must be in [0, min(N, 64)]");
  NOPE_CHECK(k == 0 || (out_topv && out_topi), "top-k outputs missing");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CUDA(cudaSetDevice(m->device));
  m->launches = 0;
  const int total = B * N;
  const int cap = std::min(m->chunk, total);
  if (m->ensure_workspace(cap, B)) return -1;
  const int hw = m->S0 * m->S0;
  const int nslab = (hw + kFinalThreads - 1) / kFinalThreads;
  float* part = nullptr;
  if (query_latent) {
    const size_t need = (size_t)total * nslab;
    if (need > m->score_partial_cap) {
      NOPE_CUDA(cudaStreamSynchronize(st));
      if (m->score_partial) cudaFree(m->score_partial);
      NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&m->score_partial), need * sizeof(float)));
      m->score_partial_cap = need;
    }
    part = m->score_partial;
  }
  if (m->prestage(ref_latent, B, st)) return -1;
  for (int h0 = 0; h0 < total; h0 += cap) {
    const int n = std::min(cap, total - h0);
    if (m->forward_chunk(poses, h0, n, N, query_latent, out_emb, part, st)) return -1;
  }
  if (query_latent && (out_sim || k > 0)) {
    float* sim = out_sim;
    if (!sim) {
      if ((size_t)total > m->sim_buf_cap) {
        NOPE_CUDA(cudaStreamSynchronize(st));
        if (m->sim_buf) cudaFree(m->sim_buf);
        NOPE_CUDA(cudaMalloc(reinterpret_cast<void**>(&m->sim_buf), (size_t)total * sizeof(float)));
        m->sim_buf_cap = total;
      }
      sim = m->sim_buf;
    }
    sim_topk_kernel<<<B, 256, 0, st>>>(part, nslab, sim, N, k, out_topv, reinterpret_cast<long long*>(out_topi),
                                       (long long)idx_base);
    NOPE_CUDA(cudaGetLastError());
    ++m->launches;
  }
  return 0;
}

int nope_ldm_debug_tap(nope_ldm_t* m, const float* ref_latent, const float* poses, int N, const char* tap,
                       float* out, int64_t out_capacity_floats, int* out_C, int* out_H, void* stream) {
  NOPE_CHECK(m && m->finalized && ref_latent && poses && tap && out, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CHECK(N <= m->chunk, "debug tap: N must fit one chunk");
  if (m->ensure_workspace(N, 1)) return -1;
  m->tap_name = tap;
  m->tap_out = out;
  m->tap_cap = out_capacity_floats;
  m->tap_hit = false;
  int rc = m->prestage(ref_latent, 1, st);
  if (!rc) rc = m->forward_chunk(poses, 0, N, N, nullptr, nullptr, nullptr, st);
  m->tap_out = nullptr;
  if (rc) return rc;
  NOPE_CUDA(cudaStreamSynchronize(st));
  NOPE_CHECK(m->tap_hit, std::string("unknown tap name: ") + tap);
  if (out_C) *out_C = m->tap_C;
  if (out_H) *out_H = m->tap_S;
  return 0;
}

int nope_ldm_run_block(nope_ldm_t* m, const char* name, const float* x0, int C0, const float* x1, int C1, int S,
                       int n, const float* poses, float* out, void* stream) {
  NOPE_CHECK(m && m->finalized && name && x0 && out && n >= 1, "bad argument");
  NOPE_CHECK(S == 8 || S == 16 || S == 32, "side must be 8, 16 or 32");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CUDA(cudaSetDevice(m->device));
  if (m->ensure_workspace(std::max(n, 1), 1)) return -1;
  NOPE_CHECK(n <= m->cap, "run_block: n exceeds the workspace");
  const std::string nm = name;
  // stage the inputs in XA / XB (NHWC fp16); results land in XC
  nchw_f32_to_nhwc_f16_kernel<<<ew_grid((long long)n * C0 * S * S), 256, 0, st>>>(x0, m->XA, n, C0, S * S);
  if (x1) nchw_f32_to_nhwc_f16_kernel<<<ew_grid((long long)n * C1 * S * S), 256, 0, st>>>(x1, m->XB, n, C1, S * S);
  NOPE_CUDA(cudaGetLastError());
  int Co = 0, So = S;
  if (m->convs.count(nm + ".c1")) {
    if (m->resblock(nm, m->XA, C0, x1 ? m->XB : nullptr, x1 ? C1 : 0, m->XC, S, n, st)) return -1;
    Co = m->convs.at(nm + ".c2").cout;
  } else if (m->convs.count(nm + ".qkv")) {
    NOPE_CHECK(poses != nullptr && x1 == nullptr, "transformer block: poses required, one input");
    if (m->cross_terms(poses, n, st)) return -1;
    if (m->stats(m->XA, C0, nullptr, 0, S, n, m->S_out, st)) return -1;
    if (m->transformer(nm, m->XA, m->XC, C0, S, n, m->cb, st)) return -1;
    Co = C0;
  } else if (m->convs.count(nm)) {
    const LdmConv& L = m->convs.at(nm);
    NOPE_CHECK(x1 == nullptr && L.cin == C0 && (L.mode == 3 || L.mode == 4), "run_block: not a resample conv");
    So = L.mode == 3 ? 2 * S : S / 2;
    if (m->conv(L, m->XA, m->XC, So, n, st)) return -1;
    Co = L.cout;
  } else {
    return fail(std::string("run_block: unknown module ") + nm);
  }
  nhwc_f16_to_nchw_f32_kernel<<<ew_grid((long long)n * Co * So * So), 256, 0, st>>>(m->XC, out, n, Co, So * So);
  NOPE_CUDA(cudaGetLastError());
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int nope_op_mh_attention(int impl, const float* qkv, float* out, int n_img, int n_tok, int C, void* stream) {
  NOPE_CHECK(qkv && out && n_img >= 1 && n_tok >= 64 && n_tok % 64 == 0 && C % 64 == 0 && C >= 64,
             "bad arguments (n_tok and C must be multiples of 64)");
  NOPE_CHECK(impl == 0 || impl == 1, "impl must be 0 (tcgen05) or 1 (CUDA cores)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  nope_ldm e;    // only the attention staging buffers are used; freed by the destructor
  e.attn_impl = impl;
  const size_t tok = (size_t)n_img * n_tok;
  __half *q16 = nullptr, *o16 = nullptr;
  if (e.ws_half(&q16, tok * 3 * C) || e.ws_half(&o16, tok * C) || e.ws_half(&e.Vt, tok * C)) return -1;
  // [n_img, n_tok, 3C] fp32 is already token-major: a plain fp32 -> fp16 cast ("NCHW" with hw = 1)
  nchw_f32_to_nhwc_f16_kernel<<<ew_grid((long long)tok * 3 * C), 256, 0, st>>>(qkv, q16, (int)tok, 3 * C, 1);
  NOPE_CUDA(cudaGetLastError());
  if (e.attention(q16, o16, C, n_tok, n_img, st)) return -1;
  nhwc_f16_to_nchw_f32_kernel<<<ew_grid((long long)tok * C), 256, 0, st>>>(o16, out, (int)tok, C, 1);
  NOPE_CUDA(cudaGetLastError());
  NOPE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------
// VSD evaluation: depth renders + fused VSD error (vsd.cuh)
// ---------------------------------------------------------------------------------
namespace {
struct VsdLayout {
  size_t info, cam, big, counter, total;
};
int vsd_plan(const int64_t* mesh_voff, const int64_t* mesh_foff, int M, const int* mesh_ids, int P,
             std::vector<VsdRenderInfo>* infos, VsdLayout* L) {
  NOPE_CHECK(mesh_voff && mesh_foff && mesh_ids, "null argument");
  NOPE_CHECK(M >= 1 && P >= 1 && P <= 65535, "need M >= 1 meshes and 1 <= P <= 65535 renders");
  NOPE_CHECK(mesh_voff[0] == 0 && mesh_foff[0] == 0, "mesh offsets must start at 0");
  for (int m = 0; m < M; ++m) {
    NOPE_CHECK(mesh_voff[m + 1] > mesh_voff[m] && mesh_foff[m + 1] > mesh_foff[m],
               "mesh offsets must increase strictly (every mesh needs vertices and faces)");
    NOPE_CHECK(mesh_voff[m + 1] - mesh_voff[m] <= INT32_MAX && mesh_foff[m + 1] - mesh_foff[m] <= INT32_MAX,
               "a mesh has more than 2^31 - 1 vertices or faces");
  }
  long long nv = 0, nf = 0;
  if (infos) infos->resize(P);
  for (int p = 0; p < P; ++p) {
    const int m = mesh_ids[p];
    NOPE_CHECK(m >= 0 && m < M, "mesh id " + std::to_string(m) + " of render " + std::to_string(p) +
                                    " is outside [0, " + std::to_string(M) + ")");
    VsdRenderInfo ri;
    ri.nv = (int)(mesh_voff[m + 1] - mesh_voff[m]);
    ri.nf = (int)(mesh_foff[m + 1] - mesh_foff[m]);
    ri.vbase = mesh_voff[m];
    ri.fbase = mesh_foff[m];
    ri.wbase = nv;
    if (infos) (*infos)[p] = ri;
    nv += ri.nv;
    nf += ri.nf;
  }
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  L->info = 0;
  L->cam = up(sizeof(VsdRenderInfo) * (size_t)P);
  L->big = L->cam + up(sizeof(double) * 3 * (size_t)nv);
  L->counter = L->big + up(sizeof(int2) * (size_t)nf);
  L->total = L->counter + 256;
  return 0;
}
}  // namespace

extern "C" {

int64_t nope_vsd_workspace_bytes(const int64_t* mesh_voff, const int64_t* mesh_foff, int M, const int* mesh_ids,
                                 int P) {
  VsdLayout L;
  if (vsd_plan(mesh_voff, mesh_foff, M, mesh_ids, P, nullptr, &L)) return -1;
  return (int64_t)L.total;
}

int nope_vsd_render(const float* verts, const int* faces, const int64_t* mesh_voff, const int64_t* mesh_foff, int M,
                    const int* mesh_ids, const float* poses, const double* intrinsics, int P, int H, int W,
                    float znear, float zfar, void* workspace, int64_t workspace_bytes, float* depth, void* stream) {
  NOPE_CHECK(H >= 1 && W >= 1 && (int64_t)H * W <= INT32_MAX, "image size must satisfy 1 <= H*W <= 2^31 - 1");
  NOPE_CHECK(verts && faces && poses && intrinsics && depth, "null argument");
  NOPE_CHECK(znear > 0.f && zfar > znear, "need 0 < znear < zfar");
  std::vector<VsdRenderInfo> infos;
  VsdLayout L;
  if (vsd_plan(mesh_voff, mesh_foff, M, mesh_ids, P, &infos, &L)) return -1;
  NOPE_CHECK(workspace && workspace_bytes >= (int64_t)L.total,
             "workspace smaller than nope_vsd_workspace_bytes (" + std::to_string(L.total) + " bytes)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  auto* info = reinterpret_cast<VsdRenderInfo*>(ws + L.info);
  auto* cam = reinterpret_cast<double*>(ws + L.cam);
  auto* big = reinterpret_cast<int2*>(ws + L.big);
  auto* n_big = reinterpret_cast<unsigned int*>(ws + L.counter);
  NOPE_CUDA(cudaMemcpyAsync(info, infos.data(), sizeof(VsdRenderInfo) * P, cudaMemcpyHostToDevice, st));
  NOPE_CUDA(cudaMemsetAsync(n_big, 0, sizeof(unsigned int), st));
  int max_nv = 0, max_nf = 0;
  for (const auto& ri : infos) {
    max_nv = std::max(max_nv, ri.nv);
    max_nf = std::max(max_nf, ri.nf);
  }
  const size_t n_px = (size_t)P * H * W;
  auto* zbuf = reinterpret_cast<unsigned int*>(depth);
  const int ew = (int)std::min<size_t>((n_px + 255) / 256, 4096);
  vsd_fill_kernel<<<ew, 256, 0, st>>>(zbuf, n_px, 0x7f800000u);
  NOPE_CUDA(cudaGetLastError());
  vsd_vertex_kernel<<<dim3(std::min((max_nv + 255) / 256, 1024), P), 256, 0, st>>>(verts, poses, info, cam);
  NOPE_CUDA(cudaGetLastError());
  vsd_face_kernel<<<dim3((max_nf + 127) / 128, P), 128, 0, st>>>(faces, cam, info, intrinsics, H, W, znear, zfar,
                                                                 zbuf, big, n_big);
  NOPE_CUDA(cudaGetLastError());
  vsd_big_face_kernel<<<kVsdBigTriCtas, 256, 0, st>>>(faces, cam, info, intrinsics, H, W, znear, zfar, zbuf, big,
                                                       n_big);
  NOPE_CUDA(cudaGetLastError());
  vsd_finish_kernel<<<ew, 256, 0, st>>>(zbuf, n_px);
  NOPE_CUDA(cudaGetLastError());
  return 0;
}

int nope_vsd_error(const uint16_t* depth_raw, double depth_scale, const double* intrinsics, const float* depth_gt,
                   const float* depth_est, int F, int k, int H, int W, float delta, double tau, int64_t* out_counts,
                   double* out_err, void* stream) {
  NOPE_CHECK(depth_raw && intrinsics && depth_gt && depth_est && out_counts && out_err, "null argument");
  NOPE_CHECK(F >= 1 && F <= 65535 && k >= 1 && k <= 65535 && (int64_t)F * k <= INT32_MAX,
             "need 1 <= F, k <= 65535 and F*k <= 2^31 - 1");
  NOPE_CHECK(H >= 1 && W >= 1 && (int64_t)H * W <= INT32_MAX, "image size must satisfy 1 <= H*W <= 2^31 - 1");
  NOPE_CHECK(depth_scale > 0.0, "depth_scale must be positive");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  NOPE_CUDA(cudaMemsetAsync(out_counts, 0, sizeof(int64_t) * 3 * (size_t)F * k, st));
  const int slices = (int)(((int64_t)H * W + kVsdErrPixelsPerCta - 1) / kVsdErrPixelsPerCta);
  vsd_error_kernel<<<dim3(slices, k, F), 256, 0, st>>>(depth_raw, depth_scale, intrinsics, depth_gt, depth_est, k,
                                                       H, W, delta, tau,
                                                       reinterpret_cast<unsigned long long*>(out_counts));
  NOPE_CUDA(cudaGetLastError());
  vsd_error_finish_kernel<<<(F * k + 255) / 256, 256, 0, st>>>(
      reinterpret_cast<const unsigned long long*>(out_counts), F * k, out_err);
  NOPE_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
