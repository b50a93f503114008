// Denoiser networks of the YOND path on B200: UNetSeeInDark, GuidedResUnet, SNRnet.
//   reference: archs/Unet.py:4-104, :288-378, :380-470; archs/modules.py:117-125, :163-233; archs/__init__.py:10-17.
// The handle owns device copies of the weights, repacked once from the reference's state_dict layout
// (utils/utils.py:160-209) into the tensor-core kernels' layout; activations live in a caller-provided workspace.
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

#include "conv_tc.cuh"
#include "net_kernels.cuh"

namespace {

struct LayerW {
  int mode = 0, Cin0 = 0, Cin1 = 0, Cout = 0;
  std::string wkey, bkey;
  std::string wkey2, bkey2;  // CONV_UPSC: the 1x1 shortcut conv folded behind the transposed conv (wkey / bkey)
  int wcin = 0;  // input channels of the SOURCE weight tensor when the layer uses only its first Cin0 + Cin1 (0: all)
  bf16* w = nullptr;
  bf16* wpaired = nullptr;  // 32 -> 32 channel 3x3 layers: pixel-pair pack (conv_tc_pack_paired)
  float* bias = nullptr;
};

struct Bump {  // workspace carve-up; with base == nullptr it only measures
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* b) : base(reinterpret_cast<uint8_t*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 1024);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

}  // namespace

struct yond_net {
  int arch = 0, in_nc = 4, out_nc = 4, nf = 32, res = 1, norm = 0, conv_impl = 0;
  std::vector<std::string> keys;
  std::map<std::string, std::vector<int64_t>> shapes;
  std::map<std::string, std::vector<float>> host;
  std::map<std::string, float*> f32;   // device copies of small fp32 tensors, torch layout
  std::map<std::string, LayerW> conv;  // tensor-core layers by module name
  float* head_w = nullptr;             // [9][4][nf]
  float* tail_w = nullptr;             // [nf][4]
  bool finalized = false;
  // live profiling of the tensor-core conv launches
  int profile = 0;
  std::vector<cudaEvent_t> events;
  size_t ev_used = 0;
  double acc_ms = 0, acc_flops = 0, pending_flops = 0;
  int acc_launches = 0;
  // side stream for the conditioning vectors: they depend only on t and run beside the first layer
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int ch(int lvl) const { return nf << lvl; }
};

namespace {

void add_key(yond_net* n, const std::string& k, std::vector<int64_t> shape) {
  n->keys.push_back(k);
  n->shapes[k] = std::move(shape);
}
void add_conv_keys(yond_net* n, const std::string& name, int cout, int cin, int k) {
  add_key(n, name + ".weight", {cout, cin, k, k});
  add_key(n, name + ".bias", {cout});
}
void add_convT_keys(yond_net* n, const std::string& name, int cin, int cout) {
  add_key(n, name + ".weight", {cin, cout, 2, 2});
  add_key(n, name + ".bias", {cout});
}
void add_layer(yond_net* n, const std::string& name, int mode, int cin0, int cin1, int cout) {
  LayerW L;
  L.mode = mode;
  L.Cin0 = cin0;
  L.Cin1 = cin1;
  L.Cout = cout;
  L.wkey = name + ".weight";
  L.bkey = name + ".bias";
  n->conv[name] = L;
}

// state_dict keys in the reference's registration order + the tensor-core layer table
void describe(yond_net* n) {
  const int nf = n->nf, cin = n->in_nc, cout = n->out_nc;
  if (n->arch == YOND_ARCH_SELFRES || n->arch == YOND_ARCH_GSELF) {
    // SelfResUNet archs/comp.py:745-776 (Res :830-838, RUP :804-813, LR :709-717) / GuidedSelfUnet :852-883 (GLR :912-926, GRes :936-946,
    // GUP :956-966); depth 5
    const bool gsu = n->arch == YOND_ARCH_GSELF;
    auto glr = [&](const std::string& p, int co, int k) {  // conv + the conditioning MLPs, in GLR's registration order
      add_conv_keys(n, p + ".block", co, co, k);
      add_conv_keys(n, p + ".gamma.0", co, 1, 1);
      add_conv_keys(n, p + ".gamma.2", co, co, 1);
      add_conv_keys(n, p + ".beta.1", co, co, 1);
      add_layer(n, p + ".block", k == 3 ? CONV_3X3_S1 : CONV_1X1, co, 0, co);
    };
    auto res = [&](const std::string& p, int ci, int co, int k, bool tc_shortcut) {
      add_conv_keys(n, p + ".conv_1.block.0", co, co, k);
      add_layer(n, p + ".conv_1.block.0", k == 3 ? CONV_3X3_S1 : CONV_1X1, co, 0, co);
      if (gsu) {
        glr(p + ".conv_2", co, k);
      } else {
        add_conv_keys(n, p + ".conv_2.block.0", co, co, k);
        add_layer(n, p + ".conv_2.block.0", k == 3 ? CONV_3X3_S1 : CONV_1X1, co, 0, co);
      }
      if (ci != co) {
        add_conv_keys(n, p + ".short_cut.0", co, ci, 1);
        if (tc_shortcut) {  // 1x1 on cat[up (2 nf), skip (nf)], or on the 2 nf feature part of cat[up, input]
          add_layer(n, p + ".short_cut.0", CONV_1X1, 2 * nf, ci == 3 * nf ? nf : 0, co);
          n->conv[p + ".short_cut.0"].wcin = ci;
        }
      }
    };
    res("head", cin, nf, 3, false);  // its 4 -> nf shortcut runs on the float32 input (head kernel, centre tap only)
    for (int i = 0; i < 5; ++i) {
      if (gsu) glr("down_path." + std::to_string(i), nf, 3);
      else res("down_path." + std::to_string(i), nf, nf, 3, false);
    }
    for (int i = 0; i < 5; ++i) res("up_path." + std::to_string(i), i == 0 ? 2 * nf : (i == 4 ? 2 * nf + cin : 3 * nf), 2 * nf, 3, true);
    res("last", 2 * nf, 2 * nf, 1, false);
    add_conv_keys(n, "out", cout, 2 * nf, 1);
  } else if (n->arch == YOND_ARCH_UNET) {  // archs/Unet.py:17-52
    int prev = cin;
    for (int l = 1; l <= 5; ++l) {
      const int c = n->ch(l - 1);
      const std::string a = "conv" + std::to_string(l) + "_1", b = "conv" + std::to_string(l) + "_2";
      add_conv_keys(n, a, c, prev, 3);
      add_conv_keys(n, b, c, c, 3);
      if (l > 1) add_layer(n, a, CONV_3X3_S1, prev, 0, c);
      add_layer(n, b, CONV_3X3_S1, c, 0, c);
      prev = c;
    }
    for (int i = 0; i < 4; ++i) {
      const int c = n->ch(3 - i);
      const std::string l = std::to_string(6 + i);
      add_convT_keys(n, "upv" + l, 2 * c, c);
      add_conv_keys(n, "conv" + l + "_1", c, 2 * c, 3);
      add_conv_keys(n, "conv" + l + "_2", c, c, 3);
      add_layer(n, "upv" + l, CONVT_2X2, 2 * c, 0, c);
      add_layer(n, "conv" + l + "_1", CONV_3X3_S1, c, c, c);
      add_layer(n, "conv" + l + "_2", CONV_3X3_S1, c, 0, c);
    }
    add_conv_keys(n, "conv10_1", cout, nf, 1);
  } else {  // GuidedResUnet archs/Unet.py:393-421 / SNRnet :301-329; blocks archs/modules.py:163-218
    const bool guided = n->arch == YOND_ARCH_GUIDED || n->arch == YOND_ARCH_RES2;  // ResBlock registers the same gamma / beta modules
    auto block = [&](const std::string& p, int ci, int co) {
      add_conv_keys(n, p + ".conv1", co, co, 3);
      add_conv_keys(n, p + ".conv2", co, co, 3);
      if (guided) {
        add_conv_keys(n, p + ".gamma.0", co, 1, 1);
        add_conv_keys(n, p + ".gamma.2", co, co, 1);
        add_conv_keys(n, p + ".beta.1", co, co, 1);
      } else {
        add_conv_keys(n, p + ".sfm1.0", co, 1, 1);
        add_conv_keys(n, p + ".sfm1.2", co, co, 1);
        add_conv_keys(n, p + ".sfm2.0", co, 1, 1);
        add_conv_keys(n, p + ".sfm2.2", co, co, 1);
      }
      if (ci != co) {
        add_conv_keys(n, p + ".short_cut.0", co, ci, 1);
        add_layer(n, p + ".short_cut.0", CONV_1X1, co, co, co);  // input = cat[up, skip], co channels each
      }
      add_layer(n, p + ".conv1", CONV_3X3_S1, co, 0, co);
      add_layer(n, p + ".conv2", CONV_3X3_S1, co, 0, co);
    };
    add_conv_keys(n, "conv_in", nf, cin, 3);
    for (int l = 1; l <= 4; ++l) {
      const int c = n->ch(l - 1);
      block("conv" + std::to_string(l), c, c);
      add_conv_keys(n, "pool" + std::to_string(l) + ".conv", 2 * c, c, 3);
      add_layer(n, "pool" + std::to_string(l) + ".conv", CONV_3X3_S2, c, 0, 2 * c);
    }
    block("conv5", n->ch(4), n->ch(4));
    for (int i = 0; i < 4; ++i) {
      const int c = n->ch(3 - i);
      const std::string l = std::to_string(6 + i);
      add_convT_keys(n, "upv" + l, 2 * c, c);
      add_layer(n, "upv" + l, CONVT_2X2, 2 * c, 0, c);
      block("conv" + l, 2 * c, c);
      if (c <= 64) {  // up-sampling + 1x1 shortcut on cat[up, skip] as ONE layer (weights resident in shared memory)
        add_layer(n, "conv" + l + ".upsc", CONV_UPSC, 2 * c, c, c);
        LayerW& F = n->conv["conv" + l + ".upsc"];
        F.wkey = "upv" + l + ".weight";
        F.bkey = "upv" + l + ".bias";
        F.wkey2 = "conv" + l + ".short_cut.0.weight";
        F.bkey2 = "conv" + l + ".short_cut.0.bias";
      }
    }
    add_conv_keys(n, "conv10", cout, nf, 1);
  }
}

void free_device(yond_net* n) {
  for (auto& kv : n->f32) cudaFree(kv.second);
  n->f32.clear();
  for (auto& kv : n->conv) {
    if (kv.second.w) cudaFree(kv.second.w);
    if (kv.second.wpaired) cudaFree(kv.second.wpaired);
    kv.second.w = kv.second.wpaired = nullptr;
    kv.second.bias = nullptr;
  }
  if (n->head_w) cudaFree(n->head_w);
  if (n->tail_w) cudaFree(n->tail_w);
  n->head_w = n->tail_w = nullptr;
  n->finalized = false;
}

// torch layout -> [cbg][tap][N][CB] bf16 (K-major tiles the weight TMA map walks)
std::vector<bf16> pack_weights(const LayerW& L, const std::vector<float>& w) {
  const int Cin = L.Cin0 + L.Cin1, CB = conv_tc_channel_block(L.Cin0, L.Cin1);
  const int taps = (L.mode == CONV_3X3_S1 || L.mode == CONV_3X3_S2) ? 9 : 1;
  const int N = L.mode == CONVT_2X2 ? 4 * L.Cout : L.Cout;
  std::vector<bf16> out((size_t)taps * Cin * N);
  for (int cbg = 0; cbg < Cin / CB; ++cbg)
    for (int tap = 0; tap < taps; ++tap)
      for (int nn = 0; nn < N; ++nn)
        for (int j = 0; j < CB; ++j) {
          const int ci = cbg * CB + j;
          float v;
          if (L.mode == CONVT_2X2) {  // (Cin, Cout, 2, 2); n = (a*2+b)*Cout + co
            const int q = nn / L.Cout, co = nn % L.Cout;
            v = w[(((size_t)ci * L.Cout + co) * 2 + (q >> 1)) * 2 + (q & 1)];
          } else {  // (Cout, Cin, k, k); tap = r*k + s
            v = w[((size_t)nn * (L.wcin ? L.wcin : Cin) + ci) * taps + tap];
          }
          out[(((size_t)cbg * taps + tap) * N + nn) * CB + j] = __float2bfloat16_rn(v);
        }
  return out;
}

// CONV_UPSC: fold ConvTranspose2d(2x2, s2) into the 1x1 shortcut that follows it on cat[up, skip].
//   Wt (Cl, C, 2, 2), bt (C);  Wsc (C, 2C, 1, 1), bsc (C)
//   part A [cb][n = (a*2+b)*C + co][CB] = sum_m Wsc[co][m] * Wt[cl][m][a][b]      (float64 accumulation, one bf16 rounding)
//   part B [cb][co][CB]                 = Wsc[co][C + cs]
//   bias'[co] = bsc[co] + sum_m Wsc[co][m] * bt[m]
std::vector<bf16> pack_upsc(const LayerW& L, const std::vector<float>& wt, const std::vector<float>& bt, const std::vector<float>& wsc,
                            const std::vector<float>& bsc, std::vector<float>* bias_out) {
  const int C = L.Cout, Cl = L.Cin0, CB = conv_tc_channel_block(L.Cin0, L.Cin1);
  std::vector<bf16> out((size_t)Cl * 4 * C + (size_t)C * C);
  for (int cb = 0; cb < Cl / CB; ++cb)
    for (int q = 0; q < 4; ++q)
      for (int co = 0; co < C; ++co)
        for (int j = 0; j < CB; ++j) {
          const int cl = cb * CB + j;
          double acc = 0.0;
          for (int m = 0; m < C; ++m) acc += (double)wsc[(size_t)co * 2 * C + m] * (double)wt[(((size_t)cl * C + m) * 2 + (q >> 1)) * 2 + (q & 1)];
          out[(((size_t)cb * 4 * C) + (size_t)q * C + co) * CB + j] = __float2bfloat16_rn((float)acc);
        }
  const size_t offB = (size_t)Cl * 4 * C;
  for (int cb = 0; cb < C / CB; ++cb)
    for (int co = 0; co < C; ++co)
      for (int j = 0; j < CB; ++j) out[offB + ((size_t)cb * C + co) * CB + j] = __float2bfloat16_rn(wsc[(size_t)co * 2 * C + C + cb * CB + j]);
  bias_out->resize(C);
  for (int co = 0; co < C; ++co) {
    double acc = bsc[co];
    for (int m = 0; m < C; ++m) acc += (double)wsc[(size_t)co * 2 * C + m] * (double)bt[m];
    (*bias_out)[co] = (float)acc;
  }
  return out;
}

int upload_f32(yond_net* n, const std::string& key) {
  const std::vector<float>& h = n->host[key];
  float* d = nullptr;
  YOND_CUDA_CHECK(cudaMalloc(&d, h.size() * sizeof(float)));
  YOND_CUDA_CHECK(cudaMemcpy(d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
  n->f32[key] = d;
  return YOND_OK;
}

int finalize(yond_net* n) {
  if (n->finalized) return YOND_OK;
  for (const auto& k : n->keys)
    if (!n->host.count(k)) return yond_set_error(YOND_ERR_INVALID, "network tensor '%s' has not been set", k.c_str());
  free_device(n);
  for (const auto& k : n->keys) {
    const bool is_tc_weight = k.size() > 7 && k.compare(k.size() - 7, 7, ".weight") == 0 && n->conv.count(k.substr(0, k.size() - 7));
    if (!is_tc_weight) {
      int rc = upload_f32(n, k);
      if (rc) return rc;
    }
  }
  for (auto& kv : n->conv) {
    LayerW& L = kv.second;
    if (L.mode == CONV_UPSC) {
      std::vector<float> fb;
      std::vector<bf16> packed = pack_upsc(L, n->host[L.wkey], n->host[L.bkey], n->host[L.wkey2], n->host[L.bkey2], &fb);
      YOND_CUDA_CHECK(cudaMalloc(&L.w, packed.size() * sizeof(bf16)));
      YOND_CUDA_CHECK(cudaMemcpy(L.w, packed.data(), packed.size() * sizeof(bf16), cudaMemcpyHostToDevice));
      const std::string fk = kv.first + ".bias(folded)";
      n->host[fk] = fb;
      int rc = upload_f32(n, fk);
      n->host.erase(fk);
      if (rc) return rc;
      L.bias = n->f32[fk];
      continue;
    }
    std::vector<bf16> packed = pack_weights(L, n->host[L.wkey]);
    YOND_CUDA_CHECK(cudaMalloc(&L.w, packed.size() * sizeof(bf16)));
    YOND_CUDA_CHECK(cudaMemcpy(L.w, packed.data(), packed.size() * sizeof(bf16), cudaMemcpyHostToDevice));
    if (L.mode == CONV_3X3_S1 && L.Cin0 == 32 && L.Cin1 == 0 && L.Cout == 32) {
      std::vector<bf16> pp(kConvPairedElems);
      conv_tc_pack_paired(n->host[L.wkey].data(), pp.data());
      YOND_CUDA_CHECK(cudaMalloc(&L.wpaired, pp.size() * sizeof(bf16)));
      YOND_CUDA_CHECK(cudaMemcpy(L.wpaired, pp.data(), pp.size() * sizeof(bf16), cudaMemcpyHostToDevice));
    }
    L.bias = n->f32[L.bkey];
  }
  if (n->arch == YOND_ARCH_SELFRES || n->arch == YOND_ARCH_GSELF) {  // head shortcut (nf,4,1,1) as the centre tap of a 3x3; out (4,2nf,1,1) -> [ci][4]; input part of the last shortcut
    const std::vector<float>& hw = n->host["head.short_cut.0.weight"];
    std::vector<float> h((size_t)36 * n->nf, 0.f);
    for (int co = 0; co < n->nf; ++co)
      for (int ci = 0; ci < 4; ++ci) h[((size_t)4 * 4 + ci) * n->nf + co] = hw[(size_t)co * 4 + ci];
    YOND_CUDA_CHECK(cudaMalloc(&n->head_w, h.size() * sizeof(float)));
    YOND_CUDA_CHECK(cudaMemcpy(n->head_w, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    const int c2 = 2 * n->nf;
    const std::vector<float>& tw = n->host["out.weight"];
    std::vector<float> t((size_t)c2 * 4);
    for (int co = 0; co < 4; ++co)
      for (int ci = 0; ci < c2; ++ci) t[(size_t)ci * 4 + co] = tw[(size_t)co * c2 + ci];
    YOND_CUDA_CHECK(cudaMalloc(&n->tail_w, t.size() * sizeof(float)));
    YOND_CUDA_CHECK(cudaMemcpy(n->tail_w, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
    const std::vector<float>& sw = n->host["up_path.4.short_cut.0.weight"];  // (2nf, 2nf + 4): the last 4 input channels = network input
    std::vector<float> win((size_t)c2 * 4);
    for (int co = 0; co < c2; ++co)
      for (int ci = 0; ci < 4; ++ci) win[(size_t)co * 4 + ci] = sw[(size_t)co * (c2 + 4) + c2 + ci];
    const std::string ik = "up_path.4.short_cut.0.weight(input part)";
    n->host[ik] = win;
    int rc = upload_f32(n, ik);
    n->host.erase(ik);
    if (rc) return rc;
  } else {  // head: (nf,4,3,3) -> [tap][ci][co];  tail: (4,nf,1,1) -> [ci][4]
    const std::string hk = n->arch == YOND_ARCH_UNET ? "conv1_1.weight" : "conv_in.weight";
    const std::string tk = n->arch == YOND_ARCH_UNET ? "conv10_1.weight" : "conv10.weight";
    const std::vector<float>& hw = n->host[hk];
    std::vector<float> h((size_t)36 * n->nf);
    for (int co = 0; co < n->nf; ++co)
      for (int ci = 0; ci < 4; ++ci)
        for (int t = 0; t < 9; ++t) h[((size_t)t * 4 + ci) * n->nf + co] = hw[((size_t)co * 4 + ci) * 9 + t];
    YOND_CUDA_CHECK(cudaMalloc(&n->head_w, h.size() * sizeof(float)));
    YOND_CUDA_CHECK(cudaMemcpy(n->head_w, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    const std::vector<float>& tw = n->host[tk];
    std::vector<float> t((size_t)n->nf * 4);
    for (int co = 0; co < 4; ++co)
      for (int ci = 0; ci < n->nf; ++ci) t[(size_t)ci * 4 + co] = tw[(size_t)co * n->nf + ci];
    YOND_CUDA_CHECK(cudaMalloc(&n->tail_w, t.size() * sizeof(float)));
    YOND_CUDA_CHECK(cudaMemcpy(n->tail_w, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  n->finalized = true;
  return YOND_OK;
}

double layer_flops(const LayerW& L, int B, int Hin, int Win) {
  const double cin = L.Cin0 + L.Cin1;
  switch (L.mode) {
    case CONV_3X3_S1: return 2.0 * B * Hin * Win * 9.0 * cin * L.Cout;
    case CONV_3X3_S2: return 2.0 * B * (Hin / 2) * (Win / 2) * 9.0 * cin * L.Cout;
    case CONV_1X1: return 2.0 * B * Hin * Win * cin * L.Cout;
    case CONV_UPSC:  // the algorithmic work of the two reference layers it replaces (transposed conv + 1x1 on 2 Cout channels)
      return 2.0 * B * Hin * Win * L.Cin0 * 4.0 * L.Cout + 2.0 * B * (2.0 * Hin) * (2.0 * Win) * 2.0 * L.Cout * L.Cout;
    default: return 2.0 * B * Hin * Win * cin * 4.0 * L.Cout;  // CONVT_2X2
  }
}

struct TailArgs {  // fused output conv of the last tensor-core layer (ConvLayer::tail_*)
  const float* w;
  const float* b;
  const float* z;
  const float* ub;
  float* y;
  int res;
};

struct Runner {
  yond_net* n;
  cudaStream_t s;
  int rc = YOND_OK;
  double flops = 0;
  bool dry = false;  // only count FLOPs / workspace
  // One tensor-core conv layer on `B` images (pointers already offset to the first image).
  void conv(const std::string& name, int B, int Hin, int Win, const bf16* src0, const bf16* src1, const float* scale,
            const float* shift, int act, float slope, const bf16* res, bf16* out0, bf16* out1, const TailArgs* tail = nullptr) {
    const LayerW& L = n->conv.at(name);
    const double f = layer_flops(L, B, Hin, Win);
    flops += f;
    if (dry || rc) return;
    ConvLayer c{};
    c.mode = L.mode;
    c.B = B;
    c.Hin = Hin;
    c.Win = Win;
    c.Cin0 = L.Cin0;
    c.Cin1 = L.Cin1;
    c.src0 = src0;
    c.src1 = src1;
    c.Cout = L.Cout;
    c.wpacked = L.w;
    c.wpaired = L.wpaired;
    c.bias = L.bias;
    c.scale = scale;
    c.shift = shift;
    c.act = act;
    c.slope = slope;
    c.res = res;
    c.out0 = out0;
    c.out1 = out1;
    if (tail) {
      c.tail_w = tail->w; c.tail_b = tail->b; c.tail_z = tail->z; c.tail_ub = tail->ub; c.tail_y = tail->y; c.tail_res = tail->res;
    }
    const bool prof = n->profile && n->ev_used + 2 <= n->events.size();
    if (prof) cudaEventRecord(n->events[n->ev_used], s);
    rc = n->conv_impl == 1 ? conv_ref_launch(c, s) : conv_tc_launch(c, s);
    if (prof) {
      cudaEventRecord(n->events[n->ev_used + 1], s);
      n->ev_used += 2;
      n->pending_flops += f;
    }
  }
};

// SelfResUNet.forward (archs/comp.py:778-802): every layer is a tensor-core conv (3x3 / 1x1 + LeakyReLU(0.1) [+ residual]); the two
// 4-channel 1x1 pieces (head shortcut on the input, input part of the last up-level shortcut) stay in float32.
int forward_selfres(yond_net* n, const float* z, const float* ub, const float* tvec, float* y, int B, int H, int W, void* ws, size_t* ws_bytes,
                    double* flops, cudaStream_t s) {
  const bool dry = ws == nullptr;
  const bool gsu = n->arch == YOND_ARCH_GSELF;
  YOND_REQUIRE(H % 32 == 0 && W % 32 == 0, "SelfResUNet: H, W must be multiples of 32 (five 2x2 poolings); got %d x %d", H, W);
  if (!dry && gsu && tvec == nullptr) return yond_set_error(YOND_ERR_INVALID, "guided network needs the per-sample t vector");
  YOND_REQUIRE(!(gsu && n->res), "GuidedSelfUnet: res must be 0 (archs/comp.py:904-905 adds a 2nf-channel tensor to the output)");
  Bump bump(ws);
  Runner R;
  R.n = n;
  R.s = s;
  R.dry = dry;
  const int nf = n->nf, c2 = 2 * nf;
  const float slope = 0.1f;
  const float* ubn = n->norm ? ub : nullptr;
  auto px = [&](int lv) { return (size_t)(H >> lv) * (W >> lv); };
  auto buf = [&](int lv, int C) { return bump.take<bf16>((size_t)B * px(lv) * C); };
#define RUN(expr)                                       \
  do {                                                  \
    if (!dry && R.rc == YOND_OK) R.rc = (expr);         \
  } while (0)
  // conditioning vectors of the 12 GLRs (GuidedSelfUnet): head.conv_2, down_path.0-4, up_path.0-4.conv_2, last.conv_2
  float* va[12] = {nullptr};
  float* vb[12] = {nullptr};
  if (gsu) {
    FilmAll all{};
    all.n = 12;
    for (int k = 0; k < 12; ++k) {
      const int C = (k >= 1 && k <= 5) || k == 0 ? nf : c2;
      const std::string p = k == 0 ? "head.conv_2" : (k <= 5 ? "down_path." + std::to_string(k - 1) : (k <= 10 ? "up_path." + std::to_string(k - 6) + ".conv_2" : "last.conv_2"));
      va[k] = bump.take<float>((size_t)B * C);
      vb[k] = bump.take<float>((size_t)B * C);
      if (!dry) {
        FilmWeights& fw = all.fw[k];
        fw.w0 = n->f32[p + ".gamma.0.weight"]; fw.b0 = n->f32[p + ".gamma.0.bias"];
        fw.w2 = n->f32[p + ".gamma.2.weight"]; fw.b2 = n->f32[p + ".gamma.2.bias"];
        fw.w3 = n->f32[p + ".beta.1.weight"];  fw.b3 = n->f32[p + ".beta.1.bias"];
        all.C[k] = C;
        all.out_a[k] = va[k];
        all.out_b[k] = vb[k];
      }
    }
    RUN(film_launch(all, tvec, ubn, B, 1, s));
  }
  auto film_of = [&](const std::string& p) {
    if (p == "head") return 0;
    if (p == "last") return 11;
    return 6 + (p.back() - '0');  // up_path.i
  };
  auto res_block = [&](const std::string& p, int lv, int C, const bf16* x, bf16* t, bf16* out) {  // out = LR|GLR(LR(x)) + x
    R.conv(p + ".conv_1.block.0", B, H >> lv, W >> lv, x, nullptr, nullptr, nullptr, ACT_LRELU, slope, nullptr, t, nullptr);
    if (gsu) {
      const int k = film_of(p);
      R.conv(p + ".conv_2.block", B, H >> lv, W >> lv, t, nullptr, va[k], vb[k], ACT_LRELU, slope, x, out, nullptr);
    } else {
      R.conv(p + ".conv_2.block.0", B, H >> lv, W >> lv, t, nullptr, nullptr, nullptr, ACT_LRELU, slope, x, out, nullptr);
    }
  };
  bf16* x0 = buf(0, nf);
  bf16* t0 = buf(0, nf);
  bf16* h = buf(0, nf);
  RUN(head_conv_launch(z, ubn, n->head_w, dry ? nullptr : n->f32["head.short_cut.0.bias"], B, H, W, nf, 1.0f, x0, nullptr, s));
  res_block("head", 0, nf, x0, t0, h);
  bf16* pool[5];
  for (int i = 0; i < 5; ++i) {
    pool[i] = buf(i + 1, nf);
    bf16* t = buf(i + 1, nf);
    bf16* hn = buf(i + 1, nf);
    RUN(maxpool2_launch(h, pool[i], B, H >> i, W >> i, nf, s));
    if (gsu)  // one GLR, no residual
      R.conv("down_path." + std::to_string(i) + ".block", B, H >> (i + 1), W >> (i + 1), pool[i], nullptr, va[1 + i], vb[1 + i], ACT_LRELU, slope,
             nullptr, hn, nullptr);
    else
      res_block("down_path." + std::to_string(i), i + 1, nf, pool[i], t, hn);
    h = hn;
  }
  for (int i = 0; i < 5; ++i) {
    const int lv = 4 - i, hl = H >> (lv + 1), wl = W >> (lv + 1);  // h lives at level lv + 1
    const std::string p = "up_path." + std::to_string(i);
    bf16* c = buf(lv, c2);
    if (i == 0) {  // cat[up(h) (nf), pool_3 (nf)]: identity shortcut
      RUN(upcat_launch(h, pool[3], c, B, hl, wl, nf, nf, s));
    } else {
      bf16* upx = buf(lv, c2);
      RUN(upcat_launch(h, nullptr, upx, B, hl, wl, c2, 0, s));
      if (i < 4) {  // 1x1 on cat[up (2 nf), pool (nf)]
        R.conv(p + ".short_cut.0", B, H >> lv, W >> lv, upx, pool[3 - i], nullptr, nullptr, ACT_NONE, 0.f, nullptr, c, nullptr);
      } else {      // 1x1 on cat[up (2 nf), network input (4)]: feature part on the tensor cores, input part in float32
        R.conv(p + ".short_cut.0", B, H, W, upx, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, c, nullptr);
        RUN(add_in4_launch(c, n->f32["up_path.4.short_cut.0.weight(input part)"], z, ubn, B, H, W, c2, s));
      }
    }
    bf16* t = buf(lv, c2);
    bf16* yb = buf(lv, c2);
    res_block(p, lv, c2, c, t, yb);
    h = yb;
  }
  bf16* tl = buf(0, c2);
  bf16* l = buf(0, c2);
  res_block("last", 0, c2, h, tl, l);
  RUN(tail_conv_launch(l, n->tail_w, dry ? nullptr : n->f32["out.bias"], z, ubn, n->res, B, H, W, c2, y, s));
#undef RUN
  if (ws_bytes) *ws_bytes = align_up(bump.off, 1024);
  if (flops) *flops = R.flops + 2.0 * B * H * W * (4.0 * nf + 4.0 * c2 + 4.0 * c2);
  return R.rc;
}

// One forward pass; with ws == nullptr only measures workspace bytes and FLOPs.
//
// Every layer runs once over the whole batch.  The two full-resolution levels hold ~85 % of the activation bytes, and running
// them in sub-batches small enough for a producer's output to still be in the 126 MB L2 when its consumer reads it was
// measured on B200 (bench.py, 1280 blocks): the split costs more in launch tails than L2 residency returns (43.7 ms/step
// unsplit vs 49-60 ms at 16-48 blocks).
int forward_impl(yond_net* n, const float* z, const float* ub, const float* t, float* y, int B, int H, int W, void* ws,
                 size_t* ws_bytes, double* flops, cudaStream_t s) {
  if (n->arch == YOND_ARCH_SELFRES || n->arch == YOND_ARCH_GSELF) return forward_selfres(n, z, ub, t, y, B, H, W, ws, ws_bytes, flops, s);
  const bool dry = ws == nullptr;
  Bump bump(ws);
  Runner R;
  R.n = n;
  R.s = s;
  R.dry = dry;
  const int nf = n->nf;
  const float* ubn = n->norm ? ub : nullptr;
  const bool unet = n->arch == YOND_ARCH_UNET;
  const bool guided = n->arch == YOND_ARCH_GUIDED;
  const bool res2 = n->arch == YOND_ARCH_RES2;  // GuidedResUnet's graph without conditioning
  if (!dry && !unet && !res2 && t == nullptr) return yond_set_error(YOND_ERR_INVALID, "guided network needs the per-sample t vector");
  const double head_tail_flops = 2.0 * B * H * W * (36.0 * nf + 4.0 * nf);
  auto px = [&](int lv) { return (size_t)(H >> lv) * (W >> lv); };
  const bool fuse_up = !n->conv_impl;  // the CUDA-core cross-check path keeps the two reference layers
  auto buf = [&](int lv, int C) { return bump.take<bf16>((size_t)B * px(lv) * C); };

#define RUN(expr)                                       \
  do {                                                  \
    if (!dry && R.rc == YOND_OK) R.rc = (expr);         \
  } while (0)

  // ---- conditioning vectors of the 9 blocks (one launch, whole batch, on the side stream) ----
  bool film_pending = false;
  auto film_join = [&]() {
    if (film_pending) {
      film_pending = false;
      if (cudaStreamWaitEvent(s, n->ev_join, 0) != cudaSuccess && R.rc == YOND_OK)
        R.rc = yond_set_error(YOND_ERR_CUDA, "cudaStreamWaitEvent(film) failed");
    }
  };
  float* va[10] = {nullptr};
  float* vb[10] = {nullptr};
  if (!unet && !res2) {
    FilmAll all{};
    all.n = 9;
    for (int l = 1; l <= 9; ++l) {
      const int lv = l <= 5 ? l - 1 : 9 - l, C = n->ch(lv);
      va[l] = bump.take<float>((size_t)B * C);
      vb[l] = bump.take<float>((size_t)B * C);
      if (!dry) {
        const std::string p = "conv" + std::to_string(l);
        FilmWeights& fw = all.fw[l - 1];
        if (guided) {
          fw.w0 = n->f32[p + ".gamma.0.weight"]; fw.b0 = n->f32[p + ".gamma.0.bias"];
          fw.w2 = n->f32[p + ".gamma.2.weight"]; fw.b2 = n->f32[p + ".gamma.2.bias"];
          fw.w3 = n->f32[p + ".beta.1.weight"];  fw.b3 = n->f32[p + ".beta.1.bias"];
        } else {
          fw.w0 = n->f32[p + ".sfm1.0.weight"]; fw.b0 = n->f32[p + ".sfm1.0.bias"];
          fw.w2 = n->f32[p + ".sfm1.2.weight"]; fw.b2 = n->f32[p + ".sfm1.2.bias"];
          fw.w3 = n->f32[p + ".sfm2.0.weight"]; fw.b3 = n->f32[p + ".sfm2.0.bias"];
          fw.w4 = n->f32[p + ".sfm2.2.weight"]; fw.b4 = n->f32[p + ".sfm2.2.bias"];
        }
        all.C[l - 1] = C;
        all.out_a[l - 1] = va[l];
        all.out_b[l - 1] = vb[l];
      }
    }
    if (!dry && R.rc == YOND_OK) {
      if (!n->side) {
        YOND_CUDA_CHECK(cudaStreamCreateWithFlags(&n->side, cudaStreamNonBlocking));
        YOND_CUDA_CHECK(cudaEventCreateWithFlags(&n->ev_fork, cudaEventDisableTiming));
        YOND_CUDA_CHECK(cudaEventCreateWithFlags(&n->ev_join, cudaEventDisableTiming));
      }
      YOND_CUDA_CHECK(cudaEventRecord(n->ev_fork, s));
      YOND_CUDA_CHECK(cudaStreamWaitEvent(n->side, n->ev_fork, 0));
      R.rc = film_launch(all, t, ubn, B, guided ? 1 : 0, n->side);
      YOND_CUDA_CHECK(cudaEventRecord(n->ev_join, n->side));
      film_pending = true;
    }
  }
  // One residual block (FiLM rows are per image): x raw, xs = SiLU(x).
  auto block = [&](int l, int lv, const bf16* x, const bf16* xs, bf16* zb, bf16* out, const TailArgs* tail = nullptr) {
    const int h = H >> lv, w = W >> lv;
    const std::string p = "conv" + std::to_string(l);
    const float* a = va[l];
    const float* bb = vb[l];
    if (guided || res2) {  // z = SiLU(conv1(SiLU(x)) * tk + tb); out = conv2(z) + x   (ResUnet2: tk = 1, tb = 0)
      R.conv(p + ".conv1", B, h, w, xs, nullptr, a, bb, ACT_SILU, 0.f, nullptr, zb, nullptr);
      R.conv(p + ".conv2", B, h, w, zb, nullptr, nullptr, nullptr, ACT_NONE, 0.f, x, out, nullptr, tail);
    } else {  // SNR: z = SiLU(conv1(SiLU(x)) * a1); out = conv2(z) * a2 + x
      R.conv(p + ".conv1", B, h, w, xs, nullptr, a, nullptr, ACT_SILU, 0.f, nullptr, zb, nullptr);
      R.conv(p + ".conv2", B, h, w, zb, nullptr, bb, nullptr, ACT_NONE, 0.f, x, out, nullptr, tail);
    }
  };
  // The 1x1 output conv (+ input residual, x ub) rides in the epilogue of the last 3x3 layer: its 64 B/px input is never stored.
  const bool fuse_tail = !n->conv_impl && nf == 32 && H >= 16;
  const int C0 = n->ch(0), C1 = n->ch(1), C2 = n->ch(2), C3 = n->ch(3), C4 = n->ch(4);
  const int H1 = H >> 1, W1 = W >> 1, H2 = H >> 2, W2 = W >> 2, H3 = H >> 3, W3 = W >> 3, H4 = H >> 4, W4 = W >> 4;
  // skips of the full-resolution levels (whole batch) and the level-2 hand-over tensors
  bf16* skip0 = buf(0, C0);
  bf16* skip1 = buf(1, C1);

  if (unet) {
    bf16* p2 = buf(2, C1);  // pooled level-1 output
    bf16* a0 = buf(0, C0);
    bf16* p1 = buf(1, C0);
    bf16* a1 = buf(1, C1);
    RUN(head_conv_launch(z, ubn, n->head_w, n->f32["conv1_1.bias"], B, H, W, nf, 0.2f, a0, nullptr, s));
    R.conv("conv1_2", B, H, W, a0, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, skip0, nullptr);
    RUN(maxpool2_launch(skip0, p1, B, H, W, C0, s));
    R.conv("conv2_1", B, H1, W1, p1, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, a1, nullptr);
    R.conv("conv2_2", B, H1, W1, a1, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, skip1, nullptr);
    RUN(maxpool2_launch(skip1, p2, B, H1, W1, C1, s));
    bf16* a2 = buf(2, C2); bf16* c3 = buf(2, C2); bf16* p3 = buf(3, C2);
    bf16* a3 = buf(3, C3); bf16* c4 = buf(3, C3); bf16* p4 = buf(4, C3);
    bf16* a4 = buf(4, C4); bf16* c5 = buf(4, C4);
    R.conv("conv3_1", B, H2, W2, p2, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, a2, nullptr);
    R.conv("conv3_2", B, H2, W2, a2, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c3, nullptr);
    RUN(maxpool2_launch(c3, p3, B, H2, W2, C2, s));
    R.conv("conv4_1", B, H3, W3, p3, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, a3, nullptr);
    R.conv("conv4_2", B, H3, W3, a3, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c4, nullptr);
    RUN(maxpool2_launch(c4, p4, B, H3, W3, C3, s));
    R.conv("conv5_1", B, H4, W4, p4, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, a4, nullptr);
    R.conv("conv5_2", B, H4, W4, a4, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c5, nullptr);
    bf16* u6 = buf(3, C3); bf16* t6 = buf(3, C3); bf16* c6 = buf(3, C3);
    R.conv("upv6", B, H4, W4, c5, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u6, nullptr);
    R.conv("conv6_1", B, H3, W3, u6, c4, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, t6, nullptr);
    R.conv("conv6_2", B, H3, W3, t6, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c6, nullptr);
    bf16* u7 = buf(2, C2); bf16* t7 = buf(2, C2); bf16* c7 = buf(2, C2);
    R.conv("upv7", B, H3, W3, c6, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u7, nullptr);
    R.conv("conv7_1", B, H2, W2, u7, c3, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, t7, nullptr);
    R.conv("conv7_2", B, H2, W2, t7, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c7, nullptr);
    bf16* u8 = buf(1, C1); bf16* t8 = buf(1, C1); bf16* c8 = buf(1, C1);
    bf16* u9 = buf(0, C0); bf16* t9 = buf(0, C0); bf16* c9 = buf(0, C0);
    R.conv("upv8", B, H2, W2, c7, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u8, nullptr);
    R.conv("conv8_1", B, H1, W1, u8, skip1, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, t8, nullptr);
    R.conv("conv8_2", B, H1, W1, t8, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c8, nullptr);
    R.conv("upv9", B, H1, W1, c8, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u9, nullptr);
    R.conv("conv9_1", B, H, W, u9, skip0, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, t9, nullptr);
    if (fuse_tail) {
      const TailArgs ta{n->tail_w, dry ? nullptr : n->f32["conv10_1.bias"], z, ubn, y, n->res};
      R.conv("conv9_2", B, H, W, t9, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c9, nullptr, &ta);
    } else {
      R.conv("conv9_2", B, H, W, t9, nullptr, nullptr, nullptr, ACT_LRELU, 0.2f, nullptr, c9, nullptr);
      RUN(tail_conv_launch(c9, n->tail_w, n->f32["conv10_1.bias"], z, ubn, n->res, B, H, W, nf, y, s));
    }
  } else {
    bf16* x2 = buf(2, C2);   // pool2 output (raw) and its SiLU: inputs of the level-2 block
    bf16* x2s = buf(2, C2);
    bf16* x0 = buf(0, C0); bf16* x0s = buf(0, C0); bf16* z0 = buf(0, C0);
    bf16* x1 = buf(1, C1); bf16* x1s = buf(1, C1); bf16* z1 = buf(1, C1);
    RUN(head_conv_launch(z, ubn, n->head_w, n->f32["conv_in.bias"], B, H, W, nf, res2 ? 0.2f : 0.01f, x0, x0s, s));
    film_join();
    block(1, 0, x0, x0s, z0, skip0);
    // stride-2 conv, no activation (modules.py:117-125); the dual store feeds the next block
    R.conv("pool1.conv", B, H, W, skip0, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x1, x1s);
    block(2, 1, x1, x1s, z1, skip1);
    R.conv("pool2.conv", B, H1, W1, skip1, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x2, x2s);
    bf16* zb2 = buf(2, C2); bf16* c3 = buf(2, C2);
    bf16* x3 = buf(3, C3); bf16* x3s = buf(3, C3); bf16* zb3 = buf(3, C3); bf16* c4 = buf(3, C3);
    bf16* x4 = buf(4, C4); bf16* x4s = buf(4, C4); bf16* zb4 = buf(4, C4); bf16* c5 = buf(4, C4);
    block(3, 2, x2, x2s, zb2, c3);
    R.conv("pool3.conv", B, H2, W2, c3, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x3, x3s);
    block(4, 3, x3, x3s, zb3, c4);
    R.conv("pool4.conv", B, H3, W3, c4, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x4, x4s);
    block(5, 4, x4, x4s, zb4, c5);
    bf16* u6 = buf(3, C3); bf16* c6 = buf(3, C3);
    R.conv("upv6", B, H4, W4, c5, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u6, nullptr);
    R.conv("conv6.short_cut.0", B, H3, W3, u6, c4, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x3, x3s);  // x3/x3s are free again
    block(6, 3, x3, x3s, zb3, c6);
    bf16* u7 = buf(2, C2); bf16* c7 = buf(2, C2);
    R.conv("upv7", B, H3, W3, c6, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u7, nullptr);
    R.conv("conv7.short_cut.0", B, H2, W2, u7, c3, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x2, x2s);
    block(7, 2, x2, x2s, zb2, c7);
    bf16* u8 = buf(1, C1); bf16* c8 = buf(1, C1);
    bf16* u9 = buf(0, C0); bf16* c9 = buf(0, C0);
    if (fuse_up && n->conv.count("conv8.upsc")) {
      R.conv("conv8.upsc", B, H2, W2, c7, skip1, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x1, x1s);
    } else {
      R.conv("upv8", B, H2, W2, c7, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u8, nullptr);
      R.conv("conv8.short_cut.0", B, H1, W1, u8, skip1, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x1, x1s);
    }
    block(8, 1, x1, x1s, z1, c8);
    if (fuse_up && n->conv.count("conv9.upsc")) {
      R.conv("conv9.upsc", B, H1, W1, c8, skip0, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x0, x0s);
    } else {
      R.conv("upv9", B, H1, W1, c8, nullptr, nullptr, nullptr, ACT_NONE, 0.f, nullptr, u9, nullptr);
      R.conv("conv9.short_cut.0", B, H, W, u9, skip0, nullptr, nullptr, ACT_NONE, 0.f, nullptr, x0, x0s);
    }
    if (fuse_tail) {
      const TailArgs ta{n->tail_w, dry ? nullptr : n->f32["conv10.bias"], z, ubn, y, n->res};
      block(9, 0, x0, x0s, z0, c9, &ta);
    } else {
      block(9, 0, x0, x0s, z0, c9);
      RUN(tail_conv_launch(c9, n->tail_w, n->f32["conv10.bias"], z, ubn, n->res, B, H, W, nf, y, s));
    }
  }
  film_join();
#undef RUN
  if (ws_bytes) *ws_bytes = align_up(bump.off, 1024);
  if (flops) *flops = R.flops + head_tail_flops;
  return R.rc;
}

}  // namespace

extern "C" {

int yond_net_create(int arch, int in_nc, int out_nc, int nf, int res, int norm, yond_net_t** out) {
  YOND_REQUIRE(out != nullptr, "yond_net_create: null output");
  YOND_REQUIRE(arch >= YOND_ARCH_UNET && arch <= YOND_ARCH_GSELF, "yond_net_create: unknown arch %d", arch);
  YOND_REQUIRE(in_nc == 4 && out_nc == 4, "yond_net_create: only packed-Bayer nets (in_nc = out_nc = 4, nframes = 1) are built");
  YOND_REQUIRE(nf >= 32 && nf % 32 == 0, "yond_net_create: nf must be a multiple of 32 (got %d)", nf);
  yond_net* n = new yond_net();
  n->arch = arch;
  n->in_nc = in_nc;
  n->out_nc = out_nc;
  n->nf = nf;
  n->res = res;
  n->norm = norm;
  describe(n);
  *out = n;
  return YOND_OK;
}

void yond_net_destroy(yond_net_t* n) {
  if (!n) return;
  free_device(n);
  for (auto e : n->events) cudaEventDestroy(e);
  if (n->ev_fork) cudaEventDestroy(n->ev_fork);
  if (n->ev_join) cudaEventDestroy(n->ev_join);
  if (n->side) cudaStreamDestroy(n->side);
  delete n;
}

int yond_net_set_tensor(yond_net_t* n, const char* key, const float* host_data, const int64_t* shape, int ndim) {
  YOND_REQUIRE(n && key && host_data, "yond_net_set_tensor: null argument");
  auto it = n->shapes.find(key);
  if (it == n->shapes.end()) return yond_set_error(YOND_ERR_INVALID, "unexpected state-dict key '%s'", key);
  const std::vector<int64_t>& exp = it->second;
  bool ok = (int)exp.size() == ndim;
  size_t numel = 1;
  for (int i = 0; ok && i < ndim; ++i) ok = exp[i] == shape[i];
  for (auto d : exp) numel *= (size_t)d;
  if (!ok) return yond_set_error(YOND_ERR_INVALID, "shape mismatch for '%s'", key);
  n->host[key].assign(host_data, host_data + numel);
  n->finalized = false;
  return YOND_OK;
}

int yond_net_missing(yond_net_t* n, char* missing, size_t cap) {
  int cnt = 0;
  std::string s;
  for (const auto& k : n->keys)
    if (!n->host.count(k)) {
      ++cnt;
      s += k + ";";
    }
  if (missing && cap) {
    snprintf(missing, cap, "%s", s.c_str());
  }
  return cnt;
}

int yond_net_num_keys(yond_net_t* n) { return (int)n->keys.size(); }
const char* yond_net_key(yond_net_t* n, int i) { return (i >= 0 && i < (int)n->keys.size()) ? n->keys[i].c_str() : nullptr; }
int yond_net_key_shape(yond_net_t* n, int i, int64_t* shape4) {
  if (i < 0 || i >= (int)n->keys.size()) return -1;
  const std::vector<int64_t>& s = n->shapes[n->keys[i]];
  for (size_t d = 0; d < s.size(); ++d) shape4[d] = s[d];
  return (int)s.size();
}

size_t yond_net_workspace_bytes(yond_net_t* n, int B, int H, int W) {
  size_t bytes = 0;
  forward_impl(n, nullptr, nullptr, nullptr, nullptr, B, H, W, nullptr, &bytes, nullptr, nullptr);
  // extras of the NCHW surface: z, y (B,H,W,4) f32 and ub (B)
  return bytes + 2 * align_up((size_t)B * H * W * 4 * sizeof(float), 1024) + align_up((size_t)B * sizeof(float), 1024) + 4096;
}

double yond_net_flops(yond_net_t* n, int B, int H, int W) {
  double f = 0;
  forward_impl(n, nullptr, nullptr, nullptr, nullptr, B, H, W, nullptr, nullptr, &f, nullptr);
  return f;
}

int yond_net_set_conv_impl(yond_net_t* n, int impl) {
  n->conv_impl = impl == 2 ? 2 : (impl ? 1 : 0);  // 2: tensor-core kernels with the layer fusions off (A/B checks)
  return YOND_OK;
}

int yond_net_forward(yond_net_t* n, const float* z, const float* ub, const float* t, float* y, int B, int H, int W,
                     void* workspace, size_t workspace_bytes, void* stream) {
  YOND_REQUIRE(n && z && y && workspace, "yond_net_forward: null argument");
  YOND_REQUIRE(B > 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, "yond_net_forward: H,W must be multiples of 16 (got %d,%d)", H, W);
  YOND_REQUIRE(!n->norm || ub, "yond_net_forward: norm=1 needs ub");
  YOND_REQUIRE((uintptr_t)workspace % 1024 == 0, "yond_net_forward: workspace must be 1024-byte aligned");
  int rc = finalize(n);
  if (rc) return rc;
  size_t need = 0;
  forward_impl(n, nullptr, nullptr, nullptr, nullptr, B, H, W, nullptr, &need, nullptr, nullptr);
  YOND_REQUIRE(workspace_bytes >= need, "yond_net_forward: workspace too small (%zu < %zu)", workspace_bytes, need);
  return forward_impl(n, z, ub, t, y, B, H, W, workspace, nullptr, nullptr, (cudaStream_t)stream);
}

int yond_net_forward_nchw(yond_net_t* n, const float* x, const float* t, float* y, int B, int H, int W, void* workspace,
                          size_t workspace_bytes, void* stream) {
  YOND_REQUIRE(n && x && y && workspace, "yond_net_forward_nchw: null argument");
  YOND_REQUIRE((uintptr_t)workspace % 1024 == 0, "yond_net_forward_nchw: workspace must be 1024-byte aligned");
  YOND_REQUIRE(workspace_bytes >= yond_net_workspace_bytes(n, B, H, W), "yond_net_forward_nchw: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
  const size_t img = align_up((size_t)B * H * W * 4 * sizeof(float), 1024);
  float* z = reinterpret_cast<float*>(base);
  float* yy = reinterpret_cast<float*>(base + img);
  float* ub = reinterpret_cast<float*>(base + 2 * img);
  uint8_t* rest = base + 2 * img + align_up((size_t)B * sizeof(float), 1024);
  int rc = nchw_to_nhwc4_launch(x, z, ub, B, H, W, s);
  if (rc) return rc;
  rc = yond_net_forward(n, z, ub, t, yy, B, H, W, rest, workspace_bytes - (rest - base), stream);
  if (rc) return rc;
  return nhwc4_to_nchw_launch(yy, y, B, H, W, s);
}

int yond_conv2d(int mode, int impl, int B, int Hin, int Win, int Cin0, int Cin1, const void* src0, const void* src1, int Cout,
                const float* weight_host, const float* bias, const float* scale, const float* shift, int act, float slope,
                const void* res, void* out0, void* out1, void* stream) {
  YOND_REQUIRE(mode >= 0 && mode <= 3 && weight_host && src0 && out0 && bias, "yond_conv2d: bad arguments");
  LayerW L;
  L.mode = mode;
  L.Cin0 = Cin0;
  L.Cin1 = Cin1;
  L.Cout = Cout;
  const int taps = (mode == CONV_3X3_S1 || mode == CONV_3X3_S2) ? 9 : 1;
  const size_t nw = (size_t)taps * (Cin0 + Cin1) * Cout * (mode == CONVT_2X2 ? 4 : 1);
  std::vector<float> w(weight_host, weight_host + nw);
  std::vector<bf16> packed = pack_weights(L, w);
  bf16* dw = nullptr;
  YOND_CUDA_CHECK(cudaMalloc(&dw, packed.size() * sizeof(bf16)));
  YOND_CUDA_CHECK(cudaMemcpy(dw, packed.data(), packed.size() * sizeof(bf16), cudaMemcpyHostToDevice));
  bf16* dwp = nullptr;
  if (mode == CONV_3X3_S1 && Cin0 == 32 && Cin1 == 0 && Cout == 32) {
    std::vector<bf16> pp(kConvPairedElems);
    conv_tc_pack_paired(weight_host, pp.data());
    YOND_CUDA_CHECK(cudaMalloc(&dwp, pp.size() * sizeof(bf16)));
    YOND_CUDA_CHECK(cudaMemcpy(dwp, pp.data(), pp.size() * sizeof(bf16), cudaMemcpyHostToDevice));
  }
  ConvLayer c{};
  c.wpaired = dwp;
  c.mode = mode; c.B = B; c.Hin = Hin; c.Win = Win; c.Cin0 = Cin0; c.Cin1 = Cin1;
  c.src0 = (const bf16*)src0; c.src1 = (const bf16*)src1; c.Cout = Cout; c.wpacked = dw; c.bias = bias;
  c.scale = scale; c.shift = shift; c.act = act; c.slope = slope; c.res = (const bf16*)res;
  c.out0 = (bf16*)out0; c.out1 = (bf16*)out1;
  int rc = impl ? conv_ref_launch(c, (cudaStream_t)stream) : conv_tc_launch(c, (cudaStream_t)stream);
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  cudaFree(dw);
  if (dwp) cudaFree(dwp);
  if (rc) return rc;
  if (e != cudaSuccess) return yond_set_error(YOND_ERR_CUDA, "yond_conv2d: kernel failed: %s", cudaGetErrorString(e));
  return YOND_OK;
}

int yond_net_profile(yond_net_t* n, int enable) {
  n->profile = enable;
  if (enable && n->events.empty()) {
    n->events.resize(32768);
    for (auto& e : n->events) YOND_CUDA_CHECK(cudaEventCreate(&e));
  }
  return YOND_OK;
}

int yond_net_profile_read(yond_net_t* n, double* conv_ms, double* conv_flops, int* launches, int reset) {
  if (n->ev_used) {
    YOND_CUDA_CHECK(cudaEventSynchronize(n->events[n->ev_used - 1]));
    for (size_t i = 0; i + 1 < n->ev_used; i += 2) {
      float ms = 0;
      YOND_CUDA_CHECK(cudaEventElapsedTime(&ms, n->events[i], n->events[i + 1]));
      n->acc_ms += ms;
    }
    n->acc_launches += (int)(n->ev_used / 2);
    n->acc_flops += n->pending_flops;
    n->ev_used = 0;
    n->pending_flops = 0;
  }
  if (conv_ms) *conv_ms = n->acc_ms;
  if (conv_flops) *conv_flops = n->acc_flops;
  if (launches) *launches = n->acc_launches;
  if (reset) {
    n->acc_ms = n->acc_flops = 0;
    n->acc_launches = 0;
  }
  return YOND_OK;
}

}  // extern "C"
