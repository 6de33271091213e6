// Pipeline of one m3_infer call: TextEncoder -> duration predictor -> length regulator ->
// coupling flow -> HiFi-GAN -> peak-normalised int16 (SURVEY.md Appendix A; the ONNX graph
// the reference runs at mimic3_tts/voice.py:230, plus utils.py:237-244).
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstring>

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "../../include/m3b200.h"
#include "kernels.h"

namespace m3 {

// ======================================================================================
// memory helpers
// ======================================================================================
void Arena::reserve(size_t bytes) {
  used = 0;
  if (bytes <= cap) return;
  if (base) cudaFree(base);
  base = nullptr;
  cap = 0;
  size_t want = bytes + bytes / 8 + (1 << 20);
  M3_CUDA(cudaMalloc(&base, want));
  cap = want;
}
Arena::~Arena() {
  if (base) cudaFree(base);
}
void PinnedBuf::reserve(size_t bytes) {
  if (bytes <= cap) return;
  if (p) cudaFreeHost(p);
  p = nullptr;
  cap = 0;
  size_t want = bytes + bytes / 8 + 4096;
  M3_CUDA(cudaMallocHost(&p, want));
  cap = want;
}
PinnedBuf::~PinnedBuf() {
  if (p) cudaFreeHost(p);
}
Context::Context(int dev) : device(dev) {
  M3_CUDA(cudaSetDevice(dev));
  M3_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  M3_CUDA(cudaEventCreate(&ev0));
  M3_CUDA(cudaEventCreate(&ev1));
}
Context::~Context() {
  cudaSetDevice(device);
  for (auto e : marks) cudaEventDestroy(e);
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  if (stream) cudaStreamDestroy(stream);
}
Context* Voice::acquire() {
  std::lock_guard<std::mutex> lk(mu);
  if (!idle.empty()) {
    Context* c = idle.back();
    idle.pop_back();
    return c;
  }
  all.emplace_back(new Context(dv->device));
  return all.back().get();
}
void Voice::release(Context* c) {
  std::lock_guard<std::mutex> lk(mu);
  idle.push_back(c);
}
DeviceVoice::~DeviceVoice() {
  if (slab || slab16) cudaSetDevice(device);
  if (slab) cudaFree(slab);
  if (slab16) cudaFree(slab16);
}

// ======================================================================================
// weight packing: PyTorch layouts -> channels-last GEMM operands, one device slab
// ======================================================================================
namespace {

struct Packer {
  std::vector<float> host;
  size_t add(const std::vector<float>& v) {
    size_t off = (host.size() + 63) & ~size_t(63);
    host.resize(off + v.size());
    std::copy(v.begin(), v.end(), host.begin() + off);
    return off;
  }
};

struct Pending {
  const float** slot;
  size_t off;
};

struct Builder {
  const HostVoice& hv;
  Packer pk;
  std::vector<Pending> fix;
  std::vector<uint16_t> h16;  // tensor-core operands
  int tc_fmt = 0;
  int64_t n_params = 0;
  explicit Builder(const HostVoice& h) : hv(h) {}

  uint16_t cvt16(float f) const {
    if (tc_fmt == 1) {
      __nv_bfloat16 h = __float2bfloat16_rn(f);
      return *reinterpret_cast<uint16_t*>(&h);
    }
    __half h = __float2half_rn(f);
    return *reinterpret_cast<uint16_t*>(&h);
  }

  // fp16 hi/lo split packing of W[tap][k][n] for rowgemm_tc_kernel:
  // [chunk][K block][tap][hi|lo][4][nc][8]
  void rows_pack(RowTcW& t, const std::vector<float>& W, int taps, int K, int N) {
    t.ok = false;
    if (!rowgemm_tc_supported(K, taps)) return;
    const int KB = 32, NCc = rowgemm_tc_nc(N, taps);
    t.nc = NCc;
    const int chunks = (N + NCc - 1) / NCc, nkb = K / KB;
    while (h16.size() % 64) h16.push_back(0);
    t.woff = h16.size();
    const size_t o = h16.size();
    h16.resize(o + rowgemm_tc_weight_elems(K, N, taps, NCc), 0);
    for (int c = 0; c < chunks; ++c)
      for (int kb = 0; kb < nkb; ++kb)
        for (int tap = 0; tap < taps; ++tap)
          for (int kk = 0; kk < KB; ++kk)
            for (int j = 0; j < NCc; ++j) {
              const int n = c * NCc + j;
              if (n >= N) continue;
              const float w = W[(size_t(tap) * K + kb * KB + kk) * N + n];
              const __half hi = __float2half_rn(w);
              const __half lo = __float2half_rn((w - __half2float(hi)) * 2048.f);
              const size_t blk = ((size_t(c) * nkb + kb) * taps + tap) * 2;
              const size_t in_blk = (size_t(kk / 8) * NCc + j) * 8 + (kk & 7);
              h16[o + (blk + 0) * (KB * NCc) + in_blk] = *reinterpret_cast<const uint16_t*>(&hi);
              h16[o + (blk + 1) * (KB * NCc) + in_blk] = *reinterpret_cast<const uint16_t*>(&lo);
            }
    t.ok = true;
  }

  // Pack logical weights W[tap][k][n] (n < Ncols) for conv_tc_kernel.  gate: the Ncols = 2*N
  // columns are (a | b) halves and every chunk carries NC/2 a-columns followed by their b-columns.
  void tc_pack(TcConvW& t, const std::vector<float>& W, int taps, int K, int N, int dil, bool gate) {
    t.ok = false;
    const int ncols = gate ? 2 * N : N;
    int best = 0;
    long best_pad = -1;
    // two M tiles per CTA; only when no width fits that, one (the default generator's K = 512 upsampler)
    for (int m_tiles = 2; m_tiles >= 1 && !best; --m_tiles)
      for (int nc : {128, 96, 64, 32}) {
        if (gate && nc % 64) continue;
        if (!conv_tc_supported(K, nc, taps, dil, m_tiles)) continue;
        const int per = gate ? nc / 2 : nc;
        const long padded = long((N + per - 1) / per) * per;
        if (best_pad < 0 || padded < best_pad) {
          best_pad = padded;
          best = nc;
        }
      }
    if (!best) return;
    const int NC = best, per = gate ? NC / 2 : NC;
    const int chunks = (N + per - 1) / per;
    while (h16.size() % 64) h16.push_back(0);
    t.woff = h16.size();
    const size_t o = h16.size();
    h16.resize(o + size_t(chunks) * taps * K * NC, 0);
    for (int c = 0; c < chunks; ++c)
      for (int tap = 0; tap < taps; ++tap)
        for (int k = 0; k < K; ++k)
          for (int j = 0; j < NC; ++j) {
            int col;
            if (gate) {
              const int ch = c * per + (j % per);
              if (ch >= N) continue;
              col = (j < per ? 0 : N) + ch;
            } else {
              col = c * NC + j;
              if (col >= N) continue;
            }
            h16[o + ((size_t(c) * taps + tap) * (K / 8) + k / 8) * NC * 8 + size_t(j) * 8 + (k & 7)] =
                cvt16(W[(size_t(tap) * K + k) * ncols + col]);
          }
    t.ok = true;
    t.K = K;
    t.NC = NC;
    t.n_chunks = chunks;
    t.N = N;
    t.taps = taps;
  }

  void place(const float** slot, const std::vector<float>& v) { fix.push_back({slot, pk.add(v)}); }

  // Conv1d weight (Cout, Cin, k) -> [k][Cin][Cout]
  // tc: 0 = fp32 SIMT only, 1 = also pack for the tensor-core conv, 2 = gated (cout = 2 * channels),
  //     3 = token-level GEMM: fp16 hi/lo split packing (rowgemm_tc_kernel)
  // dil: the dilation the tensor-core conv will run at (its shared-memory fit depends on it)
  void conv(Lin& l, const std::string& base, int cout, int cin, int k, bool need_bias = true, int tc = 0, int dil = 1) {
    const OnnxTensor& w = hv.need(base + ".weight", {cout, cin, k});
    std::vector<float> t(size_t(k) * cin * cout);
    for (int o = 0; o < cout; ++o)
      for (int i = 0; i < cin; ++i)
        for (int j = 0; j < k; ++j) t[(size_t(j) * cin + i) * cout + o] = w.f32[(size_t(o) * cin + i) * k + j];
    if (tc == 3) rows_pack(l.rtc, t, k, cin, cout);
    else if (tc && cin % 16 == 0 && (tc == 2 ? (cout / 2) % 16 == 0 : cout % 4 == 0))
      tc_pack(l.tc, t, k, cin, tc == 2 ? cout / 2 : cout, dil, tc == 2);
    place(&l.w, t);
    n_params += int64_t(t.size());
    l.cin = cin;
    l.cout = cout;
    l.taps = k;
    l.b = nullptr;
    if (const OnnxTensor* b = hv.maybe(base + ".bias")) {
      if (b->numel() != cout) throw EngineError(3, "generator.onnx: '" + base + ".bias' has wrong size");
      place(&l.b, b->f32);
      n_params += cout;
    } else if (need_bias) {
      throw EngineError(3, "generator.onnx: missing initializer '" + base + ".bias'");
    }
  }
  void vec(const float** slot, const std::string& name, int n) {
    const OnnxTensor& t = hv.need(name, {});
    if (t.numel() != n)
      throw EngineError(3, "generator.onnx: '" + name + "' has " + std::to_string(t.numel()) + " elements, expected " +
                               std::to_string(n));
    place(slot, t.f32);
    n_params += n;
  }
  void dds(DDSW& d, const std::string& p, int ch) {
    for (int i = 0; i < 3; ++i) {
      const std::string is = std::to_string(i);
      const OnnxTensor& w = hv.need(p + ".convs_sep." + is + ".weight", {ch, 1, 3});
      std::vector<float> t(size_t(3) * ch);
      for (int c = 0; c < ch; ++c)
        for (int j = 0; j < 3; ++j) t[size_t(j) * ch + c] = w.f32[size_t(c) * 3 + j];
      place(&d.sep_w[i], t);
      n_params += 3 * ch;
      vec(&d.sep_b[i], p + ".convs_sep." + is + ".bias", ch);
      conv(d.c1x1[i], p + ".convs_1x1." + is, ch, ch, 1, true, 3);
      vec(&d.n1g[i], p + ".norms_1." + is + ".gamma", ch);
      vec(&d.n1b[i], p + ".norms_1." + is + ".beta", ch);
      vec(&d.n2g[i], p + ".norms_2." + is + ".gamma", ch);
      vec(&d.n2b[i], p + ".norms_2." + is + ".beta", ch);
    }
  }
};

}  // namespace

PackedVoice pack_voice(const HostVoice& hv) {
  PackedVoice pv;
  pv.dv.reset(new DeviceVoice());
  DeviceVoice& dv = *pv.dv;
  dv.cfg = hv.cfg;
  const VoiceConfig& c = hv.cfg;
  Builder B(hv);
  {
    // tensor-core operand format: fp16 (default; 11-bit significand keeps the waveform within
    // 1e-4 RMS of fp32) or bf16 (M3B200_TC_FORMAT=bf16).  Accumulation is always fp32.
    const char* fe = getenv("M3B200_TC_FORMAT");
    dv.tc_fmt = (fe && std::string(fe) == "bf16") ? 1 : 0;
    B.tc_fmt = dv.tc_fmt;
    const char* fs = getenv("M3B200_FORCE_SIMT");
    dv.use_tc = !(fs && *fs && *fs != '0');
    const char* ft = getenv("M3B200_TEXT_SIMT");
    dv.use_rows_tc = dv.use_tc && !(ft && *ft && *ft != '0');
  }
  const int H = c.hidden, I = c.inter, Ff = c.filter;
  const int dk = H / c.n_heads;

  // ---- text encoder
  {
    const OnnxTensor& e = hv.need("enc_p.emb.weight", {});
    if (e.dims.size() != 2 || e.dims[1] != H)
      throw EngineError(3, "generator.onnx: enc_p.emb.weight does not match hidden_channels");
    if (c.num_symbols > 0 && e.dims[0] != c.num_symbols)
      throw EngineError(3, "generator.onnx: enc_p.emb.weight rows != config.json model.num_symbols");
    dv.cfg.num_symbols = int(e.dims[0]);
    B.place(&dv.emb, e.f32);
    B.n_params += e.numel();
  }
  dv.enc.resize(c.n_layers);
  for (int l = 0; l < c.n_layers; ++l) {
    EncLayerW& L = dv.enc[l];
    const std::string a = "enc_p.encoder.attn_layers." + std::to_string(l);
    {  // q | k | v concatenated along Cout
      std::vector<float> w(size_t(H) * 3 * H), b(3 * H);
      const char* names[3] = {".conv_q", ".conv_k", ".conv_v"};
      for (int s = 0; s < 3; ++s) {
        const OnnxTensor& t = hv.need(a + names[s] + ".weight", {H, H, 1});
        const OnnxTensor& tb = hv.need(a + names[s] + ".bias", {H});
        for (int o = 0; o < H; ++o) {
          for (int i = 0; i < H; ++i) w[size_t(i) * 3 * H + s * H + o] = t.f32[size_t(o) * H + i];
          b[s * H + o] = tb.f32[o];
        }
      }
      B.rows_pack(L.qkv.rtc, w, 1, H, 3 * H);
      B.place(&L.qkv.w, w);
      B.place(&L.qkv.b, b);
      L.qkv.cin = H;
      L.qkv.cout = 3 * H;
      L.qkv.taps = 1;
      B.n_params += int64_t(w.size() + b.size());
    }
    B.conv(L.o, a + ".conv_o", H, H, 1, true, 3);
    {
      const OnnxTensor& ek = hv.need(a + ".emb_rel_k", {});
      const OnnxTensor& ev = hv.need(a + ".emb_rel_v", {});
      if (ek.dims.size() != 3 || ek.dims[0] != 1 || ek.dims[2] != dk || ek.dims != ev.dims || (ek.dims[1] & 1) == 0)
        throw EngineError(3, "generator.onnx: unexpected emb_rel_k/emb_rel_v shape (heads must share, odd window)");
      dv.window = int(ek.dims[1] - 1) / 2;
      B.place(&L.ek, ek.f32);
      B.place(&L.ev, ev.f32);
      B.n_params += 2 * ek.numel();
    }
    B.vec(&L.g1, "enc_p.encoder.norm_layers_1." + std::to_string(l) + ".gamma", H);
    B.vec(&L.b1, "enc_p.encoder.norm_layers_1." + std::to_string(l) + ".beta", H);
    B.vec(&L.g2, "enc_p.encoder.norm_layers_2." + std::to_string(l) + ".gamma", H);
    B.vec(&L.b2, "enc_p.encoder.norm_layers_2." + std::to_string(l) + ".beta", H);
    const std::string f = "enc_p.encoder.ffn_layers." + std::to_string(l);
    B.conv(L.ffn1, f + ".conv_1", Ff, H, c.kernel_size, true, 3);
    B.conv(L.ffn2, f + ".conv_2", H, Ff, c.kernel_size, true, 3);
  }
  B.conv(dv.enc_proj, "enc_p.proj", 2 * I, H, 1, true, 3);

  // ---- speaker embedding & conditioning layers (collected into one G -> n_cond GEMM)
  const OnnxTensor* embg = hv.maybe("emb_g.weight");
  dv.has_emb_g = embg != nullptr;
  int G = 0;
  if (embg) {
    if (embg->dims.size() != 2) throw EngineError(3, "generator.onnx: emb_g.weight must be 2-D");
    G = int(embg->dims[1]);
    if (c.n_speakers > 1 && embg->dims[0] != c.n_speakers)
      throw EngineError(3, "generator.onnx: emb_g.weight rows != config.json model.n_speakers");
    dv.cfg.n_speakers = int(embg->dims[0]);
    B.place(&dv.emb_g, embg->f32);
    B.n_params += embg->numel();
  }
  std::vector<std::pair<std::string, int>> cond_layers;  // (module, width)
  auto add_cond = [&](const std::string& mod, int width) -> int {
    if (!G) return -1;
    if (!hv.maybe(mod + ".weight")) return -1;
    int off = 0;
    for (auto& p : cond_layers) off += p.second;
    cond_layers.emplace_back(mod, width);
    return off;
  };

  // ---- duration predictor
  dv.use_sdp = c.use_sdp && hv.maybe("dp.flows.0.m") != nullptr;
  if (c.use_sdp && !dv.use_sdp && !hv.maybe("dp.conv_1.weight"))
    throw EngineError(3, "generator.onnx: use_sdp is set but neither dp.flows.0.m nor dp.conv_1.weight exists");
  if (dv.use_sdp) {
    const int Fd = H;
    dv.dp_ch = Fd;
    B.conv(dv.dp_pre, "dp.pre", Fd, H, 1, true, 3);
    B.conv(dv.dp_proj, "dp.proj", Fd, Fd, 1, true, 3);
    B.dds(dv.dp_dds, "dp.convs", Fd);
    dv.dp_cond_off = add_cond("dp.cond", Fd);
    const OnnxTensor& m = hv.need("dp.flows.0.m", {2, 1});
    const OnnxTensor& ls = hv.need("dp.flows.0.logs", {2, 1});
    dv.ea_m[0] = m.f32[0]; dv.ea_m[1] = m.f32[1];
    dv.ea_logs[0] = ls.f32[0]; dv.ea_logs[1] = ls.f32[1];
    B.n_params += 4;
    // flows = [EA, CF1, Flip, CF2, Flip, CF3, Flip, CF4, Flip]; reverse drops CF1 ("useless vflow")
    for (int n : {7, 5, 3}) {
      const std::string p = "dp.flows." + std::to_string(n);
      dv.cflows.emplace_back();
    }
    int idx = 0;
    for (int n : {7, 5, 3}) {
      const std::string p = "dp.flows." + std::to_string(n);
      ConvFlowW& cf = dv.cflows[idx++];
      const OnnxTensor& pw = hv.need(p + ".pre.weight", {Fd, 1, 1});
      B.place(&cf.pre_w, pw.f32);
      B.vec(&cf.pre_b, p + ".pre.bias", Fd);
      B.n_params += Fd;
      B.dds(cf.dds, p + ".convs", Fd);
      B.conv(cf.proj, p + ".proj", 29, Fd, 1, true, 3);
    }
  } else {
    const OnnxTensor& w1 = hv.need("dp.conv_1.weight", {});
    if (w1.dims.size() != 3 || w1.dims[1] != H) throw EngineError(3, "generator.onnx: bad dp.conv_1.weight shape");
    const int Fd = int(w1.dims[0]), k = int(w1.dims[2]);
    dv.dp_ch = Fd;
    B.conv(dv.dpp_c1, "dp.conv_1", Fd, H, k);
    B.conv(dv.dpp_c2, "dp.conv_2", Fd, Fd, k);
    B.conv(dv.dpp_proj, "dp.proj", 1, Fd, 1);
    B.vec(&dv.dpp_g1, "dp.norm_1.gamma", Fd);
    B.vec(&dv.dpp_b1, "dp.norm_1.beta", Fd);
    B.vec(&dv.dpp_g2, "dp.norm_2.gamma", Fd);
    B.vec(&dv.dpp_b2, "dp.norm_2.beta", Fd);
    dv.dp_cond_off = add_cond("dp.cond", H);
  }

  // ---- flow (ResidualCouplingBlock): modules flows.{0,2,4,..}; applied in reverse
  {
    int nflows = 0;
    while (hv.maybe("flow.flows." + std::to_string(2 * nflows) + ".pre.weight")) ++nflows;
    if (!nflows) throw EngineError(3, "generator.onnx: no flow.flows.N.pre.weight found");
    const OnnxTensor& pw = hv.need("flow.flows.0.pre.weight", {});
    if (pw.dims.size() != 3 || pw.dims[1] != I / 2) throw EngineError(3, "generator.onnx: bad flow pre shape");
    const int Hf = int(pw.dims[0]);
    int nl = 0;
    while (hv.maybe("flow.flows.0.enc.in_layers." + std::to_string(nl) + ".weight")) ++nl;
    if (!nl) throw EngineError(3, "generator.onnx: flow WN in_layers missing (weight-norm not resolved?)");
    const OnnxTensor& iw = hv.need("flow.flows.0.enc.in_layers.0.weight", {});
    dv.flow_hidden = Hf;
    dv.flow_layers = nl;
    dv.flow_kernel = int(iw.dims[2]);
    for (int f = nflows - 1; f >= 0; --f) {
      const std::string p = "flow.flows." + std::to_string(2 * f);
      dv.couplings.emplace_back();
    }
    int idx = 0;
    for (int f = nflows - 1; f >= 0; --f) {
      const std::string p = "flow.flows." + std::to_string(2 * f);
      CouplingW& cw = dv.couplings[idx++];
      B.conv(cw.pre, p + ".pre", Hf, I / 2, 1, true, 1);
      B.conv(cw.post, p + ".post", I / 2, Hf, 1, true, 1);
      cw.in.resize(nl);
      cw.rs.resize(nl);
      for (int i = 0; i < nl; ++i) {
        B.conv(cw.in[i], p + ".enc.in_layers." + std::to_string(i), 2 * Hf, Hf, dv.flow_kernel, true, 2);
        B.conv(cw.rs[i], p + ".enc.res_skip_layers." + std::to_string(i), i < nl - 1 ? 2 * Hf : Hf, Hf, 1, true, 1);
      }
      cw.cond_off = add_cond(p + ".enc.cond_layer", 2 * Hf * nl);
    }
  }

  // ---- fused coupling-layer packing (tensor cores): weights in the kernel's schedule order
  {
    const int Hf = dv.flow_hidden, nl = dv.flow_layers, half = I / 2;
    const int nfl = int(dv.couplings.size());
    if (flow_tc_supported(Hf, half, nl, dv.flow_kernel)) {
      for (int a = 0; a < nfl; ++a) {  // a = application order; module = flows.{2*(nfl-1-a)}
        CouplingW& cw = dv.couplings[a];
        const std::string p = "flow.flows." + std::to_string(2 * (nfl - 1 - a));
        const bool rev = ((a + 1) & 1) != 0;  // odd number of Flips so far: halves swapped and reversed
        cw.ftc.x0_coff = rev ? half : 0;
        cw.ftc.x1_coff = rev ? 0 : half;
        auto perm = [&](int ch) { return rev ? half - 1 - ch : ch; };
        while (B.h16.size() % 64) B.h16.push_back(0);
        cw.ftc.woff = B.h16.size();
        auto stage = [&](int K, auto&& wfun) {  // wfun(k, j) -> weight of input k, stage column j
          const size_t o = B.h16.size();
          B.h16.resize(o + size_t(K) * 64, 0);
          for (int k = 0; k < K; ++k)
            for (int j = 0; j < 64; ++j) B.h16[o + (size_t(k / 8) * 64 + j) * 8 + (k & 7)] = B.cvt16(wfun(k, j));
        };
        const OnnxTensor& wpre = hv.need(p + ".pre.weight", {Hf, half, 1});
        const OnnxTensor& bpre = hv.need(p + ".pre.bias", {Hf});
        for (int cc = 0; cc < Hf / 64; ++cc)
          stage(half, [&](int k, int j) { return wpre.f32[size_t(64 * cc + j) * half + perm(k)]; });
        std::vector<float> inb(size_t(nl) * 2 * Hf), cumb(size_t(nl) * Hf), skb(Hf, 0.f), pob(half);
        std::vector<float> run(bpre.f32.begin(), bpre.f32.end());
        for (int i = 0; i < nl; ++i) {
          const std::string is = std::to_string(i);
          const OnnxTensor& win = hv.need(p + ".enc.in_layers." + is + ".weight", {2 * Hf, Hf, dv.flow_kernel});
          const OnnxTensor& bin = hv.need(p + ".enc.in_layers." + is + ".bias", {2 * Hf});
          const int rsn = i < nl - 1 ? 2 * Hf : Hf;
          const OnnxTensor& wrs = hv.need(p + ".enc.res_skip_layers." + is + ".weight", {rsn, Hf, 1});
          const OnnxTensor& brs = hv.need(p + ".enc.res_skip_layers." + is + ".bias", {rsn});
          for (int n = 0; n < 2 * Hf; ++n) inb[size_t(i) * 2 * Hf + n] = bin.f32[n];
          for (int n = 0; n < Hf; ++n) cumb[size_t(i) * Hf + n] = run[n];
          for (int cc = 0; cc < Hf / 32; ++cc)
            for (int tap = 0; tap < dv.flow_kernel; ++tap)
              stage(Hf, [&](int k, int j) {
                const int ch = (j < 32 ? 0 : Hf) + 32 * cc + (j & 31);
                return win.f32[(size_t(ch) * Hf + k) * dv.flow_kernel + tap];
              });
          for (int cc = 0; cc < rsn / 64; ++cc)
            stage(Hf, [&](int k, int j) { return wrs.f32[size_t(64 * cc + j) * Hf + k]; });
          if (i < nl - 1) {
            for (int n = 0; n < Hf; ++n) run[n] += brs.f32[n];
            for (int n = 0; n < Hf; ++n) skb[n] += brs.f32[Hf + n];
          } else {
            for (int n = 0; n < Hf; ++n) skb[n] += brs.f32[n];
          }
        }
        const OnnxTensor& wpo = hv.need(p + ".post.weight", {half, Hf, 1});
        const OnnxTensor& bpo = hv.need(p + ".post.bias", {half});
        for (int cc = 0; cc < (half + 63) / 64; ++cc)
          stage(Hf, [&](int k, int j) {
            const int n = 64 * cc + j;
            return n < half ? wpo.f32[size_t(perm(n)) * Hf + k] : 0.f;
          });
        for (int n = 0; n < half; ++n) pob[n] = bpo.f32[perm(n)];
        B.place(&cw.ftc.in_bias, inb);
        B.place(&cw.ftc.cum_bias, cumb);
        B.place(&cw.ftc.skip_bias, skb);
        B.place(&cw.ftc.post_bias, pob);
        cw.ftc.ok = true;

        // ---- second-generation stream (kernels_tc_flow2.cu): every block [K/8][N][8] with K x N = 192 x 96 or 96 x 192
        if (flow2_tc_supported(Hf, half, nl, dv.flow_kernel)) {
          while (B.h16.size() % 64) B.h16.push_back(0);
          cw.ftc.woff2 = B.h16.size();
          auto block = [&](int K, int N, auto&& wfun) {  // wfun(k, n) -> weight of input k, output column n
            const size_t o = B.h16.size();
            B.h16.resize(o + size_t(K) * N, 0);
            for (int k = 0; k < K; ++k)
              for (int n = 0; n < N; ++n) B.h16[o + (size_t(k / 8) * N + n) * 8 + (k & 7)] = B.cvt16(float(wfun(k, n)));
          };
          block(half, Hf, [&](int k, int n) { return wpre.f32[size_t(n) * half + perm(k)]; });
          std::vector<double> mb(half, 0.0);
          for (int n = 0; n < half; ++n) {
            double acc = bpo.f32[perm(n)];
            for (int sidx = 0; sidx < Hf; ++sidx) acc += double(wpo.f32[size_t(perm(n)) * Hf + sidx]) * double(skb[sidx]);
            mb[n] = acc;
          }
          for (int i = 0; i < nl; ++i) {
            const std::string is = std::to_string(i);
            const OnnxTensor& win = hv.need(p + ".enc.in_layers." + is + ".weight", {2 * Hf, Hf, dv.flow_kernel});
            const int rsn = i < nl - 1 ? 2 * Hf : Hf;
            const OnnxTensor& wrs = hv.need(p + ".enc.res_skip_layers." + is + ".weight", {rsn, Hf, 1});
            for (int cc = 0; cc < Hf / 48; ++cc)
              for (int tap = 0; tap < dv.flow_kernel; ++tap)
                block(Hf, 96, [&](int k, int j) {
                  const int ch = (j < 48 ? 0 : Hf) + 48 * cc + (j % 48);
                  return win.f32[(size_t(ch) * Hf + k) * dv.flow_kernel + tap];
                });
            if (i < nl - 1)
              for (int kh = 0; kh < 2; ++kh)
                block(Hf / 2, Hf, [&](int k, int n) { return wrs.f32[size_t(n) * Hf + kh * (Hf / 2) + k]; });
            // m-update: W'[n][k] = sum_s W_post[perm(n)][s] . W_skip_i[s][k]  (fp64 on the host, one rounding to 16 bits)
            const size_t skip_row0 = i < nl - 1 ? size_t(Hf) : 0;
            std::vector<double> wp(size_t(half) * Hf, 0.0);
            for (int n = 0; n < half; ++n)
              for (int sidx = 0; sidx < Hf; ++sidx) {
                const double a = wpo.f32[size_t(perm(n)) * Hf + sidx];
                const float* wrow = &wrs.f32[(skip_row0 + sidx) * Hf];
                double* dst = &wp[size_t(n) * Hf];
                for (int k = 0; k < Hf; ++k) dst[k] += a * double(wrow[k]);
              }
            block(Hf, half, [&](int k, int n) { return wp[size_t(n) * Hf + k]; });
          }
          std::vector<float> mbf(mb.begin(), mb.end());
          B.place(&cw.ftc.m_bias, mbf);
          cw.ftc.ok2 = B.h16.size() - cw.ftc.woff2 == flow2_tc_weight_elems(nl);
        }
      }
    }
  }

  // ---- HiFi-GAN decoder
  {
    const int C0 = c.up_init;
    B.conv(dv.dec_pre, "dec.conv_pre", C0, I, 7, true, 1);
    dv.dec_cond_off = add_cond("dec.cond", C0);
    const int nk = int(c.rb_kernels.size());
    dv.ups.resize(c.up_rates.size());
    dv.rbs.resize(c.up_rates.size() * nk);
    for (size_t i = 0; i < c.up_rates.size(); ++i) {
      UpW& u = dv.ups[i];
      u.cin = C0 >> i;
      u.cout = C0 >> (i + 1);
      u.k = c.up_kernels[i];
      u.u = c.up_rates[i];
      if ((u.k - u.u) < 0 || ((u.k - u.u) & 1))
        throw EngineError(3, "config.json: upsample kernel/rate pair not supported (need k >= u, k-u even)");
      u.pad = (u.k - u.u) / 2;
      u.ntaps = (u.k + u.u - 1) / u.u;
      const OnnxTensor& w = hv.need("dec.ups." + std::to_string(i) + ".weight", {u.cin, u.cout, u.k});
      std::vector<float> t(size_t(u.u) * u.ntaps * u.cin * u.cout, 0.f);
      for (int j1 = 0; j1 < u.u; ++j1)
        for (int mp = 0; mp < u.ntaps; ++mp) {
          const int m = u.ntaps - 1 - mp, j = j1 + m * u.u;
          if (j >= u.k) continue;
          for (int ci = 0; ci < u.cin; ++ci)
            for (int co = 0; co < u.cout; ++co)
              t[((size_t(j1) * u.ntaps + mp) * u.cin + ci) * u.cout + co] = w.f32[(size_t(ci) * u.cout + co) * u.k + j];
        }
      if (u.cin % 16 == 0 && u.cout % 4 == 0) {
        // logical [tap m'][ci][phase*Cout + co] for the polyphase GEMM (N = u * Cout)
        std::vector<float> lw(size_t(u.ntaps) * u.cin * u.u * u.cout, 0.f);
        for (int j1 = 0; j1 < u.u; ++j1)
          for (int mp = 0; mp < u.ntaps; ++mp)
            for (int ci = 0; ci < u.cin; ++ci)
              for (int co = 0; co < u.cout; ++co)
                lw[(size_t(mp) * u.cin + ci) * (u.u * u.cout) + j1 * u.cout + co] =
                    t[((size_t(j1) * u.ntaps + mp) * u.cin + ci) * u.cout + co];
        B.tc_pack(u.tc, lw, u.ntaps, u.cin, u.u * u.cout, 1, false);
      }
      B.place(&u.w, t);
      B.n_params += w.numel();
      B.vec(&u.b, "dec.ups." + std::to_string(i) + ".bias", u.cout);
      // ResBlock1 stage on tensor cores: every conv of the stage is also packed for conv_tc_kernel, or none is
      bool rb1_tc = c.resblock != "2" && nk >= 1 && nk <= 4;
      if (rb1_tc) {
        const int nd = int(c.rb_dils[0].size());
        int ks[4] = {}, dl[4][3] = {};
        for (int j = 0; j < nk; ++j) {
          ks[j] = c.rb_kernels[j];
          if (int(c.rb_dils[j].size()) != nd || nd > 3) rb1_tc = false;
          for (int d = 0; d < nd && d < 3; ++d) dl[j][d] = c.rb_dils[j][d];
        }
        rb1_tc = rb1_tc && mrf1_tc_supported(u.cout, nk, nd, ks, dl);
      }
      for (int j = 0; j < nk; ++j) {
        // NOTE: Builder records the address of every pointer slot, so the Lin objects must
        // already sit at their final address (pre-sized vectors, no copies afterwards).
        ResBlockW& rb = dv.rbs[i * nk + j];
        rb.k = c.rb_kernels[j];
        rb.dil = c.rb_dils[j];
        const std::string rp = "dec.resblocks." + std::to_string(i * nk + j);
        rb.c1.resize(rb.dil.size());
        if (c.resblock != "2") rb.c2.resize(rb.dil.size());
        for (size_t d = 0; d < rb.dil.size(); ++d) {
          if (c.resblock == "2") {
            B.conv(rb.c1[d], rp + ".convs." + std::to_string(d), u.cout, u.cout, rb.k);
          } else {
            B.conv(rb.c1[d], rp + ".convs1." + std::to_string(d), u.cout, u.cout, rb.k, true, rb1_tc ? 1 : 0, rb.dil[d]);
            B.conv(rb.c2[d], rp + ".convs2." + std::to_string(d), u.cout, u.cout, rb.k, true, rb1_tc ? 1 : 0);
          }
        }
      }
    }
    const int cl = C0 >> c.up_rates.size();
    const OnnxTensor& pw = hv.need("dec.conv_post.weight", {});
    if (pw.dims.size() != 3 || pw.dims[0] != 1 || pw.dims[1] != cl)
      throw EngineError(3, "generator.onnx: bad dec.conv_post.weight shape");
    dv.post_k = int(pw.dims[2]);
    dv.post_c = cl;
    std::vector<float> t(size_t(dv.post_k) * cl);
    for (int ci = 0; ci < cl; ++ci)
      for (int j = 0; j < dv.post_k; ++j) t[size_t(j) * cl + ci] = pw.f32[size_t(ci) * dv.post_k + j];
    B.place(&dv.post_w, t);
    B.n_params += pw.numel();
  }

  // ---- tensor-core operands of the MRF stages: per conv [tap][Cin/8][Cout][8], 16-bit
  std::vector<uint16_t>& h16 = B.h16;
  {
    auto cvt = [&](float f) -> uint16_t { return B.cvt16(f); };
    const int nk = int(c.rb_kernels.size());
    dv.mrf.resize(c.up_rates.size());
    for (size_t i = 0; i < c.up_rates.size(); ++i) {
      MrfStageW& ms = dv.mrf[i];
      const int C = c.up_init >> (i + 1);
      int ks[4] = {0, 0, 0, 0};
      int nd = nk ? int(c.rb_dils[0].size()) : 0;
      bool uniform = c.resblock == "2" && nk <= 4;
      for (int j = 0; j < nk && j < 4; ++j) {
        ks[j] = c.rb_kernels[j];
        if (int(c.rb_dils[j].size()) != nd) uniform = false;
      }
      int HX = 0, HY = 0;
      for (int j = 0; j < nk && uniform; ++j) {
        HX = std::max(HX, c.rb_dils[j][0] * (c.rb_kernels[j] - 1) / 2);
        if (nd > 1) HY = std::max(HY, c.rb_dils[j][1] * (c.rb_kernels[j] - 1) / 2);
      }
      if (!uniform || !mrf_tc_supported(C, nk, nd, ks, std::max(HX, HY))) continue;
      ms.ok = true;
      ms.nk = nk;
      ms.nd = nd;
      ms.HX = HX;
      ms.HY = HY;
      ms.H = HY;
      std::vector<float> late(C, 0.f);
      for (int j = 0; j < nk; ++j)
        for (int d = 0; d < nd; ++d) {
          const std::string nm = "dec.resblocks." + std::to_string(i * nk + j) + ".convs." + std::to_string(d);
          const int k = c.rb_kernels[j];
          const OnnxTensor& w = hv.need(nm + ".weight", {C, C, k});
          const OnnxTensor& bsrc = hv.need(nm + ".bias", {C});
          if (d >= 1)
            for (int ch = 0; ch < C; ++ch) late[ch] += bsrc.f32[ch];
          while (h16.size() % 64) h16.push_back(0);
          ms.woff[j][d] = h16.size();
          const size_t o = h16.size();
          h16.resize(o + size_t(k) * C * C);
          for (int tap = 0; tap < k; ++tap)
            for (int ci = 0; ci < C; ++ci)
              for (int co = 0; co < C; ++co)
                h16[o + ((size_t(tap) * (C / 8) + ci / 8) * C + co) * 8 + (ci & 7)] = cvt(w.f32[(size_t(co) * C + ci) * k + tap]);
        }
      B.place(&ms.late_bias, late);
    }
  }

  // ---- fused last stage (ConvTranspose + MRF + conv_post): extra operand packings
  if (!c.up_rates.empty() && !dv.mrf.empty()) {
    const size_t li = c.up_rates.size() - 1;
    const UpW& u = dv.ups[li];
    const MrfStageW& ms = dv.mrf[li];
    const int C = u.cout;
    if (ms.ok && dv.post_c == C && dv.post_k == 7 &&
        dec_last_supported(C, u.cin, u.k, u.u, ms.nk, ms.nd, ms.HX, ms.HY)) {
      const OnnxTensor& w = hv.need("dec.ups." + std::to_string(li) + ".weight", {u.cin, u.cout, u.k});
      while (B.h16.size() % 64) B.h16.push_back(0);
      dv.dec_last.up_woff = B.h16.size();
      {  // conv over the zero-stuffed input: W'[jj][ci][co] = w[ci][co][k-1-jj], layout [jj][cin/8][C][8]
        const size_t o = B.h16.size();
        B.h16.resize(o + size_t(u.k) * u.cin * C, 0);
        for (int jj = 0; jj < u.k; ++jj)
          for (int ci = 0; ci < u.cin; ++ci)
            for (int co = 0; co < C; ++co)
              B.h16[o + ((size_t(jj) * (u.cin / 8) + ci / 8) * C + co) * 8 + (ci & 7)] =
                  B.cvt16(w.f32[(size_t(ci) * u.cout + co) * u.k + (u.k - 1 - jj)]);
      }
      const OnnxTensor& pw = hv.need("dec.conv_post.weight", {1, C, 7});
      while (B.h16.size() % 64) B.h16.push_back(0);
      dv.dec_last.post_woff = B.h16.size();
      {  // [tap][C/8][16][8], output column 0 is the real one
        const size_t o = B.h16.size();
        B.h16.resize(o + size_t(7) * C * 16, 0);
        for (int tap = 0; tap < 7; ++tap)
          for (int ci = 0; ci < C; ++ci)
            B.h16[o + ((size_t(tap) * (C / 8) + ci / 8) * 16 + 0) * 8 + (ci & 7)] = B.cvt16(pw.f32[size_t(ci) * 7 + tap]);
      }
      dv.dec_last.ok = true;

      // ---- persistent fused kernel: every operand of the stage in one blob (polyphase transposed conv)
      DecLastW& dl = dv.dec_last;
      bool shape_ok = ms.nk == 3 && ms.nd == 2 && u.k == 2 * u.u;
      if (shape_ok) {
        for (int j = 0; j < 3; ++j) {
          dl.HYb[j] = std::max(c.rb_dils[j][1] * (c.rb_kernels[j] - 1) / 2, j == 0 ? 3 : 0);
        }
        while (B.h16.size() % 64) B.h16.push_back(0);
        dl.blob_off = B.h16.size();
        auto here = [&] {
          while (B.h16.size() % 64) B.h16.push_back(0);
          return unsigned((B.h16.size() - dl.blob_off) * 2);
        };
        dl.f_up = here();
        {
          const int N = u.u * C;
          const size_t o = B.h16.size();
          B.h16.resize(o + size_t(2) * u.cin * N, 0);
          for (int d = 0; d < 2; ++d)
            for (int ci = 0; ci < u.cin; ++ci)
              for (int ph = 0; ph < u.u; ++ph)
                for (int co = 0; co < C; ++co)
                  B.h16[o + ((size_t(d) * (u.cin / 8) + ci / 8) * N + ph * C + co) * 8 + (ci & 7)] =
                      B.cvt16(w.f32[(size_t(ci) * u.cout + co) * u.k + (u.u * d + ph)]);
        }
        for (int j = 0; j < 3; ++j)
          for (int d = 0; d < 2; ++d) {
            const unsigned off = here();
            (d == 0 ? dl.f_c1 : dl.f_c2)[j] = off;
            const size_t n = size_t(c.rb_kernels[j]) * C * C;
            const size_t src = ms.woff[j][d], o = B.h16.size();
            B.h16.resize(o + n);
            std::copy(B.h16.begin() + src, B.h16.begin() + src + n, B.h16.begin() + o);
          }
        dl.f_post = here();
        {
          const size_t n = size_t(7) * C * 16, src = dl.post_woff, o = B.h16.size();
          B.h16.resize(o + n);
          std::copy(B.h16.begin() + src, B.h16.begin() + src + n, B.h16.begin() + o);
        }
        dl.blob_bytes = here();
        dl.f_postp = here();
        {  // conv_post for the phase-major kernel (kernels.h: kDecPostPlanesBytes); the v2 kernel never loads past blob_bytes
          const size_t o = B.h16.size();
          B.h16.resize(o + kDecPostPlanesBytes / 2, 0);
          int pair = 0;
          for (int sh = -1; sh <= 1; ++sh)
            for (int pi = 0; pi < 4; ++pi) {
              if ((sh < 0 && pi == 0) || (sh > 0 && pi == 3)) continue;
              for (int php = 0; php < 4; ++php) {
                const int tap = 4 * sh + pi - php + 3;
                if (tap < 0 || tap > 6) continue;
                for (int ci = 0; ci < C; ++ci)
                  B.h16[o + ((size_t(pair) * (C / 8) + ci / 8) * 16 + php) * 8 + (ci & 7)] = B.cvt16(pw.f32[size_t(ci) * 7 + tap]);
              }
              ++pair;
            }
        }
        dl.fused_ok = dec_fused_supported(C, u.cin, u.k, u.u, ms.nk, ms.nd, ms.HX, dl.HYb, dl.blob_bytes);
        dl.planes_ok = dl.fused_ok && dec_planes_supported(C, u.cin, u.k, u.u, ms.nk, ms.nd, ms.HX, dl.HYb, dl.f_post + kDecPostPlanesBytes);
      }
    }
  }

  // ---- conditioning GEMM [G][n_cond]
  if (G && !cond_layers.empty()) {
    int n = 0;
    for (auto& p : cond_layers) n += p.second;
    dv.n_cond = n;
    std::vector<float> w(size_t(G) * n), b(n);
    int off = 0;
    for (auto& p : cond_layers) {
      const OnnxTensor& t = hv.need(p.first + ".weight", {p.second, G, 1});
      const OnnxTensor& tb = hv.need(p.first + ".bias", {p.second});
      for (int o = 0; o < p.second; ++o) {
        for (int g = 0; g < G; ++g) w[size_t(g) * n + off + o] = t.f32[size_t(o) * G + g];
        b[off + o] = tb.f32[o];
      }
      off += p.second;
      B.n_params += t.numel() + tb.numel();
    }
    B.place(&dv.cond_all.w, w);
    B.place(&dv.cond_all.b, b);
    dv.cond_all.cin = G;
    dv.cond_all.cout = n;
    dv.cond_all.taps = 1;
  }
  dv.cfg.gin = G;

  dv.n_params = B.n_params;
  dv.slab_floats = B.pk.host.size();
  pv.f32 = std::move(B.pk.host);
  pv.h16 = std::move(B.h16);
  pv.fix.reserve(B.fix.size());
  for (auto& f : B.fix) pv.fix.emplace_back(f.slot, f.off);
  pv.pack_flags = pack_flags_string();
  return pv;
}

// Everything pack_voice reads from the environment (part of the weight-cache key: a blob packed under other
// switches must not be picked up).
std::string pack_flags_string() {
  auto env = [](const char* n) {
    const char* e = getenv(n);
    return std::string(e ? e : "");
  };
  return "fmt=" + env("M3B200_TC_FORMAT") + ";simt=" + env("M3B200_FORCE_SIMT") + ";text_simt=" + env("M3B200_TEXT_SIMT") +
         ";rows_nc=" + env("M3B200_ROWGEMM_NC");
}

void require_sm100(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    throw EngineError(M3_ERR_NOGPU, "no CUDA device visible: libm3b200 has no CPU fallback");
  }
  if (device < 0 || device >= n) throw EngineError(M3_ERR_INVALID, "device ordinal out of range");
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (major != 10)
    throw EngineError(M3_ERR_NOGPU, "device " + std::to_string(device) + " is compute capability " +
                                        std::to_string(major) + ".x; this library carries sm_100a code only");
}

// Upload of the two slabs (everything before this is host-only, so model errors surface without a GPU).
void upload_slabs(DeviceVoice& dv, int device, const float* f32, size_t n_f32, const uint16_t* h16, size_t n_h16) {
  require_sm100(device);
  M3_CUDA(cudaSetDevice(device));
  dv.device = device;
  dv.slab_floats = n_f32;
  M3_CUDA(cudaMalloc(&dv.slab, std::max<size_t>(n_f32, 1) * sizeof(float)));
  M3_CUDA(cudaMemcpy(dv.slab, f32, n_f32 * sizeof(float), cudaMemcpyHostToDevice));
  if (n_h16) {
    M3_CUDA(cudaMalloc(&dv.slab16, n_h16 * sizeof(uint16_t)));
    M3_CUDA(cudaMemcpy(dv.slab16, h16, n_h16 * sizeof(uint16_t), cudaMemcpyHostToDevice));
  }
}

std::unique_ptr<DeviceVoice> upload_voice(PackedVoice&& pv, int device) {
  upload_slabs(*pv.dv, device, pv.f32.data(), pv.f32.size(), pv.h16.data(), pv.h16.size());
  for (auto& f : pv.fix) *f.first = pv.dv->slab + f.second;
  return std::move(pv.dv);
}

std::unique_ptr<DeviceVoice> build_device_voice(const HostVoice& hv, int device) {
  return upload_voice(pack_voice(hv), device);
}

// ======================================================================================
// the pipeline
// ======================================================================================
namespace {

struct Segs {
  const int* off;
  const int* len;
  int n;
  int max_len;
};

struct Run {
  DeviceVoice& dv;
  Context& cx;
  cudaStream_t st;
  Result* res;
  bool debug;
  bool timing = false;
  mutable std::vector<std::string> mark_names;

  // stage boundary: time between consecutive marks is reported as "ms:<name of the later mark>"
  void mark(const char* name) const {
    if (!timing) return;
    const size_t i = mark_names.size();
    if (cx.marks.size() <= i) {
      cudaEvent_t e;
      M3_CUDA(cudaEventCreate(&e));
      cx.marks.push_back(e);
    }
    M3_CUDA(cudaEventRecord(cx.marks[i], st));
    mark_names.push_back(name);
  }
  void collect_marks() const {
    if (!timing) return;
    for (size_t i = 1; i < mark_names.size(); ++i) {
      float ms = 0;
      M3_CUDA(cudaEventElapsedTime(&ms, cx.marks[i - 1], cx.marks[i]));
      DebugTensor& t = res->debug["ms:" + mark_names[i]];
      if (t.data.empty()) {
        t.rows = t.cols = 1;
        t.data.assign(1, 0.f);
      }
      t.data[0] += ms;
    }
  }

  ConvParams base_conv(const Lin& l, const float* in, int in_stride, float* out, int out_stride, const Segs& s,
                       int scale) const {
    ConvParams p;
    p.in = in;
    p.in_stride = in_stride;
    p.Cin = l.cin;
    p.W = l.w;
    p.Cout = l.cout;
    p.taps = l.taps;
    p.pad_left = (l.taps - 1) / 2;
    p.bias = l.b;
    p.out = out;
    p.out_stride = out_stride;
    p.seg_off = s.off;
    p.seg_len = s.len;
    p.in_scale = scale;
    p.out_scale = scale;
    return p;
  }
  void conv(const ConvParams& p, const Segs& s) const { launch_conv(p, s.n, s.max_len, st); }

  // token-level fp32 convs over packed rows
  const int4* rowinfo = nullptr;
  int n_rows = 0;
  const int* vmap = nullptr;
  int vrows = 0;
  void row_conv(const Lin& l, const float* in, int in_stride, float* out, int out_stride, int act = 0,
                const float* ub = nullptr, int ub_stride = 0) const {
    if (dv.use_rows_tc && l.rtc.ok && (l.taps == 1 || l.taps == 3)) {
      RowGemmTcParams q;
      q.in = in;
      q.in_stride = in_stride;
      q.K = l.cin;
      q.w = dv.slab16 + l.rtc.woff;
      q.N = l.cout;
      q.taps = l.taps;
      q.nc = l.rtc.nc;
      q.pad_left = (l.taps - 1) / 2;
      q.bias = l.b;
      q.ubias = ub;
      q.ub_stride = ub_stride;
      q.act = act;
      q.out = out;
      q.out_stride = out_stride;
      q.vmap = vmap;
      q.rowinfo = rowinfo;
      q.vrows = vrows;
      launch_rowgemm_tc(q, st);
      return;
    }
    RowConvParams p;
    p.in = in;
    p.in_stride = in_stride;
    p.Cin = l.cin;
    p.W = l.w;
    p.Cout = l.cout;
    p.taps = l.taps;
    p.pad_left = (l.taps - 1) / 2;
    p.bias = l.b;
    p.ubias = ub;
    p.ub_stride = ub_stride;
    p.act = act;
    p.out = out;
    p.out_stride = out_stride;
    p.rowinfo = rowinfo;
    p.rows = n_rows;
    launch_row_conv(p, st);
  }

  bool tc_ok(const TcConvW& t) const { return dv.use_tc && t.ok; }
  TcConvParams base_tc(const TcConvW& t, const float* bias, const float* in, int in_stride, float* out,
                       int out_stride, const Segs& s, int scale) const {
    TcConvParams p;
    p.in = in;
    p.in_stride = in_stride;
    p.K = t.K;
    p.w = dv.slab16 + t.woff;
    p.NC = t.NC;
    p.n_chunks = t.n_chunks;
    p.N = t.N;
    p.taps = t.taps;
    p.pad_left = (t.taps - 1) / 2;
    p.bias = bias;
    p.out = out;
    p.out_stride = out_stride;
    p.seg_off = s.off;
    p.seg_len = s.len;
    p.in_scale = scale;
    p.out_scale = scale;
    return p;
  }
  void tc_conv(const TcConvParams& p, const Segs& s) const { launch_conv_tc(p, dv.tc_fmt, s.n, s.max_len, st); }

  void dump(const char* name, const float* d, int64_t rows, int64_t cols) const {
    if (!debug) return;
    DebugTensor t;
    t.rows = rows;
    t.cols = cols;
    t.data.resize(size_t(rows * cols));
    M3_CUDA(cudaStreamSynchronize(st));
    M3_CUDA(cudaMemcpy(t.data.data(), d, t.data.size() * sizeof(float), cudaMemcpyDeviceToHost));
    res->debug[name] = std::move(t);
  }

  // DDSConv (modules.DDSConv [EXT]): x updated in place; tmp1/tmp2 scratch [rows][C]
  void dds(const DDSW& d, float* x, float* tmp1, float* tmp2, int C, const Segs& s, int rows) const {
    int dil = 1;
    for (int i = 0; i < 3; ++i) {
      launch_dds_sep(x, d.sep_w[i], d.sep_b[i], d.n1g[i], d.n1b[i], tmp1, C, dil, s.off, s.len, s.n, s.max_len, st);
      row_conv(d.c1x1[i], tmp1, C, tmp2, C);
      launch_layernorm(tmp2, nullptr, x, d.n2g[i], d.n2b[i], x, rows, C, 1, st);
      dil *= 3;
    }
  }
};

}  // namespace

void write_wav_header(uint8_t* h, int sample_rate, int64_t n_samples) {
  const uint32_t data = uint32_t(n_samples * 2);
  auto u32 = [&](int o, uint32_t v) {
    for (int i = 0; i < 4; ++i) h[o + i] = uint8_t(v >> (8 * i));
  };
  auto u16 = [&](int o, uint32_t v) {
    h[o] = uint8_t(v);
    h[o + 1] = uint8_t(v >> 8);
  };
  memcpy(h, "RIFF", 4);
  u32(4, 36u + data);
  memcpy(h + 8, "WAVEfmt ", 8);
  u32(16, 16u);
  u16(20, 1u);   // PCM
  u16(22, 1u);   // mono
  u32(24, uint32_t(sample_rate));
  u32(28, uint32_t(sample_rate) * 2u);
  u16(32, 2u);   // block align
  u16(34, 16u);  // bits per sample
  memcpy(h + 36, "data", 4);
  u32(40, data);
}

Result* run_inference(Voice& v, const int64_t* ids, const int64_t* lengths, int batch, int t_stride,
                      const float* scales, const int64_t* sid, uint64_t seed, uint32_t flags, const InferOpts* opts) {
  DeviceVoice& dv = *v.dv;
  const VoiceConfig& c = dv.cfg;
  const InferOpts no_opts;
  const InferOpts& o = opts ? *opts : no_opts;
  if (batch <= 0) throw EngineError(M3_ERR_INVALID, "batch must be >= 1");
  if (!ids || !lengths) throw EngineError(M3_ERR_INVALID, "ids and lengths must not be NULL");
  if (!scales && !o.row_scales) throw EngineError(M3_ERR_INVALID, "scales (or per-utterance row_scales) must not be NULL");
  if (t_stride <= 0) throw EngineError(M3_ERR_INVALID, "input has zero phonemes");
  if (dv.has_emb_g && !sid) throw EngineError(M3_ERR_INVALID, "multi-speaker voice: input 'sid' is required");
  const bool post = o.post_chain();
  if (post && (flags & M3_FLAG_KEEP_FLOAT))
    throw EngineError(M3_ERR_INVALID, "M3_FLAG_KEEP_FLOAT cannot be combined with the PCM post chain (volume / silence / WAV)");
  for (int b = 0; b < batch; ++b) {
    if (o.row_scales)
      for (int k = 0; k < 3; ++k)
        if (!std::isfinite(o.row_scales[3 * b + k]))
          throw EngineError(M3_ERR_INVALID, "row_scales[" + std::to_string(b) + "] is not finite");
    if (o.volume && !std::isfinite(o.volume[b])) throw EngineError(M3_ERR_INVALID, "volume[" + std::to_string(b) + "] is not finite");
    if ((o.lead_silence && o.lead_silence[b] < 0) || (o.trail_silence && o.trail_silence[b] < 0))
      throw EngineError(M3_ERR_INVALID, "silence[" + std::to_string(b) + "] is negative");
  }
  const float noise_scale = scales ? scales[0] : 0.f, length_scale = scales ? scales[1] : 1.f, noise_w = scales ? scales[2] : 0.f;
  const bool ids_on_device = flags & M3_FLAG_DEVICE_IDS;

  std::vector<int> tok_off(batch), tok_len(batch);
  int NT = 0, Tmax = 0;
  for (int b = 0; b < batch; ++b) {
    if (lengths[b] <= 0 || lengths[b] > t_stride)
      throw EngineError(M3_ERR_INVALID, "input_lengths[" + std::to_string(b) + "]=" + std::to_string(lengths[b]) +
                                            " outside [1, " + std::to_string(t_stride) + "]");
    tok_off[b] = NT;
    tok_len[b] = int(lengths[b]);
    NT += tok_len[b];
    Tmax = std::max(Tmax, tok_len[b]);
  }
  if (sid && dv.has_emb_g)
    for (int b = 0; b < batch; ++b)
      if (sid[b] < 0 || sid[b] >= c.n_speakers)
        throw EngineError(M3_ERR_INVALID, "sid[" + std::to_string(b) + "]=" + std::to_string(sid[b]) +
                                              " outside [0, " + std::to_string(c.n_speakers) + ")");
  if (!ids_on_device)
    for (int b = 0; b < batch; ++b)
      for (int t = 0; t < tok_len[b]; ++t) {
        const int64_t id = ids[size_t(b) * t_stride + t];
        if (id < 0 || id >= c.num_symbols)
          throw EngineError(M3_ERR_INVALID, "input[" + std::to_string(b) + "][" + std::to_string(t) + "]=" +
                                                std::to_string(id) + " outside [0, " + std::to_string(c.num_symbols) + ")");
      }

  M3_CUDA(cudaSetDevice(dv.device));
  Context* cxp = v.acquire();
  std::unique_ptr<Result> res(new Result());
  res->batch = batch;
  res->owner = &v;
  res->ctx = cxp;
  struct Lease {
    Voice& v;
    Context* c;
    bool keep = false;
    ~Lease() {
      if (!keep) v.release(c);
    }
  } lease{v, cxp};
  Context& cx = *cxp;
  cudaStream_t st = cx.stream;
  g_launch_count = 0;
  Run R{dv, cx, st, res.get(), (flags & M3_FLAG_DEBUG_TENSORS) != 0};
  R.timing = (flags & M3_FLAG_STAGE_TIMING) != 0;
  R.mark("start");

  const int H = c.hidden, I = c.inter, Ff = c.filter, Fd = dv.dp_ch;
  const int G = c.gin;

  // ---------------- phase 1 workspace (token level) ----------------
  {
    size_t fl = size_t(NT) * (size_t(H) * 3 + 3 * H + Ff + 2 * I + size_t(Fd) * 4 + 40) + size_t(batch) * (G + dv.n_cond + 8);
    size_t bytes = fl * 4 + size_t(batch) * t_stride * 8 + size_t(batch) * 64 + (1 << 16) + 512 * 64 + size_t(NT) * 16 + (size_t(NT) + batch) * 4;
    cx.a1.reserve(bytes);
  }
  Arena& A = cx.a1;
  int* d_meta = A.alloc<int>(size_t(batch) * 4 + 4);  // tok_off | tok_len | frm_off | frm_len
  int* d_tok_off = d_meta;
  int* d_tok_len = d_meta + batch;
  int* d_frm_off = d_meta + 2 * batch;
  int* d_frm_len = d_meta + 3 * batch;
  int64_t* d_ids = nullptr;
  int64_t* d_sid = A.alloc<int64_t>(batch);
  int* d_one = A.alloc<int>(4);  // {0, batch}: a single segment of `batch` rows

  // stage host inputs in pinned memory, one async copy each
  cx.h_meta.reserve(size_t(batch) * 4 * sizeof(int) + size_t(batch) * 8 + 64);
  int* hm = static_cast<int*>(cx.h_meta.p);
  memcpy(hm, tok_off.data(), batch * sizeof(int));
  memcpy(hm + batch, tok_len.data(), batch * sizeof(int));
  M3_CUDA(cudaEventRecord(cx.ev0, st));
  M3_CUDA(cudaMemcpyAsync(d_meta, hm, size_t(batch) * 2 * sizeof(int), cudaMemcpyHostToDevice, st));
  {
    int* ho = hm + 4 * batch;
    ho[0] = 0;
    ho[1] = batch;
    M3_CUDA(cudaMemcpyAsync(d_one, ho, 2 * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  if (ids_on_device) {
    d_ids = const_cast<int64_t*>(ids);
  } else {
    d_ids = A.alloc<int64_t>(size_t(batch) * t_stride);
    cx.h_in.reserve(size_t(batch) * t_stride * 8);
    memcpy(cx.h_in.p, ids, size_t(batch) * t_stride * 8);
    M3_CUDA(cudaMemcpyAsync(d_ids, cx.h_in.p, size_t(batch) * t_stride * 8, cudaMemcpyHostToDevice, st));
  }
  // per-utterance settings (Mimic3Settings of each sentence, tts.py:519-528): staged once, read by the
  // noise / duration / prior kernels instead of the scalar scales
  float* d_row_scales = nullptr;
  cx.h_opts.reserve(size_t(batch) * (3 * sizeof(float) + sizeof(long long) + sizeof(double)) + 64);
  if (o.row_scales) {
    d_row_scales = A.alloc<float>(size_t(batch) * 3);
    memcpy(cx.h_opts.p, o.row_scales, size_t(batch) * 3 * sizeof(float));
    M3_CUDA(cudaMemcpyAsync(d_row_scales, cx.h_opts.p, size_t(batch) * 3 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  Segs tok{d_tok_off, d_tok_len, batch, Tmax};
  Segs one{d_one, d_one + 1, 1, batch};
  {
    int4* d_rowinfo = A.alloc<int4>(NT);
    launch_fill_rowinfo(d_rowinfo, d_tok_off, d_tok_len, batch, Tmax, st);
    R.rowinfo = d_rowinfo;
    R.n_rows = NT;
    int* d_vmap = A.alloc<int>(size_t(NT) + batch);
    launch_fill_vmap(d_vmap, d_tok_off, d_tok_len, batch, Tmax, st);
    R.vmap = d_vmap;
    R.vrows = NT + batch;
  }

  // ---------------- speaker conditioning ----------------
  float* d_cond = nullptr;  // [batch][n_cond]
  if (dv.has_emb_g && dv.n_cond) {
    int64_t* hs = reinterpret_cast<int64_t*>(hm + 4 * batch + 8);
    memcpy(hs, sid, size_t(batch) * 8);
    M3_CUDA(cudaMemcpyAsync(d_sid, hs, size_t(batch) * 8, cudaMemcpyHostToDevice, st));
    float* d_g = A.alloc<float>(size_t(batch) * G);
    d_cond = A.alloc<float>(size_t(batch) * dv.n_cond);
    launch_gather_rows(d_sid, dv.emb_g, d_g, batch, G, st);
    ConvParams p = R.base_conv(dv.cond_all, d_g, G, d_cond, dv.n_cond, one, 1);
    R.conv(p, one);
  }
  auto ubias = [&](int off) -> const float* { return (d_cond && off >= 0) ? d_cond + off : nullptr; };

  // ---------------- A.1 text encoder ----------------
  float* x = A.alloc<float>(size_t(NT) * H);
  float* qkv = A.alloc<float>(size_t(NT) * 3 * H);
  float* att = A.alloc<float>(size_t(NT) * H);
  float* y = A.alloc<float>(size_t(NT) * H);
  float* ffn = A.alloc<float>(size_t(NT) * Ff);
  float* stats = A.alloc<float>(size_t(NT) * 2 * I);
  launch_embedding(d_ids, t_stride, dv.emb, c.num_symbols, sqrtf(float(H)), x, H, d_tok_off, d_tok_len, batch, Tmax, st);
  for (int l = 0; l < c.n_layers; ++l) {
    const EncLayerW& L = dv.enc[l];
    R.row_conv(L.qkv, x, H, qkv, 3 * H);
    launch_attention(qkv, L.ek, L.ev, att, H, c.n_heads, dv.window, d_tok_off, d_tok_len, batch, Tmax, st);
    R.row_conv(L.o, att, H, y, H);
    launch_layernorm(x, y, nullptr, L.g1, L.b1, x, NT, H, 0, st);
    // attentions.FFN "same" padding: pad_l = (k-1)//2, pad_r = k//2
    R.row_conv(L.ffn1, x, H, ffn, Ff, 1);
    R.row_conv(L.ffn2, ffn, Ff, y, H);
    launch_layernorm(x, y, nullptr, L.g2, L.b2, x, NT, H, 0, st);
  }
  R.row_conv(dv.enc_proj, x, H, stats, 2 * I);
  R.mark("text_encoder");
  R.dump("x", x, NT, H);
  R.dump("stats", stats, NT, 2 * I);

  // ---------------- A.2 duration predictor ----------------
  float* logw = A.alloc<float>(NT);
  if (dv.use_sdp) {
    float* h = A.alloc<float>(size_t(NT) * Fd);
    float* u = A.alloc<float>(size_t(NT) * Fd);
    float* t1 = A.alloc<float>(size_t(NT) * Fd);
    float* t2 = A.alloc<float>(size_t(NT) * Fd);
    float* pr = A.alloc<float>(size_t(NT) * 32);
    float* z = A.alloc<float>(size_t(NT) * 2);
    R.row_conv(dv.dp_pre, x, H, h, Fd, 0, ubias(dv.dp_cond_off), dv.n_cond);
    R.dds(dv.dp_dds, h, t1, t2, Fd, tok, NT);
    R.row_conv(dv.dp_proj, h, Fd, t1, Fd);
    float* hc = t1;  // conditioning for the conv flows
    float* s1 = h;   // h is free now: reuse as scratch
    launch_sdp_noise(z, noise_w, d_row_scales, seed, d_tok_off, d_tok_len, batch, Tmax, st);
    // z channels are never moved: `c0` tracks which physical column is logical channel 0
    int c0 = 0;
    const float inv_sqrt = 1.0f / sqrtf(float(Fd));
    for (size_t f = 0; f < dv.cflows.size(); ++f) {
      c0 ^= 1;  // Flip
      const ConvFlowW& cf = dv.cflows[f];
      launch_convflow_pre(z, c0, cf.pre_w, cf.pre_b, hc, u, NT, Fd, st);
      R.dds(cf.dds, u, s1, t2, Fd, tok, NT);
      R.row_conv(cf.proj, u, Fd, pr, 32);
      launch_rqs_inverse(z, c0 ^ 1, pr, 32, inv_sqrt, NT, st);
    }
    c0 ^= 1;  // final Flip, then ElementwiseAffine^-1; logw = logical channel 0
    launch_sdp_finish(z, c0, dv.ea_m[0], dv.ea_logs[0], logw, NT, st);
  } else {
    float* h = A.alloc<float>(size_t(NT) * std::max(Fd, H));
    float* h2 = A.alloc<float>(size_t(NT) * Fd);
    const float* xin = x;
    if (const float* ub = ubias(dv.dp_cond_off)) {  // x = x + cond(g)
      launch_add_ubias(x, ub, dv.n_cond, h, H, d_tok_off, d_tok_len, batch, Tmax, st);
      xin = h;
    }
    {
      ConvParams p = R.base_conv(dv.dpp_c1, xin, H, h2, Fd, tok, 1);
      p.act = 1;
      R.conv(p, tok);
    }
    launch_layernorm(h2, nullptr, nullptr, dv.dpp_g1, dv.dpp_b1, h2, NT, Fd, 0, st);
    float* h3 = A.alloc<float>(size_t(NT) * Fd);
    {
      ConvParams p = R.base_conv(dv.dpp_c2, h2, Fd, h3, Fd, tok, 1);
      p.act = 1;
      R.conv(p, tok);
    }
    launch_layernorm(h3, nullptr, nullptr, dv.dpp_g2, dv.dpp_b2, h3, NT, Fd, 0, st);
    R.conv(R.base_conv(dv.dpp_proj, h3, Fd, logw, 1, tok, 1), tok);
  }
  R.dump("logw", logw, NT, 1);

  // ---------------- A.0 durations -> frames ----------------
  R.mark("duration_predictor");
  int* cum = A.alloc<int>(NT);
  launch_durations(logw, 1, length_scale, d_row_scales, cum, d_frm_len, d_tok_off, d_tok_len, batch, st);
  int* h_frames = hm + 2 * batch;
  M3_CUDA(cudaMemcpyAsync(h_frames, d_frm_len, size_t(batch) * sizeof(int), cudaMemcpyDeviceToHost, st));
  M3_CUDA(cudaStreamSynchronize(st));
  std::vector<int> frm_off(batch), frm_len(batch);
  int64_t NF = 0;
  int Fmax = 0;
  for (int b = 0; b < batch; ++b) {
    frm_len[b] = h_frames[b];
    frm_off[b] = int(NF);
    NF += frm_len[b];
    Fmax = std::max(Fmax, frm_len[b]);
  }
  const int hop = c.hop();
  if (NF * hop > (int64_t(1) << 31) - 1)
    throw EngineError(M3_ERR_INVALID, "batch produces more than 2^31 samples; split the batch");
  res->frames.assign(frm_len.begin(), frm_len.end());
  res->sample_off.resize(batch + 1);
  int64_t stream_samples = 0;  // output stream: [lead silence][utterance][trail silence] per row
  for (int b = 0; b < batch; ++b) {
    if (o.lead_silence) stream_samples += o.lead_silence[b];
    res->sample_off[b] = stream_samples;
    stream_samples += int64_t(frm_len[b]) * hop;
    if (o.trail_silence) stream_samples += o.trail_silence[b];
  }
  res->sample_off[batch] = stream_samples;
  if (stream_samples > (int64_t(1) << 31) - 64)
    throw EngineError(M3_ERR_INVALID, "batch produces more than 2^31 output samples; split the batch");
  memcpy(hm + 2 * batch, frm_off.data(), batch * sizeof(int));
  memcpy(hm + 3 * batch, frm_len.data(), batch * sizeof(int));
  M3_CUDA(cudaMemcpyAsync(d_frm_off, hm + 2 * batch, size_t(batch) * 2 * sizeof(int), cudaMemcpyHostToDevice, st));
  Segs frm{d_frm_off, d_frm_len, batch, Fmax};
  if (R.debug) {
    DebugTensor t;
    t.rows = NT;
    t.cols = 1;
    std::vector<int> hc(NT);
    M3_CUDA(cudaMemcpy(hc.data(), cum, size_t(NT) * 4, cudaMemcpyDeviceToHost));
    t.data.resize(NT);
    for (int b = 0; b < batch; ++b)
      for (int t2 = 0; t2 < tok_len[b]; ++t2) {
        const int i = tok_off[b] + t2;
        t.data[i] = float(hc[i] - (t2 ? hc[i - 1] : 0));
      }
    res->debug["durations"] = std::move(t);
  }

  // ---------------- phase 2 workspace (frame level) ----------------
  const int Hf = dv.flow_hidden;
  const int C0 = c.up_init;
  {
    size_t fl = size_t(NF) * (size_t(I) + 3 * size_t(Hf) + C0);
    int scale = 1;
    for (size_t i = 0; i < dv.ups.size(); ++i) {
      scale *= dv.ups[i].u;
      fl += size_t(NF) * scale * dv.ups[i].cout * 5;  // x, y0, y1, tmp, sum
    }
    fl += size_t(NF) * hop;                 // audio
    size_t bytes = fl * 4 + size_t(stream_samples) * 2 + size_t(batch) * 32 + (1 << 16) + 512 * 64;
    cx.a2.reserve(bytes);
  }
  Arena& A2 = cx.a2;

  // ---------------- length regulator + prior sample ----------------
  float* z = A2.alloc<float>(size_t(NF) * I);
  R.mark("durations_sync");
  launch_expand(stats, I, cum, d_tok_off, d_tok_len, d_frm_off, d_frm_len, batch, Fmax, noise_scale, d_row_scales, seed, z, st);
  R.mark("expand");
  R.dump("z_p", z, NF, I);

  // ---------------- A.3 flow (reverse) ----------------
  {
    float* h = A2.alloc<float>(size_t(NF) * Hf);
    float* act = A2.alloc<float>(size_t(NF) * Hf);
    float* skip = A2.alloc<float>(size_t(NF) * Hf);
    const int half = I / 2;
    const bool fused = dv.use_tc && !dv.couplings.empty() && dv.couplings[0].ftc.ok && !getenv("M3B200_UNFUSED_FLOW");
    for (size_t f = 0; fused && f < dv.couplings.size(); ++f) {
      const CouplingW& cw = dv.couplings[f];
      FlowTcParams fp;
      fp.z = z;
      fp.z_stride = I;
      fp.x0_coff = cw.ftc.x0_coff;
      fp.x1_coff = cw.ftc.x1_coff;
      fp.Hc = Hf;
      fp.half = half;
      fp.nl = dv.flow_layers;
      fp.w = dv.slab16 + cw.ftc.woff;
      fp.in_bias = cw.ftc.in_bias;
      fp.cum_bias = cw.ftc.cum_bias;
      fp.skip_bias = cw.ftc.skip_bias;
      fp.post_bias = cw.ftc.post_bias;
      if (const float* ub = ubias(cw.cond_off)) {
        fp.cond = ub;
        fp.cond_stride = dv.n_cond;
      }
      fp.seg_off = d_frm_off;
      fp.seg_len = d_frm_len;
      if (cw.ftc.ok2 && !getenv("M3B200_FLOW_V1")) {  // second-generation kernel: fewer, wider MMAs (kernels_tc_flow2.cu)
        fp.w = dv.slab16 + cw.ftc.woff2;
        fp.post_bias = cw.ftc.m_bias;
        launch_flow2_tc(fp, dv.tc_fmt, batch, Fmax, st);
      } else {
        launch_flow_tc(fp, dv.tc_fmt, batch, Fmax, st);
      }
    }
    for (size_t f = 0; !fused && f < dv.couplings.size(); ++f) {
      const CouplingW& cw = dv.couplings[f];
      launch_flip_channels(z, int(NF), I, st);
      if (R.tc_ok(cw.pre.tc)) R.tc_conv(R.base_tc(cw.pre.tc, cw.pre.b, z, I, h, Hf, frm, 1), frm);
      else R.conv(R.base_conv(cw.pre, z, I, h, Hf, frm, 1), frm);  // x0 = z[:, :half]
      M3_CUDA(cudaMemsetAsync(skip, 0, size_t(NF) * Hf * 4, st));
      const int nl = dv.flow_layers;
      for (int i = 0; i < nl; ++i) {
        if (R.tc_ok(cw.in[i].tc)) {
          TcConvParams p = R.base_tc(cw.in[i].tc, cw.in[i].b, h, Hf, act, Hf, frm, 1);
          p.epi = TC_GATE;
          if (const float* ub = ubias(cw.cond_off)) {
            p.ubias = ub + size_t(i) * 2 * Hf;
            p.ub_stride = dv.n_cond;
          }
          R.tc_conv(p, frm);
        } else {
          ConvParams p = R.base_conv(cw.in[i], h, Hf, act, Hf, frm, 1);
          p.Cout = Hf;
          p.gate = 1;
          if (const float* ub = ubias(cw.cond_off)) {
            p.ubias = ub + size_t(i) * 2 * Hf;
            p.ub_stride = dv.n_cond;
          }
          R.conv(p, frm);
        }
        if (R.tc_ok(cw.rs[i].tc)) {
          TcConvParams p = R.base_tc(cw.rs[i].tc, cw.rs[i].b, act, Hf, h, Hf, frm, 1);
          p.epi = TC_RES_SKIP;
          if (i < nl - 1) {
            p.split = Hf;
            p.out2 = skip;
            p.out2_stride = Hf;
          } else {
            p.out = skip;
            p.out_stride = Hf;
          }
          R.tc_conv(p, frm);
        } else {
          ConvParams p = R.base_conv(cw.rs[i], act, Hf, h, Hf, frm, 1);
          p.mode = 1;
          if (i < nl - 1) {
            p.split = Hf;
            p.out2 = skip;
            p.out2_stride = Hf;
          } else {
            p.out = skip;
            p.out_stride = Hf;
          }
          R.conv(p, frm);
        }
      }
      if (R.tc_ok(cw.post.tc)) {
        TcConvParams p = R.base_tc(cw.post.tc, cw.post.b, skip, Hf, z, I, frm, 1);
        p.out_coff = half;
        p.epi = TC_SUB;  // x1 = x1 - m   (mean_only coupling)
        R.tc_conv(p, frm);
      } else {
        ConvParams p = R.base_conv(cw.post, skip, Hf, z, I, frm, 1);
        p.out_coff = half;
        p.mode = 2;  // x1 = x1 - m   (mean_only coupling)
        R.conv(p, frm);
      }
    }
  }
  R.mark("flow");
  R.dump("z", z, NF, I);

  // ---------------- A.4 HiFi-GAN ----------------
  float* cur = A2.alloc<float>(size_t(NF) * C0);
  if (R.tc_ok(dv.dec_pre.tc)) {
    TcConvParams p = R.base_tc(dv.dec_pre.tc, dv.dec_pre.b, z, I, cur, C0, frm, 1);
    if (const float* ub = ubias(dv.dec_cond_off)) {
      p.ubias = ub;
      p.ub_stride = dv.n_cond;
    }
    R.tc_conv(p, frm);
  } else {
    ConvParams p = R.base_conv(dv.dec_pre, z, I, cur, C0, frm, 1);
    if (const float* ub = ubias(dv.dec_cond_off)) {
      p.ubias = ub;
      p.ub_stride = dv.n_cond;
    }
    R.conv(p, frm);
  }
  R.mark("conv_pre");
  int scale = 1;
  const int nk = int(c.rb_kernels.size());
  const bool fuse_last = dv.use_tc && dv.dec_last.ok && !getenv("M3B200_UNFUSED_DEC");
  float* audio = A2.alloc<float>(size_t(NF) * hop);
  int16_t* pcm = A2.alloc<int16_t>(size_t(stream_samples));
  unsigned* peak = A2.alloc<unsigned>(batch);
  M3_CUDA(cudaMemsetAsync(peak, 0, size_t(batch) * 4, st));
  bool audio_done = false;
  for (size_t i = 0; i < dv.ups.size(); ++i) {
    const UpW& u = dv.ups[i];
    const int out_scale = scale * u.u;
    if (fuse_last && i + 1 == dv.ups.size() && dv.dec_last.fused_ok && !getenv("M3B200_DEC_V1")) {
      const MrfStageW& ms = dv.mrf[i];
      const DecLastW& dl = dv.dec_last;
      DecFusedParams fp;
      fp.yprev = cur;
      fp.cin = u.cin;
      fp.up_u = u.u;
      fp.up_pad = u.pad;
      fp.prev_scale = scale;
      fp.scale = out_scale;
      fp.audio = audio;
      fp.peak_bits = peak;
      fp.wblob = dv.slab16 + dl.blob_off;
      fp.w_bytes = dl.blob_bytes;
      fp.up.woff = dl.f_up;
      fp.up.taps = 2;
      fp.up.dil = -1;  // tap d reads y_prev row t - d
      fp.up.pad_left = 0;
      int hymax = 0;
      for (int j = 0; j < 3; ++j) {
        const ResBlockW& rb = dv.rbs[i * nk + j];
        fp.c1[j].woff = dl.f_c1[j];
        fp.c2[j].woff = dl.f_c2[j];
        fp.c1[j].taps = fp.c2[j].taps = rb.k;
        fp.c1[j].pad_left = fp.c2[j].pad_left = (rb.k - 1) / 2;
        fp.c1[j].dil = rb.dil[0];
        fp.c2[j].dil = rb.dil[1];
        fp.bias1[j] = rb.c1[0].b;
        fp.HYb[j] = dl.HYb[j];
        hymax = std::max(hymax, dl.HYb[j]);
      }
      fp.post.woff = dl.f_post;
      fp.post.taps = 7;
      fp.post.dil = 1;
      fp.post.pad_left = 3;
      fp.up_bias = u.b;
      fp.late_bias = ms.late_bias;
      fp.inv_nk = 1.0f / float(ms.nk);
      fp.seg_off = d_frm_off;
      fp.seg_len = d_frm_len;
      fp.HX = ms.HX;
      fp.H = ms.HX + hymax + 3;
      // M3B200_DEC_V2=1: second-generation kernel (sample-order windows); read per call so that one process can A/B them
      if (dl.planes_ok && !getenv("M3B200_DEC_V2")) {
        fp.w_bytes = dl.f_post + kDecPostPlanesBytes;  // shared-memory image: blob[0, f_post) | regrouped conv_post
        fp.post_planes_src = dl.f_postp;
        launch_dec_planes(fp, dv.tc_fmt, batch, Fmax, st);
      }
      else launch_dec_fused(fp, dv.tc_fmt, batch, Fmax, st);
      R.mark("dec_last");
      scale = out_scale;
      audio_done = true;
      break;
    }
    if (fuse_last && i + 1 == dv.ups.size()) {
      const MrfStageW& ms = dv.mrf[i];
      DecStageParams dp;
      dp.yprev = cur;
      dp.cin = u.cin;
      dp.up_u = u.u;
      dp.prev_scale = scale;
      dp.scale = out_scale;
      dp.audio = audio;
      dp.peak_bits = peak;
      dp.w16 = dv.slab16;
      int ns = 0;
      DecConv up;
      up.woff = dv.dec_last.up_woff;
      up.K = u.cin;
      up.N = u.cout;
      up.taps = u.k;
      up.dil = 1;
      up.pad_left = u.k - 1 - u.pad;
      up.kind = 0;
      dp.steps[ns++] = up;
      dp.up = up;
      for (int j = 0; j < ms.nk; ++j) {
        const ResBlockW& rb = dv.rbs[i * nk + j];
        for (int d = 0; d < ms.nd; ++d) {
          DecConv cvn;
          cvn.woff = ms.woff[j][d];
          cvn.K = u.cout;
          cvn.N = u.cout;
          cvn.taps = rb.k;
          cvn.dil = rb.dil[d];
          cvn.pad_left = (rb.k - 1) / 2;
          cvn.kind = d + 1 == ms.nd ? 2 : 1;
          cvn.rb = j;
          dp.steps[ns++] = cvn;
        }
        dp.bias0[j] = rb.c1[0].b;
      }
      DecConv po;
      po.woff = dv.dec_last.post_woff;
      po.K = u.cout;
      po.N = 16;
      po.taps = 7;
      po.dil = 1;
      po.pad_left = 3;
      po.kind = 3;
      dp.steps[ns++] = po;
      dp.nsteps = ns;
      dp.up_bias = u.b;
      dp.late_bias = ms.late_bias;
      dp.nk = ms.nk;
      dp.inv_nk = 1.0f / float(ms.nk);
      dp.seg_off = d_frm_off;
      dp.seg_len = d_frm_len;
      dp.HX = ms.HX;
      dp.HY = ms.HY;
      dp.H = ms.HX + ms.HY + 3;
      launch_dec_last(dp, u.cout, dv.tc_fmt, batch, Fmax, st);
      R.mark("dec_last");
      scale = out_scale;
      audio_done = true;
      break;
    }
    const size_t n = size_t(NF) * out_scale * u.cout;
    float* xu = A2.alloc<float>(n);
    float* yb[2] = {A2.alloc<float>(n), A2.alloc<float>(n)};
    float* tb = A2.alloc<float>(n);
    float* sum = A2.alloc<float>(n);
    if (R.tc_ok(u.tc)) {
      Segs fs{d_frm_off, d_frm_len, batch, Fmax};
      TcConvParams p = R.base_tc(u.tc, u.b, cur, u.cin, xu, u.cout, fs, scale);
      p.in_slope = 0.1f;
      p.pad_left = u.ntaps - 1;
      p.epi = TC_UPS;
      p.out_scale = out_scale;
      p.rows_extra = u.ntaps - 1;
      p.ups_u = u.u;
      p.ups_pad = u.pad;
      p.ups_cout = u.cout;
      if (ups_tc_enabled() && ups_tc_supported(p)) launch_ups_tc(p, dv.tc_fmt, batch, Fmax, st);
      else launch_conv_tc(p, dv.tc_fmt, batch, Fmax, st);
    } else {
      ConvParams p;
      p.in = cur;
      p.in_stride = u.cin;
      p.Cin = u.cin;
      p.in_slope = 0.1f;
      p.W = u.w;
      p.w_phase_stride = (long long)u.ntaps * u.cin * u.cout;
      p.Cout = u.cout;
      p.taps = u.ntaps;
      p.pad_left = u.ntaps - 1;
      p.bias = u.b;
      p.out = xu;
      p.out_stride = u.cout;
      p.seg_off = d_frm_off;
      p.seg_len = d_frm_len;
      p.in_scale = scale;
      p.out_scale = out_scale;
      p.rows_extra = u.ntaps - 1;
      p.out_mul = u.u;
      p.out_add = -u.pad;
      p.out_add_phase = 1;
      p.phases = u.u;
      launch_conv(p, batch, Fmax, st);
    }
    R.mark("upsample");
    Segs lvl{d_frm_off, d_frm_len, batch, Fmax};
    const MrfStageW& ms = dv.mrf[i];
    bool rb1_tc = dv.use_tc;  // pack_voice packed every conv of a ResBlock1 stage for the tensor cores, or none
    for (int j = 0; j < nk; ++j)
      for (size_t d = 0; d < dv.rbs[i * nk + j].c1.size(); ++d)
        rb1_tc = rb1_tc && !dv.rbs[i * nk + j].c2.empty() && dv.rbs[i * nk + j].c1[d].tc.ok && dv.rbs[i * nk + j].c2[d].tc.ok;
    if (dv.use_tc && ms.ok) {
      MrfParams mp;
      mp.x = xu;
      mp.out = sum;
      mp.w16 = dv.slab16;
      mp.nk = ms.nk;
      mp.nd = ms.nd;
      for (int j = 0; j < ms.nk; ++j) {
        const ResBlockW& rb = dv.rbs[i * nk + j];
        mp.k[j] = rb.k;
        for (int d = 0; d < ms.nd; ++d) {
          mp.dil[j][d] = rb.dil[d];
          mp.woff[j][d] = ms.woff[j][d];
          mp.bias[j][d] = rb.c1[d].b;
        }
      }
      mp.late_bias = ms.late_bias;
      mp.seg_off = d_frm_off;
      mp.seg_len = d_frm_len;
      mp.scale = out_scale;
      mp.H = ms.H;
      mp.HX = ms.HX;
      mp.HY = ms.HY;
      mp.inv_nk = 1.0f / float(ms.nk);
      const bool v1 = getenv("M3B200_MRF_V1") != nullptr;  // per-window kernel for every stage (A/B, parity tests)
      if (!v1 && mrf_ws_supported(mp, u.cout)) launch_mrf_ws(mp, dv.tc_fmt, batch, Fmax, st);
      else if (!v1 && mrf_ws128_supported(mp, u.cout)) launch_mrf_ws128(mp, dv.tc_fmt, batch, Fmax, st);
      else launch_mrf_tc(mp, u.cout, dv.tc_fmt, batch, Fmax, st);
    } else if (rb1_tc) {
      // ResBlock1 on tensor cores: one conv_tc_kernel per conv, the residual add and the 1/nk mean in the second
      // conv's epilogue; same buffers as the fp32 branch below
      for (int j = 0; j < nk; ++j) {
        const ResBlockW& rb = dv.rbs[i * nk + j];
        const float* src = xu;
        const size_t nd = rb.dil.size();
        for (size_t d = 0; d < nd; ++d) {
          const bool last = d + 1 == nd;
          // t = conv1_d(lrelu(x)) + b1; x = x + conv2_d(lrelu(t)) + b2 (each conv reads rows outside the utterance as 0)
          TcConvParams p = R.base_tc(rb.c1[d].tc, rb.c1[d].b, src, u.cout, tb, u.cout, lvl, out_scale);
          p.dil = rb.dil[d];
          p.in_slope = 0.1f;
          R.tc_conv(p, lvl);
          TcConvParams q = R.base_tc(rb.c2[d].tc, rb.c2[d].b, tb, u.cout, last ? sum : yb[d & 1], u.cout, lvl, out_scale);
          q.in_slope = 0.1f;
          q.res = src;
          q.res_stride = u.cout;
          if (last) {
            q.scale = 1.0f / float(nk);
            q.accumulate = j == 0 ? 0 : 1;
          }
          launch_conv_tc_res(q, dv.tc_fmt, lvl.n, lvl.max_len, st);
          src = yb[d & 1];
        }
      }
    } else
    for (int j = 0; j < nk; ++j) {
      const ResBlockW& rb = dv.rbs[i * nk + j];
      const float* src = xu;
      const size_t nd = rb.dil.size();
      for (size_t d = 0; d < nd; ++d) {
        const bool last = d + 1 == nd;
        if (rb.c2.empty()) {  // ResBlock2: x = x + conv_d(lrelu(x))
          ConvParams p = R.base_conv(rb.c1[d], src, u.cout, last ? sum : yb[d & 1], u.cout, lvl, out_scale);
          p.dil = rb.dil[d];
          p.pad_left = (rb.k - 1) / 2;  // in taps; the kernel multiplies by the dilation
          p.in_slope = 0.1f;
          p.res = src;
          p.res_stride = u.cout;
          if (last) {
            p.scale = 1.0f / float(nk);
            p.mode = j == 0 ? 0 : 1;
          }
          R.conv(p, lvl);
        } else {  // ResBlock1: t = conv1_d(lrelu(x)); t = conv2(lrelu(t)); x = x + t
          {
            ConvParams p = R.base_conv(rb.c1[d], src, u.cout, tb, u.cout, lvl, out_scale);
            p.dil = rb.dil[d];
            p.pad_left = (rb.k - 1) / 2;
            p.in_slope = 0.1f;
            R.conv(p, lvl);
          }
          {
            ConvParams p = R.base_conv(rb.c2[d], tb, u.cout, last ? sum : yb[d & 1], u.cout, lvl, out_scale);
            p.pad_left = (rb.k - 1) / 2;
            p.in_slope = 0.1f;
            p.res = src;
            p.res_stride = u.cout;
            if (last) {
              p.scale = 1.0f / float(nk);
              p.mode = j == 0 ? 0 : 1;
            }
            R.conv(p, lvl);
          }
        }
        src = yb[d & 1];
      }
    }
    R.mark("mrf");
    cur = sum;
    scale = out_scale;
    if (R.debug) R.dump(("mrf" + std::to_string(i)).c_str(), sum, NF * out_scale, u.cout);
  }
  if (!audio_done)
    launch_conv_post(cur, dv.post_c, dv.post_w, dv.post_k, 0.01f, audio, peak, d_frm_off, d_frm_len, hop, batch, Fmax, st);
  if (!post) {
    launch_to_int16(audio, peak, pcm, d_frm_off, d_frm_len, hop, batch, Fmax, st);
  } else {
    // PCM post chain on the device (SURVEY.md §8f rank 2): volume, inter-sentence silence, WAV framing
    long long* d_out_off = A2.alloc<long long>(batch);
    double* d_volume = o.volume ? A2.alloc<double>(batch) : nullptr;
    char* hp = static_cast<char*>(cx.h_opts.p) + ((size_t(batch) * 3 * sizeof(float) + 15) & ~size_t(15));
    long long* h_off = reinterpret_cast<long long*>(hp);
    double* h_vol = reinterpret_cast<double*>(hp + size_t(batch) * sizeof(long long));
    for (int b = 0; b < batch; ++b) h_off[b] = res->sample_off[b];
    M3_CUDA(cudaMemcpyAsync(d_out_off, h_off, size_t(batch) * sizeof(long long), cudaMemcpyHostToDevice, st));
    if (o.volume) {
      memcpy(h_vol, o.volume, size_t(batch) * sizeof(double));
      M3_CUDA(cudaMemcpyAsync(d_volume, h_vol, size_t(batch) * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if (stream_samples != NF * hop) M3_CUDA(cudaMemsetAsync(pcm, 0, size_t(stream_samples) * 2, st));
    launch_to_int16_post(audio, peak, pcm, d_frm_off, d_frm_len, hop, d_out_off, d_volume, batch, Fmax, st);
  }
  R.mark("post_int16");

  // ---------------- outputs ----------------
  const size_t NS = size_t(stream_samples);
  const size_t hdr = o.wav_header ? 44 : 0;
  res->d_pcm = pcm;
  float* h_peaks = reinterpret_cast<float*>(hm);  // reuse meta staging (tok arrays no longer needed on host)
  M3_CUDA(cudaMemcpyAsync(h_peaks, peak, size_t(batch) * 4, cudaMemcpyDeviceToHost, st));
  if (!(flags & M3_FLAG_NO_HOST_COPY)) {
    cx.h_pcm.reserve(hdr + NS * 2);
    uint8_t* hs = static_cast<uint8_t*>(cx.h_pcm.p);
    if (hdr) write_wav_header(hs, c.sample_rate, int64_t(NS));
    M3_CUDA(cudaMemcpyAsync(hs + hdr, pcm, NS * 2, cudaMemcpyDeviceToHost, st));
    res->pcm = reinterpret_cast<const int16_t*>(hs + hdr);
    res->stream = hs;
    res->stream_bytes = int64_t(hdr + NS * 2);
    if (flags & M3_FLAG_KEEP_FLOAT) {
      cx.h_audio.reserve(NS * 4);
      M3_CUDA(cudaMemcpyAsync(cx.h_audio.p, audio, NS * 4, cudaMemcpyDeviceToHost, st));
      res->audio = static_cast<const float*>(cx.h_audio.p);
    }
  }
  M3_CUDA(cudaEventRecord(cx.ev1, st));
  M3_CUDA(cudaStreamSynchronize(st));
  M3_CUDA(cudaGetLastError());
  float ms = 0;
  M3_CUDA(cudaEventElapsedTime(&ms, cx.ev0, cx.ev1));
  res->device_ms = ms;
  res->launches = g_launch_count;
  R.collect_marks();
  res->peaks.assign(h_peaks, h_peaks + batch);
  lease.keep = true;
  return res.release();
}

}  // namespace m3
