// Kernel launch interface of the engine (host side).  All activations are fp32,
// channels-last, utterances packed back to back: row r of utterance b at level L lives at
// (seg_off[b] * scale_L + r).  No padded rows exist, so VITS' mask multiplications
// (SURVEY.md Appendix A) reduce to per-utterance zero padding at segment edges, which is
// exactly the batch-1 behaviour of the reference (mimic3_tts/voice.py:180-181).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace m3 {

extern thread_local int64_t g_launch_count;  // kernels launched by this thread's current call
void post_launch(const char* what, cudaStream_t st);
// Raises a kernel's dynamic shared-memory limit to the opt-in maximum exactly once (process-wide, thread safe).
void ensure_max_dynamic_smem(const void* func);

struct ConvParams {
  // input
  const float* in = nullptr;
  int in_stride = 0, in_coff = 0, Cin = 0;
  float in_slope = 1.f;  // leaky-relu applied to the input on load (1 = identity)
  // weights [phase][tap][Cin][ldw], ldw = Cout (2*Cout when gate)
  const float* W = nullptr;
  long long w_phase_stride = 0;
  int Cout = 0, taps = 1, dil = 1, pad_left = 0;
  const float* bias = nullptr;   // [ldw]
  const float* ubias = nullptr;  // per-utterance bias [B][ub_stride] (+ column offset folded in pointer)
  int ub_stride = 0;
  // epilogue: v = acc + bias + ubias; (gate) v = tanh(va)*sigmoid(vb); v += res; v *= scale; act; mode
  int gate = 0;
  const float* res = nullptr;
  int res_stride = 0, res_coff = 0;
  float scale = 1.f;
  int act = 0;   // 0 none, 1 relu
  int mode = 0;  // 0 store, 1 accumulate (out += v), 2 subtract (out -= v)
  float* out = nullptr;
  int out_stride = 0, out_coff = 0;
  float* out2 = nullptr;  // columns >= split go to out2[col - split]
  int out2_stride = 0, split = 1 << 30;
  // segments
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
  int in_scale = 1;    // input rows per segment unit
  int out_scale = 1;   // output rows per segment unit
  int rows_extra = 0;  // GEMM rows = len*in_scale + rows_extra
  int out_mul = 1, out_add = 0, out_add_phase = 0;  // out row = t*out_mul + out_add + phase*out_add_phase
  int phases = 1;
};

void launch_conv(const ConvParams& p, int n_seg, int max_seg_len, cudaStream_t st);

// Token-level fp32 conv-as-GEMM over PACKED rows (tiles span utterance boundaries, so short
// utterances waste nothing).  rowinfo[r] = (seg_lo, seg_hi, seg_id, 0): taps outside [lo, hi) read 0.
struct RowConvParams {
  const float* in = nullptr;
  int in_stride = 0, Cin = 0;
  const float* W = nullptr;  // [taps][Cin][Cout]
  int Cout = 0, taps = 1, pad_left = 0;
  const float* bias = nullptr;
  const float* ubias = nullptr;  // [n_seg][ub_stride]
  int ub_stride = 0;
  int act = 0;  // 0 none, 1 relu
  float* out = nullptr;
  int out_stride = 0;
  const int4* rowinfo = nullptr;
  int rows = 0;
};
void launch_row_conv(const RowConvParams& p, cudaStream_t st);
void launch_fill_rowinfo(int4* rowinfo, const int* seg_off, const int* seg_len, int n_seg, int max_len,
                         cudaStream_t st);

// Fused tensor-core MRF stage (kernels_tc.cu).  Weights: 16-bit, per conv [tap][Cin/8][Cout][8].
struct MrfParams {
  const float* x = nullptr;  // [rows][C] fp32, channels-last
  float* out = nullptr;      // [rows][C] fp32
  const uint16_t* w16 = nullptr;
  unsigned long long woff[4][2] = {};  // element offset of conv (resblock j, conv d) in w16
  const float* bias[4][2] = {};
  const float* late_bias = nullptr;    // [C] = sum_j sum_{d>=1} bias[j][d]
  int k[4] = {}, dil[4][2] = {};
  int nk = 0, nd = 0;
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
  int scale = 1;
  int stride = 0;  // filled by the launcher: R - 2H
  int H = 0, HX = 0, HY = 0;
  int wg = 1;      // taps per weight-staging group (launcher)
  float inv_nk = 1.f;
  int dbg = 0;     // M3B200_MRF_DEBUG bit mask (performance experiments only; breaks results)
  int n_seg = 0, max_win = 0, nslot = 0;  // persistent kernel (kernels_tc_mrf2.cu), filled by its launcher
  long long* prof = nullptr;              // M3B200_MRF_PROFILE=1: per-role cycle counters (debug)
};
// Generic tensor-core Conv1d / polyphase ConvTranspose1d (kernels_tc.cu).
// Weights: 16-bit, [chunk][tap][K/8][NC][8] (one contiguous block per (chunk, tap): a bulk copy).
enum TcEpi { TC_STORE = 0, TC_GATE = 1, TC_RES_SKIP = 2, TC_SUB = 3, TC_UPS = 4 };
struct TcConvParams {
  const float* in = nullptr;
  int in_stride = 0, in_coff = 0, K = 0;
  float in_slope = 1.f;
  const uint16_t* w = nullptr;
  int NC = 0, n_chunks = 0, N = 0;  // N = logical output columns (gate: gated channels)
  int taps = 1, dil = 1, pad_left = 0;
  int epi = TC_STORE;
  const float* bias = nullptr;
  const float* ubias = nullptr;
  int ub_stride = 0;
  float* out = nullptr;
  int out_stride = 0, out_coff = 0;
  float* out2 = nullptr;
  int out2_stride = 0, split = 1 << 30;
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
  int in_scale = 1, out_scale = 1, rows_extra = 0;
  int ups_u = 1, ups_pad = 0, ups_cout = 0;
  int wide = 0;  // 256-bit global stores in the polyphase epilogue (set by the launcher: M3B200_WIDE_IO + alignment)
  // residual epilogue (launch_conv_tc_res only): o = (acc + bias + res) * scale; out = accumulate ? out + o : o
  const float* res = nullptr;
  int res_stride = 0;
  float scale = 1.f;
  int accumulate = 0;
};
// m_tiles: 128-row M tiles per CTA, 2 or 1.  launch_conv_tc runs 2 whenever they fit shared memory and 1 otherwise,
// so a weight packing accepted for 1 tile only (K = 512 with 2 taps, the default generator's first upsampler) runs too.
bool conv_tc_supported(int K, int NC, int taps, int dil, int m_tiles = 2);
void launch_conv_tc(const TcConvParams& p, int fmt, int n_seg, int max_seg_len, cudaStream_t st);
// conv_tc_kernel with the residual epilogue above: the second conv of a ResBlock1 dilation step
// (x = x + conv2(lrelu(t)) + b2), and for the last step the 1/nk mean into the stage sum.
void launch_conv_tc_res(const TcConvParams& p, int fmt, int n_seg, int max_seg_len, cudaStream_t st);
// Every conv of a ResBlock1 MRF stage (C channels, nk resblocks of nd dilations, kernel sizes k[j], dilations dil[j][d])
// fits conv_tc_kernel with two M tiles: C % 32 == 0, nk <= 4, nd <= 3, odd k <= 11, and the A operand of
// 256 + (k-1)*dil rows x C channels plus two weight stages within 225 KB of shared memory.  That holds for every
// k <= 11, dil <= 5 up to C = 288; C = 320 / 352 fit only up to (k-1)*dil = 39 / 7, and C >= 384 never fits.
bool mrf1_tc_supported(int C, int nk, int nd, const int* k, const int (*dil)[3]);
// kernels_tc_ups.cu: the TC_UPS case with a shared-memory bias and an early accumulator release; the default
// for the polyphase upsamplers since round 2 (bit-identical to conv_tc_kernel's TC_UPS epilogue, which
// M3B200_UPS_V1=1 selects again).
bool ups_tc_enabled();
bool ups_tc_supported(const TcConvParams& p);
void launch_ups_tc(const TcConvParams& p, int fmt, int n_seg, int max_seg_len, cudaStream_t st);

// Token-level conv-as-GEMM on tensor cores with fp16 hi/lo split operands (kernels_tc_rows.cu).
// Weights: [chunk(nc cols)][K block(32)][tap][hi|lo][4][nc][8], 16-bit; nc = rowgemm_tc_nc(N, taps).
struct RowGemmTcParams {
  const float* in = nullptr;
  int in_stride = 0, K = 0;
  const uint16_t* w = nullptr;
  int N = 0, taps = 1, pad_left = 0;
  int nc = 64;                    // output columns per CTA the weights were packed for
  const float* bias = nullptr;
  const float* ubias = nullptr;
  int ub_stride = 0;
  int act = 0;
  float* out = nullptr;
  int out_stride = 0;
  const int* vmap = nullptr;      // virtual row -> physical row, -1 for the zero row after each utterance
  const int4* rowinfo = nullptr;  // physical row -> (lo, hi, seg, 0)
  int vrows = 0;
  int wide = 0;  // 256-bit global loads / stores (set by the launcher: M3B200_WIDE_IO + alignment)
};
bool wide_io_enabled();  // M3B200_WIDE_IO (read per launch)
bool rowgemm_tc_supported(int K, int taps);
int rowgemm_tc_nc(int N, int taps);
size_t rowgemm_tc_weight_elems(int K, int N, int taps, int nc);
void launch_rowgemm_tc(const RowGemmTcParams& p, cudaStream_t st);
void launch_fill_vmap(int* vmap, const int* seg_off, const int* seg_len, int n_seg, int max_len, cudaStream_t st);

// Fused last generator stage: ConvTranspose + MRF + conv_post/tanh/peak (kernels_tc_dec.cu).
struct DecConv {
  unsigned long long woff = 0;  // element offset of [tap][K/8][N][8] in w16
  int K = 0, N = 0, taps = 1, dil = 1, pad_left = 0;
  int kind = 0;  // 0 transposed conv (zero-stuffed input), 1 resblock conv, 2 last conv of a resblock, 3 conv_post
  int rb = 0;    // resblock index (kinds 1, 2)
};
struct DecStageParams {
  const float* yprev = nullptr;  // [rows_prev][cin] fp32: previous stage output (pre-activation)
  int cin = 0, up_u = 1, prev_scale = 1, scale = 1;
  float* audio = nullptr;
  unsigned* peak_bits = nullptr;
  const uint16_t* w16 = nullptr;
  DecConv steps[12];
  int nsteps = 0;
  DecConv up;  // == steps[0]
  const float* up_bias = nullptr;
  const float* bias0[4] = {};
  const float* late_bias = nullptr;
  int nk = 0;
  float inv_nk = 1.f;
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
  int H = 0, HX = 0, HY = 0, stride = 0, wb_bytes = 16 * 1024;
};
bool dec_last_supported(int C, int cin, int up_k, int up_u, int nk, int nd, int HX, int HY);
void launch_dec_last(const DecStageParams& p, int C, int fmt, int n_seg, int max_len, cudaStream_t st);

// Persistent, warp-specialised version of the fused last stage (kernels_tc_dec2.cu).  All weights of the
// stage live in ONE contiguous 16-bit blob (byte offsets below are relative to it):
//   up   : polyphase transposed conv, per tap d in {0,1}: [cin/8][u*C][8], column ph*C+co = W[ci][co][u*d+ph]
//   c1/c2: resblock j first / second conv, [tap][C/8][C][8]
//   post : conv_post, [tap][C/8][16][8] (column 0 real)
struct DecFusedConv {
  unsigned woff = 0;
  int taps = 1, dil = 1, pad_left = 0;
};
struct DecFusedParams {
  const float* yprev = nullptr;  // [rows_prev][cin] fp32: previous stage output (pre-activation)
  int cin = 0, up_u = 1, up_pad = 0, prev_scale = 1, scale = 1;
  float* audio = nullptr;
  unsigned* peak_bits = nullptr;
  const uint16_t* wblob = nullptr;
  unsigned w_bytes = 0;
  DecFusedConv up, c1[3], c2[3], post;
  const float* up_bias = nullptr;
  const float* bias1[3] = {};
  const float* late_bias = nullptr;
  float inv_nk = 1.f;
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
  int H = 0, HX = 0, HYb[3] = {};  // HYb: halo rows of resblock j's second-conv operand buffer (>= 3 for j = 0: conv_post reuses it)
  int stride = 0, n_seg = 0, max_win = 0;  // filled by the launcher
  int HL = 0;                              // dec_planes_kernel: left halo of a window (launcher; >= H, aligns windows to the upsampling phase)
  unsigned post_planes_src = 0;            // dec_planes_kernel: byte offset in wblob of conv_post regrouped per (row shift, input plane)
  long long* prof = nullptr;               // M3B200_DEC_PROFILE=1: per-role cycle counters (debug)
};
bool dec_fused_supported(int C, int cin, int up_k, int up_u, int nk, int nd, int HX, const int* HYb, size_t w_bytes);
void launch_dec_fused(const DecFusedParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);
// Third generation (kernels_tc_dec3.cu): same blob and parameters, the stage kept in phase-major planes (u = 4, cin = 64):
// 512-sample windows, no transposition of the transposed-conv result, two issuer warps.  conv_post (one output channel)
// is regrouped: output column = output plane ph', one [C/8][16][8] block per (row shift sh, input plane pi) in the order
// sh = -1: pi 1..3, sh = 0: pi 0..3, sh = +1: pi 0..2, block column ph' = w[tap 4 sh + pi - ph' + 3] -- 20 MMAs per window
// instead of 56.  The kernel's shared-memory weight image is blob[0, post.woff) followed by those kDecPostPlanesBytes (engine.h).
bool dec_planes_supported(int C, int cin, int up_k, int up_u, int nk, int nd, int HX, const int* HYb, size_t w_bytes);
void launch_dec_planes(const DecFusedParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);

// Fused coupling layer of the flow (kernels_tc_flow.cu).  Weights: one 16-bit stream in schedule order
// (pre chunks | per layer: gate chunks x 5 taps, res chunks, skip chunks | post chunks), each stage
// [K/8][64][8]; the channel Flip is folded into pre/post packing and x0_coff / x1_coff.
struct FlowTcParams {
  float* z = nullptr;  // [frames][z_stride] fp32, updated in place (x1 half)
  int z_stride = 0, x0_coff = 0, x1_coff = 0;
  int Hc = 0, half = 0, nl = 0;
  const uint16_t* w = nullptr;
  const float* in_bias = nullptr;    // [nl][2*Hc]
  const float* cum_bias = nullptr;   // [nl][Hc]: b_pre + sum_{j<i} b_res_j
  const float* skip_bias = nullptr;  // [Hc]
  const float* post_bias = nullptr;  // [half] (flip-permuted)
  const float* cond = nullptr;       // per utterance [cond_stride], laid out like in_bias; may be null
  int cond_stride = 0;
  long long* prof = nullptr;         // M3B200_FLOW_PROFILE=1: per-role cycle counters (debug)
  const int* seg_off = nullptr;
  const int* seg_len = nullptr;
};
bool flow_tc_supported(int Hc, int half, int nl, int kernel);
void launch_flow_tc(const FlowTcParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);
// Second generation (kernels_tc_flow2.cu): same params; `w` is the v2 stream (pre K96xN192 | per layer: 4 gate chunks x 5
// taps K192xN96 (48 "a" + 48 "b" columns), [res K-halves 2 x K96xN192], m-update K192xN96 with W' = W_post.W_skip),
// `post_bias` = m_bias; skip_bias unused.
bool flow2_tc_supported(int Hc, int half, int nl, int kernel);
size_t flow2_tc_weight_elems(int nl);
void launch_flow2_tc(const FlowTcParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);

bool mrf_tc_supported(int C, int nk, int nd, const int* k, int max_halo);
// persistent warp-specialised variant for C = 64, three ResBlock2 chains (kernels_tc_mrf2.cu)
bool mrf_ws_supported(const MrfParams& p, int C);
void launch_mrf_ws(const MrfParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);
// C = 128 stage, persistent + warp-specialised (kernels_tc_mrf3.cu): chains serialised through one TMEM tile pair,
// running sum in TMEM, 16 KB half-tap weight ring.
bool mrf_ws128_supported(const MrfParams& p, int C);
void launch_mrf_ws128(const MrfParams& p, int fmt, int n_seg, int max_len, cudaStream_t st);
// fmt: 0 = fp16 operands, 1 = bf16 operands
void launch_mrf_tc(const MrfParams& p, int C, int fmt, int n_seg, int max_len, cudaStream_t st);

// out = res + act(LN(a + b)) over channels, eps 1e-5; act: 0 none, 1 erf-GELU
void launch_layernorm(const float* a, const float* b, const float* res, const float* gamma, const float* beta,
                      float* out, int rows, int C, int act, cudaStream_t st);
// y = GELU(LN(depthwise_conv_k3(x, dilation) + bias)) (DDSConv first half), segment aware
void launch_dds_sep(const float* x, const float* w /*[3][C]*/, const float* bias, const float* gamma,
                    const float* beta, float* out, int C, int dil, const int* seg_off, const int* seg_len, int n_seg,
                    int max_len, cudaStream_t st);
// out[t][c] = in[t][c] + ubias[seg][c]
void launch_add_ubias(const float* in, const float* ubias, int ub_stride, float* out, int C, const int* seg_off,
                      const int* seg_len, int n_seg, int max_len, cudaStream_t st);
void launch_embedding(const int64_t* ids, int t_stride, const float* emb, int num_symbols, float scale, float* out, int H,
                      const int* seg_off, const int* seg_len, int n_seg, int max_len, cudaStream_t st);
void launch_gather_rows(const int64_t* idx, const float* table, float* out, int n, int C, cudaStream_t st);
// relative-position multi-head self attention (window W), qkv [rows][3H]
void launch_attention(const float* qkv, const float* emb_rel_k, const float* emb_rel_v, float* out, int H,
                      int n_heads, int window, const int* seg_off, const int* seg_len, int n_seg, int max_len,
                      cudaStream_t st);
// short-sequence variant (kernels_attn.cu): whole (utterance, head) in shared memory; returns false when the
// shape does not fit and the generic kernel has to run (M3B200_ATTN_V1=1 forces that)
bool launch_attention_short(const float* qkv, const float* emb_rel_k, const float* emb_rel_v, float* out, int H,
                            int n_heads, int window, const int* seg_off, const int* seg_len, int n_seg, int max_len,
                            cudaStream_t st);
// u[t][c] = z[t][zc]*w[c] + b[c] + h[t][c]
void launch_convflow_pre(const float* z, int zc, const float* w, const float* b, const float* h, float* out,
                         int rows, int C, cudaStream_t st);
// z[t][zc] = RQS^-1(z[t][zc] | params[t][0:29] scaled)
void launch_rqs_inverse(float* z, int zc, const float* params, int pstride, float inv_sqrt_c, int rows,
                        cudaStream_t st);
// row_scales (nullable, here and below): per-utterance [noise_scale, length_scale, noise_w] overriding the scalar
void launch_sdp_noise(float* z, float noise_w, const float* row_scales, uint64_t seed, const int* seg_off,
                      const int* seg_len, int n_seg, int max_len, cudaStream_t st);
// logw = (z[:, zc] - m) * exp(-logs)
void launch_sdp_finish(const float* z, int zc, float m, float logs, float* logw, int rows, cudaStream_t st);
// durations: w_ceil = ceil(exp(logw)*length_scale); cum = inclusive scan per utterance; frames[b] = max(1, total)
void launch_durations(const float* logw, int logw_stride, float length_scale, const float* row_scales, int* cum,
                      int* frames, const int* seg_off, const int* seg_len, int n_seg, cudaStream_t st);
// z_p[frame][c] = m[tok][c] + N(0,1)*exp(logs[tok][c])*noise_scale  (stats = [m | logs], stride 2I)
void launch_expand(const float* stats, int I, const int* cum, const int* tok_off, const int* tok_len,
                   const int* frm_off, const int* frm_len, int n_seg, int max_frames, float noise_scale,
                   const float* row_scales, uint64_t seed, float* zp, cudaStream_t st);
void launch_flip_channels(float* x, int rows, int C, cudaStream_t st);
// y = tanh(conv_k(lrelu(x, slope)))  (C_out = 1, no bias) + per-utterance max|y|
void launch_conv_post(const float* x, int C, const float* w /*[k][C]*/, int k, float slope, float* audio,
                      unsigned* peak_bits, const int* seg_off, const int* seg_len, int scale, int n_seg, int max_len,
                      cudaStream_t st);
// pcm = trunc(clip(audio * 32767/max(0.01, peak)))  (mimic3_tts/utils.py:237-244)
void launch_to_int16(const float* audio, const unsigned* peak_bits, int16_t* pcm, const int* seg_off,
                     const int* seg_len, int scale, int n_seg, int max_len, cudaStream_t st);
// same + the PCM post chain (tts.py:536-543): utterance b written at out_off[b] of `stream`, optional
// audioop.mul volume factor per utterance
void launch_to_int16_post(const float* audio, const unsigned* peak_bits, int16_t* stream, const int* seg_off,
                          const int* seg_len, int scale, const long long* out_off, const double* volume, int n_seg,
                          int max_len, cudaStream_t st);

}  // namespace m3
