// Generic tensor-core Conv1d / polyphase ConvTranspose1d as an implicit GEMM (sm_100a):
//     D[t, n] = sum_tap  A[t + (tap - pad) * dil, :] . W_tap[:, n]
// rows = time (two 128-row M tiles per CTA), K = input channels, N processed in chunks of NC
// columns.  Used for the coupling-flow convolutions (WN in_layers k=5 with the gated
// tanh*sigmoid epilogue, 1x1 res/skip, pre, post), the generator's conv_pre and the
// ConvTranspose1d upsamplers (polyphase: N = stride*C_out, 2 taps).
//
// Warp-specialised, one CTA per SM:
//   warp 0      weight producer: one 1-D bulk copy (TMA engine) per (chunk, tap) block into a
//               2..4 stage smem ring, completion on mbarriers (expect_tx / complete_tx);
//   warp 1      tcgen05.mma issuer (one elected lane); frees ring stages and publishes
//               accumulators with tcgen05.commit;
//   warps 2..9  epilogue: TMEM -> registers -> fused epilogue -> global.
// The A operand (fp32 activations -> 16-bit, optional leaky-relu) is staged once per CTA in the
// interleaved layout of tc_common.cuh, so a tap is a descriptor start-address shift.
// Accumulators are double-buffered in TMEM: the epilogue of chunk c overlaps the MMAs of c+1.
#include <algorithm>
#include <stdexcept>

#include "kernels.h"
#include "tc_common.cuh"

namespace m3 {

constexpr int CT_NT = 2;  // M tiles per CTA (1 for shapes whose A operand only fits shared memory at 128 rows)
constexpr int CT_THREADS = 320;
constexpr int CT_SMEM_MAX = 225 * 1024;

// RES: residual epilogue of launch_conv_tc_res (p.epi is ignored); NT: M tiles (128 rows each) per CTA.  Template
// arguments, so that the instantiation every other caller runs (RES = false, NT = 2) compiles exactly as without them.
template <int FMT, bool RES, int NT>
__global__ void __launch_bounds__(CT_THREADS, 1) conv_tc_kernel(TcConvParams p, int stages, int rows_a) {
  constexpr int CT_R = NT * 128;  // rows per CTA
  using E = tc::Elem<FMT>;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], acc_full[2], acc_empty[2];

  const int seg = blockIdx.y;
  const int len_units = p.seg_len[seg];
  const int in_len = len_units * p.in_scale;
  const int rows = in_len + p.rows_extra;
  const int t0 = blockIdx.x * CT_R;
  if (t0 >= rows) return;
  const long long in_base = (long long)p.seg_off[seg] * p.in_scale;
  const int out_len = len_units * p.out_scale;
  const long long out_base = (long long)p.seg_off[seg] * p.out_scale;
  const int CH = p.K / 8;
  const int NC = p.NC;
  const uint32_t stage_bytes = uint32_t(p.K) * NC * 2;
  uint8_t* bufA = smem;
  uint8_t* wring = smem + ((size_t(CH) * rows_a * 16 + 127) & ~size_t(127));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tc::tmem_alloc<512>(&tmem_slot);
  if (tid == 32) {
    for (int s = 0; s < stages; ++s) {
      tc::mbar_init(&full_bar[s], 1);
      tc::mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&acc_full[b], 1);
      tc::mbar_init(&acc_empty[b], 8);
    }
    tc::mbar_fence_init();
  }
  // ---- stage the A operand: input rows [t0 - halo_l, t0 - halo_l + rows_a) x K ------------------
  // Item = (row, 8-channel chunk), chunk fastest: a warp reads whole rows (coalesced 32 B per lane);
  // rows_a is odd so the 16-byte smem stores of 8 neighbouring chunks fall into distinct banks.
  // Four items per thread are in flight at once (the loop is a chain of L2 round trips otherwise).
  {
    const int halo_l = p.pad_left * p.dil;
    const float slope = p.in_slope;
    const int items = CH * rows_a;
    auto lr = [slope](float v) { return v >= 0.f ? v : slope * v; };
    for (int i0 = tid; i0 < items; i0 += 4 * CT_THREADS) {
      float4 a[4], b[4];
      int dsti[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = i0 + u * CT_THREADS;
        a[u] = b[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        dsti[u] = -1;
        if (idx < items) {
          const int rr = idx / CH, c8 = idx - rr * CH;
          dsti[u] = c8 * rows_a + rr;
          const int ti = t0 - halo_l + rr;
          if (ti >= 0 && ti < in_len) {
            const float* src = p.in + (in_base + ti) * (long long)p.in_stride + p.in_coff + c8 * 8;
            a[u] = *reinterpret_cast<const float4*>(src);
            b[u] = *reinterpret_cast<const float4*>(src + 4);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (dsti[u] < 0) continue;
        uint4 pk;
        pk.x = E::pack2(lr(a[u].x), lr(a[u].y));
        pk.y = E::pack2(lr(a[u].z), lr(a[u].w));
        pk.z = E::pack2(lr(b[u].x), lr(b[u].y));
        pk.w = E::pack2(lr(b[u].z), lr(b[u].w));
        *reinterpret_cast<uint4*>(bufA + size_t(dsti[u]) * 16) = pk;
      }
    }
  }
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;

  if (warp == 0) {
    // ===================== producer =====================
    if (tc::elect_one()) {
      int it = 0;
      for (int c = 0; c < p.n_chunks; ++c)
        for (int tap = 0; tap < p.taps; ++tap, ++it) {
          const int s = it % stages;
          tc::mbar_wait(&empty_bar[s], (((it / stages) & 1) ^ 1));
          tc::mbar_expect_tx(&full_bar[s], stage_bytes);
          tc::bulk_g2s(wring + size_t(s) * stage_bytes, p.w + (size_t(c) * p.taps + tap) * size_t(p.K) * NC,
                       stage_bytes, &full_bar[s]);
        }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (tc::elect_one()) {
      const uint32_t idesc = tc::make_idesc(128, NC, FMT);
      const uint32_t abase = tc::smem_u32(bufA);
      int it = 0;
      for (int c = 0; c < p.n_chunks; ++c) {
        const int b = c & 1;
        tc::mbar_wait(&acc_empty[b], (((c >> 1) & 1) ^ 1));
        tc::fence_after_sync();
        for (int tap = 0; tap < p.taps; ++tap, ++it) {
          const int s = it % stages;
          tc::mbar_wait(&full_bar[s], ((it / stages) & 1));
          tc::fence_after_sync();
          const uint32_t wbase = tc::smem_u32(wring + size_t(s) * stage_bytes);
          // k-step outer, tile inner: consecutive MMAs alternate between the two accumulators
          // (a dependent accumulate chain costs ~115 cycles per instruction, tools/ubench.py)
          for (int ks = 0; ks < p.K / 16; ++ks) {
            const uint64_t bd = tc::make_desc(wbase + uint32_t(ks * 2 * NC) * 16u, uint32_t(NC) * 16u, 128u);
#pragma unroll
            for (int m = 0; m < NT; ++m) {
              const int arow = m * 128 + tap * p.dil;
              const uint64_t ad =
                  tc::make_desc(abase + uint32_t((ks * 2) * rows_a + arow) * 16u, uint32_t(rows_a) * 16u, 128u);
              tc::mma_f16_ss(tmem + uint32_t(b * NT + m) * NC, ad, bd, idesc, (tap | ks) ? 1u : 0u);
            }
          }
          tc::mma_commit(&empty_bar[s]);
        }
        tc::mma_commit(&acc_full[b]);
      }
    }
  } else {
    // ===================== epilogue (8 warps) =====================
    const int q = warp & 3;            // TMEM lane quarter this warp may touch
    const int hh = (warp - 2) >> 2;    // column half
    const uint32_t lane_base = tmem + (uint32_t(q * 32) << 16);
    for (int c = 0; c < p.n_chunks; ++c) {
      const int b = c & 1;
      tc::mbar_wait(&acc_full[b], ((c >> 1) & 1));
      tc::fence_after_sync();
      for (int m = 0; m < NT; ++m) {
        const int t = t0 + m * 128 + q * 32 + lane;
        const bool row_ok = t < rows;
        const uint32_t acc = lane_base + uint32_t(b * NT + m) * NC;
        if (!RES && p.epi == TC_GATE) {
          const int cpt = NC / 4;  // gated channels per thread
          for (int cc = 0; cc < cpt; cc += 16) {
            __syncwarp();
            const int j0 = hh * cpt + cc;
            float va[16], vb[16];
            tc::tmem_ld16(acc + j0, va);
            tc::tmem_ld16(acc + NC / 2 + j0, vb);
            tc::tmem_ld_wait();
            if (row_ok && t < out_len) {
              const long long orow = out_base + t;
              const int ch0 = c * (NC / 2) + j0;
              float o[16];
#pragma unroll
              for (int e = 0; e < 16; ++e) {
                const int ch = ch0 + e;
                float a = va[e], g = vb[e];
                if (ch < p.N) {
                  a += p.bias[ch];
                  g += p.bias[p.N + ch];
                  if (p.ubias) {
                    a += p.ubias[(long long)seg * p.ub_stride + ch];
                    g += p.ubias[(long long)seg * p.ub_stride + p.N + ch];
                  }
                }
                o[e] = tanhf(a) * (1.f / (1.f + expf(-g)));
              }
              if (ch0 + 15 < p.N) {
                float4* dst = reinterpret_cast<float4*>(p.out + orow * p.out_stride + p.out_coff + ch0);
#pragma unroll
                for (int e = 0; e < 4; ++e) dst[e] = make_float4(o[4 * e], o[4 * e + 1], o[4 * e + 2], o[4 * e + 3]);
              } else {
                for (int e = 0; e < 16; ++e)
                  if (ch0 + e < p.N) p.out[orow * p.out_stride + p.out_coff + ch0 + e] = o[e];
              }
            }
          }
        } else {
          const int cpt = NC / 2;
          for (int cc = 0; cc < cpt; cc += 16) {
            __syncwarp();
            const int j0 = hh * cpt + cc;
            float v[16];
            tc::tmem_ld16(acc + j0, v);
            tc::tmem_ld_wait();
            if (!row_ok) continue;
            const int n0 = c * NC + j0;
            if constexpr (RES) {
              // same operation order as the fp32 conv's epilogue: ((acc + bias) + res) * scale, then store or add
              if (t >= out_len) continue;
              const long long orow = out_base + t;
              float4 r[4], cur[4];
#pragma unroll
              for (int e4 = 0; e4 < 4; ++e4) {  // all operands in flight together
                const int n = n0 + e4 * 4;
                if (n >= p.N) continue;
                r[e4] = *reinterpret_cast<const float4*>(p.res + orow * p.res_stride + n);
                if (p.accumulate) cur[e4] = *reinterpret_cast<const float4*>(p.out + orow * p.out_stride + p.out_coff + n);
              }
#pragma unroll
              for (int e4 = 0; e4 < 4; ++e4) {
                const int n = n0 + e4 * 4;
                if (n >= p.N) continue;
                const float* rr = reinterpret_cast<const float*>(&r[e4]);
                float o[4];
#pragma unroll
                for (int f = 0; f < 4; ++f) o[f] = (v[e4 * 4 + f] + p.bias[n + f] + rr[f]) * p.scale;
                if (p.accumulate) {
                  o[0] += cur[e4].x;
                  o[1] += cur[e4].y;
                  o[2] += cur[e4].z;
                  o[3] += cur[e4].w;
                }
                *reinterpret_cast<float4*>(p.out + orow * p.out_stride + p.out_coff + n) = make_float4(o[0], o[1], o[2], o[3]);
              }
              continue;
            }
            if (p.epi == TC_UPS && p.wide) {
              // same mapping, one full 32-byte sector per lane and store (Cout % 8 == 0: the 8 columns of a
              // group share their phase)
#pragma unroll
              for (int e = 0; e < 16; e += 8) {
                const int n = n0 + e;
                if (n >= p.N) break;
                const int phase = n / p.ups_cout, co = n - phase * p.ups_cout;
                const int po = t * p.ups_u + phase - p.ups_pad;
                if (po < 0 || po >= out_len) continue;
                float o[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) o[k] = v[e + k] + p.bias[co + k];
                tc::stg256(p.out + (out_base + po) * p.out_stride + co, o);
              }
              continue;
            }
            if (p.epi == TC_UPS) {
              // column n = phase * Cout + co ; output row = t*u + phase - pad
#pragma unroll 1
              for (int e = 0; e < 16; e += 4) {
                const int n = n0 + e;
                if (n >= p.N) break;
                const int phase = n / p.ups_cout, co = n - phase * p.ups_cout;
                const int po = t * p.ups_u + phase - p.ups_pad;
                if (po < 0 || po >= out_len) continue;
                const float4 o = make_float4(v[e] + p.bias[co], v[e + 1] + p.bias[co + 1], v[e + 2] + p.bias[co + 2],
                                             v[e + 3] + p.bias[co + 3]);
                *reinterpret_cast<float4*>(p.out + (out_base + po) * p.out_stride + co) = o;
              }
              continue;
            }
            if (t >= out_len) continue;
            const long long orow = out_base + t;
            float4* d4[4];
            float4 cur[4];
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {  // all read-modify-write operands in flight together
              const int n = n0 + e4 * 4;
              d4[e4] = nullptr;
              if (n < p.N) {
                float* dst = n < p.split ? p.out + orow * p.out_stride + p.out_coff + n
                                         : p.out2 + orow * p.out2_stride + (n - p.split);
                d4[e4] = reinterpret_cast<float4*>(dst);
                if (p.epi != TC_STORE) cur[e4] = *d4[e4];
              }
            }
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
              if (!d4[e4]) continue;
              const int n = n0 + e4 * 4;
              float o[4];
#pragma unroll
              for (int f = 0; f < 4; ++f) {
                o[f] = v[e4 * 4 + f];
                if (p.bias) o[f] += p.bias[n + f];
                if (p.ubias) o[f] += p.ubias[(long long)seg * p.ub_stride + n + f];
              }
              if (p.epi == TC_STORE) {
                *d4[e4] = make_float4(o[0], o[1], o[2], o[3]);
              } else if (p.epi == TC_RES_SKIP) {
                *d4[e4] = make_float4(cur[e4].x + o[0], cur[e4].y + o[1], cur[e4].z + o[2], cur[e4].w + o[3]);
              } else {  // TC_SUB
                *d4[e4] = make_float4(cur[e4].x - o[0], cur[e4].y - o[1], cur[e4].z - o[2], cur[e4].w - o[3]);
              }
            }
          }
        }
      }
      __syncwarp();
      tc::fence_before_sync();
      if (lane == 0) tc::mbar_arrive(&acc_empty[b]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<512>(tmem);
}

bool conv_tc_supported(int K, int NC, int taps, int dil, int m_tiles) {
  if (K % 16 || K < 16 || K > 512) return false;
  if (NC % 32 || NC < 32 || NC > 128) return false;  // 2 buffers x 2 tiles x NC <= 512 TMEM columns
  if (m_tiles != 1 && m_tiles != CT_NT) return false;
  const size_t a_bytes = size_t(K / 8) * ((m_tiles * 128 + (taps - 1) * dil) | 1) * 16 + 128;
  const size_t stage = size_t(K) * NC * 2;
  return a_bytes + 2 * stage <= size_t(CT_SMEM_MAX);
}

bool mrf1_tc_supported(int C, int nk, int nd, const int* k, const int (*dil)[3]) {
  if (C % 32 || nk < 1 || nk > 4 || nd < 1 || nd > 3) return false;
  for (int j = 0; j < nk; ++j) {
    if (k[j] < 1 || k[j] > 11 || !(k[j] & 1)) return false;
    for (int d = 0; d < nd; ++d) {
      if (dil[j][d] < 1) return false;
      if (!conv_tc_supported(C, 32, k[j], dil[j][d])) return false;  // NC = 32 is the smallest packing
    }
  }
  return true;
}

template <bool RES, int NT>
static void launch_nt(const TcConvParams& p, int fmt, dim3 grid, size_t smem, int stages, int rows_a, cudaStream_t st) {
  ensure_max_dynamic_smem(fmt ? reinterpret_cast<const void*>(conv_tc_kernel<1, RES, NT>)
                              : reinterpret_cast<const void*>(conv_tc_kernel<0, RES, NT>));
  if (fmt) conv_tc_kernel<1, RES, NT><<<grid, CT_THREADS, smem, st>>>(p, stages, rows_a);
  else conv_tc_kernel<0, RES, NT><<<grid, CT_THREADS, smem, st>>>(p, stages, rows_a);
}

template <bool RES>
static void launch_conv_tc_impl(const TcConvParams& p_in, int fmt, int n_seg, int max_seg_len, cudaStream_t st) {
  TcConvParams p = p_in;
  p.wide = (!RES && p.epi == TC_UPS && wide_io_enabled() && p.ups_cout % 8 == 0 && p.out_stride % 8 == 0 &&
            (reinterpret_cast<uintptr_t>(p.out) & 31u) == 0)
               ? 1
               : 0;
  const int rows = max_seg_len * p.in_scale + p.rows_extra;
  if (rows <= 0 || n_seg <= 0) return;
  // two M tiles per CTA whenever two weight stages fit next to the A operand, else one (e.g. K = 512 polyphase upsampler)
  int nt = CT_NT, rows_a = 0, stages = 0;
  size_t a_bytes = 0;
  const size_t stage = size_t(p.K) * p.NC * 2;
  for (; nt >= 1; --nt) {
    rows_a = (nt * 128 + (p.taps - 1) * p.dil) | 1;  // odd row pitch: conflict-free chunk-major smem stores
    a_bytes = (size_t(p.K / 8) * rows_a * 16 + 127) & ~size_t(127);
    stages = a_bytes < size_t(CT_SMEM_MAX) ? std::min(4, int((size_t(CT_SMEM_MAX) - a_bytes) / stage)) : 0;
    if (stages >= 2) break;
  }
  if (nt < 1) throw std::runtime_error("conv_tc: shape does not fit shared memory");
  // >= 120 KB keeps a single CTA per SM (each CTA owns all 512 TMEM columns)
  const size_t smem = std::max(a_bytes + stages * stage, size_t(120 * 1024));
  const int R = nt * 128;
  dim3 grid((rows + R - 1) / R, n_seg);
  if (nt == CT_NT) launch_nt<RES, CT_NT>(p, fmt, grid, smem, stages, rows_a, st);
  else launch_nt<RES, 1>(p, fmt, grid, smem, stages, rows_a, st);
  post_launch(RES ? "conv_tc_kernel(res)" : "conv_tc_kernel", st);
}

void launch_conv_tc(const TcConvParams& p, int fmt, int n_seg, int max_seg_len, cudaStream_t st) {
  launch_conv_tc_impl<false>(p, fmt, n_seg, max_seg_len, st);
}

void launch_conv_tc_res(const TcConvParams& p, int fmt, int n_seg, int max_seg_len, cudaStream_t st) {
  if (!p.res || !p.bias || p.N % 16 || p.res_stride % 4 || p.out_stride % 4 || p.out_coff % 4)
    throw std::runtime_error("conv_tc_res: needs res and bias, N % 16 == 0 and 16-byte aligned rows");
  launch_conv_tc_impl<true>(p, fmt, n_seg, max_seg_len, st);
}

}  // namespace m3
