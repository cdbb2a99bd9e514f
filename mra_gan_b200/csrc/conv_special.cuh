// Tensor-core lowering of the two degenerate-channel layers of the generator:
//
//   STEM  Conv3d(1 -> Co, k, pad 0) on the replication-padded image   (networks3D.py:185-187)
//   HEAD  Conv3d(Ci -> 1, k, pad 0) on the replication-padded features (networks3D.py:211-213)
//
// A direct implicit GEMM would have K = k^3 with Cin = 1 (stem) or N = 1 (head): hopeless for the MMA.
// Instead the (kh, kw) taps are folded into a 64-wide channel axis, c = kh*8 + kw (k <= 8):
//
//   stem fprop : E[n,d,h,w,c]   = x[n,d,h+kh,w+kw]                       (expand_hw, sgn = +1)
//                y              = GATHER_{kd}(E, B[kd][co][c])           (Cin=64 conv with a (k,1,1) kernel)
//   stem wgrad : dWe[kd][co][c] = WGRAD(dy, E)  -> scatter back to dw[(kd,kh,kw)][co]
//   stem dgrad : Z[n,d',h,w,c]  = GATHER_{kd}(dy, B^T)  ; dx[n,d',h',w'] = sum_c Z[n,d',h'-kh,w'-kw,c]  (shift_sum, sgn = -1)
//   head fprop : Z[n,d,h',w',c] = GATHER_{kd}(x, B[kd][c][ci]) ; y = act(bias + sum_c Z[n,d,h+kh,w+kw,c]) (shift_sum, sgn = +1)
//   head dgrad : E'[n,d,h',w',c] = dy[n,d,h'-kh,w'-kw] (expand_hw, sgn = -1) ; dx = GATHER_{kd}(E', B^T)
//   head wgrad : dWe[kd][c][ci] = WGRAD(E', x)  -> scatter back to dw[(kd,kh,kw)][ci]
//
// so all six run on gather_tc_kernel / wgrad_tc_kernel; the helpers here are small HBM-bound kernels.
// Cost: K efficiency k^2/64 (77 % for k = 7) and one extra 64-channel intermediate (E or Z) per call.
#pragma once
#include "common.cuh"
#include "conv_plan.h"
#include "conv_tc_halo.cuh"

namespace mra {
namespace special {

// out[n,d,ho,wo,kh*8+kw] = src[n,d,ho+sgn*kh+off,wo+sgn*kw+off] (0 out of range / kh,kw >= k).
// One block = a band of kExpandBand output lines of one (n, d) plane: the band + 7 source lines it touches are staged
// in shared memory once (zero outside the volume; line l holds source columns j + base, base = off - (sgn < 0 ? 7 : 0)),
// then one thread per (wo, kh) writes 8 channels = 16 B; a warp writes 512 contiguous bytes.  The 8 source values of an
// item are consecutive in the staged line (ascending for sgn > 0, descending for sgn < 0): they are fetched as five
// aligned 32-bit words and cut out with one funnel shift / byte permute per output word (the first version read them
// as 8 scalar bf16 and was bound by instruction issue at 2.7 TB/s of stores).
constexpr int kExpandBand = 16;
__global__ void __launch_bounds__(256) expand_hw_kernel(const bf16* __restrict__ src, bf16* __restrict__ out, long long rows /*N*D*/,
                                                         int Hs, int Ws, int Ho, int Wo, int k, int sgn, int off, int pitch) {
  extern __shared__ uint32_t s_words[];              // [kExpandBand + 7][pitch / 2]
  const int pw = pitch >> 1;                         // words per staged line
  const int nbands = (Ho + kExpandBand - 1) / kExpandBand;
  const long long nwork = rows * nbands;
  const int base = off - (sgn < 0 ? 7 : 0);
  // zero masks for kw >= k inside output word i (kw = 2i, 2i + 1)
  uint32_t wmask[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) wmask[i] = (2 * i < k ? 0x0000ffffu : 0u) | (2 * i + 1 < k ? 0xffff0000u : 0u);
  for (long long wk = blockIdx.x; wk < nwork; wk += gridDim.x) {
    const int bi = (int)(wk % nbands);
    const long long r = wk / nbands;
    const int ho0 = bi * kExpandBand, nlo = min(kExpandBand, Ho - ho0);
    // staged line l <-> source line hs = hs0 + l;  output line ho uses line (ho - ho0) + (sgn > 0 ? kh : 7 - kh)
    const int hs0 = ho0 + off - (sgn < 0 ? 7 : 0);
    const int nl = nlo + 7;
    __syncthreads();                                 // previous band fully written out
    bf16* sl = reinterpret_cast<bf16*>(s_words);
    for (int l = 0; l < nl; ++l) {
      const int hs = hs0 + l;
      const bf16* gl = src + (r * Hs + hs) * (long long)Ws;
      for (int j = threadIdx.x; j < pitch; j += blockDim.x) {
        const int ws = j + base;
        bf16 v = __float2bfloat16_rn(0.f);
        if (hs >= 0 && hs < Hs && ws >= 0 && ws < Ws) v = gl[ws];
        sl[l * pitch + j] = v;
      }
    }
    __syncthreads();
    for (int lo = 0; lo < nlo; ++lo) {
      uint4* oline = reinterpret_cast<uint4*>(out + ((r * Ho + ho0 + lo) * (long long)Wo) * 64);
      for (int i = threadIdx.x; i < Wo * 8; i += blockDim.x) {
        const int kh = i & 7, wo = i >> 3;
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (kh < k) {
          const int l = lo + (sgn > 0 ? kh : 7 - kh);
          const int e0 = wo;                         // lowest staged column of the item (columns e0 .. e0 + 7)
          const uint32_t* w = s_words + l * pw + (e0 >> 1);
          const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3], w4 = w[4];
          if (sgn > 0) {
            const uint32_t sh = (uint32_t)(e0 & 1) * 16u;
            o.x = __funnelshift_r(w0, w1, sh); o.y = __funnelshift_r(w1, w2, sh);
            o.z = __funnelshift_r(w2, w3, sh); o.w = __funnelshift_r(w3, w4, sh);
          } else if (e0 & 1) {                       // descending from column e0 + 7: (lo of w[4-i], hi of w[3-i])
            o.x = __byte_perm(w4, w3, 0x7610); o.y = __byte_perm(w3, w2, 0x7610);
            o.z = __byte_perm(w2, w1, 0x7610); o.w = __byte_perm(w1, w0, 0x7610);
          } else {                                   // descending, even start: halves of w[3-i] swapped
            o.x = __byte_perm(w3, 0u, 0x1032); o.y = __byte_perm(w2, 0u, 0x1032);
            o.z = __byte_perm(w1, 0u, 0x1032); o.w = __byte_perm(w0, 0u, 0x1032);
          }
          o.x &= wmask[0]; o.y &= wmask[1]; o.z &= wmask[2]; o.w &= wmask[3];
        }
        oline[i] = o;
      }
    }
  }
}

// out[n,d,ho,wo] = act(bias + sum_{kh,kw<k} Z[n,d,ho+sgn*kh+off,wo+sgn*kw+off,kh*8+kw])
// One block = a band of output lines of one (n, d) plane.  Every Z line of the band is read from global memory ONCE
// (coalesced cp.async) into a padded shared-memory line (position pitch 33 words: conflict-free column reads);
// thread wo then adds the line's k*k contributions to the <= 8 output lines that are still open, which it keeps in
// registers (a statically rotated window of 8 partial sums).
// SGN and K are COMPILE-TIME parameters: the window slot of an output line is ((u - SGN*kh) mod 8) with u, kh unrolled,
// i.e. a constant only when the sign is one -- the first version took sgn and k as kernel arguments, which made acc[] a
// run-time indexed array in LOCAL memory (146 LDL/STL in its SASS, 80 registers, ~800 predicate instructions) and the
// kernel ran at 2.1 TB/s.  CHECKW = false when the host has shown that every wo + SGN*kw + off lies inside the Z line.
template <typename TO, int SGN, int K, bool CHECKW>
__global__ void __launch_bounds__(256) shift_sum_kernel(const bf16* __restrict__ Z, TO* __restrict__ out, long long rows, int Hz,
                                                         int Wz, int Ho, int Wo, int off, const float* __restrict__ bias, int act,
                                                         float slope, int band) {
  static_assert(K >= 1 && K <= 8 && (SGN == 1 || SGN == -1), "shift_sum: window of 8 lines");
  extern __shared__ uint32_t s_z[];                  // 2 x [Wz][33] words: 64 bf16 of one position + 1 pad word
  const float b = bias ? bias[0] : 0.f;
  const int nbands = (Ho + band - 1) / band;
  const long long nwork = rows * nbands;
  const int wo = threadIdx.x;                        // Wo <= blockDim.x (host)
  const int buf_words = Wz * 33;
  for (long long wk = blockIdx.x; wk < nwork; wk += gridDim.x) {
    const int bi = (int)(wk % nbands);
    const long long r = wk / nbands;
    const int ho0 = bi * band, ho1 = min(Ho, ho0 + band);
    // Z lines that feed output lines [ho0, ho1): hz = ho + SGN*kh + off, kh in [0, K)
    const int hz_lo = SGN > 0 ? ho0 + off : ho0 - (K - 1) + off;
    const int hz_hi = SGN > 0 ? ho1 - 1 + (K - 1) + off : ho1 - 1 + off;       // inclusive
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    // Z lines are double-buffered: while line hz is being added up, line hz + 1 streams into the other buffer with
    // cp.async (4-byte pieces: the 33-word pitch that makes the column reads conflict-free is not 16-byte aligned; a
    // warp moves the 128 contiguous bytes of one position per instruction)
    // (a warp copies whole positions -- 32 words -- and walks them with two pointer increments per copy: the first version
    // recomputed (i >> 5) * 33 + (i & 31) and the 64-bit global address per element, 13 instructions per 4-byte copy, three
    // times the cost of the additions the kernel is there for; ncu showed it no faster than its predecessor at 177 us)
    auto stage = [&](int hz, uint32_t* dst) {
      if (hz >= 0 && hz < Hz && hz <= hz_hi) {
        const int nw = (int)(blockDim.x >> 5), wp = (int)(threadIdx.x >> 5), ln = (int)(threadIdx.x & 31);
        const uint32_t* gp = reinterpret_cast<const uint32_t*>(Z + ((r * Hz + hz) * (long long)Wz) * 64) + wp * 32 + ln;
        uint32_t sa = (uint32_t)__cvta_generic_to_shared(dst + wp * 33 + ln);
        const uint32_t sstep = (uint32_t)nw * 33u * 4u;
        const int gstep = nw * 32;
#pragma unroll 4
        for (int pz = wp; pz < Wz; pz += nw) {
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(gp) : "memory");
          sa += sstep; gp += gstep;
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    __syncthreads();                                 // the previous band is done with both buffers
    stage(hz_lo, s_z);
    int cur = 0;
    // the lines are processed in groups of 8 so that the rotating window index is static
    for (int hz0 = hz_lo; hz0 <= hz_hi; hz0 += 8) {
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int hz = hz0 + u;
        if (hz > hz_hi) break;
        const uint32_t* s_cur = s_z + cur * buf_words;
        stage(hz + 1, s_z + (cur ^ 1) * buf_words);   // that buffer was last read before the barrier closing line hz - 1
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        if (wo < Wo) {
          if (hz >= 0 && hz < Hz) {                  // (block-uniform) a line outside Z contributes zeros
            // contributions of line hz: to output line ho = hz - off - SGN*kh, kept in slot (u - SGN*kh) mod 8
#pragma unroll
            for (int kh = 0; kh < K; ++kh) {
              float s = 0.f;
#pragma unroll
              for (int kw = 0; kw < K; ++kw) {
                const int wz = wo + SGN * kw + off;
                if (!CHECKW || (unsigned)wz < (unsigned)Wz) {
                  const uint32_t wrd = s_cur[wz * 33 + ((kh * 8 + kw) >> 1)];
                  s += __uint_as_float((kw & 1) ? (wrd & 0xffff0000u) : (wrd << 16));
                }
              }
              acc[((u - SGN * kh) % 8 + 8) % 8] += s;
            }
          }
          // the output line completed by this Z line: for SGN > 0 it is ho = hz - off - (K-1) (its last contributor is
          // kh = K-1); for SGN < 0 it is ho = hz - off (last contributor kh = 0)
          const int ho_done = SGN > 0 ? hz - off - (K - 1) : hz - off;
          constexpr int kDoneShift = SGN > 0 ? K - 1 : 0;
          float& a_done = acc[((u - kDoneShift) % 8 + 8) % 8];
          if (ho_done >= ho0 && ho_done < ho1)
            out[(r * Ho + ho_done) * (long long)Wo + wo] = from_f<TO>(apply_act(a_done + b, act, slope));
          a_done = 0.f;
        }
        __syncthreads();                             // line hz fully consumed: its buffer may be refilled
        cur ^= 1;
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
}

// src [k^3][C] (the packed weight of a layer whose other channel count is 1)
//   mode 0: dst[kd][ch][c] = src[(kd,kh,kw)][ch]      mode 1: dst[kd][c][ch] = src[(kd,kh,kw)][ch]     (c = kh*8+kw)
__global__ void wexp_kernel(const bf16* __restrict__ src, bf16* __restrict__ dst, int k, int C, int mode) {
  const int total = k * C * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int kd, ch, c;
    if (mode == 0) { c = i % 64; ch = (i / 64) % C; kd = i / (64 * C); }
    else           { ch = i % C; c = (i / C) % 64; kd = i / (64 * C); }
    const int kh = c >> 3, kw = c & 7;
    bf16 v = __float2bfloat16_rn(0.f);
    if (kh < k && kw < k) v = src[((long long)(kd * k + kh) * k + kw) * C + ch];
    dst[i] = v;
  }
}
// dw[(kd,kh,kw)][ch] += dWe (mode 0: dWe[kd][ch][c], mode 1: dWe[kd][c][ch])
__global__ void wunexp_kernel(const float* __restrict__ dwe, float* __restrict__ dw, int k, int C, int mode) {
  const int total = k * k * k * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ch = i % C;
    const int t = i / C;
    const int kw = t % k, kh = (t / k) % k, kd = t / (k * k);
    const int c = kh * 8 + kw;
    const float v = mode == 0 ? dwe[((long long)kd * C + ch) * 64 + c] : dwe[((long long)kd * 64 + c) * C + ch];
    dw[i] += v;
  }
}

// PatchGAN layer 0 (networks3D.py:392): Conv3d(1 -> Co, k4, s2, p1).  With Cin = 1 and k^3 <= 64 the whole
// receptive field fits one 64-wide channel axis: E[n,o,(kd,kh,kw)] = x[n, o*s - p + k] (im2col), after which
// the layer is a 1x1x1 convolution (one GEMM tap) on the tensor cores; dgrad is the GEMM followed by col2im.
// (Index arithmetic is 32-bit with one tap decode per thread: the first version spent ~250 instructions per 16-byte
// store on 64-bit divisions and ran at 0.5 TB/s; positions are checked to fit 31 bits on the host.)
__global__ void __launch_bounds__(256) im2col1_kernel(const bf16* __restrict__ x, bf16* __restrict__ E, int N, int Di, int Hi, int Wi,
                                                       int Do, int Ho, int Wo, int k, int s, int p) {
  const unsigned total = (unsigned)N * Do * Ho * Wo * 8u;         // one thread = 8 consecutive channels
  const int taps = k * k * k;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int c0 = (int)(i & 7u) * 8;
    unsigned q = i >> 3;
    const int ow = (int)(q % (unsigned)Wo); q /= (unsigned)Wo;
    const int oh = (int)(q % (unsigned)Ho); q /= (unsigned)Ho;
    const int od = (int)(q % (unsigned)Do);
    const int n = (int)(q / (unsigned)Do);
    int kw = c0 % k, kh = (c0 / k) % k, kd = c0 / (k * k);        // taps c0 .. c0 + 7 walk (kd, kh, kw) incrementally
    const bf16* xn = x + (long long)n * Di * Hi * Wi;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[j] = 0.f;
      if (c0 + j < taps) {
        const int d = od * s - p + kd, h = oh * s - p + kh, w = ow * s - p + kw;
        if ((unsigned)d < (unsigned)Di && (unsigned)h < (unsigned)Hi && (unsigned)w < (unsigned)Wi)
          v[j] = __bfloat162float(xn[(d * Hi + h) * Wi + w]);
      }
      if (++kw == k) { kw = 0; if (++kh == k) { kh = 0; ++kd; } }
    }
    Vec8<bf16>::store(E + (long long)(i >> 3) * 64 + c0, v);
  }
}
// dx[n,i] = sum over (o, k) with o*s - p + k == i of dE[n,o,(kd,kh,kw)].  Per dim only ceil(k/s) output coordinates can
// reach an input voxel: o = (i + p) / s - j, tap = (i + p) - o*s.
__global__ void __launch_bounds__(256) col2im1_kernel(const bf16* __restrict__ dE, bf16* __restrict__ dx, int N, int Di, int Hi, int Wi,
                                                       int Do, int Ho, int Wo, int k, int s, int p,
                                                       const float* __restrict__ bias, int act, float slope) {
  const float bv = bias ? bias[0] : 0.f;
  const unsigned total = (unsigned)N * Di * Hi * Wi;
  const int R = (k + s - 1) / s;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    unsigned q = i;
    const int w = (int)(q % (unsigned)Wi); q /= (unsigned)Wi;
    const int h = (int)(q % (unsigned)Hi); q /= (unsigned)Hi;
    const int d = (int)(q % (unsigned)Di);
    const int n = (int)(q / (unsigned)Di);
    const bf16* En = dE + (long long)n * Do * Ho * Wo * 64;
    const int od0 = (d + p) / s, oh0 = (h + p) / s, ow0 = (w + p) / s;
    float acc = 0.f;
    for (int jd = 0; jd < R; ++jd) {
      const int od = od0 - jd, kd = d + p - od * s;
      if (od < 0 || od >= Do || kd >= k) continue;
      for (int jh = 0; jh < R; ++jh) {
        const int oh = oh0 - jh, kh = h + p - oh * s;
        if (oh < 0 || oh >= Ho || kh >= k) continue;
        const bf16* Er = En + ((long long)(od * Ho + oh) * Wo) * 64 + (kd * k + kh) * k;
        for (int jw = 0; jw < R; ++jw) {
          const int ow = ow0 - jw, kw = w + p - ow * s;
          if (ow < 0 || ow >= Wo || kw >= k) continue;
          acc += __bfloat162float(Er[ow * 64 + kw]);
        }
      }
    }
    dx[i] = __float2bfloat16_rn(apply_act(acc + bv, act, slope));
  }
}
// B[co][c] = w[c][co] (c < taps, else 0)  /  BT[c][co]  /  dw[t][co] += dWe[co][t]
__global__ void im2col_w_kernel(const bf16* __restrict__ w, bf16* __restrict__ B, int taps, int C, int transpose) {
  const int total = C * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int ch, c;
    if (!transpose) { c = i % 64; ch = i / 64; } else { ch = i % C; c = i / C; }
    B[i] = c < taps ? w[(long long)c * C + ch] : __float2bfloat16_rn(0.f);
  }
}
__global__ void im2col_dw_kernel(const float* __restrict__ dwe, float* __restrict__ dw, int taps, int C) {
  const int total = taps * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ch = i % C, t = i / C;
    dw[i] += dwe[(long long)ch * 64 + t];
  }
}

inline int launch_expand_hw(const bf16* src, bf16* out, long long rows, int Hs, int Ws, int Ho, int Wo, int k, int sgn, int off,
                            cudaStream_t st) {
  const long long nwork = rows * ((Ho + kExpandBand - 1) / kExpandBand);
  long long grid = nwork < (long long)num_sms() * 8 ? nwork : (long long)num_sms() * 8;
  if (grid < 1) grid = 1;
  // staged line: Wo + 8 columns + 2 of slack for the fifth word; an odd number of words per line spreads the 8 lines
  // a warp reads (one per kh) over the banks
  int pitch = (Wo + 10 + 1) & ~1;
  if (((pitch >> 1) & 1) == 0) pitch += 2;
  const size_t smem = (size_t)(kExpandBand + 7) * pitch * sizeof(bf16);
  MRA_REQUIRE(smem <= 48 * 1024, "expand_hw: line too long (Wo = %d)", Wo);
  expand_hw_kernel<<<(unsigned)grid, 256, smem, st>>>(src, out, rows, Hs, Ws, Ho, Wo, k, sgn, off, pitch);
  MRA_LAUNCH_CHECK();
  return 0;
}
// Launch geometry of shift_sum: blocks of round_up(Wo, 32) threads (one thread per output column -- the first version
// always ran 256, half of them idle for a 128-wide line, and its 80 registers x 256 threads allowed 3 blocks per SM);
// bands sized to the resident block count: rows = 256 planes (batch 2 x 128) on 148 x 6 slots -> 3 bands of 43 lines =
// 768 items in one wave, instead of 1024 items of 32 lines in 2.3 waves.  A band re-reads the K - 1 Z lines it shares
// with its neighbour (L2 hits).
// Two line buffers of Wz positions x 33 words: 67.6 KB for the widest line the stem / head lowerings accept (256).
inline size_t shift_sum_smem(int Wz) { return (size_t)2 * Wz * 33 * sizeof(uint32_t); }
template <typename TO, int SGN, int K, bool CHECKW>
inline int launch_shift_sum_t(const bf16* Z, TO* out, long long rows, int Hz, int Wz, int Ho, int Wo, int off, const float* bias,
                              int act, float slope, cudaStream_t st) {
  auto kern = shift_sum_kernel<TO, SGN, K, CHECKW>;
  int threads = ((Wo + 31) / 32) * 32;
  if (threads < 64) threads = 64;
  const size_t smem = shift_sum_smem(Wz);
  MRA_REQUIRE(smem <= max_optin_smem(), "shift_sum: Z line does not fit shared memory (Wz = %d)", Wz);
  // resident blocks per SM for this (kernel, block size, shared memory): asked once per configuration (host-side query,
  // no stream work; the first call of a configuration happens in the eager warm-up steps, before any graph capture)
  static std::mutex mu;
  static std::map<std::pair<int, size_t>, int> occ_cache;
  static bool attr_set = false;
  int occ = 0;
  {
    std::lock_guard<std::mutex> lk(mu);
    if (!attr_set) {                                 // lines wider than 186 positions need more than the default 48 KB
      MRA_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_optin_smem()));
      attr_set = true;
    }
    auto key = std::make_pair(threads, smem);
    auto it = occ_cache.find(key);
    if (it == occ_cache.end()) {
      MRA_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
      if (occ < 1) occ = 1;
      occ_cache[key] = occ;
    } else {
      occ = it->second;
    }
  }
  const long long slots = (long long)num_sms() * occ;
  // bands per plane: minimise (rounds of the block-cyclic schedule) x (Z lines per band, K - 1 of them re-read)
  int band = Ho;
  long long best = -1;
  for (int nb = 1; nb <= (Ho + 7) / 8; ++nb) {
    const int bd = (Ho + nb - 1) / nb;
    const long long items = rows * ((Ho + bd - 1) / bd);
    const long long cost = ((items + slots - 1) / slots) * (bd + K - 1);
    if (best < 0 || cost < best) { best = cost; band = bd; }
  }
  const long long nwork = rows * ((Ho + band - 1) / band);
  long long grid = nwork < slots ? nwork : slots;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, threads, smem, st>>>(Z, out, rows, Hz, Wz, Ho, Wo, off, bias, act, slope, band);
  MRA_LAUNCH_CHECK();
  return 0;
}
inline int launch_shift_sum(const bf16* Z, bf16* out, long long rows, int Hz, int Wz, int Ho, int Wo, int k, int sgn, int off,
                            const float* bias, int act, float slope, cudaStream_t st) {
  MRA_REQUIRE(Wo <= 256 && k >= 1 && k <= 8 && (sgn == 1 || sgn == -1), "shift_sum: line longer than a block (Wo = %d) or k = %d", Wo, k);
  // does any (wo, kw) fall outside the Z line?
  const int wlo = sgn > 0 ? off : off - (k - 1), whi = sgn > 0 ? Wo - 1 + (k - 1) + off : Wo - 1 + off;
  const bool check_w = wlo < 0 || whi >= Wz;
#define MRA_SS_CASE(KK)                                                                                                          \
  case KK:                                                                                                                       \
    if (sgn > 0) {                                                                                                               \
      if (check_w) return launch_shift_sum_t<bf16, 1, KK, true>(Z, out, rows, Hz, Wz, Ho, Wo, off, bias, act, slope, st);        \
      return launch_shift_sum_t<bf16, 1, KK, false>(Z, out, rows, Hz, Wz, Ho, Wo, off, bias, act, slope, st);                    \
    }                                                                                                                            \
    if (check_w) return launch_shift_sum_t<bf16, -1, KK, true>(Z, out, rows, Hz, Wz, Ho, Wo, off, bias, act, slope, st);         \
    return launch_shift_sum_t<bf16, -1, KK, false>(Z, out, rows, Hz, Wz, Ho, Wo, off, bias, act, slope, st);
  switch (k) {
    MRA_SS_CASE(1) MRA_SS_CASE(2) MRA_SS_CASE(3) MRA_SS_CASE(4) MRA_SS_CASE(5) MRA_SS_CASE(6) MRA_SS_CASE(7) MRA_SS_CASE(8)
  }
#undef MRA_SS_CASE
  return ::mra::fail(-1, "shift_sum: unsupported k = %d", k);
}

struct Workspace {
  char* base; size_t size, off;
  void* take(size_t bytes) {
    off = (off + 255) & ~size_t(255);
    if (off + bytes > size) return nullptr;
    void* p = base + off;
    off += bytes;
    return p;
  }
};

inline bool stem_eligible(const mra_conv_desc& d) {
  return d.dtype == MRA_BF16 && !(d.flags & MRA_CONV_FORCE_NAIVE) && !d.transposed && d.stride == 1 && d.pad == 0 &&
         d.cin == 1 && d.k >= 2 && d.k <= 8 && d.win <= 256 && tc::tc_channels_ok(d.cout);
}
inline bool head_eligible(const mra_conv_desc& d) {
  return d.dtype == MRA_BF16 && !(d.flags & MRA_CONV_FORCE_NAIVE) && !d.transposed && d.stride == 1 && d.pad >= 0 &&
         d.pad < d.k && d.cout == 1 && d.k >= 2 && d.k <= 8 && d.win <= 256 && tc::tc_channels_ok(d.cin);
}

inline bool im2col_eligible(const mra_conv_desc& d) {
  // (the im2col / col2im helpers index with 32 bits)
  if ((long long)d.n * d.dout * d.hout * d.wout * 8 >= (1ll << 32) || (long long)d.n * d.din * d.hin * d.win >= (1ll << 31))
    return false;
  return d.dtype == MRA_BF16 && !(d.flags & MRA_CONV_FORCE_NAIVE) && !d.transposed && d.cin == 1 &&
         d.k * d.k * d.k <= 64 && tc::tc_channels_ok(d.cout) && !(d.stride == 1 && d.pad == 0 && d.k >= 2);
}
// ConvTranspose3d(C -> 1, k, s, p) (the UNet's outermost up-convolution, networks3D.py:312-316) is, operand for operand,
// the mirror Conv3d(1 -> C, k, s, p) with the roles of x and y swapped:
//   convT fprop(x, w)  = mirror dgrad(dy := x)  (+ bias, activation)      convT dgrad(dy) = mirror fprop(x := dy)
//   convT wgrad(x, dy) = mirror wgrad(x := dy, dy := x)
// and the packed weights coincide byte for byte ([taps][1][C] vs [taps][C][1]).  So it rides the im2col lowering.
inline mra_conv_desc convT1_mirror(const mra_conv_desc& d) {
  mra_conv_desc m = d;
  m.cin = 1; m.cout = d.cin;
  m.din = d.dout; m.hin = d.hout; m.win = d.wout;
  m.dout = d.din; m.hout = d.hin; m.wout = d.win;
  m.transposed = 0; m.act = MRA_ACT_NONE;
  return m;
}
inline bool convT1_eligible(const mra_conv_desc& d) {
  if (!d.transposed || d.cout != 1 || d.dtype != MRA_BF16 || (d.flags & MRA_CONV_FORCE_NAIVE)) return false;
  const mra_conv_desc m = convT1_mirror(d);
  // the mirror must be a valid convolution (output_padding < stride guarantees it) that the im2col path accepts
  if ((m.din + 2 * m.pad - m.k) / m.stride + 1 != m.dout || (m.hin + 2 * m.pad - m.k) / m.stride + 1 != m.hout ||
      (m.win + 2 * m.pad - m.k) / m.stride + 1 != m.wout)
    return false;
  return im2col_eligible(m);
}
inline GeomEx im2col_geom(const mra_conv_desc& d) {    // E [N][Do][Ho][Wo][64] -> y [N][Do][Ho][Wo][Co], 1x1x1
  GeomEx g;
  g.n = d.n; g.cin = 64; g.cout = d.cout;
  for (int i = 0; i < 3; ++i) { g.k[i] = 1; g.pad[i] = 0; }
  g.in[0] = g.out[0] = d.dout; g.in[1] = g.out[1] = d.hout; g.in[2] = g.out[2] = d.wout;
  g.stride = 1; g.transposed = 0;
  return g;
}

// expanded-geometry helpers
inline GeomEx stem_geom(const mra_conv_desc& d) {      // x := E [N][Din][Hout][Wout][64] -> y [N][Dout][Hout][Wout][Co]
  GeomEx g;
  g.n = d.n; g.cin = 64; g.cout = d.cout;
  g.in[0] = d.din; g.in[1] = d.hout; g.in[2] = d.wout;
  g.out[0] = d.dout; g.out[1] = d.hout; g.out[2] = d.wout;
  g.k[0] = d.k; g.k[1] = 1; g.k[2] = 1;
  g.pad[0] = g.pad[1] = g.pad[2] = 0;
  g.stride = 1; g.transposed = 0;
  return g;
}
inline GeomEx head_geom(const mra_conv_desc& d) {      // x [N][Din][Hin][Win][Ci] -> Z [N][Dout][Hin][Win][64]
  GeomEx g;
  g.n = d.n; g.cin = d.cin; g.cout = 64;
  g.in[0] = d.din; g.in[1] = d.hin; g.in[2] = d.win;
  g.out[0] = d.dout; g.out[1] = d.hin; g.out[2] = d.win;
  g.k[0] = d.k; g.k[1] = 1; g.k[2] = 1;
  g.pad[0] = d.pad; g.pad[1] = g.pad[2] = 0;      // (kh, kw) zero padding is applied by shift_sum / expand_hw
  g.stride = 1; g.transposed = 0;
  return g;
}

inline size_t a256(size_t v) { return (v + 255) & ~size_t(255); }
inline size_t workspace_bytes(const mra_conv_desc& d, int which);
inline size_t workspace_bytes_convT1(const mra_conv_desc& d) { return workspace_bytes(convT1_mirror(d), 0); }
inline size_t workspace_bytes(const mra_conv_desc& d, int which) {
  if (convT1_eligible(d)) return workspace_bytes_convT1(d);
  const size_t wexp = a256((size_t)d.k * 64 * (d.cin == 1 ? d.cout : d.cin) * 2);
  const size_t dwe = a256((size_t)d.k * 64 * (d.cin == 1 ? d.cout : d.cin) * 4);
  if (im2col_eligible(d)) {
    const size_t e = a256((size_t)d.n * d.dout * d.hout * d.wout * 64 * 2);
    return e + a256((size_t)64 * d.cout * 4) + 512;
  }
  if (stem_eligible(d)) {
    const size_t e = (size_t)d.n * d.din * d.hout * d.wout * 64;
    if (which == 0) return a256(e * 2) + wexp + 512;
    if (which == 1) return a256(e * 2) + wexp + 512;
    return a256(e * 2) + dwe + 512;
  }
  if (head_eligible(d)) {
    const size_t z = (size_t)d.n * d.dout * d.hin * d.win * 64;
    if (which == 0) return a256(z * 2) + wexp + 512;
    if (which == 1) return a256(z * 2) + wexp + 512;
    return a256(z * 2) + dwe + 512;
  }
  return 0;
}

inline unsigned sgrid(long long n) {
  long long b = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

#define MRA_WS_TAKE(var, type, bytes)                                                      \
  type* var = reinterpret_cast<type*>(ws.take(bytes));                                      \
  MRA_REQUIRE(var != nullptr, "workspace too small (need mra_conv3d_workspace_size bytes)")

inline int im2col_fprop(const mra_conv_desc& d, const void* x, const void* w, const float* bias, void* y, double* stats,
                        void* wsp, size_t wsb, cudaStream_t st) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long pos = (long long)d.n * d.dout * d.hout * d.wout;
  MRA_WS_TAKE(E, bf16, (size_t)pos * 64 * 2);
  MRA_WS_TAKE(B, bf16, (size_t)64 * d.cout * 2);
  if (!(d.flags & MRA_CONV_WS_REUSE)) {
    im2col1_kernel<<<sgrid(pos * 8), 256, 0, st>>>((const bf16*)x, E, d.n, d.din, d.hin, d.win, d.dout, d.hout, d.wout, d.k, d.stride, d.pad);
    MRA_LAUNCH_CHECK();
  }
  im2col_w_kernel<<<sgrid(64 * d.cout), 256, 0, st>>>((const bf16*)w, B, d.k * d.k * d.k, d.cout, 0);
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(im2col_geom(d), 0, plan), "im2col plan");
  tc::GatherRun R{E, B, 1, bias, y, 1, d.act, d.slope, stats};
  return tc::run_gather_tc(plan, R, st);
}
inline int im2col_wgrad(const mra_conv_desc& d, const void* x, const void* dy, float* dw, void* wsp, size_t wsb, cudaStream_t st) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long pos = (long long)d.n * d.dout * d.hout * d.wout;
  MRA_WS_TAKE(E, bf16, (size_t)pos * 64 * 2);
  MRA_WS_TAKE(dWe, float, (size_t)64 * d.cout * 4);
  if (!(d.flags & MRA_CONV_WS_REUSE)) {
    im2col1_kernel<<<sgrid(pos * 8), 256, 0, st>>>((const bf16*)x, E, d.n, d.din, d.hin, d.win, d.dout, d.hout, d.wout, d.k, d.stride, d.pad);
    MRA_LAUNCH_CHECK();
  }
  MRA_CHECK_CUDA(cudaMemsetAsync(dWe, 0, (size_t)64 * d.cout * 4, st));
  WgradPlan plan;
  MRA_REQUIRE(build_wgrad_plan(im2col_geom(d), plan), "im2col wgrad plan");
  if (int rc = tc::run_wgrad_tc(plan, E, dy, dWe, st)) return rc;           // dWe[co][c]
  im2col_dw_kernel<<<sgrid((long long)d.k * d.k * d.k * d.cout), 256, 0, st>>>(dWe, dw, d.k * d.k * d.k, d.cout);
  MRA_LAUNCH_CHECK();
  return 0;
}
inline int im2col_dgrad(const mra_conv_desc& d, const void* dy, const void* wT, void* dx, void* wsp, size_t wsb, cudaStream_t st,
                        const float* bias = nullptr, int act = MRA_ACT_NONE, float slope = 0.f) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long pos = (long long)d.n * d.dout * d.hout * d.wout;
  MRA_WS_TAKE(dE, bf16, (size_t)pos * 64 * 2);
  MRA_WS_TAKE(BT, bf16, (size_t)64 * d.cout * 2);
  im2col_w_kernel<<<sgrid(64 * d.cout), 256, 0, st>>>((const bf16*)wT, BT, d.k * d.k * d.k, d.cout, 1);    // [c][co]
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(im2col_geom(d), 1, plan), "im2col dgrad plan");
  tc::GatherRun R{dy, BT, 1, nullptr, dE, 1, MRA_ACT_NONE, 0.f, nullptr};
  if (int rc = tc::run_gather_tc(plan, R, st)) return rc;
  col2im1_kernel<<<sgrid((long long)d.n * d.din * d.hin * d.win), 256, 0, st>>>(dE, (bf16*)dx, d.n, d.din, d.hin, d.win, d.dout, d.hout,
                                                                                  d.wout, d.k, d.stride, d.pad, bias, act, slope);
  MRA_LAUNCH_CHECK();
  return 0;
}


inline int stem_fprop(const mra_conv_desc& d, const void* x, const void* w, const float* bias, void* y, double* stats,
                      void* wsp, size_t wsb, cudaStream_t st) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.din;
  MRA_WS_TAKE(E, bf16, (size_t)rows * d.hout * d.wout * 64 * 2);
  MRA_WS_TAKE(B, bf16, (size_t)d.k * d.cout * 64 * 2);
  MRA_REQUIRE(launch_expand_hw((const bf16*)x, E, rows, d.hin, d.win, d.hout, d.wout, d.k, +1, 0, st) == 0, "expand_hw launch");
  wexp_kernel<<<sgrid((long long)d.k * d.cout * 64), 256, 0, st>>>((const bf16*)w, B, d.k, d.cout, 0);
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(stem_geom(d), 0, plan), "stem plan");
  tc::GatherRun R{E, B, d.k, bias, y, 1, d.act, d.slope, stats};
  return tc::run_gather_tc(plan, R, st);
}

inline int stem_wgrad(const mra_conv_desc& d, const void* x, const void* dy, float* dw, void* wsp, size_t wsb, cudaStream_t st) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.din;
  MRA_WS_TAKE(E, bf16, (size_t)rows * d.hout * d.wout * 64 * 2);
  MRA_WS_TAKE(dWe, float, (size_t)d.k * d.cout * 64 * 4);
  if (!(d.flags & MRA_CONV_WS_REUSE))
    MRA_REQUIRE(launch_expand_hw((const bf16*)x, E, rows, d.hin, d.win, d.hout, d.wout, d.k, +1, 0, st) == 0, "expand_hw launch");
  MRA_CHECK_CUDA(cudaMemsetAsync(dWe, 0, (size_t)d.k * d.cout * 64 * 4, st));
  WgradPlan plan;
  MRA_REQUIRE(build_wgrad_plan(stem_geom(d), plan), "stem wgrad plan");
  if (int rc = tc::run_wgrad_tc(plan, E, dy, dWe, st)) return rc;
  wunexp_kernel<<<sgrid((long long)d.k * d.k * d.k * d.cout), 256, 0, st>>>(dWe, dw, d.k, d.cout, 0);
  MRA_LAUNCH_CHECK();
  return 0;
}

inline int stem_dgrad(const mra_conv_desc& d, const void* dy, const void* wT, void* dx, void* wsp, size_t wsb, cudaStream_t st) {
  MRA_REQUIRE(shift_sum_smem(d.wout) <= max_optin_smem(), "stem dgrad: Z line does not fit shared memory (W = %d)", d.wout);
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.din;
  MRA_WS_TAKE(Z, bf16, (size_t)rows * d.hout * d.wout * 64 * 2);                    // bf16, see head_fprop
  MRA_WS_TAKE(BT, bf16, (size_t)d.k * d.cout * 64 * 2);
  wexp_kernel<<<sgrid((long long)d.k * d.cout * 64), 256, 0, st>>>((const bf16*)wT, BT, d.k, d.cout, 1);   // [kd][c][co]
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(stem_geom(d), 1, plan), "stem dgrad plan");
  tc::GatherRun R{dy, BT, d.k, nullptr, Z, 1, MRA_ACT_NONE, 0.f, nullptr};
  if (int rc = tc::run_gather_tc(plan, R, st)) return rc;
  if (int rc = launch_shift_sum(Z, (bf16*)dx, rows, d.hout, d.wout, d.hin, d.win, d.k, -1, 0, nullptr, MRA_ACT_NONE, 0.f, st)) return rc;
  return 0;
}

inline int head_fprop(const mra_conv_desc& d, const void* x, const void* w, const float* bias, void* y, void* wsp, size_t wsb,
                      cudaStream_t st) {
  MRA_REQUIRE(shift_sum_smem(d.win) <= max_optin_smem(), "head fprop: Z line does not fit shared memory (W = %d)", d.win);
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.dout;
  // Z (the per-(kh,kw) partial sums over kd and ci) is stored in bf16: its 49 terms per output are summed in fp32
  // by shift_sum, so the rounding noise stays at the level of the bf16 output itself while the traffic halves
  MRA_WS_TAKE(Z, bf16, (size_t)rows * d.hin * d.win * 64 * 2);
  MRA_WS_TAKE(B, bf16, (size_t)d.k * d.cin * 64 * 2);
  wexp_kernel<<<sgrid((long long)d.k * d.cin * 64), 256, 0, st>>>((const bf16*)w, B, d.k, d.cin, 1);       // [kd][c][ci]
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(head_geom(d), 0, plan), "head plan");
  tc::GatherRun R{x, B, d.k, nullptr, Z, 1, MRA_ACT_NONE, 0.f, nullptr};
  if (int rc = tc::run_gather_tc(plan, R, st)) return rc;
  if (int rc = launch_shift_sum(Z, (bf16*)y, rows, d.hin, d.win, d.hout, d.wout, d.k, +1, -d.pad, bias, d.act, d.slope, st)) return rc;
  return 0;
}

inline int head_dgrad(const mra_conv_desc& d, const void* dy, const void* wT, void* dx, void* wsp, size_t wsb, cudaStream_t st,
                      double* nstats = nullptr, const void* aux = nullptr, float aux_nslope = 0.f) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.dout;
  MRA_WS_TAKE(E, bf16, (size_t)rows * d.hin * d.win * 64 * 2);
  MRA_WS_TAKE(BT, bf16, (size_t)d.k * d.cin * 64 * 2);
  if (!(d.flags & MRA_CONV_WS_REUSE))
    MRA_REQUIRE(launch_expand_hw((const bf16*)dy, E, rows, d.hout, d.wout, d.hin, d.win, d.k, -1, d.pad, st) == 0, "expand_hw launch");
  wexp_kernel<<<sgrid((long long)d.k * d.cin * 64), 256, 0, st>>>((const bf16*)wT, BT, d.k, d.cin, 0);      // [kd][ci][c]
  MRA_LAUNCH_CHECK();
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(head_geom(d), 1, plan), "head dgrad plan");
  tc::GatherRun R{E, BT, d.k, nullptr, dx, 1, MRA_ACT_NONE, 0.f, nstats};
  R.aux = aux; R.aux_nslope = aux_nslope;
  return tc::run_gather_tc(plan, R, st);
}

inline int head_wgrad(const mra_conv_desc& d, const void* x, const void* dy, float* dw, void* wsp, size_t wsb, cudaStream_t st) {
  Workspace ws{(char*)wsp, wsb, 0};
  const long long rows = (long long)d.n * d.dout;
  MRA_WS_TAKE(E, bf16, (size_t)rows * d.hin * d.win * 64 * 2);
  MRA_WS_TAKE(dWe, float, (size_t)d.k * d.cin * 64 * 4);
  MRA_REQUIRE(launch_expand_hw((const bf16*)dy, E, rows, d.hout, d.wout, d.hin, d.win, d.k, -1, d.pad, st) == 0, "expand_hw launch");
  MRA_CHECK_CUDA(cudaMemsetAsync(dWe, 0, (size_t)d.k * d.cin * 64 * 4, st));
  WgradPlan plan;
  MRA_REQUIRE(build_wgrad_plan(head_geom(d), plan), "head wgrad plan");
  if (int rc = tc::run_wgrad_tc(plan, x, E, dWe, st)) return rc;      // dWe[kd][c][ci]
  wunexp_kernel<<<sgrid((long long)d.k * d.k * d.k * d.cin), 256, 0, st>>>(dWe, dw, d.k, d.cin, 1);
  MRA_LAUNCH_CHECK();
  return 0;
}

}  // namespace special
}  // namespace mra
