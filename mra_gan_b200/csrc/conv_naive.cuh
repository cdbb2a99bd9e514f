// CUDA-core direct convolution kernels (any channel count / kernel size): the fp32 parity path and
// the fall-back for shapes the tcgen05 path does not take.  They index straight from the conv
// descriptor -- deliberately NOT through conv_plan.h -- so the two implementations cross-check.
#pragma once
#include "common.cuh"

namespace mra {

struct NaiveGatherP {
  const void* a; const void* b; const float* bias; void* out;
  int N, Ck, Cn;
  int Ad, Ah, Aw;      // A spatial dims
  int Od, Oh, Ow;      // out spatial dims
  int k, s, p;
  int transposed_mode; // 0: a_pos = o*s - p + t ; 1: a_pos = (o + p - t)/s when divisible
  int act; float slope;
};

// One thread per output element (n, od, oh, ow, cn), cn fastest.  B is [taps][Cn][Ck].
template <typename T, bool VEC>
__global__ void __launch_bounds__(256) naive_gather_kernel(const NaiveGatherP P) {
  const long long total = (long long)P.N * P.Od * P.Oh * P.Ow * P.Cn;
  const T* __restrict__ A = reinterpret_cast<const T*>(P.a);
  const T* __restrict__ B = reinterpret_cast<const T*>(P.b);
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int cn = (int)(idx % P.Cn);
    long long r = idx / P.Cn;
    const int ow = (int)(r % P.Ow); r /= P.Ow;
    const int oh = (int)(r % P.Oh); r /= P.Oh;
    const int od = (int)(r % P.Od);
    const int n = (int)(r / P.Od);
    float acc = 0.f;
    for (int kd = 0; kd < P.k; ++kd) {
      int ad;
      if (!P.transposed_mode) ad = od * P.s - P.p + kd;
      else { int v = od + P.p - kd; if (v % P.s) continue; ad = v / P.s; }
      if (ad < 0 || ad >= P.Ad) continue;
      for (int kh = 0; kh < P.k; ++kh) {
        int ah;
        if (!P.transposed_mode) ah = oh * P.s - P.p + kh;
        else { int v = oh + P.p - kh; if (v % P.s) continue; ah = v / P.s; }
        if (ah < 0 || ah >= P.Ah) continue;
        for (int kw = 0; kw < P.k; ++kw) {
          int aw;
          if (!P.transposed_mode) aw = ow * P.s - P.p + kw;
          else { int v = ow + P.p - kw; if (v % P.s) continue; aw = v / P.s; }
          if (aw < 0 || aw >= P.Aw) continue;
          const T* ap = A + ((((long long)n * P.Ad + ad) * P.Ah + ah) * P.Aw + aw) * P.Ck;
          const T* bp = B + ((long long)((kd * P.k + kh) * P.k + kw) * P.Cn + cn) * P.Ck;
          if (VEC) {
            for (int c = 0; c < P.Ck; c += 8) {
              float av[8], bv[8];
              Vec8<T>::load(ap + c, av);
              Vec8<T>::load(bp + c, bv);
#pragma unroll
              for (int j = 0; j < 8; ++j) acc = fmaf(av[j], bv[j], acc);
            }
          } else {
            for (int c = 0; c < P.Ck; ++c) acc = fmaf(to_f(ap[c]), to_f(bp[c]), acc);
          }
        }
      }
    }
    if (P.bias) acc += P.bias[cn];
    acc = apply_act(acc, P.act, P.slope);
    reinterpret_cast<T*>(P.out)[idx] = from_f<T>(acc);
  }
}

template <typename T>
int launch_naive_gather(const NaiveGatherP& P, cudaStream_t st) {
  const long long total = (long long)P.N * P.Od * P.Oh * P.Ow * P.Cn;
  if (total == 0) return 0;
  const int threads = 256;
  long long blocks = (total + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 64;
  if (blocks > cap) blocks = cap;
  const bool vec = (P.Ck % 8) == 0;
  if (vec) naive_gather_kernel<T, true><<<(unsigned)blocks, threads, 0, st>>>(P);
  else naive_gather_kernel<T, false><<<(unsigned)blocks, threads, 0, st>>>(P);
  MRA_LAUNCH_CHECK();
  return 0;
}

struct NaiveWgradP {
  const void* x; const void* dy; float* dw;
  int N, Cin, Cout;
  int Xd, Xh, Xw;     // x dims
  int Yd, Yh, Yw;     // dy dims
  int k, s, p;
  int transposed;     // 0: x_pos = y_pos*s - p + t ; 1: y_pos = x_pos*s - p + t
  int chunks;         // position chunks per sample (atomic partial sums)
};

// One thread per (tap, co, ci) x (n, position chunk); ci fastest.  dw[tap][co][ci] += partial.
template <typename T>
__global__ void __launch_bounds__(256) naive_wgrad_kernel(const NaiveWgradP P) {
  const int taps = P.k * P.k * P.k;
  const long long per = (long long)taps * P.Cout * P.Cin;
  const long long total = per * P.N * P.chunks;
  const T* __restrict__ X = reinterpret_cast<const T*>(P.x);
  const T* __restrict__ DY = reinterpret_cast<const T*>(P.dy);
  // dense position space: y positions for conv, x positions for convT
  const int Qd = P.transposed ? P.Xd : P.Yd, Qh = P.transposed ? P.Xh : P.Yh, Qw = P.transposed ? P.Xw : P.Yw;
  const int Sd = P.transposed ? P.Yd : P.Xd, Sh = P.transposed ? P.Yh : P.Xh, Sw = P.transposed ? P.Yw : P.Xw;
  const long long Q = (long long)Qd * Qh * Qw;
  const long long qchunk = (Q + P.chunks - 1) / P.chunks;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long e = idx % per;
    long long r = idx / per;
    const int chunk = (int)(r % P.chunks);
    const int n = (int)(r / P.chunks);
    const int ci = (int)(e % P.Cin); e /= P.Cin;
    const int co = (int)(e % P.Cout);
    const int t = (int)(e / P.Cout);
    const int kw = t % P.k, kh = (t / P.k) % P.k, kd = t / (P.k * P.k);
    const long long q0 = chunk * qchunk;
    const long long q1 = (q0 + qchunk < Q) ? q0 + qchunk : Q;
    float acc = 0.f;
    for (long long q = q0; q < q1; ++q) {
      const int qw = (int)(q % Qw);
      const int qh = (int)((q / Qw) % Qh);
      const int qd = (int)(q / ((long long)Qw * Qh));
      const int sd = qd * P.s - P.p + kd, sh = qh * P.s - P.p + kh, sw = qw * P.s - P.p + kw;
      if (sd < 0 || sd >= Sd || sh < 0 || sh >= Sh || sw < 0 || sw >= Sw) continue;
      const long long qoff = ((long long)n * Qd + qd) * Qh * Qw + (long long)qh * Qw + qw;
      const long long soff = (((long long)n * Sd + sd) * Sh + sh) * Sw + sw;
      float xv, gv;
      if (!P.transposed) { gv = to_f(DY[qoff * P.Cout + co]); xv = to_f(X[soff * P.Cin + ci]); }
      else               { xv = to_f(X[qoff * P.Cin + ci]);   gv = to_f(DY[soff * P.Cout + co]); }
      acc = fmaf(xv, gv, acc);
    }
    atomicAdd(P.dw + ((long long)t * P.Cout + co) * P.Cin + ci, acc);
  }
}

template <typename T>
int launch_naive_wgrad(NaiveWgradP P, cudaStream_t st) {
  const long long per = (long long)P.k * P.k * P.k * P.Cout * P.Cin;
  const long long Q = P.transposed ? (long long)P.Xd * P.Xh * P.Xw : (long long)P.Yd * P.Yh * P.Yw;
  if (per == 0 || Q == 0 || P.N == 0) return 0;
  // enough threads to fill the machine a few times over, but keep chunks >= 64 positions
  long long want = (long long)num_sms() * 2048 * 4;
  long long chunks = (want + per * P.N - 1) / (per * P.N);
  if (chunks < 1) chunks = 1;
  long long maxchunks = (Q + 63) / 64;
  if (chunks > maxchunks) chunks = maxchunks;
  P.chunks = (int)chunks;
  const long long total = per * P.N * chunks;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 64;
  if (blocks > cap) blocks = cap;
  naive_wgrad_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(P);
  MRA_LAUNCH_CHECK();
  return 0;
}

// dbias[c] += sum over rows of dy[row][c]   (rows = N*D*H*W)
// Each block stores its partial sums in part[blockIdx.y][blockIdx.x][32]; colsum_finish_kernel adds them in block order,
// so dbias is the same in every run (one fp32 atomicAdd per block summed them in timing order).
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ dy, long long rows, int C,
                                                      float* __restrict__ part) {
  const int c = blockIdx.y * 32 + (threadIdx.x & 31);
  const int lane_row = threadIdx.x >> 5;           // 8 row lanes
  float acc = 0.f;
  if (c < C)
    for (long long r = blockIdx.x * 8LL + lane_row; r < rows; r += (long long)gridDim.x * 8)
      acc += to_f(dy[r * C + c]);
  __shared__ float sm[8][33];
  sm[lane_row][threadIdx.x & 31] = acc;
  __syncthreads();
  if (lane_row == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += sm[i][threadIdx.x & 31];
    part[((long long)blockIdx.y * gridDim.x + blockIdx.x) * 32 + threadIdx.x] = s;
  }
}
__global__ void __launch_bounds__(256) colsum_finish_kernel(const float* __restrict__ part, int blocks, int C,
                                                            float* __restrict__ out) {
  // one warp per channel; lane l adds blocks l, l + 32, ... in order, then the 32 lane sums are added in lane order
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  __shared__ float sm[8][32];
  float s = 0.f;
  if (c < C)
    for (int b = lane; b < blocks; b += 32) s += part[((long long)(c >> 5) * blocks + b) * 32 + (c & 31)];
  sm[threadIdx.x >> 5][lane] = s;
  __syncwarp();
  if (c < C && lane == 0) {
    float t = 0.f;
    for (int i = 0; i < 32; ++i) t += sm[threadIdx.x >> 5][i];
    out[c] += t;
  }
}

template <typename T>
int launch_colsum(const void* dy, long long rows, int C, float* out, cudaStream_t st) {
  if (rows == 0 || C == 0) return 0;
  long long bx = (rows + 8 * 64 - 1) / (8 * 64);
  if (bx > 1024) bx = 1024;
  if (bx < 1) bx = 1;
  const unsigned groups = (unsigned)((C + 31) / 32);
  float* part = nullptr;                             // stream-ordered: capture-safe, freed after the finishing pass
  MRA_CHECK_CUDA(cudaMallocAsync((void**)&part, (size_t)groups * bx * 32 * sizeof(float), st));
  colsum_kernel<T><<<dim3((unsigned)bx, groups), 256, 0, st>>>(reinterpret_cast<const T*>(dy), rows, C, part);
  MRA_LAUNCH_CHECK();
  colsum_finish_kernel<<<(unsigned)((C + 7) / 8), 256, 0, st>>>(part, (int)bx, C, out);
  MRA_LAUNCH_CHECK();
  MRA_CHECK_CUDA(cudaFreeAsync(part, st));
  return 0;
}

}  // namespace mra
