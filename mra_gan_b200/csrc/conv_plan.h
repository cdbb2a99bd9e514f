// Host-side planning of the implicit-GEMM convolution launches (pure C++, no CUDA calls).
//
// Every conv-family op (Conv3d / ConvTranspose3d, fprop / dgrad / wgrad) is lowered to one of two
// generic device computations:
//
//   GATHER   out[n, l*ostep + o0, cn] = sum_{tap, ck} A[n, l*astep + tap.d, ck] * B[tap.widx][cn][ck]
//            (l ranges over a "launch space" of positions; out-of-range A reads are zero)
//              conv  fprop : one launch, astep = stride, tap.d = t - pad,        B = w
//              convT dgrad : same with A = dy,                                   B = wT
//              conv  dgrad : A = dy, B = wT; stride 1: tap.d = pad - t; stride 2: one launch per
//              convT fprop : A = x,  B = w;  output parity phase r (o = 2l + r) holding the taps with
//                                            (r + pad - t) even, tap.d = (r + pad - t)/2, astep = 1
//
//   WGRAD    dW[tap][cm][cn] = sum_{n, q} Mop[n, pos_m, cm] * Nop[n, pos_n, cn]
//            where one operand is read at the dense position q and the other at q*sstep + tap.d:
//              conv  : M = dy (dense, q over y), N = x  (shifted, tap.d = t - pad)
//              convT : M = dy (shifted),          N = x  (dense, q over x)
//
// mra_conv_plan_describe() serialises a plan as int32 words (see describe()) so the CPU tests can
// emulate it against torch's conv3d / conv_transpose3d without a GPU.
#pragma once
#include <stdint.h>
#include <stdlib.h>
#include <vector>

#include "../../include/mra_gan_b200.h"

namespace mra {

struct Tap {
  int dd, dh, dw;  // coordinate offset added to (l * astep)
  int widx;        // weight slab index (kd*k + kh)*k + kw
};

struct GatherLaunch {
  int o0[3];    // output coordinate offset (d, h, w)
  int ostep;    // output coordinate step
  int dims[3];  // launch-space extent (d, h, w)
  int astep;    // A coordinate step
  std::vector<Tap> taps;
  int box[3];   // tile box (d, h, w), product 128
};

struct GatherPlan {
  int n, ck, cn;      // batch, reduction channels, output channels
  int adims[3];       // A spatial dims
  int odims[3];       // output spatial dims
  std::vector<GatherLaunch> launches;
};

// One wgrad launch: a list of filter taps processed `gpi` at a time by one CTA (the accumulators of
// all taps of an item live side by side in TMEM, so the dense operand is loaded once per item).
// With share == K (K taps of a (K,1,1) filter, the stem / head lowerings) all taps read ONE box extended by K - 1
// planes along d -- tap kd starts kd planes into it -- instead of K separate boxes (a third of the bytes at K = 7).
// With share == 2 consecutive taps form pairs that read the SAME shared-memory box of the shifted
// operand (box extended by `ext`), each through its own row shift -- the halo is loaded once.
struct WgradLaunch {
  int share;                 // taps per shared box: 1, 2 or the whole (K,1,1) chain
  int gpi;                   // taps per item (multiple of share)
  int ext[3];                // box extension (d, h, w) of the shifted operand's box (zeros when share == 1)
  std::vector<int> taps;     // indices into WgradPlan::taps, item by item
  std::vector<Tap> origin;   // per entry: offset of its box origin (shared by both taps of a pair); widx unused
};

struct WgradPlan {
  int n, cm, cn;      // dW is [taps][cm][cn] with cm = cout, cn = cin
  int qdims[3];       // dense position space
  int mdims[3], ndims[3];
  int sstep;          // stride applied to q for the shifted operand
  int m_is_shifted;   // 1: dy (M side) is the shifted operand (ConvTranspose3d)
  std::vector<Tap> taps;
  int box[3];         // K-block box (d, h, w), product 64
  int ncc;            // 64-channel chunks of the shifted operand per tap (accumulator width = 64 * ncc)
  std::vector<WgradLaunch> launches;
};

// Pick power-of-two box extents (d,h,w) with product `total` minimising the padded volume of the
// launch space; ties prefer a longer w (contiguous) run.  `maxw` bounds the w extent (TMA boxDim<=256
// after multiplying by the element stride).
inline void choose_box(const int dims[3], int total, int maxw, int box[3]) {
  long long best = -1;
  int bb[3] = {1, 1, total};
  for (int bd = 1; bd <= total; bd <<= 1)
    for (int bh = 1; bd * bh <= total; bh <<= 1) {
      int bw = total / (bd * bh);
      if (bw > maxw) continue;
      long long pd = (long long)((dims[0] + bd - 1) / bd) * bd;
      long long ph = (long long)((dims[1] + bh - 1) / bh) * bh;
      long long pw = (long long)((dims[2] + bw - 1) / bw) * bw;
      long long vol = pd * ph * pw;
      bool better = best < 0 || vol < best ||
                    (vol == best && (bw > bb[2] || (bw == bb[2] && bh > bb[1])));
      if (better) { best = vol; bb[0] = bd; bb[1] = bh; bb[2] = bw; }
    }
  box[0] = bb[0]; box[1] = bb[1]; box[2] = bb[2];
}

// Extended geometry: per-axis kernel extent and zero padding (the public descriptor is cubic; the
// stem / head lowerings in conv_special.cuh use (7,1,1) kernels on channel-expanded tensors).
struct GeomEx {
  int n, cin, cout;
  int in[3], out[3];   // x / y spatial dims (d, h, w)
  int k[3], pad[3];
  int stride;
  int transposed;
};

inline GeomEx geom_from_desc(const mra_conv_desc& d) {
  GeomEx g;
  g.n = d.n; g.cin = d.cin; g.cout = d.cout;
  g.in[0] = d.din; g.in[1] = d.hin; g.in[2] = d.win;
  g.out[0] = d.dout; g.out[1] = d.hout; g.out[2] = d.wout;
  for (int i = 0; i < 3; ++i) { g.k[i] = d.k; g.pad[i] = d.pad; }
  g.stride = d.stride; g.transposed = d.transposed;
  return g;
}

inline bool build_gather_plan(const GeomEx& d, int which, GatherPlan& P) {
  // which: 0 = fprop (A = x, out = y), 1 = dgrad (A = dy, out = dx)
  const int s = d.stride;
  if (s != 1 && s != 2) return false;
  const bool fprop = which == 0;
  P.n = d.n;
  P.ck = fprop ? d.cin : d.cout;
  P.cn = fprop ? d.cout : d.cin;
  for (int i = 0; i < 3; ++i) {
    P.adims[i] = fprop ? d.in[i] : d.out[i];
    P.odims[i] = fprop ? d.out[i] : d.in[i];
  }
  // direct addressing: A coord = o*s - p + t.  Used by conv fprop and convT dgrad.
  const bool direct = (fprop && !d.transposed) || (!fprop && d.transposed);
  const int K0 = d.k[0], K1 = d.k[1], K2 = d.k[2];
  auto widx = [&](int a, int b, int c) { return (a * K1 + b) * K2 + c; };
  P.launches.clear();
  if (direct || s == 1) {
    GatherLaunch L;
    for (int i = 0; i < 3; ++i) { L.o0[i] = 0; L.dims[i] = P.odims[i]; }
    L.ostep = 1; L.astep = direct ? s : 1;
    for (int kd = 0; kd < K0; ++kd) for (int kh = 0; kh < K1; ++kh) for (int kw = 0; kw < K2; ++kw) {
      if (direct) L.taps.push_back(Tap{kd - d.pad[0], kh - d.pad[1], kw - d.pad[2], widx(kd, kh, kw)});
      else        L.taps.push_back(Tap{d.pad[0] - kd, d.pad[1] - kh, d.pad[2] - kw, widx(kd, kh, kw)});
    }
    choose_box(L.dims, 128, 256 / L.astep, L.box);
    P.launches.push_back(L);
  } else {
    for (int rd = 0; rd < 2; ++rd) for (int rh = 0; rh < 2; ++rh) for (int rw = 0; rw < 2; ++rw) {
      const int r[3] = {rd, rh, rw};
      GatherLaunch L;
      bool empty = false;
      for (int i = 0; i < 3; ++i) {
        L.o0[i] = r[i];
        L.dims[i] = (P.odims[i] - r[i] + 1) / 2;
        if (L.dims[i] <= 0) empty = true;
      }
      if (empty) continue;
      L.ostep = 2; L.astep = 1;
      for (int kd = 0; kd < K0; ++kd) {
        if ((rd + d.pad[0] - kd) & 1) continue;
        for (int kh = 0; kh < K1; ++kh) {
          if ((rh + d.pad[1] - kh) & 1) continue;
          for (int kw = 0; kw < K2; ++kw) {
            if ((rw + d.pad[2] - kw) & 1) continue;
            L.taps.push_back(Tap{(rd + d.pad[0] - kd) / 2, (rh + d.pad[1] - kh) / 2, (rw + d.pad[2] - kw) / 2,
                                 widx(kd, kh, kw)});
          }
        }
      }
      if (L.taps.empty()) continue;
      choose_box(L.dims, 128, 256, L.box);
      P.launches.push_back(L);
    }
  }
  return true;
}
inline bool build_gather_plan(const mra_conv_desc& d, int which, GatherPlan& P) {
  return build_gather_plan(geom_from_desc(d), which, P);
}

inline void wgrad_add_launch(WgradPlan& P, const std::vector<int>& idx, int share, int gpi, int ed, int eh, int ew) {
  if (idx.empty()) return;
  WgradLaunch L;
  L.share = share; L.gpi = gpi; L.ext[0] = ed; L.ext[1] = eh; L.ext[2] = ew;
  L.taps = idx;
  for (size_t i = 0; i < idx.size(); ++i) {
    const Tap& a = P.taps[idx[i - i % share]];                     // first tap of a box set holds the minimum offsets
    L.origin.push_back(Tap{a.dd, a.dh, a.dw, 0});
  }
  P.launches.push_back(L);
}

inline bool build_wgrad_plan(const GeomEx& d, WgradPlan& P) {
  const int s = d.stride;
  if (s != 1 && s != 2) return false;
  P.n = d.n; P.cm = d.cout; P.cn = d.cin;
  for (int i = 0; i < 3; ++i) {
    P.mdims[i] = d.out[i];         // M operand = dy
    P.ndims[i] = d.in[i];          // N operand = x
    P.qdims[i] = d.transposed ? d.in[i] : d.out[i];
  }
  P.sstep = s;
  P.m_is_shifted = d.transposed ? 1 : 0;
  P.taps.clear();
  for (int kd = 0; kd < d.k[0]; ++kd) for (int kh = 0; kh < d.k[1]; ++kh) for (int kw = 0; kw < d.k[2]; ++kw)
    P.taps.push_back(Tap{kd - d.pad[0], kh - d.pad[1], kw - d.pad[2], (kd * d.k[1] + kh) * d.k[2] + kw});
  choose_box(P.qdims, 64, 256 / s, P.box);
  // ---- launch structure (tensor-core kernel only; channel counts in 64-channel chunks) ----
  P.launches.clear();
  const int cs = d.transposed ? d.cout : d.cin;          // channels of the shifted operand
  P.ncc = cs % 256 == 0 ? 4 : (cs % 128 == 0 ? 2 : 1);
  const int cap = 8 / P.ncc;                             // taps whose accumulators fit TMEM (512 columns)
  const int K0 = d.k[0], K1 = d.k[1], K2 = d.k[2];
  auto ti = [&](int a, int b, int c) { return (a * K1 + b) * K2 + c; };
  std::vector<int> wpairs, hpairs, rest;
  // (K,1,1) filters (channel-expanded stem / head): one d-extended box for all K taps, 4x4x4 K-blocks so that the
  // extension (K - 1 planes of 16 positions) stays small next to the 64 positions of the block itself
  if (s == 1 && K1 == 1 && K2 == 1 && K0 >= 3 && K0 <= cap && getenv("MRA_WGRAD_NO_DCHAIN") == nullptr) {
    P.box[0] = 4; P.box[1] = 4; P.box[2] = 4;
    std::vector<int> all;
    for (int kd = 0; kd < K0; ++kd) all.push_back(ti(kd, 0, 0));
    wgrad_add_launch(P, all, K0, K0, K0 - 1, 0, 0);
    return true;
  }
  const bool can_share = s == 1 && P.box[2] % 16 == 0 && cap >= 2;
  if (can_share) {
    std::vector<int> left;                               // taps left over after pairing along w
    for (int kd = 0; kd < K0; ++kd) for (int kh = 0; kh < K1; ++kh) {
      int kw = 0;
      for (; kw + 1 < K2; kw += 2) { wpairs.push_back(ti(kd, kh, kw)); wpairs.push_back(ti(kd, kh, kw + 1)); }
      if (kw < K2) left.push_back(ti(kd, kh, kw));
    }
    // the leftovers all have kw = K2-1: pair them along h
    const bool no_hpairs = getenv("MRA_WGRAD_NO_HPAIRS") != nullptr;
    if (no_hpairs) rest = left;
    for (int kd = 0; kd < K0 && (K2 & 1) && !no_hpairs; ++kd) {
      int kh = 0;
      for (; kh + 1 < K1; kh += 2) { hpairs.push_back(ti(kd, kh, K2 - 1)); hpairs.push_back(ti(kd, kh + 1, K2 - 1)); }
      if (kh < K1) rest.push_back(ti(kd, kh, K2 - 1));
    }
  } else {
    for (int i = 0; i < (int)P.taps.size(); ++i) rest.push_back(i);
  }
  const int gshare = cap - (cap & 1);
  wgrad_add_launch(P, wpairs, 2, gshare, 0, 0, 1);
  wgrad_add_launch(P, hpairs, 2, gshare, 0, 1, 0);
  // unshared taps: each tap needs its own ncc boxes per stage; 4 / ncc taps = 256 accumulator columns = one MMA
  const int gsolo = P.ncc >= 4 ? 1 : 4 / P.ncc;
  wgrad_add_launch(P, rest, 1, gsolo, 0, 0, 0);
  return true;
}
inline bool build_wgrad_plan(const mra_conv_desc& d, WgradPlan& P) { return build_wgrad_plan(geom_from_desc(d), P); }

// Serialisation for mra_conv_plan_describe():
//  gather: [0, n, ck, cn, adims[3], odims[3], nlaunch, then per launch:
//           o0[3], ostep, dims[3], astep, box[3], ntaps, ntaps x (dd, dh, dw, widx)]
//  wgrad : [1, n, cm, cn, qdims[3], mdims[3], ndims[3], sstep, m_is_shifted, box[3], ntaps,
//           ntaps x (dd, dh, dw, widx), ncc, nlaunch, per launch: share, gpi, ext[3], n, n x (tap, odd, odh, odw)]
inline int describe(const GatherPlan& P, int32_t* out, int cap) {
  std::vector<int32_t> v = {0, P.n, P.ck, P.cn};
  for (int i = 0; i < 3; ++i) v.push_back(P.adims[i]);
  for (int i = 0; i < 3; ++i) v.push_back(P.odims[i]);
  v.push_back((int)P.launches.size());
  for (const auto& L : P.launches) {
    for (int i = 0; i < 3; ++i) v.push_back(L.o0[i]);
    v.push_back(L.ostep);
    for (int i = 0; i < 3; ++i) v.push_back(L.dims[i]);
    v.push_back(L.astep);
    for (int i = 0; i < 3; ++i) v.push_back(L.box[i]);
    v.push_back((int)L.taps.size());
    for (const auto& t : L.taps) { v.push_back(t.dd); v.push_back(t.dh); v.push_back(t.dw); v.push_back(t.widx); }
  }
  if ((int)v.size() > cap) return -2;
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  return (int)v.size();
}
inline int describe(const WgradPlan& P, int32_t* out, int cap) {
  std::vector<int32_t> v = {1, P.n, P.cm, P.cn};
  for (int i = 0; i < 3; ++i) v.push_back(P.qdims[i]);
  for (int i = 0; i < 3; ++i) v.push_back(P.mdims[i]);
  for (int i = 0; i < 3; ++i) v.push_back(P.ndims[i]);
  v.push_back(P.sstep); v.push_back(P.m_is_shifted);
  for (int i = 0; i < 3; ++i) v.push_back(P.box[i]);
  v.push_back((int)P.taps.size());
  for (const auto& t : P.taps) { v.push_back(t.dd); v.push_back(t.dh); v.push_back(t.dw); v.push_back(t.widx); }
  // launch structure: ncc, nlaunch, then per launch: share, gpi, ext[3], n, n x (tap index, origin dd, dh, dw)
  v.push_back(P.ncc); v.push_back((int)P.launches.size());
  for (const auto& L : P.launches) {
    v.push_back(L.share); v.push_back(L.gpi);
    for (int i = 0; i < 3; ++i) v.push_back(L.ext[i]);
    v.push_back((int)L.taps.size());
    for (size_t i = 0; i < L.taps.size(); ++i) {
      v.push_back(L.taps[i]); v.push_back(L.origin[i].dd); v.push_back(L.origin[i].dh); v.push_back(L.origin[i].dw);
    }
  }
  if ((int)v.size() > cap) return -2;
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  return (int)v.size();
}

}  // namespace mra
