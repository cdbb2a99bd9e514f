// extern "C" entry points of libmra_b200.so (see include/mra_gan_b200.h for the contract).
#include <stdarg.h>

#include "common.cuh"
#include "conv_naive.cuh"
#include "conv_plan.h"
#include "conv_tc_halo.cuh"
#include "conv_tc_phase.cuh"
#include "conv_special.cuh"
#include "misc.cuh"
#include "norm.cuh"
#include "norm_stream.cuh"

namespace mra {
thread_local std::string g_last_error;
std::atomic<long long> g_launch_count{0};
}
using namespace mra;

#define DISPATCH_DTYPE(dt, ...)                                  \
  do {                                                           \
    if ((dt) == MRA_F32) { typedef float T; __VA_ARGS__; }       \
    else if ((dt) == MRA_BF16) { typedef bf16 T; __VA_ARGS__; }  \
    else return fail(-1, "unknown dtype %d", (int)(dt));         \
  } while (0)

static int check_conv(const mra_conv_desc* d) {
  MRA_REQUIRE(d != nullptr, "null conv descriptor");
  MRA_REQUIRE(d->n > 0 && d->cin > 0 && d->cout > 0 && d->k > 0, "bad conv sizes");
  MRA_REQUIRE(d->stride == 1 || d->stride == 2, "stride must be 1 or 2 (got %d)", d->stride);
  MRA_REQUIRE(d->dtype == MRA_F32 || d->dtype == MRA_BF16, "unknown dtype %d", (int)d->dtype);
  const int in[3] = {d->din, d->hin, d->win}, out[3] = {d->dout, d->hout, d->wout};
  for (int i = 0; i < 3; ++i) {
    MRA_REQUIRE(in[i] > 0 && out[i] > 0, "bad conv spatial dims");
    if (!d->transposed) {
      const int e = (in[i] + 2 * d->pad - d->k) / d->stride + 1;
      MRA_REQUIRE(e == out[i], "conv output dim %d: expected %d got %d", i, e, out[i]);
    } else {
      const int lo = (in[i] - 1) * d->stride - 2 * d->pad + d->k;   // output_padding in [0, stride)
      MRA_REQUIRE(out[i] >= lo && out[i] < lo + d->stride, "convT output dim %d: %d not in [%d,%d)", i, out[i], lo,
                  lo + d->stride);
    }
  }
  return 0;
}

static NaiveGatherP naive_params(const mra_conv_desc& d, int which, const void* a, const void* b, const float* bias,
                                 void* out) {
  NaiveGatherP P;
  const bool fprop = which == 0;
  P.a = a; P.b = b; P.bias = bias; P.out = out;
  P.N = d.n; P.Ck = fprop ? d.cin : d.cout; P.Cn = fprop ? d.cout : d.cin;
  if (fprop) { P.Ad = d.din; P.Ah = d.hin; P.Aw = d.win; P.Od = d.dout; P.Oh = d.hout; P.Ow = d.wout; }
  else       { P.Ad = d.dout; P.Ah = d.hout; P.Aw = d.wout; P.Od = d.din; P.Oh = d.hin; P.Ow = d.win; }
  P.k = d.k; P.s = d.stride; P.p = d.pad;
  const bool direct = (fprop && !d.transposed) || (!fprop && d.transposed);
  P.transposed_mode = direct ? 0 : 1;
  P.act = fprop ? d.act : MRA_ACT_NONE; P.slope = d.slope;
  return P;
}

extern "C" {

int mra_version(void) { return 100; }
long long mra_debug_launch_count(void) { return g_launch_count.load(); }
const char* mra_last_error(void) { return g_last_error.c_str(); }

size_t mra_conv3d_workspace_size(const mra_conv_desc* d, int which) {
  if (!d) return 0;
  if (special::stem_eligible(*d) || special::head_eligible(*d) || special::im2col_eligible(*d) || special::convT1_eligible(*d))
    return special::workspace_bytes(*d, which);
  if (which == 0 || which == 1) return tc::ksplit_workspace_bytes(*d, which);     // fp32 partial sums of the split-K gather
  return 0;
}

int mra_conv3d_lowering(const mra_conv_desc* d) {
  if (!d) return 0;
  if (special::im2col_eligible(*d)) return 3;
  if (special::convT1_eligible(*d)) return 2;      // wgrad builds im2col(dy), dgrad reuses it
  if (special::stem_eligible(*d)) return 1;
  if (special::head_eligible(*d)) return 2;
  return 0;
}

int mra_conv3d_uses_tensor_cores(const mra_conv_desc* d, int which) {
  if (!d) return 0;
  if (special::stem_eligible(*d) || special::head_eligible(*d) || special::im2col_eligible(*d) || special::convT1_eligible(*d))
    return 1;
  if (which == 2) return tc::wgrad_eligible(*d) ? 1 : 0;
  return tc::gather_eligible(*d, which) ? 1 : 0;
}

int mra_conv3d_fprop(const mra_conv_desc* d, const void* x, const void* w, const float* bias, void* y, double* stats,
                     void* workspace, size_t workspace_bytes, mra_stream_t stream) {
  if (int rc = check_conv(d)) return rc;
  MRA_REQUIRE(x != nullptr && w != nullptr && y != nullptr, "mra_conv3d_fprop: null operand (x, w and y are mandatory)");
  cudaStream_t st = (cudaStream_t)stream;
  if (stats) MRA_CHECK_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * d->n * d->cout, st));
  if (special::im2col_eligible(*d)) return special::im2col_fprop(*d, x, w, bias, y, stats, workspace, workspace_bytes, st);
  if (special::stem_eligible(*d)) return special::stem_fprop(*d, x, w, bias, y, stats, workspace, workspace_bytes, st);
  if (special::convT1_eligible(*d) || special::head_eligible(*d)) {
    // single-channel outputs: no epilogue statistics in these lowerings, so they come from a pass over the stored y
    MRA_REQUIRE(!stats || d->act == MRA_ACT_NONE, "stats are defined on the pre-activation output only");
    if (special::convT1_eligible(*d)) {
      if (int rc = special::im2col_dgrad(special::convT1_mirror(*d), x, w, y, workspace, workspace_bytes, st, bias, d->act, d->slope))
        return rc;
    } else if (int rc = special::head_fprop(*d, x, w, bias, y, workspace, workspace_bytes, st)) {
      return rc;
    }
    if (!stats) return 0;
    mra_norm_desc nd;
    memset(&nd, 0, sizeof(nd));
    nd.n = d->n; nd.c = d->cout; nd.d = d->dout; nd.h = d->hout; nd.w = d->wout; nd.res_pad = -1; nd.dtype = d->dtype;
    return mra_inorm_stats(&nd, y, stats, stream);
  }
  if (tc::gather_eligible(*d, 0)) {
    bool split = false;
    if (int rc = tc::run_gather_tc(*d, 0, x, w, bias, y, stats, st, nullptr, 0.f, workspace, workspace_bytes, &split)) return rc;
    if (split && stats) {                          // the split-K path leaves the statistics to the exact pass over y
      MRA_REQUIRE(d->act == MRA_ACT_NONE, "stats are defined on the pre-activation output only");
      mra_norm_desc nd;
      memset(&nd, 0, sizeof(nd));
      nd.n = d->n; nd.c = d->cout; nd.d = d->dout; nd.h = d->hout; nd.w = d->wout; nd.res_pad = -1; nd.dtype = d->dtype;
      return mra_inorm_stats(&nd, y, stats, stream);
    }
    return 0;
  }
  NaiveGatherP P = naive_params(*d, 0, x, w, bias, y);
  DISPATCH_DTYPE(d->dtype, { if (int rc = launch_naive_gather<T>(P, st)) return rc; });
  if (stats) {
    MRA_REQUIRE(d->act == MRA_ACT_NONE, "stats are defined on the pre-activation output only");
    mra_norm_desc nd;
    memset(&nd, 0, sizeof(nd));
    nd.n = d->n; nd.c = d->cout; nd.d = d->dout; nd.h = d->hout; nd.w = d->wout; nd.res_pad = -1; nd.dtype = d->dtype;
    return mra_inorm_stats(&nd, y, stats, stream);
  }
  return 0;
}

int mra_conv3d_dgrad(const mra_conv_desc* d, const void* dy, const void* wT, void* dx, void* workspace,
                     size_t workspace_bytes, mra_stream_t stream) {
  if (int rc = check_conv(d)) return rc;
  MRA_REQUIRE(dy != nullptr && wT != nullptr && dx != nullptr, "mra_conv3d_dgrad: null operand (dy, wT and dx are mandatory)");
  cudaStream_t st = (cudaStream_t)stream;
  if (special::im2col_eligible(*d)) return special::im2col_dgrad(*d, dy, wT, dx, workspace, workspace_bytes, st);
  if (special::convT1_eligible(*d))
    return special::im2col_fprop(special::convT1_mirror(*d), dy, wT, nullptr, dx, nullptr, workspace, workspace_bytes, st);
  if (special::stem_eligible(*d)) return special::stem_dgrad(*d, dy, wT, dx, workspace, workspace_bytes, st);
  if (special::head_eligible(*d)) return special::head_dgrad(*d, dy, wT, dx, workspace, workspace_bytes, st);
  if (tc::gather_eligible(*d, 1)) {
    bool split = false;
    return tc::run_gather_tc(*d, 1, dy, wT, nullptr, dx, nullptr, st, nullptr, 0.f, workspace, workspace_bytes, &split);
  }
  NaiveGatherP P = naive_params(*d, 1, dy, wT, nullptr, dx);
  DISPATCH_DTYPE(d->dtype, { if (int rc = launch_naive_gather<T>(P, st)) return rc; });
  return 0;
}

// dgrad + the statistics pass of the InstanceNorm backward in front of this conv (see EpiArgs::aux)
static bool dgrad_nstats_ok(const mra_conv_desc& d) {
  if (d.dtype != MRA_BF16 || (d.flags & MRA_CONV_FORCE_NAIVE)) return false;
  if (special::im2col_eligible(d) || special::convT1_eligible(d) || special::stem_eligible(d)) return false;
  if (special::head_eligible(d)) return true;
  return tc::gather_eligible(d, 1);
}
int mra_conv3d_dgrad_nstats_supported(const mra_conv_desc* d) { return d && dgrad_nstats_ok(*d) ? 1 : 0; }

int mra_conv3d_dgrad_nstats(const mra_conv_desc* d, const void* dy, const void* wT, void* dx, const void* y_act, int norm_act,
                            float norm_slope, double* sums, void* workspace, size_t workspace_bytes, mra_stream_t stream) {
  if (int rc = check_conv(d)) return rc;
  MRA_REQUIRE(dy != nullptr && wT != nullptr && dx != nullptr, "mra_conv3d_dgrad_nstats: null operand (dy, wT and dx are mandatory)");
  MRA_REQUIRE(y_act != nullptr && sums != nullptr, "dgrad_nstats needs the norm output and a sums buffer");
  MRA_REQUIRE(dgrad_nstats_ok(*d), "this layer's dgrad does not run on the tensor-core gather kernels");
  float nslope;
  if (norm_act == MRA_ACT_NONE) nslope = 1.f;
  else if (norm_act == MRA_ACT_RELU) nslope = 0.f;
  else if (norm_act == MRA_ACT_LRELU && norm_slope >= 0.f && norm_slope <= 1.f) nslope = norm_slope;
  else return fail(-1, "dgrad_nstats: activation %d (slope %g) is not piecewise linear", norm_act, (double)norm_slope);
  cudaStream_t st = (cudaStream_t)stream;
  const int cn = d->cin;                                    // channels of dx = channels of the norm
  MRA_CHECK_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * d->n * cn, st));
  if (special::head_eligible(*d)) return special::head_dgrad(*d, dy, wT, dx, workspace, workspace_bytes, st, sums, y_act, nslope);
  return tc::run_gather_tc(*d, 1, dy, wT, nullptr, dx, sums, st, y_act, nslope);
}

int mra_conv3d_wgrad(const mra_conv_desc* d, const void* x, const void* dy, float* dw, float* dbias,
                     void* workspace, size_t workspace_bytes, mra_stream_t stream) {
  if (int rc = check_conv(d)) return rc;
  MRA_REQUIRE(dy != nullptr && (x != nullptr || dw == nullptr), "mra_conv3d_wgrad: null operand (dy always, x when dw is asked for)");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t wn = (size_t)d->k * d->k * d->k * d->cout * d->cin;
  if (!(d->flags & MRA_CONV_ACCUMULATE)) {
    if (dw) MRA_CHECK_CUDA(cudaMemsetAsync(dw, 0, wn * sizeof(float), st));
    if (dbias) MRA_CHECK_CUDA(cudaMemsetAsync(dbias, 0, (size_t)d->cout * sizeof(float), st));
  }
  if (dw) {
    if (special::im2col_eligible(*d)) {
      if (int rc = special::im2col_wgrad(*d, x, dy, dw, workspace, workspace_bytes, st)) return rc;
    } else if (special::convT1_eligible(*d)) {
      if (int rc = special::im2col_wgrad(special::convT1_mirror(*d), dy, x, dw, workspace, workspace_bytes, st)) return rc;
    } else if (special::stem_eligible(*d)) {
      if (int rc = special::stem_wgrad(*d, x, dy, dw, workspace, workspace_bytes, st)) return rc;
    } else if (special::head_eligible(*d)) {
      if (int rc = special::head_wgrad(*d, x, dy, dw, workspace, workspace_bytes, st)) return rc;
    } else if (tc::wgrad_eligible(*d)) {
      if (int rc = tc::run_wgrad_tc(*d, x, dy, dw, st)) return rc;
    } else {
      NaiveWgradP P;
      P.x = x; P.dy = dy; P.dw = dw; P.N = d->n; P.Cin = d->cin; P.Cout = d->cout;
      P.Xd = d->din; P.Xh = d->hin; P.Xw = d->win; P.Yd = d->dout; P.Yh = d->hout; P.Yw = d->wout;
      P.k = d->k; P.s = d->stride; P.p = d->pad; P.transposed = d->transposed; P.chunks = 1;
      DISPATCH_DTYPE(d->dtype, { if (int rc = launch_naive_wgrad<T>(P, st)) return rc; });
    }
  }
  if (dbias) {
    const long long rows = (long long)d->n * d->dout * d->hout * d->wout;
    DISPATCH_DTYPE(d->dtype, { if (int rc = launch_colsum<T>(dy, rows, d->cout, dbias, st)) return rc; });
  }
  return 0;
}

int mra_pack_weight_t(const void* w, int src_dtype, void* wT, int dst_dtype, int taps, int cout, int cin,
                      mra_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MRA_REQUIRE(taps > 0 && cout > 0 && cin > 0 && taps <= 65535, "bad pack sizes");
  dim3 grid((cin + 31) / 32, (cout + 31) / 32, taps), block(32, 8);
  if (src_dtype == MRA_F32 && dst_dtype == MRA_F32)
    pack_weight_t_kernel<float, float><<<grid, block, 0, st>>>((const float*)w, (float*)wT, cout, cin);
  else if (src_dtype == MRA_F32 && dst_dtype == MRA_BF16)
    pack_weight_t_kernel<float, bf16><<<grid, block, 0, st>>>((const float*)w, (bf16*)wT, cout, cin);
  else if (src_dtype == MRA_BF16 && dst_dtype == MRA_BF16)
    pack_weight_t_kernel<bf16, bf16><<<grid, block, 0, st>>>((const bf16*)w, (bf16*)wT, cout, cin);
  else return fail(-1, "unsupported pack dtype combination %d -> %d", src_dtype, dst_dtype);
  MRA_LAUNCH_CHECK();
  return 0;
}

int mra_convert(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t numel, mra_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (numel <= 0) return 0;
  const unsigned g = ew_grid(numel);
  if (src_dtype == MRA_F32 && dst_dtype == MRA_BF16)
    convert_kernel<float, bf16><<<g, 256, 0, st>>>((const float*)src, (bf16*)dst, numel);
  else if (src_dtype == MRA_BF16 && dst_dtype == MRA_F32)
    convert_kernel<bf16, float><<<g, 256, 0, st>>>((const bf16*)src, (float*)dst, numel);
  else if (src_dtype == MRA_F32 && dst_dtype == MRA_F32)
    convert_kernel<float, float><<<g, 256, 0, st>>>((const float*)src, (float*)dst, numel);
  else if (src_dtype == MRA_BF16 && dst_dtype == MRA_BF16)
    convert_kernel<bf16, bf16><<<g, 256, 0, st>>>((const bf16*)src, (bf16*)dst, numel);
  else return fail(-1, "unsupported convert %d -> %d", src_dtype, dst_dtype);
  MRA_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------ norm family
static int check_norm(const mra_norm_desc* d) {
  MRA_REQUIRE(d != nullptr, "null norm descriptor");
  MRA_REQUIRE(d->n > 0 && d->c > 0 && d->d > 0 && d->h > 0 && d->w > 0, "bad norm sizes");
  MRA_REQUIRE(d->c <= 2048, "channel count %d too large", d->c);
  MRA_REQUIRE(d->pad >= 0 && d->res_pad >= -1, "bad pad");
  return 0;
}
#define DISPATCH_NORM(d, ...)                                                       \
  do {                                                                              \
    const bool vec8 = ((d)->c % 8) == 0;                                            \
    if ((d)->dtype == MRA_F32) { typedef float T; if (vec8) { constexpr int VEC = 8; __VA_ARGS__; } else { constexpr int VEC = 1; __VA_ARGS__; } } \
    else if ((d)->dtype == MRA_BF16) { typedef bf16 T; if (vec8) { constexpr int VEC = 8; __VA_ARGS__; } else { constexpr int VEC = 1; __VA_ARGS__; } } \
    else return fail(-1, "unknown dtype %d", (int)(d)->dtype);                      \
  } while (0)

int mra_inorm_stats(const mra_norm_desc* d, const void* x, double* stats, mra_stream_t stream) {
  if (int rc = check_norm(d)) return rc;
  DISPATCH_NORM(d, return (norm_stats_launch<T, VEC>(*d, x, stats, (cudaStream_t)stream)));
  return 0;
}

int mra_inorm_act_pad_fwd(const mra_norm_desc* d, const void* x, const double* stats, const void* residual, void* y,
                          float* mean, float* rstd, float* running_mean, float* running_var, mra_stream_t stream) {
  if (int rc = check_norm(d)) return rc;
  MRA_REQUIRE(d->use_running || (long long)d->d * d->h * d->w > 1,
              "InstanceNorm needs more than 1 spatial element per channel in training mode");
  MRA_REQUIRE((d->res_pad >= 0) == (residual != nullptr), "residual pointer / res_pad mismatch");
  MRA_REQUIRE(d->use_running != 1 || (running_mean && running_var), "eval-mode norm needs running stats");
  MRA_REQUIRE(d->use_running >= 0 && d->use_running <= 2, "bad use_running mode %d", (int)d->use_running);
  DISPATCH_NORM(d, return (ns::norm_fwd_launch_v2<T, VEC>(*d, x, stats, residual, y, mean, rstd, running_mean, running_var,
                                                   (cudaStream_t)stream)));
  return 0;
}

int mra_inorm_act_pad_bwd(const mra_norm_desc* d, const void* gy, const void* x, const float* mean, const float* rstd,
                          void* dx, void* dres, double* sums, mra_stream_t stream) {
  if (int rc = check_norm(d)) return rc;
  MRA_REQUIRE(!dres || d->res_pad >= 0, "dres requested without a residual");
  DISPATCH_NORM(d, return (ns::norm_bwd_launch_v2<T, VEC>(*d, gy, x, mean, rstd, dx, dres, sums, (cudaStream_t)stream)));
  return 0;
}

int mra_inorm_act_pad_bwd_stats(const mra_norm_desc* d, const void* gy, const void* x, const float* mean, const float* rstd,
                                double* sums, mra_stream_t stream) {
  if (int rc = check_norm(d)) return rc;
  DISPATCH_NORM(d, return (ns::norm_bwd_launch_v2<T, VEC>(*d, gy, x, mean, rstd, nullptr, nullptr, sums, (cudaStream_t)stream, 1)));
  return 0;
}

int mra_inorm_act_pad_bwd_apply(const mra_norm_desc* d, const void* gy, const void* x, const float* mean, const float* rstd,
                                const double* sums, void* dx, void* dres, mra_stream_t stream) {
  if (int rc = check_norm(d)) return rc;
  MRA_REQUIRE(!dres || d->res_pad >= 0, "dres requested without a residual");
  DISPATCH_NORM(d, return (ns::norm_bwd_launch_v2<T, VEC>(*d, gy, x, mean, rstd, dx, dres, const_cast<double*>(sums),
                                                         (cudaStream_t)stream, 2)));
  return 0;
}

int mra_act_fwd(const void* x, void* y, int64_t numel, int act, float slope, int dtype, mra_stream_t stream) {
  if (numel <= 0) return 0;
  DISPATCH_DTYPE(dtype, (act_fwd_kernel<T><<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>((const T*)x, (T*)y, numel, act, slope)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_act_bwd(const void* dy, const void* y, void* dx, int64_t numel, int act, float slope, int dtype,
                mra_stream_t stream) {
  if (numel <= 0) return 0;
  DISPATCH_DTYPE(dtype, (act_bwd_kernel<T><<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>((const T*)dy, (const T*)y, (T*)dx, numel, act, slope)));
  MRA_LAUNCH_CHECK();
  return 0;
}

int mra_cat2_act_fwd(const void* a, const void* b, void* out, int64_t positions, int ca, int cb, int act, float slope, int dtype,
                     mra_stream_t stream) {
  MRA_REQUIRE(a && b && out && ca > 0 && cb > 0, "mra_cat2_act_fwd: bad arguments");
  if (positions <= 0) return 0;
  const bool v8 = dtype == MRA_BF16 && ca % 8 == 0 && cb % 8 == 0;
  const int vec = v8 ? 8 : 1;
  const long long items = positions * (long long)((ca + cb) / vec);
  if (v8) cat2_act_fwd_kernel<bf16, 8><<<ew_grid(items, 1), 256, 0, (cudaStream_t)stream>>>((const bf16*)a, (const bf16*)b, (bf16*)out, items, ca / 8, cb / 8, act, slope);
  else DISPATCH_DTYPE(dtype, (cat2_act_fwd_kernel<T, 1><<<ew_grid(items), 256, 0, (cudaStream_t)stream>>>((const T*)a, (const T*)b, (T*)out, items, ca, cb, act, slope)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_cat2_act_bwd(const void* dout, const void* out, void* da, void* db, int64_t positions, int ca, int cb, int act, float slope,
                     int dtype, mra_stream_t stream) {
  MRA_REQUIRE(dout && out && (da || db) && ca > 0 && cb > 0, "mra_cat2_act_bwd: bad arguments");
  MRA_REQUIRE(act == MRA_ACT_NONE || act == MRA_ACT_RELU || act == MRA_ACT_LRELU, "mra_cat2_act_bwd: activation %d", act);
  if (positions <= 0) return 0;
  const bool v8 = dtype == MRA_BF16 && ca % 8 == 0 && cb % 8 == 0;
  const int vec = v8 ? 8 : 1;
  const long long items = positions * (long long)((ca + cb) / vec);
  if (v8) cat2_act_bwd_kernel<bf16, 8><<<ew_grid(items, 1), 256, 0, (cudaStream_t)stream>>>((const bf16*)dout, (const bf16*)out, (bf16*)da, (bf16*)db, items, ca / 8, cb / 8, act, slope);
  else DISPATCH_DTYPE(dtype, (cat2_act_bwd_kernel<T, 1><<<ew_grid(items), 256, 0, (cudaStream_t)stream>>>((const T*)dout, (const T*)out, (T*)da, (T*)db, items, ca, cb, act, slope)));
  MRA_LAUNCH_CHECK();
  return 0;
}

int mra_mask_scale(const void* x, const unsigned char* keep, void* y, int64_t numel, float scale, int dtype,
                   mra_stream_t stream) {
  if (numel <= 0) return 0;
  MRA_REQUIRE(x && keep && y, "mra_mask_scale: null pointer");
  DISPATCH_DTYPE(dtype, (mask_scale_kernel<T><<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>((const T*)x, keep, (T*)y, numel, scale)));
  MRA_LAUNCH_CHECK();
  return 0;
}

static mra_norm_desc pad_desc(int n, int d, int h, int w, int c, int pad, int dtype) {
  mra_norm_desc nd;
  memset(&nd, 0, sizeof(nd));
  nd.n = n; nd.c = c; nd.d = d; nd.h = h; nd.w = w; nd.pad = pad; nd.res_pad = -1; nd.dtype = dtype;
  return nd;
}
int mra_reppad_fwd(const void* x, void* y, int n, int d, int h, int w, int c, int pad, int dtype, mra_stream_t stream) {
  mra_norm_desc nd = pad_desc(n, d, h, w, c, pad, dtype);
  if (int rc = check_norm(&nd)) return rc;
  const mra_norm_desc* dp = &nd;
  DISPATCH_NORM(dp, {
    NormP P = make_norm_params(nd, VEC);
    const long long items = (long long)(d + 2 * pad) * (h + 2 * pad) * (w + 2 * pad) * P.G;
    dim3 grid(grid_for(items, 1024, (16 + n - 1) / n), n);
    reppad_fwd_kernel<T, VEC><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, (T*)y, P);
  });
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_reppad_bwd(const void* gy, void* dx, int n, int d, int h, int w, int c, int pad, int dtype, mra_stream_t stream) {
  mra_norm_desc nd = pad_desc(n, d, h, w, c, pad, dtype);
  if (int rc = check_norm(&nd)) return rc;
  const mra_norm_desc* dp = &nd;
  DISPATCH_NORM(dp, {
    NormP P = make_norm_params(nd, VEC);
    dim3 grid(grid_for(P.V * P.G, 1024, (16 + n - 1) / n), n);
    reppad_bwd_kernel<T, VEC><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)gy, (T*)dx, P);
  });
  MRA_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------ losses / optimiser
int mra_loss_fwd(int kind, const void* a, const void* b, float target, int64_t numel, int dtype, double* acc,
                 mra_stream_t stream) {
  MRA_REQUIRE(kind >= 0 && kind <= 2, "unknown loss kind %d", kind);
  MRA_REQUIRE(kind != MRA_LOSS_L1 || b != nullptr, "L1 needs two operands");
  if (numel <= 0) return 0;
  unsigned g = ew_grid(numel, 16);
  DISPATCH_DTYPE(dtype, (loss_fwd_kernel<T><<<g, 256, 0, (cudaStream_t)stream>>>(kind, (const T*)a, (const T*)b, target, numel, acc)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_loss_bwd(int kind, const void* a, const void* b, float target, int64_t numel, int dtype, const float* gout,
                 float scale, void* da, mra_stream_t stream) {
  MRA_REQUIRE(kind >= 0 && kind <= 2, "unknown loss kind %d", kind);
  if (numel <= 0) return 0;
  DISPATCH_DTYPE(dtype, (loss_bwd_kernel<T><<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(kind, (const T*)a, (const T*)b, target, numel, gout, scale, (T*)da)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_corr_sums(const void* x, const void* y, int64_t numel, int dtype, double* acc, mra_stream_t stream) {
  if (numel <= 0) return 0;
  DISPATCH_DTYPE(dtype, (corr_sums_kernel<T><<<ew_grid(numel, 16), 256, 0, (cudaStream_t)stream>>>((const T*)x, (const T*)y, numel, acc)));
  MRA_LAUNCH_CHECK();
  return 0;
}

static int adam_launch(const mra_adam_tensor* tensors, int count, float lr, float beta1, float beta2, float eps, float step_size,
                       float bc2_sqrt, const float* hyper, cudaStream_t st) {
  int i = 0;
  while (i < count) {
    AdamBatch B;
    memset(&B, 0, sizeof(B));
    B.lr = lr; B.b1 = beta1; B.b2 = beta2; B.eps = eps;
    B.step_size = step_size;
    B.bc2_sqrt = bc2_sqrt;
    B.hyper = hyper;
    long long blocks = 0;
    int c = 0;
    for (; c < MRA_ADAM_MAX_TENSORS && i < count; ++i) {
      const mra_adam_tensor& t = tensors[i];
      if (t.numel <= 0) continue;
      B.p[c] = t.p; B.g[c] = t.g; B.m[c] = t.m; B.v[c] = t.v; B.shadow[c] = (bf16*)t.shadow; B.numel[c] = t.numel;
      B.block_start[c] = blocks;
      blocks += (t.numel + MRA_ADAM_ELEMS_PER_BLOCK - 1) / MRA_ADAM_ELEMS_PER_BLOCK;
      ++c;
    }
    B.block_start[c] = blocks;
    B.count = c;
    if (c == 0) continue;
    adam_kernel<<<(unsigned)blocks, 256, 0, st>>>(B);
    MRA_LAUNCH_CHECK();
  }
  return 0;
}

int mra_adam_multi(const mra_adam_tensor* tensors, int count, float lr, float beta1, float beta2, float eps, int step,
                   mra_stream_t stream) {
  MRA_REQUIRE(count >= 0 && step >= 1, "bad adam arguments");
  const double bc1 = 1.0 - pow((double)beta1, step), bc2 = 1.0 - pow((double)beta2, step);
  return adam_launch(tensors, count, lr, beta1, beta2, eps, (float)((double)lr / bc1), (float)sqrt(bc2), nullptr,
                     (cudaStream_t)stream);
}

int mra_adam_multi_dev(const mra_adam_tensor* tensors, int count, const float* hyper, mra_stream_t stream) {
  MRA_REQUIRE(count >= 0 && hyper != nullptr, "bad adam arguments");
  return adam_launch(tensors, count, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f, hyper, (cudaStream_t)stream);
}

int mra_adam_advance(double* state, float* hyper, mra_stream_t stream) {
  MRA_REQUIRE(state != nullptr && hyper != nullptr, "bad adam_advance arguments");
  adam_advance_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(state, hyper);
  MRA_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------ sliding window helpers
int mra_window_extract(const float* vol, int X, int Y, int Z, int i0, int j0, int k0, int px, int py, int pz,
                       void* patch, int dtype, mra_stream_t stream) {
  MRA_REQUIRE(i0 >= 0 && j0 >= 0 && k0 >= 0 && i0 + px <= X && j0 + py <= Y && k0 + pz <= Z, "window out of range");
  const long long n = (long long)px * py * pz;
  DISPATCH_DTYPE(dtype, (window_extract_kernel<T><<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>(vol, Y, Z, i0, j0, k0, px, py, pz, (T*)patch)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_window_accumulate(const void* pred, int dtype, float* label, float* weight, int X, int Y, int Z, int i0, int j0,
                          int k0, int px, int py, int pz, mra_stream_t stream) {
  MRA_REQUIRE(i0 >= 0 && j0 >= 0 && k0 >= 0 && i0 + px <= X && j0 + py <= Y && k0 + pz <= Z, "window out of range");
  const long long n = (long long)px * py * pz;
  DISPATCH_DTYPE(dtype, (window_accumulate_kernel<T><<<ew_grid(n), 256, 0, (cudaStream_t)stream>>>((const T*)pred, label, weight, Y, Z, i0, j0, k0, px, py, pz)));
  MRA_LAUNCH_CHECK();
  return 0;
}
int mra_window_finalize(float* label, const float* weight, int64_t numel, mra_stream_t stream) {
  if (numel <= 0) return 0;
  window_finalize_kernel<<<ew_grid(numel), 256, 0, (cudaStream_t)stream>>>(label, weight, numel);
  MRA_LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------ introspection
int mra_conv_plan_describe(const mra_conv_desc* d, int which, int32_t* out, int cap) {
  if (int rc = check_conv(d)) return rc;
  if (which == 2) {
    WgradPlan P;
    MRA_REQUIRE(build_wgrad_plan(*d, P), "unsupported geometry");
    return describe(P, out, cap);
  }
  GatherPlan P;
  MRA_REQUIRE(build_gather_plan(*d, which, P), "unsupported geometry");
  return describe(P, out, cap);
}

// CPU walk of the persistent schedules (see include/mra_gan_b200.h).
int mra_debug_schedule(const mra_conv_desc* d, int which, int units, int single, int32_t* out, int cap) {
  if (int rc = check_conv(d)) return rc;
  MRA_REQUIRE(out != nullptr && cap >= 16, "mra_debug_schedule: no output buffer");
  int n = 0;
  auto put = [&](long long v) { if (n < cap) out[n] = (int32_t)v; ++n; };
  if (which == 2) {
    WgradPlan plan;
    MRA_REQUIRE(build_wgrad_plan(*d, plan), "unsupported geometry");
    MRA_REQUIRE(tc::tc_channels_ok(plan.cm) && tc::tc_channels_ok(plan.cn) && !plan.launches.empty(),
                "shape not eligible for the tensor-core wgrad path");
    tc::WgradP P;
    memset(&P, 0, sizeof(P));
    const bool pair = tc::wgrad_fill_geometry(plan, P);
    const long long kblocks = (long long)P.tilesW * P.tilesH * P.tilesD * plan.n;
    MRA_REQUIRE(tc::wgrad_fill_schedule(plan, kblocks, P), "wgrad plan: too many taps or tap groups");
    long long nunits = units;
    if (nunits <= 0) {
      if (pair) nunits = (num_sms() & ~1) / 2;
      else { nunits = num_sms(); if (P.total_cost < nunits * 4) nunits = (P.total_cost + 3) / 4; if (nunits < 1) nunits = 1; }
    }
    put(2); put(pair); put(P.m_tiles); put(P.n_tiles); put(P.n_groups); put(P.n_items); put(kblocks); put(nunits);
    put(P.total_cost & 0x7fffffff); put(P.total_cost >> 31);
    for (int g = 0; g < P.n_groups; ++g) {
      put(P.grp[g].tap0); put(P.grp[g].ntaps); put(P.grp[g].gpi); put(P.grp[g].item0); put(P.grp[g].n_items);
    }
    const int at = n;
    put(0);
    int nseg = 0;
    for (int u = 0; u < (int)nunits; ++u) {
      tc::WSegIter it; tc::WSeg sg;
      tc::wseg_begin(P, kblocks, it, u, (int)nunits);
      while (tc::wseg_next(P, kblocks, it, sg)) {
        put(u); put(sg.item); put(sg.mt); put(sg.nt); put(sg.g); put(sg.tap0); put(sg.ntap); put(sg.kb0); put(sg.kb1);
        ++nseg;
      }
    }
    if (at < cap) out[at] = nseg;
    MRA_REQUIRE(n <= cap, "mra_debug_schedule: %d words needed, cap %d", n, cap);
    return n;
  }
  MRA_REQUIRE(which == 0 || which == 1, "which must be 0, 1 or 2");
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(*d, which, plan), "unsupported geometry");
  put(1);
  const int at_nl = n;
  put(0);
  int nl = 0;
  for (size_t li = 0; li < plan.launches.size(); ++li) {
    const GatherLaunch& L = plan.launches[li];
    tc::HaloP P;
    memset(&P, 0, sizeof(P));
    if (!tc::halo_setup(L, plan.n, plan.ck, plan.cn, single == 0, P, units)) continue;
    tc::halo_fill_skip(P, plan.adims[0]);
    const int pair = P.pair;
    int nu = units > 0 ? units : (pair ? num_sms() / 2 : num_sms());
    if (P.total_work < nu) nu = P.total_work;
    put((int)li); put(pair); put(P.mode); put(P.N); put(P.Dl); put(P.Hl); put(P.Wl); put(P.Wb); put(P.Cn); put(P.n_tile);
    put(P.n_tiles); put(P.total_tiles); put(P.split_from); put(P.total_work); put(nu); put(P.skip); put(P.kd); put(P.nsub);
    const int at = n;
    put(0);
    int nrec = 0;
    for (int u = 0; u < nu; ++u)
      for (int r = 0; r < (pair ? 2 : 1); ++r)
        for (int w = u; w < P.total_work; w += nu)
          for (int sub = 0; sub < P.nsub; ++sub) {
            const tc::HaloTile t = tc::halo_decode(P, w, pair, r, sub);
            int tb, coff;
            tc::halo_stats_key(P, t, tb, coff);
            int live = 0;
            for (int td = 0; td < P.kd && td < 31; ++td) if (tc::halo_plane_live(P, t.d0, td, pair)) live |= 1 << td;
            put(u); put(r); put(w); put(t.n); put(t.d); put(t.n0); put(t.width); put(t.h0); put(t.w0); put(t.f0); put(tb); put(coff);
            put(live); put(sub); put(t.rot_kc0 * 1000000 + t.rot_td0 * 10000 + t.rot_t);
            ++nrec;
          }
    if (at < cap) out[at] = nrec;
    ++nl;
  }
  if (at_nl < cap) out[at_nl] = nl;
  MRA_REQUIRE(n <= cap, "mra_debug_schedule: %d words needed, cap %d", n, cap);
  return n;
}

// Reads (and optionally clears) the tensor-core kernels' device error flag.  Synchronises the
// device: debugging / test use only.  0 = no error, else the code of the first timed-out wait.
int mra_debug_tc_error(int reset) {
  int* flag = tc::tc_err_flag();
  if (!flag) return -1;
  int v = 0;
  if (cudaMemcpy(&v, flag, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  if (reset && v) cudaMemset(flag, 0, sizeof(int));
  return v;
}

// Reads (and optionally clears) the tensor-core kernels' debug cycle counters (8 x uint64).  Synchronises.
int mra_debug_counters(unsigned long long* out, int reset) {
  unsigned long long* buf = tc::tc_dbg_counters();
  if (!buf || !out) return -1;
  if (cudaMemcpy(out, buf, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  if (reset) cudaMemset(buf, 0, 8 * sizeof(unsigned long long));
  return 0;
}

}  // extern "C"
