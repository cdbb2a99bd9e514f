// tcgen05 / TMEM / TMA implicit-GEMM convolution kernels for sm_100a (bf16 operands, fp32 accumulate).
//
// This file holds the PTX wrappers, the shared epilogue, gather_tc_kernel and wgrad_tc_kernel; the halo-plane and
// column variants of the gather computation live in conv_tc_halo.cuh / conv_tc_col.cuh (see conv_plan.h for the
// lowering every conv-family op goes through).
//
//  gather_tc_kernel : D[128 positions][n_tile channels] = sum_{tap, kchunk} A_tap[128][64] * B_tap[n_tile][64]^T
//     A tile  = one 5-D TMA box (64 ch, bw, bh, bd, 1) of the channels-last activation tensor per filter
//               tap (zero fill out of bounds gives the implicit zero padding; element strides give
//               stride-2), landing in shared memory as 128 rows x 128 B, SWIZZLE_128B  -> K-major A.
//     B tile  = 2-D TMA box (64, n_tile) of the packed weights [tap*Cn + cn][ck]        -> K-major B.
//     MMA     = tcgen05.mma.cta_group::1.kind::f16, M=128, N=n_tile (128 for paired phases), K=16, 4 per
//               64-channel chunk, issued by one elected thread; accumulators live in TMEM (up to 8 buffers).
//     Work    = (spatial tile) for a plain launch; (spatial tile, parity phase) or (tile, phase pair) when the 8
//               phases of a stride-2 dgrad-form plan are merged into one launch.
//     Epilogue= 8 warps, two per TMEM lane quadrant: tcgen05.ld 32x32b.x32 -> bias/activation, optional
//               per-(n,channel) sum / sum-of-squares for the following InstanceNorm (kept per thread across tiles
//               when a warp owns one 32-column chunk, warp transpose-reduce otherwise; one fp64 atomic per channel
//               and CTA), convert, 64 B vector stores.
//
//  wgrad_tc_kernel  : dW[tap][128 cm][n_tile cn] += sum_{positions} Mop[pos][cm] * Nop[pos'][cn]
//     both operands are position-major in memory, i.e. MN-major for the MMA: each 64-channel chunk of
//     a 64-position K-block is one TMA box landing as 64 rows x 128 B (SWIZZLE_128B); descriptors use
//     the MN-major canonical layout (LBO = chunk stride, SBO = 1 KiB).  Stream-K over position blocks, fp32
//     red.global.add epilogue.  <true>: cta_group::2 CTA pairs (M = 256, each CTA loads half of the shifted chunks).
//
// Warp roles (gather kernels): warps 0..7 = epilogue, then the TMA producer(s), the TMEM allocator + MMA issuer last
// (scheduler priority); wgrad: warp 0 = TMA producer, 1 = TMEM allocator + MMA issuer, 2..5 = epilogue.  Rings of
// shared-memory stages are guarded by full/empty mbarriers; every wait is bounded and reports through an error flag
// instead of hanging the GPU.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "conv_plan.h"

namespace mra {
namespace tc {

constexpr int kThreads = 192;                    // wgrad kernel: producer, MMA, 4 epilogue warps
// Gather kernels: warps 0..7 = epilogue (two per TMEM lane quadrant, quadrant = warp % 4), then the TMA producer(s),
// and the MMA issuer LAST: the warp scheduler of an SM sub-partition favours the highest warp id among eligible
// warps, so the single thread that feeds the tensor pipe must not sit below the epilogue warps it shares a
// scheduler with.
constexpr int kEpiWarps = 8;
constexpr int kProdWarp = kEpiWarps;             // TMA producer (A and B boxes / weight ring)
constexpr int kMmaWarp = kEpiWarps + 1;          // gather_tc / gather_col: TMEM allocator + MMA issuer
constexpr int kThreadsGather = 32 * 12;         // 3 whole warpgroups: 0..7 epilogue, 8 producer, 9 MMA, 10..11 idle
// Register split between the warpgroups (setmaxnreg): the kernels are compiled for 384 threads = 168 registers per
// thread at entry; the two epilogue warpgroups then grow to kRegsEpi, the producer / MMA warpgroup shrinks to
// kRegsOther (2 * 128 * 224 + 128 * 56 = 64 512 <= 65 536).  The epilogue with statistics keeps ~200 values live
// (accumulator chunk, partial sums, addresses); at 168 registers it spilled loop-carried scalars, and with the L1
// cut to a few KB by the shared-memory carve-out every reload was an L2 round trip inside the epilogue's critical path
// (profiles/r02_col_stem_ncu.txt: 3.4 M local loads per launch, 46 % L1 hit rate, long-scoreboard stalls).
// (The instruction sits at the head of every role branch: ptxas takes the limit of the code that follows from it.)
constexpr int kRegsEpi = 224, kRegsOther = 56;
__device__ __forceinline__ void regs_epilogue() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsEpi)); }
__device__ __forceinline__ void regs_other() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsOther)); }
constexpr int kMaxTaps = 64;
constexpr uint32_t kABytes = 128 * 128;          // 128 rows x 64 bf16

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One elected lane of a fully active warp.  Unlike `lane == 0`, ptxas knows that exactly one thread runs the
// guarded region, so per-thread values can be moved to the uniform registers UTCHMMA / UTMALDG need with a plain
// R2UR instead of a per-instruction ELECT / BROADCAST "waterfall" loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// non-blocking probe of a phase (never suspends the thread): used to "peek" at the next stage's barrier so that
// the probe's latency overlaps the MMA issue of the current stage
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: returns false (and raises the error flag) instead of hanging
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
#pragma unroll 1
  for (uint32_t it = 0; it < (1u << 24); ++it)
    if (mbar_try_wait(bar, parity)) return true;
  if (err) atomicExch(err, code);
  return false;
}
// polling variant (mbarrier.test_wait never suspends the thread)
__device__ __forceinline__ bool mbar_wait_poll(uint64_t* bar, uint32_t parity, int* err, int code) {
#pragma unroll 1
  for (uint32_t it = 0; it < (1u << 26); ++it)
    if (mbar_test_wait(bar, parity)) return true;
  if (err) atomicExch(err, code);
  return false;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptors (cute::UMMA::SmemDescriptor bit layout, version 1 = Blackwell)
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version | [61,64) layout (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t desc_kmajor_sw128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t desc_mnmajor_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32, a=b=BF16, M=128, N=n
__host__ __device__ constexpr uint32_t make_idesc(int n, int a_mn_major, int b_mn_major, int m = 128) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// 256-bit global stores / loads (sm_100: STG.E.ENL2.256): an epilogue thread owns 64 contiguous bytes of an output row
// while its neighbours' rows are >= 128 B away, so every store instruction touches 32 different sectors; with 32-byte
// pieces each of them is written whole (no partial-sector merge in L2) by half as many instructions as with 16-byte ones.
__device__ __forceinline__ void st_global_v8(void* p, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t a4,
                                             uint32_t a5, uint32_t a6, uint32_t a7) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"l"(p), "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(a4), "r"(a5), "r"(a6), "r"(a7) : "memory");
}

// Sum over the 32 lanes of each of 32 per-lane values; lane j ends up with column j's total.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16, n = 16; off >= 1; off >>= 1, n >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
      const float send = hi ? v[i] : v[i + n];
      const float keep = hi ? v[i + n] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}


// ------------------------------------------------------------------ shared epilogue of the gather kernels
// Instruction footprint matters: the epilogue warps run next to the single MMA-issuing thread, and a fully
// unrolled epilogue (hundreds of KB of SASS) evicts that thread's loop from the instruction cache every tile.
// So the 32-column chunk loop stays ROLLED, the per-chunk InstanceNorm partial sums live in a small per-thread
// array indexed at run time, and the transcendental activations are out of line.
struct EpiArgs {
  void* out; int out_bf16;
  const float* bias;
  int act; float slope;
  bool stats;
  // Norm-BACKWARD statistics (dgrad launches whose output is the gradient gy of a fused InstanceNorm -> activation ->
  // replication pad): aux = that norm's stored output y (the conv's own input: same shape and strides as `out`).  The
  // per-(n, channel) sums then are  S0 = sum gy * act'(xhat)  and  S1 = sum gy * act'(xhat) * xhat  -- for the
  // piecewise-linear activations y = max(xhat, s xhat) these are  sum gy * (y > 0 ? 1 : s)  and  sum gy * y  exactly,
  // and summing over the PADDED positions equals summing the folded gradient over the interior ones (y's halo holds
  // replicated values).  They replace the statistics pass of the norm backward (2 of its 5 tensor sweeps).
  const void* aux; float aux_nslope;
};
__device__ __noinline__ float act_slow(float v, int act) {
  return act == MRA_ACT_TANH ? tanhf(v) : 1.f / (1.f + expf(-v));
}
// One accumulator tile -> bias / stats / activation / store.  A warp owns the 32 TMEM lanes of its quadrant and the
// 32-column chunks c = c_begin, c_begin + c_step, ... < nchunks (two warps share a quadrant and take alternate
// chunks).  `release` is called once this warp's TMEM reads of the tile are done (also when it owns no chunk).
//
// InstanceNorm statistics, two flavours:
//   * defer (the warp owns at most ONE chunk, i.e. n_tile <= 64): every thread adds its row's 32 values and
//     squares into fp32 registers d1 / d2 across all tiles of the CTA; the 32-lane transpose-reduce happens once
//     per flush instead of once per tile (it is ~2/3 of the epilogue's instructions, and with N = 64 the epilogue,
//     not the tensor pipe, bounds the small-K launches);
//   * otherwise per tile: warp transpose-reduce, fp64 per-lane partials st_s / st_q.
//
// Dual-plane tiles (gather_col_kernel with 64 output channels): the accumulator is 128 columns wide, columns
// [0, 64) belong to output plane p and [64, 128) to plane p + 1 (`dual_stride` elements further, validity
// `valid_hi`); TMEM chunk c then maps to channel chunk c & 1 of plane c >> 1.
// kMode (compile time, one kernel instantiation each): 0 = no statistics -- the per-thread / per-lane partial sums do
// not exist at all, which is what keeps the dgrad-type launches free of register spills (with the shared-memory
// carve-out at its maximum the L1 is a few KB: a spilled loop variable costs an L2 round trip in the epilogue's
// critical path) --, 1 = InstanceNorm statistics of the output, 2 = norm-backward statistics against E.aux.
// Per-lane fp64 partial sums of the (at most 4) channel chunks a warp owns, slot k <-> channel chunk c_begin + k * c_step.
// Registers with a predicated update per slot: an array indexed by the (run-time) chunk would live in local memory,
// and with the L1 squeezed to a few KB by the shared-memory carve-out every update was an L2 round trip.
struct EpiStats {
  double s[4], q[4];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int i = 0; i < 4; ++i) { s[i] = 0.0; q[i] = 0.0; }
  }
  __device__ __forceinline__ void add(int k, double a, double b) {
#pragma unroll
    for (int i = 0; i < 4; ++i) if (i == k) { s[i] += a; q[i] += b; }
  }
};
// kMode 2: the 32 bf16 aux values of one chunk (64 B of this thread's row), fetched AHEAD of their use: the first chunk
// of a tile before the wait for its accumulator (epilogue_aux_first), every further chunk while the previous one is
// processed -- inside the epilogue a dependent global load costs its full L2 / HBM latency per chunk otherwise.
struct AuxRegs { uint32_t w[16]; };
__device__ __forceinline__ void aux_load(const EpiArgs& E, long long elem, bool valid, AuxRegs& a) {
  if (valid) {
    const char* p = reinterpret_cast<const char*>(reinterpret_cast<const bf16*>(E.aux) + elem);
#pragma unroll
    for (int i = 0; i < 2; ++i)
      asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                   : "=r"(a.w[8 * i]), "=r"(a.w[8 * i + 1]), "=r"(a.w[8 * i + 2]), "=r"(a.w[8 * i + 3]), "=r"(a.w[8 * i + 4]),
                     "=r"(a.w[8 * i + 5]), "=r"(a.w[8 * i + 6]), "=r"(a.w[8 * i + 7])
                   : "l"(p + 32 * i));
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) a.w[i] = 0u;
  }
}
// the first chunk of a warp's tile: call BEFORE waiting for the accumulator (kMode 2, bf16 output only)
template <int kMode>
__device__ __forceinline__ void epilogue_aux_first(const EpiArgs& E, int c_begin, int nchunks, bool valid, long long obase,
                                                   bool dual, AuxRegs& a) {
  if constexpr (kMode == 2) {
    if (E.out_bf16 && c_begin < nchunks) aux_load(E, obase + (dual ? (c_begin & 1) : c_begin) * 32, valid, a);
  }
}
template <int kMode, typename Release>
__device__ __forceinline__ void epilogue_tile(const EpiArgs& E, uint32_t t_addr, int c_begin, int c_step, int nchunks, bool valid,
                                              long long obase, int n0, int lane, EpiStats& st, int slot0, bool defer,
                                              float (&d1)[32], float (&d2)[32], AuxRegs& ax, Release release, bool dual = false,
                                              long long dual_stride = 0, bool valid_hi = false) {
  const bool lin_act = E.act == MRA_ACT_RELU || E.act == MRA_ACT_LRELU;
  const float nslope = E.act == MRA_ACT_RELU ? 0.f : E.slope;
  if (c_begin >= nchunks) { release(); return; }
  const bool valid_lo = valid;
#pragma unroll 1
  for (int ct = c_begin; ct < nchunks; ct += c_step) {
    const int c = dual ? (ct & 1) : ct;                 // channel chunk
    const int c0 = c * 32;
    if (dual) valid = (ct >> 1) ? valid_hi : valid_lo;
    const long long obase_c = obase + ((dual && (ct >> 1)) ? dual_stride : 0);
    uint32_t r[32];
    tmem_ld32(t_addr + (uint32_t)(ct * 32), r);
    AuxRegs nx;
    if constexpr (kMode == 2) {                          // next chunk's aux values: in flight while this chunk is processed
      const int ctn = ct + c_step;
      if (E.out_bf16 && ctn < nchunks) {
        const bool vn = dual ? ((ctn >> 1) ? valid_hi : valid_lo) : valid_lo;
        aux_load(E, obase + ((dual && (ctn >> 1)) ? dual_stride : 0) + (dual ? (ctn & 1) : ctn) * 32, vn, nx);
      }
    }
    tmem_wait_ld();
    if (ct + c_step >= nchunks) release();
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
    if (E.bias) {
      const float4* b4 = reinterpret_cast<const float4*>(E.bias + n0 + c0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    }
    if constexpr (kMode == 2) {
      // aux is consumed 8 values at a time (never more than 8 extra live registers); the deferred flavour adds straight
      // into d1 / d2, the per-tile flavour builds the two arrays of the transpose-reduce
      const float ns = E.aux_nslope;
      if (defer) {
        if (valid) {
          if (E.out_bf16) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float a0 = __uint_as_float(ax.w[i] << 16), a1 = __uint_as_float(ax.w[i] & 0xffff0000u);
              const float g0 = v[2 * i], g1 = v[2 * i + 1];
              d1[2 * i] += a0 > 0.f ? g0 : g0 * ns; d2[2 * i] = fmaf(g0, a0, d2[2 * i]);
              d1[2 * i + 1] += a1 > 0.f ? g1 : g1 * ns; d2[2 * i + 1] = fmaf(g1, a1, d2[2 * i + 1]);
            }
          } else {
            const float4* ap = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(E.aux) + obase_c + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 u = __ldg(ap + i);
              const float a4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float g = v[4 * i + k];
                d1[4 * i + k] += a4[k] > 0.f ? g : g * ns; d2[4 * i + k] = fmaf(g, a4[k], d2[4 * i + k]);
              }
            }
          }
        }
      } else {
        float s1[32], s2[32];
        if (valid) {
          if (E.out_bf16) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float a0 = __uint_as_float(ax.w[i] << 16), a1 = __uint_as_float(ax.w[i] & 0xffff0000u);
              const float g0 = v[2 * i], g1 = v[2 * i + 1];
              s1[2 * i] = a0 > 0.f ? g0 : g0 * ns; s2[2 * i] = g0 * a0;
              s1[2 * i + 1] = a1 > 0.f ? g1 : g1 * ns; s2[2 * i + 1] = g1 * a1;
            }
          } else {
            const float4* ap = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(E.aux) + obase_c + c0);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 u = __ldg(ap + i);
              const float a4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float g = v[4 * i + k];
                s1[4 * i + k] = a4[k] > 0.f ? g : g * ns; s2[4 * i + k] = g * a4[k];
              }
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) { s1[i] = 0.f; s2[i] = 0.f; }
        }
        const float a1 = warp_colsum32(s1, lane), a2 = warp_colsum32(s2, lane);
        st.add(slot0 + (c - c_begin) / c_step, (double)a1, (double)a2);
      }
    } else if constexpr (kMode == 1) {
      if (defer) {
        if (valid) {
#pragma unroll
          for (int i = 0; i < 32; ++i) { d1[i] += v[i]; d2[i] = fmaf(v[i], v[i], d2[i]); }
        }
      } else {
        float s1[32], s2[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) { s1[i] = valid ? v[i] : 0.f; s2[i] = s1[i] * s1[i]; }
        const float a1 = warp_colsum32(s1, lane), a2 = warp_colsum32(s2, lane);
        st.add(slot0 + (c - c_begin) / c_step, (double)a1, (double)a2);
      }
    }
    if constexpr (kMode == 2) ax = nx;
    if (lin_act) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = v[i] > 0.f ? v[i] : v[i] * nslope;
    } else if (E.act != MRA_ACT_NONE) {
#pragma unroll 1
      for (int i = 0; i < 32; ++i) {
        // dynamic index into a register array would spill; go through a select chain on a rotating copy instead
        float x = v[0];
#pragma unroll
        for (int k = 1; k < 32; ++k) x = (k == i) ? v[k] : x;
        const float y = act_slow(x, E.act);
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = (k == i) ? y : v[k];
      }
    }
    if (valid) {
      if (E.out_bf16) {
        char* o = reinterpret_cast<char*>(reinterpret_cast<bf16*>(E.out) + obase_c + c0);
#pragma unroll
        for (int i = 0; i < 2; ++i)
          st_global_v8(o + 32 * i, pack_bf16x2(v[16 * i], v[16 * i + 1]), pack_bf16x2(v[16 * i + 2], v[16 * i + 3]),
                       pack_bf16x2(v[16 * i + 4], v[16 * i + 5]), pack_bf16x2(v[16 * i + 6], v[16 * i + 7]),
                       pack_bf16x2(v[16 * i + 8], v[16 * i + 9]), pack_bf16x2(v[16 * i + 10], v[16 * i + 11]),
                       pack_bf16x2(v[16 * i + 12], v[16 * i + 13]), pack_bf16x2(v[16 * i + 14], v[16 * i + 15]));
      } else {
        float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(E.out) + obase_c + c0);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
    }
  }
}
// Add the CTA's per-chunk partial sums to stats[n][Cn][2] and clear them.  The four quadrant warps that own a chunk
// first combine their per-lane partials through shared memory, so a flush costs ONE fp64 atomic per channel and CTA:
// all CTAs flush at the same moment (kernel end), and same-address atomics are serialised by the L2 at ~50 ns each
// -- with one atomic per WARP (592 per address) that tail was 30 us per launch.
// Called by all epilogue warps at the same points of the tile sequence (named barrier 1 + group, 128 threads).
typedef double EpiRed[2][4][32][2];              // [chunk group][quadrant][lane][sum, sum of squares]
constexpr size_t kEpiRedBytes = sizeof(EpiRed);  // static shared memory of the gather kernels
__device__ __forceinline__ void epilogue_flush_stats(double* stats, int n, int Cn, int n0, int q, int c_begin, int c_step,
                                                     int nchunks, int lane, EpiStats& st, bool defer,
                                                     float (&d1)[32], float (&d2)[32], EpiRed& red) {
  if (n < 0) return;
  if (defer && c_begin < nchunks) {
    const float a1 = warp_colsum32(d1, lane), a2 = warp_colsum32(d2, lane);
    st.add(0, (double)a1, (double)a2);
#pragma unroll
    for (int i = 0; i < 32; ++i) { d1[i] = 0.f; d2[i] = 0.f; }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c_begin + k * c_step;
    if (c < nchunks) {                                   // same for all 128 threads of the group
      red[c_begin][q][lane][0] = st.s[k];
      red[c_begin][q][lane][1] = st.q[k];
      st.s[k] = 0.0; st.q[k] = 0.0;
      asm volatile("bar.sync %0, 128;" ::"r"(1 + c_begin) : "memory");
      if (q == 0) {
        const double a = red[c_begin][0][lane][0] + red[c_begin][1][lane][0] + red[c_begin][2][lane][0] + red[c_begin][3][lane][0];
        const double b = red[c_begin][0][lane][1] + red[c_begin][1][lane][1] + red[c_begin][2][lane][1] + red[c_begin][3][lane][1];
        double* sp = stats + ((long long)n * Cn + n0 + c * 32 + lane) * 2;
        atomicAdd(sp, a);
        atomicAdd(sp + 1, b);
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + c_begin) : "memory");
    }
  }
}
// per-warp epilogue state shared by the three gather kernels
struct EpiWarp {
  int q, c_begin;                  // TMEM lane quadrant (warp % 4), first chunk of this warp
  __device__ __forceinline__ EpiWarp(int warp) : q(warp & 3), c_begin(warp >> 2) {}
};

// ------------------------------------------------------------------ gather (fprop / dgrad) kernel
struct GatherP {
  int tilesW, tilesH, tilesD;
  int bw, bh, bd;
  int Dl, Hl, Wl;
  int astep;
  int Cn, n_tile, n_tiles, kchunks, ntaps;
  int total_tiles;                  // N * tilesD * tilesH * tilesW * n_tiles
  int ostep, od0, oh0, ow0;
  long long osn, osd, osh, osw;     // output strides in elements
  void* out;
  int out_bf16;
  const float* bias;
  int act;
  float slope;
  double* stats;                    // [N][Cn][2] or null
  const void* aux; float aux_nslope; // norm-backward statistics (EpiArgs::aux)
  int* err;
  int stages;
  int nbuf;                         // accumulator buffers in TMEM: 512 / n_tile, at most 8 (small tiles: the buffer
                                    // turnaround MMA -> commit -> epilogue -> release is ~1 us, far more than their MMAs)
  uint32_t tmem_cols;               // nbuf accumulator buffers of n_tile columns (power of two >= 32)
  int8_t tdd[kMaxTaps], tdh[kMaxTaps], tdw[kMaxTaps];
  int16_t twi[kMaxTaps];
  int debug;                        // bit 1: cycle counters into dbg (see tc_dbg_counters)
  unsigned long long* dbg;
  // Merged parity phases (stride-2 dgrad-form plans): ONE launch walks (spatial tile, phase) work items, so the 8
  // phases of a tile run back to back on neighbouring SMs and re-read the input tile from L2 instead of HBM.
  int nph;                          // work items per spatial tile: 1 (plain launch), 8 (phases) or 4 (phase pairs)
  int16_t ph_tap0[9];               // item p uses entries [ph_tap0[p], ph_tap0[p + 1]) of the tap arrays
  int8_t ph_od[8], ph_oh[8], ph_ow[8];   // output coordinate offsets of item p
  // Phase pairs (n_tile = 64 only: an N = 64 MMA costs 54.5 clk where 32 would be ideal, N = 128 the ideal 64): the two
  // phases that differ in the parity of w share a 128-column accumulator (columns [0, 64) = even w, [64, 128) = odd w,
  // adjacent output positions).  A tap entry is then one A offset with the weight slab of either phase or of both:
  // both -> one N = 128 MMA over the two slabs stacked in the stage, one -> N = 64 into its half.
  int pair;
  int16_t twi2[kMaxTaps];           // second phase's slab of the entry (-1: none; then twi may be -1 instead)
  uint8_t eacc[kMaxTaps];           // 1: the entry's columns were already written by an earlier entry (accumulate)
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

struct TileCoord { int n, lw0, lh0, ld0, n0, ph; };
// phase of work item `tile` of a merged launch: rotated with the spatial index so that every CTA of the persistent
// schedule sees all phases (they carry 1..8 taps) equally often
__device__ __forceinline__ int tile_phase(const GatherP& P, int tile) {
  return P.nph == 8 ? ((tile & 7) + (tile >> 3)) & 7 : (P.nph == 4 ? ((tile & 3) + (tile >> 2)) & 3 : 0);
}
__device__ __forceinline__ TileCoord decode_tile(const GatherP& P, int tile) {
  TileCoord t;
  t.ph = tile_phase(P, tile);
  if (P.nph == 8) tile >>= 3; else if (P.nph == 4) tile >>= 2;
  const int nt = tile % P.n_tiles; tile /= P.n_tiles;
  const int tw = tile % P.tilesW; tile /= P.tilesW;
  const int th = tile % P.tilesH; tile /= P.tilesH;
  const int td = tile % P.tilesD;
  t.n = tile / P.tilesD;
  t.lw0 = tw * P.bw; t.lh0 = th * P.bh; t.ld0 = td * P.bd; t.n0 = nt * P.n_tile;
  return t;
}

// Persistent: gridDim.x CTAs (one per SM) walk the work-item list with stride gridDim.x.  The accumulator is
// multi-buffered in TMEM (P.nbuf) so the epilogue of item j overlaps the MMAs of the following items; InstanceNorm
// statistics are accumulated per CTA and flushed with one fp64 atomic per channel when the sample index changes
// (instead of per tile).
template <int kMode>         // epilogue statistics mode, see epilogue_tile
__global__ void __launch_bounds__(kThreadsGather, 1)
gather_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ GatherP P) {
  pdl_launch_dependents();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t slab_bytes = (uint32_t)P.n_tile * 128u;
  const uint32_t b_bytes = P.pair ? 2u * slab_bytes : slab_bytes;
  const uint32_t stage_bytes = kABytes + b_bytes;
  const int acc_cols = P.pair ? 2 * P.n_tile : P.n_tile;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
  uint64_t* empty_bar = full_bar + P.stages;
  uint64_t* acc_full = empty_bar + P.stages;      // [nbuf]
  uint64_t* acc_empty = acc_full + P.nbuf;        // [nbuf]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + P.nbuf);

  __shared__ EpiRed epi_red;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < P.nbuf; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                  // prologue done: from here on global memory is touched

  if (warp >= kEpiWarps) {            // third warpgroup: producers, MMA issuer, idle warps -- one setmaxnreg for all of it
  regs_other();
  if (warp == kProdWarp) {
    if (elect_one()) {
      uint32_t git = 0;                                    // global k-iteration counter (stage ring position)
      bool ok = true;
      const bool prof = (P.debug & 2) != 0;
      long long t_wait = 0, t_begin = prof ? clock64() : 0;
      int s = 0;
      uint32_t ph = 0;
      (void)git;
      for (int tile = blockIdx.x; tile < P.total_tiles && ok; tile += gridDim.x) {
        const TileCoord t = decode_tile(P, tile);
        int tap = P.ph_tap0[t.ph], kc = 0;
        const int iters = (P.ph_tap0[t.ph + 1] - tap) * P.kchunks;
        for (int it = 0; it < iters; ++it) {
          const long long tw0 = prof ? clock64() : 0;
          if (!mbar_wait(&empty_bar[s], ph ^ 1u, P.err, 1)) { ok = false; break; }
          if (prof) t_wait += clock64() - tw0;
          uint8_t* sa = smem + (size_t)s * stage_bytes;
          const int w1 = P.twi[tap], w2 = P.pair ? P.twi2[tap] : -1;
          mbar_expect_tx(&full_bar[s], kABytes + ((w1 >= 0 && w2 >= 0) ? 2u * slab_bytes : slab_bytes));
          tma_load_5d(sa, &tmA, &full_bar[s], kc * 64, t.lw0 * P.astep + P.tdw[tap], t.lh0 * P.astep + P.tdh[tap],
                      t.ld0 * P.astep + P.tdd[tap], t.n);
          tma_load_2d(sa + kABytes, &tmB, &full_bar[s], kc * 64, (w1 >= 0 ? w1 : w2) * P.Cn + t.n0);
          if (w1 >= 0 && w2 >= 0) tma_load_2d(sa + kABytes + slab_bytes, &tmB, &full_bar[s], kc * 64, w2 * P.Cn + t.n0);
          if (++s == P.stages) { s = 0; ph ^= 1u; }
          if (++kc == P.kchunks) { kc = 0; ++tap; }
        }
      }
      if (prof) { atomicAdd(P.dbg + 0, (unsigned long long)t_wait); atomicAdd(P.dbg + 1, (unsigned long long)(clock64() - t_begin)); }
    }
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      const uint32_t idesc1 = make_idesc(P.n_tile, 0, 0), idesc2 = make_idesc(2 * P.n_tile, 0, 0);
      const uint64_t desc0 = desc_kmajor_sw128(0);
      const uint32_t smem_u = smem_u32(smem) >> 4, stage_u = stage_bytes >> 4;
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      int j = 0;
      const bool prof = (P.debug & 2) != 0;
      long long t_wait = 0, t_wacc = 0, t_begin = prof ? clock64() : 0;
      int buf = 0;
      uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < P.total_tiles && ok; tile += gridDim.x, ++j) {
        const long long ta0 = prof ? clock64() : 0;
        if (!mbar_wait(&acc_empty[buf], aph ^ 1u, P.err, 4)) { ok = false; break; }   // epilogue drained this buffer
        if (prof) t_wacc += clock64() - ta0;
        tc_fence_after();
        const uint32_t d_tmem0 = tmem_base + (uint32_t)(buf * acc_cols);
        // single issuing thread: no divisions, descriptors advance by constants (16-byte units)
        const int tph = tile_phase(P, tile);
        int tap = P.ph_tap0[tph], kc = 0;
        const int iters = (P.ph_tap0[tph + 1] - tap) * P.kchunks;
        for (int it = 0; it < iters; ++it) {
          const long long tw0 = prof ? clock64() : 0;
          if (!mbar_wait(&full_bar[s], ph, P.err, 2)) { ok = false; break; }
          if (prof) t_wait += clock64() - tw0;
          tc_fence_after();
          const uint32_t sa_u = smem_u + (uint32_t)s * stage_u;
          const uint64_t ad = desc0 | (uint64_t)(sa_u & 0x3FFFu);
          const uint64_t bd = desc0 | (uint64_t)((sa_u + (kABytes >> 4)) & 0x3FFFu);
          uint32_t idesc = idesc1, d_tmem = d_tmem0, acc = (uint32_t)(it != 0);
          if (P.pair) {                            // entry = one A offset x the slab(s) of the even-w / odd-w phase
            const bool has1 = P.twi[tap] >= 0, has2 = P.twi2[tap] >= 0;
            idesc = (has1 && has2) ? idesc2 : idesc1;
            d_tmem = d_tmem0 + (has1 ? 0u : (uint32_t)P.n_tile);
            acc = (uint32_t)(P.eacc[tap] != 0 || kc != 0);
          }
          umma_f16(d_tmem, ad, bd, idesc, acc);
          umma_f16(d_tmem, ad + 2, bd + 2, idesc, 1u);
          umma_f16(d_tmem, ad + 4, bd + 4, idesc, 1u);
          umma_f16(d_tmem, ad + 6, bd + 6, idesc, 1u);
          umma_commit(&empty_bar[s]);
          if (++s == P.stages) { s = 0; ph ^= 1u; }
          if (++kc == P.kchunks) { kc = 0; ++tap; }
        }
        if (ok) umma_commit(&acc_full[buf]);
        if (++buf == P.nbuf) { buf = 0; aph ^= 1u; }
      }
      if (prof) {
        atomicAdd(P.dbg + 2, (unsigned long long)t_wait); atomicAdd(P.dbg + 3, (unsigned long long)(clock64() - t_begin));
        atomicAdd(P.dbg + 6, (unsigned long long)t_wacc); atomicAdd(P.dbg + 5, 1ull);
      }
    }
  }
  } else {
    // epilogue warps 0..7 -> TMEM lane quadrant (warp % 4), alternate 32-column chunks
    regs_epilogue();
    const EpiWarp W(warp);
    const int q = W.q;
    const int row = q * 32 + lane;
    const int rw = row % P.bw, rh = (row / P.bw) % P.bh, rd = row / (P.bw * P.bh);
    const int nchunks = P.n_tile / 32;
    const bool defer = kMode != 0 && nchunks <= 2;
    EpiStats st;                             // per-lane running sums of this warp's chunks
    st.clear();
    float d1[32], d2[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) { d1[i] = 0.f; d2[i] = 0.f; }
    int st_n = -1, st_n0 = 0;
    const EpiArgs E{P.out, P.out_bf16, P.bias, P.act, P.slope, P.stats != nullptr, P.aux, P.aux_nslope};
    int buf = 0;
    uint32_t aph = 0;
    bool ok = true;
    for (int tile = blockIdx.x; tile < P.total_tiles && ok; tile += gridDim.x) {
      const TileCoord t = decode_tile(P, tile);
      const int lw = t.lw0 + rw, lh = t.lh0 + rh, ld = t.ld0 + rd;
      const bool valid = lw < P.Wl && lh < P.Hl && ld < P.Dl;
      const long long obase = (long long)t.n * P.osn + (long long)(ld * P.ostep + P.ph_od[t.ph]) * P.osd +
                              (long long)(lh * P.ostep + P.ph_oh[t.ph]) * P.osh +
                              (long long)(lw * P.ostep + P.ph_ow[t.ph]) * P.osw + t.n0;
      if (kMode != 0 && (t.n != st_n || t.n0 != st_n0)) {
        epilogue_flush_stats(P.stats, st_n, P.Cn, st_n0, W.q, W.c_begin, 2, nchunks, lane, st, defer, d1, d2, epi_red);
        st_n = t.n; st_n0 = t.n0;
      }
      AuxRegs ax;
      epilogue_aux_first<kMode>(E, W.c_begin, acc_cols / 32, valid, obase, P.pair != 0, ax);
      ok = mbar_wait(&acc_full[buf], aph, P.err, 3);
      if (!ok) break;
      tc_fence_after();
      const long long te0 = (P.debug & 2) ? clock64() : 0;
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * acc_cols);
      uint64_t* rel_bar = &acc_empty[buf];
      epilogue_tile<kMode>(E, t_addr, W.c_begin, 2, acc_cols / 32, valid, obase, t.n0, lane, st, 0, defer, d1, d2, ax, [&]() {
        tc_fence_before();                      // accumulator fully read: hand the buffer back to the MMA warp
        __syncwarp();
        if (lane == 0) mbar_arrive(rel_bar);
      }, P.pair != 0, P.osw, valid);
      if ((P.debug & 2) && threadIdx.x == 0) atomicAdd(P.dbg + 4, (unsigned long long)(clock64() - te0));
      if (++buf == P.nbuf) { buf = 0; aph ^= 1u; }
    }
    if (kMode != 0) epilogue_flush_stats(P.stats, st_n, P.Cn, st_n0, W.q, W.c_begin, 2, nchunks, lane, st, defer, d1, d2, epi_red);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, P.tmem_cols);
}

// ---- cta_group::2 (CTA pair) flavours of the PTX wrappers.  In pair mode two CTAs of a cluster (one TPC) each
// own a 128-row tile and HALF of the weight slab; the leader (cluster rank 0) issues one M = 256 MMA for both,
// so every CTA streams only half of the weights from L2.  TMA loads of both CTAs signal the LEADER's barrier
// (peer bit 24 of the shared::cluster address cleared), tcgen05.commit multicasts to both CTAs' barriers.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <bool kPair>
__device__ __forceinline__ void tma_load_5d_g(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2, int c3,
                                              int c4) {
  if constexpr (kPair) {
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
  } else {
    tma_load_5d(dst, tm, bar, c0, c1, c2, c3, c4);
  }
}
template <bool kPair>
__device__ __forceinline__ void tma_load_2d_g(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
  if constexpr (kPair) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
  } else {
    tma_load_2d(dst, tm, bar, c0, c1);
  }
}
template <bool kPair>
__device__ __forceinline__ void umma_commit_g(uint64_t* bar) {
  if constexpr (kPair) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
  } else {
    umma_commit(bar);
  }
}
template <bool kPair>
__device__ __forceinline__ void umma_f16_g(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kPair) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    umma_f16(d_tmem, adesc, bdesc, idesc, accumulate);
  }
}
// arrive on the barrier at the same offset in the pair's leader CTA
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__host__ __device__ constexpr uint32_t make_idesc_m(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}


// ------------------------------------------------------------------ wgrad kernel
// D[tap][m][n] = sum_{positions q} Dense[q][m] * Shifted[q*sstep + tap][n]
//   Dense   = the operand read at the K-block positions themselves (dy for Conv3d, x for ConvTranspose3d),
//   Shifted = the other one (x for Conv3d, dy for ConvTranspose3d).
// Work item = (item, 128-row m tile, n tile of 64*ncc channels).  An item is up to 8/ncc filter taps whose
// accumulators sit side by side in TMEM (<= 512 columns), so the dense tile of a K-block (64 positions) is
// loaded once for all of them.  Taps come in up to 4 GROUPS; in a group with share == 2 two taps that are
// neighbours along w (or h) read ONE shared-memory box of the shifted operand, extended by one column (row):
// the UMMA descriptor of the second tap simply starts `rshift` rows later (the SWIZZLE_128B pattern is a
// function of the absolute shared-memory address, so row-shifted starts are legal; verified by
// tools/halo_probe.cu).  Both operands are position-major = MN-major for the MMA.
// Scheduling is stream-K: the (work item x K-block) space, weighted by taps per item, is cut into
// gridDim.x equal contiguous ranges (one CTA per SM, one wave); a CTA whose range crosses a work-item
// boundary flushes its accumulators (fp32 red.global.add) and continues with the next item.
// A work item that several CTAs share is not added piece by piece in timing order (fp32 addition is not associative, so dw
// would change from run to run): each piece stores its partial tile in P.part, and wgrad_fixup_kernel adds the pieces of
// the item to dw in K order once the launch is complete.  An item that one CTA does alone is added straight away.
constexpr int kMaxWGroups = 4;
struct WGroup {
  int tap0, ntaps;                  // range in the launch-ordered tap arrays
  int item0, n_items;               // range of items
  int gpi, share;                   // taps per item, taps per box set
  int pitch_w, pitch_h;             // rows per h line / per d plane of a shifted-operand box
  int box_tx;                       // bytes one 64-channel box delivers
  long long cost0;                  // stream-K cost of all work items of the groups before this one
};
struct WgradP {
  int tilesW, tilesH, tilesD;       // K-block boxes per dim of the dense position space
  int bw, bh, bd;                   // K-block box (product 64)
  int N;
  int sstep;
  int Km, Kn;                       // channels of the dense / shifted operand
  int m_chunks;                     // 64-channel chunks of the dense operand per m tile (1 or 2)
  int ncc;                          // 64-channel chunks of the shifted operand per tap
  int box_bytes;                    // shared-memory slot of one 64-channel shifted box (multiple of 1024, max over groups)
  int sets_max;                     // box sets per stage slot (max over groups)
  int n_groups, n_items, m_tiles, n_tiles;
  long long total_cost;             // sum over work items of taps(item) * K-blocks
  float* dw;
  long long tap_stride, m_stride, n_stride;   // element strides of dw[tap][m][n] in memory
  float* part;                      // partial tiles of shared items: [CTA][0: the piece that starts the CTA's range,
  int part_cols;                    //   1: the piece that ends it][128 rows][part_cols]
  int* err;
  int stages;
  uint32_t tmem_cols;
  WGroup grp[kMaxWGroups];
  int8_t odd[kMaxTaps], odh[kMaxTaps], odw[kMaxTaps];   // box origin offset per tap (launch order)
  int16_t rshift[kMaxTaps];                             // row shift of the tap inside its box
  int16_t twi[kMaxTaps];                                // weight slab index of the tap
  int debug;                                            // bit 0: skip the global reductions, bit 1: cycle counters
  unsigned long long* dbg;
};
struct WMaps { CUtensorMap m[kMaxWGroups]; };

constexpr uint32_t kChunkBytes = 64 * 128;       // 64 positions x 64 bf16
constexpr size_t kWgradFlushBytes = 4 * 4096;    // transposing buffers of the 4 epilogue warps (see the flush)

// One contiguous piece of a CTA's stream-K range that lies inside a single work item.
struct WSeg { int item, mt, nt, g, tap0, ntap, kb0, kb1; };
struct WSegIter {
  long long pos, end, woff;
  int work;
};
__host__ __device__ __forceinline__ int wg_item_group(const WgradP& P, int item) {
  int g = 0;
  while (g + 1 < P.n_groups && item >= P.grp[g + 1].item0) ++g;
  return g;
}
__host__ __device__ __forceinline__ int wg_item_ntap(const WgradP& P, int g, int item) {
  const WGroup& G = P.grp[g];
  return min(G.gpi, G.ntaps - (item - G.item0) * G.gpi);
}
__host__ __device__ __forceinline__ void wseg_begin(const WgradP& P, long long kblocks, WSegIter& it, int unit, int nunits) {
  const long long share = (P.total_cost + nunits - 1) / nunits;
  it.pos = (long long)unit * share;
  it.end = min(it.pos + share, P.total_cost);
  const int per_item = P.m_tiles * P.n_tiles;
  const int n_work = P.n_items * per_item;
  // First work item that ends after it.pos, in O(groups): inside a group every item carries gpi taps except possibly the
  // last one, so the cumulative cost is piecewise linear.  (A linear walk over the work items cost the last CTAs of the
  // deep UNet layers -- 512 to 2048 items of 4 K-blocks -- ~100 us of single-thread integer code before their first load:
  // those launches took 0.11 - 0.26 ms whatever their size.)
  int g = 0;
  while (g + 1 < P.n_groups && P.grp[g + 1].cost0 <= it.pos) ++g;
  const WGroup& G = P.grp[g];
  const long long span_full = (long long)G.gpi * kblocks;
  const int items_full = G.ntaps / G.gpi;                          // items with gpi taps
  const long long works_full = (long long)items_full * per_item;
  const long long off = it.pos - G.cost0;
  long long wl;                                                    // work index inside the group
  if (off < works_full * span_full) {
    wl = off / span_full;
    it.woff = G.cost0 + wl * span_full;
  } else {
    const long long span_part = (long long)(G.ntaps - items_full * G.gpi) * kblocks;
    const long long rem = off - works_full * span_full;
    wl = works_full + (span_part > 0 ? rem / span_part : 0);
    it.woff = G.cost0 + works_full * span_full + (wl - works_full) * span_part;
  }
  it.work = G.item0 * per_item + (int)wl;
  if (it.work > n_work) it.work = n_work;
}
__host__ __device__ __forceinline__ bool wseg_next(const WgradP& P, long long kblocks, WSegIter& it, WSeg& sg) {
  const int per_item = P.m_tiles * P.n_tiles;
  const int n_work = P.n_items * per_item;
  while (it.pos < it.end && it.work < n_work) {
    const int item = it.work / per_item;
    const int g = wg_item_group(P, item);
    const int ntap = wg_item_ntap(P, g, item);
    const long long span = (long long)ntap * kblocks;
    const long long lo = it.pos, hi = min(it.end, it.woff + span);
    const int kb0 = (int)((lo - it.woff) / ntap);
    const int kb1 = hi == it.woff + span ? (int)kblocks : (int)((hi - it.woff) / ntap);
    const int w = it.work;
    it.pos = hi;
    if (hi == it.woff + span) { it.woff += span; ++it.work; }
    if (kb1 > kb0) {
      const int rem = w - item * per_item;
      sg.item = item; sg.mt = rem / P.n_tiles; sg.nt = rem - sg.mt * P.n_tiles; sg.g = g;
      sg.tap0 = P.grp[g].tap0 + (item - P.grp[g].item0) * P.grp[g].gpi; sg.ntap = ntap; sg.kb0 = kb0; sg.kb1 = kb1;
      return true;
    }
  }
  return false;
}

// kPair: two CTAs of a cluster form one cta_group::2 unit.  Each CTA owns one 128-row m tile (M = 256 per MMA) and loads
// only HALF of the shifted operand's channel chunks -- the tensor core reads the other half from the partner's shared
// memory -- so the L2 -> SM traffic per FLOP drops by a third (G.rb wgrad was bound by exactly that traffic).
template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmM, const __grid_constant__ WMaps tmN,
                const __grid_constant__ WgradP P) {
  pdl_launch_dependents();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kCtas = kPair ? 2 : 1;
  const int rank = kPair ? (int)cluster_ctarank() : 0;
  const bool leader = rank == 0;
  const int unit = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int nunits = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int ncc_l = P.ncc / kCtas;                           // shifted-operand chunks held by this CTA
  const uint32_t m_bytes = 2 * kChunkBytes;                  // the m tile always owns two chunk slots
  const uint32_t set_bytes = (uint32_t)ncc_l * (uint32_t)P.box_bytes;
  const uint32_t stage_bytes = m_bytes + (uint32_t)P.sets_max * set_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)P.stages * stage_bytes);
  uint64_t* empty_bar = full_bar + P.stages;
  uint64_t* acc_full = empty_bar + P.stages;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);
  uint8_t* flush_stage = smem + (size_t)P.stages * stage_bytes + 256;      // 4 epilogue warps x 4 KB (kWgradFlushBytes)

  const int boxes_per_sample = P.tilesW * P.tilesH * P.tilesD;
  const long long kblocks = (long long)boxes_per_sample * P.N;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmM);
    for (int g = 0; g < P.n_groups; ++g) prefetch_tmap(&tmN.m[g]);
    for (int s = 0; s < P.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 4 * kCtas);
    fence_barrier_init();
  }
  if (P.m_chunks == 1) {
    // the second chunk slot of the m tile is never loaded: keep it finite (its rows are discarded)
    for (int s = 0; s < P.stages; ++s) {
      uint4* z = reinterpret_cast<uint4*>(smem + (size_t)s * stage_bytes + kChunkBytes);
      for (int i = threadIdx.x; i < (int)(kChunkBytes / 16); i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  if (warp == 1) {
    if constexpr (kPair) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(P.tmem_cols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      tmem_alloc(tmem_slot, P.tmem_cols);
    }
  }
  tc_fence_before();
  if constexpr (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                  // prologue done: from here on global memory is touched
  const bool prof = (P.debug & 2) != 0;

  if (warp == 0) {
    // ---- TMA producer: lane j issues box j of every stage (box 0..m_chunks-1 dense, then the shifted boxes)
    WSegIter it; WSeg sg;
    wseg_begin(P, kblocks, it, unit, nunits);
    int s = 0;
    uint32_t ph = 0;
    long long t_wait = 0, t_begin = prof ? clock64() : 0;
    bool ok = true;
    while (ok && wseg_next(P, kblocks, it, sg)) {
      const WGroup& G = P.grp[sg.g];
      const int nsets = (sg.ntap + G.share - 1) / G.share;
      const int nboxes = P.m_chunks + nsets * ncc_l;
      // bytes landing per stage in the whole unit (pair: both CTAs' boxes complete on the leader's barrier)
      const uint32_t tx_bytes = ((uint32_t)P.m_chunks * kChunkBytes + (uint32_t)(nsets * ncc_l) * (uint32_t)G.box_tx) * kCtas;
      const int mt = kPair ? 2 * sg.mt + rank : sg.mt;
      // this lane's box
      const bool active = lane < nboxes;
      const bool dense = lane < P.m_chunks;
      int c0 = 0, ow = 0, oh = 0, od = 0, step = 1;
      uint32_t soff = 0;
      const CUtensorMap* tm = &tmM;
      if (active) {
        if (dense) { c0 = mt * 128 + 64 * lane; soff = (uint32_t)lane * kChunkBytes; }
        else {
          const int bi = lane - P.m_chunks, bs = bi / ncc_l, j = bi - bs * ncc_l;
          const int t = sg.tap0 + bs * G.share;
          c0 = sg.nt * P.ncc * 64 + 64 * (rank * ncc_l + j); ow = P.odw[t]; oh = P.odh[t]; od = P.odd[t]; step = P.sstep;
          soff = m_bytes + (uint32_t)bs * set_bytes + (uint32_t)j * (uint32_t)P.box_bytes;
          tm = &tmN.m[sg.g];
        }
      }
      // K-block coordinates, advanced incrementally
      int n = sg.kb0 / boxes_per_sample;
      int r = sg.kb0 - n * boxes_per_sample;
      int tw = r % P.tilesW; r /= P.tilesW;
      int th = r % P.tilesH;
      int td = r / P.tilesH;
      for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
        const long long tw0 = prof ? clock64() : 0;
        if (!mbar_wait(&empty_bar[s], ph ^ 1u, P.err, 11)) { ok = false; break; }
        if (prof) t_wait += clock64() - tw0;
        if (lane == 0 && leader) mbar_expect_tx(&full_bar[s], tx_bytes);
        __syncwarp();
        if (active)
          tma_load_5d_g<kPair>(smem + (size_t)s * stage_bytes + soff, tm, &full_bar[s], c0, tw * P.bw * step + ow,
                               th * P.bh * step + oh, td * P.bd * step + od, n);
        if (++tw == P.tilesW) { tw = 0; if (++th == P.tilesH) { th = 0; if (++td == P.tilesD) { td = 0; ++n; } } }
        if (++s == P.stages) { s = 0; ph ^= 1u; }
      }
    }
    if (prof && lane == 0) { atomicAdd(P.dbg + 0, (unsigned long long)t_wait); atomicAdd(P.dbg + 1, (unsigned long long)(clock64() - t_begin)); }
  } else if (warp == 1) {
    if (elect_one() && leader) {
      WSegIter it; WSeg sg;
      wseg_begin(P, kblocks, it, unit, nunits);
      const uint32_t smem_u = smem_u32(smem) >> 4, stage_u = stage_bytes >> 4;
      int s = 0;
      uint32_t ph = 0;
      int nseg = 0;
      bool ok = true;
      long long t_wait = 0, t_begin = prof ? clock64() : 0;
      while (ok && wseg_next(P, kblocks, it, sg)) {
        const WGroup& G = P.grp[sg.g];
        // row of the shifted box that pairs with dense row 16*j (dense rows are (d, h, w) over the K-block box)
        uint32_t rowmap[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 16 * j;
          const int kw_ = k % P.bw, kh_ = (k / P.bw) % P.bh, kd_ = k / (P.bw * P.bh);
          rowmap[j] = (uint32_t)(kd_ * G.pitch_h + kh_ * G.pitch_w + kw_);
        }
        if (nseg > 0) {                                   // the epilogue must have drained the previous item
          if (!mbar_wait(acc_empty, (uint32_t)(nseg - 1) & 1u, P.err, 15)) { ok = false; break; }
          tc_fence_after();
        }
        // Per-segment table of the MMAs of one K-block: everything that does not depend on the stage is folded
        // into constants (descriptor offsets in 16-byte units), so the per-stage loop of this single issuing
        // thread is a wait, a handful of adds and the MMAs.
        // taps per MMA: unshared boxes sit back to back (chunk stride = box size); the taps of a d-chain (share > 2,
        // one chunk each) are the SAME box entered 16*n rows later, i.e. "chunks" with a stride of one plane: up to four
        // of them form one N = 256 MMA (N = 64 MMAs run at 59 % of the tensor-pipe rate)
        const bool chain = G.share > 2 && P.ncc == 1 && sg.ntap > 1;
        const uint32_t chain_lbo = chain ? (uint32_t)(P.rshift[sg.tap0 + 1] - P.rshift[sg.tap0]) * 128u : 0u;
        const int tpm = G.share == 1 ? (P.ncc >= 4 ? 1 : 4 / P.ncc) : (chain ? 4 : 1);
        uint32_t m_boff[8], m_dcol[8], m_idesc[8];
        const int nmma = (sg.ntap + tpm - 1) / tpm;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int g = i * tpm;
          const int nt = max(1, min(tpm, sg.ntap - g));
          const int gi = min(g, sg.ntap - 1);
          m_boff[i] = (m_bytes + (uint32_t)(gi / G.share) * set_bytes + (uint32_t)P.rshift[sg.tap0 + gi] * 128u) >> 4;
          m_dcol[i] = (uint32_t)(gi * P.ncc * 64);
          m_idesc[i] = make_idesc(nt * P.ncc * 64, 1, 1, 128 * kCtas);
        }
        const uint64_t a_desc0 = desc_mnmajor_sw128(0, kChunkBytes);
        const uint64_t b_desc0 = desc_mnmajor_sw128(0, chain ? chain_lbo : (uint32_t)P.box_bytes);
        const uint32_t rm0 = rowmap[0] * 8u, rm1 = rowmap[1] * 8u, rm2 = rowmap[2] * 8u, rm3 = rowmap[3] * 8u;
        for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
          const long long tw0 = prof ? clock64() : 0;
          if (!mbar_wait(&full_bar[s], ph, P.err, 12)) { ok = false; break; }
          if (prof) t_wait += clock64() - tw0;
          tc_fence_after();
          const uint32_t sa_u = smem_u + (uint32_t)s * stage_u;
          const uint64_t ad = a_desc0 | (uint64_t)(sa_u & 0x3FFFu);
          const uint32_t accf = (uint32_t)(kb != sg.kb0);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (i >= nmma) break;
            const uint32_t d_tmem = tmem_base + m_dcol[i];
            const uint32_t bu = sa_u + m_boff[i];
            const uint32_t id = m_idesc[i];
            umma_f16_g<kPair>(d_tmem, ad, b_desc0 | (uint64_t)((bu + rm0) & 0x3FFFu), id, accf);
            umma_f16_g<kPair>(d_tmem, ad + 128, b_desc0 | (uint64_t)((bu + rm1) & 0x3FFFu), id, 1u);
            umma_f16_g<kPair>(d_tmem, ad + 256, b_desc0 | (uint64_t)((bu + rm2) & 0x3FFFu), id, 1u);
            umma_f16_g<kPair>(d_tmem, ad + 384, b_desc0 | (uint64_t)((bu + rm3) & 0x3FFFu), id, 1u);
          }
          umma_commit_g<kPair>(&empty_bar[s]);
          if (++s == P.stages) { s = 0; ph ^= 1u; }
        }
        if (ok) umma_commit_g<kPair>(acc_full);
        ++nseg;
      }
      if (prof) {
        atomicAdd(P.dbg + 2, (unsigned long long)t_wait); atomicAdd(P.dbg + 3, (unsigned long long)(clock64() - t_begin));
        atomicAdd(P.dbg + 5, 1ull);
      }
    }
  } else {
    const int q = warp & 3;
    const int ml = q * 32 + lane;
    WSegIter it; WSeg sg;
    wseg_begin(P, kblocks, it, unit, nunits);
    int nseg = 0;
    long long t_epi = 0;
    const int ncols = P.ncc * 64;
    while (wseg_next(P, kblocks, it, sg)) {
      if (!mbar_wait(acc_full, (uint32_t)nseg & 1u, P.err, 13)) break;
      tc_fence_after();
      const long long te0 = prof ? clock64() : 0;
      const int m = (kPair ? 2 * sg.mt + rank : sg.mt) * 128 + ml;
      const int n0 = sg.nt * ncols;
      const bool valid = ml < 64 * P.m_chunks && m < P.Km && !(P.debug & 1);
      float* slot = nullptr;                               // a piece of a shared item: its partial tile, row ml
      if (sg.kb0 > 0 || sg.kb1 < kblocks)
        slot = P.part + (((long long)blockIdx.x * 2 + (sg.kb1 < kblocks ? 1 : 0)) * 128 + ml) * P.part_cols;
      for (int g = 0; g < sg.ntap; ++g) {
        float* obase = P.dw + (long long)P.twi[sg.tap0 + g] * P.tap_stride + (long long)m * P.m_stride;
        for (int c0 = 0; c0 < ncols; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * ncols + c0), r);
          tmem_wait_ld();
          if (slot && P.n_stride != 1) {
            float4* o = reinterpret_cast<float4*>(slot + g * ncols + c0);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              o[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                 __uint_as_float(r[4 * j + 3]));
            continue;
          }
          if (P.n_stride == 1) {
            // A thread owns accumulator ROW ml and 32 consecutive columns = 128 B of one dw row; its neighbours' rows are
            // m_stride floats away, so a red.v4 straight from the registers touched 32 half-used sectors per warp
            // instruction (tools/red_probe.cu: 2.1 TB/s device-wide against 3.9 TB/s for contiguous lanes, and the flush
            // is the tail of every wgrad launch: nothing overlaps it).  The 32 x 32 block is therefore transposed
            // through 4 KB of shared memory per warp (16-byte pieces, XOR-swizzled by the row: conflict-free both ways)
            // and leaves as 8 instructions that each cover four whole 128-byte lines.
            float4* stg = reinterpret_cast<float4*>(flush_stage) + q * 256;
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              stg[lane * 8 + (j ^ (lane & 7))] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                             __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
            __syncwarp();
            const int ch = lane & 7;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int row = i * 4 + (lane >> 3);                     // row of this warp's 32-row quadrant
              const int mr = q * 32 + row;
              const float4 v = stg[row * 8 + (ch ^ (row & 7))];
              if (slot) {                                              // a piece of a shared item: its partial tile
                *reinterpret_cast<float4*>(slot + (long long)(mr - ml) * P.part_cols + g * ncols + c0 + ch * 4) = v;
              } else if (mr < 64 * P.m_chunks && m - ml + mr < P.Km && !(P.debug & 1)) {
                float* o = obase + (long long)(mr - ml) * P.m_stride + n0 + c0 + ch * 4;
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                             : "memory");
              }
            }
          } else if (!valid) {
            continue;
          } else {
            // fully unrolled: with a partial unroll r[] is indexed at run time, which puts the whole chunk into LOCAL memory --
            // eight STL.128 per chunk and thread ahead of the branch, i.e. also on the n_stride == 1 path above
#pragma unroll
            for (int j = 0; j < 32; ++j)
              asm volatile("red.global.add.f32 [%0], %1;" ::"l"(obase + (long long)(n0 + c0 + j) * P.n_stride),
                           "f"(__uint_as_float(r[j]))
                           : "memory");
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if constexpr (kPair) mbar_arrive_leader(acc_empty); else mbar_arrive(acc_empty); }   // accumulators are free
      if (prof) t_epi += clock64() - te0;
      ++nseg;
    }
    if (prof && threadIdx.x == 64) atomicAdd(P.dbg + 4, (unsigned long long)t_epi);
  }
  tc_fence_before();
  if constexpr (kPair) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    if constexpr (kPair)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(P.tmem_cols) : "memory");
    else
      tmem_dealloc(tmem_base, P.tmem_cols);
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// channels-last bf16 activation [N][D][H][W][C] -> 5-D map (C, W, H, D, N), box (64, bw*s, bh*s, bd*s, 1)
inline int make_act_map(CUtensorMap* tm, const void* base, int N, int D, int H, int W, int C, int bw, int bh, int bd,
                        int step) {
  EncodeTiledFn fn = get_encode_fn();
  MRA_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
  cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2,
                           (cuuint64_t)D * H * W * C * 2};
  cuuint32_t box[5] = {64, (cuuint32_t)(bw * step), (cuuint32_t)(bh * step), (cuuint32_t)(bd * step), 1};
  cuuint32_t es[5] = {1, (cuuint32_t)step, (cuuint32_t)step, (cuuint32_t)step, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MRA_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(activation) failed: %d (dims %d %d %d %d %d box %d %d %d step %d)",
              (int)r, C, W, H, D, N, bw, bh, bd, step);
  return 0;
}
// packed weights [rows][Ck] bf16 -> 2-D map, box (64, box_rows)
inline int make_weight_map(CUtensorMap* tm, const void* base, long long rows, int Ck, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  MRA_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)Ck, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)Ck * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MRA_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
  return 0;
}

inline uint32_t pow2_cols(int n) { uint32_t c = 32; while ((int)c < n) c <<= 1; return c; }
constexpr size_t kSmemLimit = 227 * 1024;

// device-side error flag shared by all TC launches (checked lazily by mra_tc_error_check)
inline int* tc_err_flag() {
  static int* flag = nullptr;
  if (!flag) {
    if (cudaMalloc(&flag, sizeof(int)) != cudaSuccess) return nullptr;
    cudaMemset(flag, 0, sizeof(int));
  }
  return flag;
}

// device-side cycle counters for pipeline diagnosis (filled only when a kernel runs with a debug bit set):
// [0] producer cycles waiting for a free stage, [1] producer total, [2] MMA cycles waiting for data,
// [3] MMA total, [4] epilogue cycles, [5] CTAs counted
inline unsigned long long* tc_dbg_counters() {
  static unsigned long long* buf = nullptr;
  if (!buf) {
    if (cudaMalloc(&buf, 8 * sizeof(unsigned long long)) != cudaSuccess) return nullptr;
    cudaMemset(buf, 0, 8 * sizeof(unsigned long long));
  }
  return buf;
}

inline int pick_n_tile(int cn) {
  if (cn % 256 == 0) return 256;
  if (cn % 128 == 0) return 128;
  if (cn % 64 == 0) return 64;
  return 0;
}

inline bool gather_eligible(const mra_conv_desc& d, int which) {
  if (d.dtype != MRA_BF16 || (d.flags & MRA_CONV_FORCE_NAIVE)) return false;
  const int ck = which == 0 ? d.cin : d.cout, cn = which == 0 ? d.cout : d.cin;
  if (ck % 64 != 0 || pick_n_tile(cn) == 0) return false;
  if (d.k * d.k * d.k > kMaxTaps) return false;
  if (d.stride != 1 && d.stride != 2) return false;
  return true;
}
inline bool wgrad_eligible(const mra_conv_desc& d) {
  if (d.dtype != MRA_BF16 || (d.flags & MRA_CONV_FORCE_NAIVE)) return false;
  if (d.cout % 64 != 0 || d.cin % 64 != 0) return false;
  if (d.k * d.k * d.k > kMaxTaps) return false;
  if (d.stride != 1 && d.stride != 2) return false;
  return true;
}

struct GatherRun {
  const void* a;        // activations (bf16, channels-last)
  const void* b;        // packed weights [slabs][cn][ck] (bf16)
  int slabs;            // number of weight slabs addressed by tap.widx
  const float* bias;
  void* out;
  int out_bf16;         // 1: bf16 output, 0: fp32 output
  int act;
  float slope;
  double* stats;
  const void* aux = nullptr;   // with stats: norm-backward statistics against this tensor (EpiArgs::aux)
  float aux_nslope = 0.f;
};

// Can the launches of a plan run as ONE merged launch?  8 parity phases over the same launch space (the stride-2
// dgrad-form plans of conv_plan.h), unit A step, one tile box, <= kMaxTaps taps in total.
inline bool gather_mergeable(const GatherPlan& plan) {
  if (plan.launches.size() != 8 || getenv("MRA_GATHER_NOMERGE")) return false;
  const GatherLaunch& L0 = plan.launches[0];
  size_t taps = 0;
  for (const GatherLaunch& L : plan.launches) {
    if (L.astep != 1 || L.ostep != L0.ostep) return false;
    for (int i = 0; i < 3; ++i)
      if (L.dims[i] != L0.dims[i] || L.box[i] != L0.box[i] || L.o0[i] < -128 || L.o0[i] > 127) return false;
    taps += L.taps.size();
  }
  return taps <= (size_t)kMaxTaps;
}

// One launch of gather_tc_kernel (one TMA box per filter tap): a single GatherLaunch of the plan, or all 8 parity
// phases merged (`nl` = 8 consecutive launches starting at `Ls`); with 64 output channels the merged phases are
// paired along w (see GatherP::pair).
struct PairEntry { int dd, dh, dw, w1, w2; };
inline bool build_phase_pairs(const GatherLaunch* Ls, int slabs, std::vector<std::vector<PairEntry>>& items, int (*o0)[3]) {
  bool used[8] = {false, false, false, false, false, false, false, false};
  items.clear();
  for (int a = 0; a < 8; ++a) {
    if (used[a]) continue;
    int b = -1;
    for (int c = 0; c < 8; ++c)
      if (c != a && !used[c] && Ls[c].o0[0] == Ls[a].o0[0] && Ls[c].o0[1] == Ls[a].o0[1] && abs(Ls[c].o0[2] - Ls[a].o0[2]) == 1) b = c;
    if (b < 0) return false;
    int lo = Ls[a].o0[2] < Ls[b].o0[2] ? a : b, hi = lo == a ? b : a;
    used[a] = used[b] = true;
    std::vector<PairEntry> both, only1, only2;
    for (const Tap& t : Ls[lo].taps) {
      if (t.widx >= slabs) return false;
      int w2 = -1;
      for (const Tap& u : Ls[hi].taps) if (u.dd == t.dd && u.dh == t.dh && u.dw == t.dw) w2 = u.widx;
      (w2 >= 0 ? both : only1).push_back(PairEntry{t.dd, t.dh, t.dw, t.widx, w2});
    }
    for (const Tap& u : Ls[hi].taps) {
      if (u.widx >= slabs) return false;
      bool shared = false;
      for (const Tap& t : Ls[lo].taps) if (u.dd == t.dd && u.dh == t.dh && u.dw == t.dw) shared = true;
      if (!shared) only2.push_back(PairEntry{u.dd, u.dh, u.dw, -1, u.widx});
    }
    std::vector<PairEntry> e = both;                    // N = 128 entries first: they initialise both halves at once
    e.insert(e.end(), only1.begin(), only1.end());
    e.insert(e.end(), only2.begin(), only2.end());
    const int idx = (int)items.size();
    for (int i = 0; i < 3; ++i) o0[idx][i] = Ls[lo].o0[i];
    items.push_back(e);
  }
  return items.size() == 4;
}

inline int run_gather_v1_launch(const GatherPlan& plan, const GatherLaunch* Ls, int nl, const GatherRun& R, const CUtensorMap& tmB,
                                int n_tile, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    MRA_CHECK_CUDA(cudaFuncSetAttribute(gather_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute(gather_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute(gather_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    attr_set = true;
  }
  const GatherLaunch& L = Ls[0];
  MRA_REQUIRE(nl == 1 || nl == 8, "gather launch: 1 or 8 phases");
  GatherP P;
  memset(&P, 0, sizeof(P));
  std::vector<std::vector<PairEntry>> pairs;
  int pair_o0[4][3];
  if (nl == 8 && n_tile == 64 && plan.cn == 64 && getenv("MRA_GATHER_NOPAIR") == nullptr && build_phase_pairs(Ls, R.slabs, pairs, pair_o0)) {
    size_t ne = 0;
    for (const auto& e : pairs) ne += e.size();
    P.pair = ne <= (size_t)kMaxTaps ? 1 : 0;
  }
  const int items = P.pair ? 4 : nl;
  P.bd = L.box[0]; P.bh = L.box[1]; P.bw = L.box[2];
  P.Dl = L.dims[0]; P.Hl = L.dims[1]; P.Wl = L.dims[2];
  P.tilesD = (P.Dl + P.bd - 1) / P.bd; P.tilesH = (P.Hl + P.bh - 1) / P.bh; P.tilesW = (P.Wl + P.bw - 1) / P.bw;
  P.astep = L.astep;
  P.Cn = plan.cn; P.n_tile = n_tile; P.n_tiles = plan.cn / n_tile; P.kchunks = plan.ck / 64;
  const long long total_tiles = (long long)plan.n * P.tilesD * P.tilesH * P.tilesW * P.n_tiles * items;
  MRA_REQUIRE(total_tiles < (1ll << 31), "too many tiles");
  P.total_tiles = (int)total_tiles;
  P.ostep = L.ostep; P.od0 = L.o0[0]; P.oh0 = L.o0[1]; P.ow0 = L.o0[2];
  P.osw = plan.cn;
  P.osh = (long long)plan.odims[2] * P.osw;
  P.osd = (long long)plan.odims[1] * P.osh;
  P.osn = (long long)plan.odims[0] * P.osd;
  P.out = R.out; P.out_bf16 = R.out_bf16;
  P.bias = R.bias; P.act = R.act; P.slope = R.slope;
  P.stats = R.stats; P.aux = R.aux; P.aux_nslope = R.aux_nslope; P.err = tc_err_flag();
  { const char* e = getenv("MRA_GATHER_DEBUG"); P.debug = e ? atoi(e) : 0; }
  P.dbg = tc_dbg_counters();
  P.nph = items;
  int nt = 0;
  if (P.pair) {
    for (int p = 0; p < 4; ++p) {
      P.ph_tap0[p] = (int16_t)nt;
      P.ph_od[p] = (int8_t)pair_o0[p][0]; P.ph_oh[p] = (int8_t)pair_o0[p][1]; P.ph_ow[p] = (int8_t)pair_o0[p][2];
      bool init1 = false, init2 = false;
      for (const PairEntry& e : pairs[p]) {
        MRA_REQUIRE(e.dd >= -128 && e.dd < 128, "tap out of range");
        P.tdd[nt] = (int8_t)e.dd; P.tdh[nt] = (int8_t)e.dh; P.tdw[nt] = (int8_t)e.dw;
        P.twi[nt] = (int16_t)e.w1; P.twi2[nt] = (int16_t)e.w2;
        if (e.w1 >= 0 && e.w2 >= 0) { MRA_REQUIRE(init1 == init2, "pair entry order"); P.eacc[nt] = init1 ? 1 : 0; init1 = init2 = true; }
        else if (e.w1 >= 0) { P.eacc[nt] = init1 ? 1 : 0; init1 = true; }
        else { P.eacc[nt] = init2 ? 1 : 0; init2 = true; }
        ++nt;
      }
      MRA_REQUIRE(init1 && init2, "pair item without taps for one phase");
    }
    P.ph_tap0[4] = (int16_t)nt;
  } else {
    for (int p = 0; p < nl; ++p) {
      const GatherLaunch& Lp = Ls[p];
      P.ph_tap0[p] = (int16_t)nt;
      P.ph_od[p] = (int8_t)Lp.o0[0]; P.ph_oh[p] = (int8_t)Lp.o0[1]; P.ph_ow[p] = (int8_t)Lp.o0[2];
      for (const Tap& t : Lp.taps) {
        MRA_REQUIRE(nt < kMaxTaps, "too many taps for the tensor-core path");
        MRA_REQUIRE(t.dd >= -128 && t.dd < 128 && t.widx < R.slabs, "tap out of range");
        P.tdd[nt] = (int8_t)t.dd; P.tdh[nt] = (int8_t)t.dh; P.tdw[nt] = (int8_t)t.dw;
        P.twi[nt] = (int16_t)t.widx; P.twi2[nt] = -1;
        ++nt;
      }
    }
    P.ph_tap0[nl] = (int16_t)nt;
  }
  P.ntaps = nt;
  const int acc_cols = P.pair ? 2 * n_tile : n_tile;
  const size_t stage_bytes = kABytes + (size_t)acc_cols * 128;
  int stages = (int)((kSmemLimit - 2048 - kEpiRedBytes) / stage_bytes);
  if (stages > 6) stages = 6;
  P.stages = stages;
  P.nbuf = 512 / acc_cols > 8 ? 8 : 512 / acc_cols;
  { const char* e = getenv("MRA_GATHER_NBUF"); if (e && atoi(e) >= 2 && atoi(e) <= P.nbuf) P.nbuf = atoi(e); }
  P.tmem_cols = pow2_cols(P.nbuf * acc_cols);
  const size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/;
  CUtensorMap tmA;
  if (int rc = make_act_map(&tmA, R.a, plan.n, plan.adims[0], plan.adims[1], plan.adims[2], plan.ck, P.bw, P.bh, P.bd,
                            P.astep))
    return rc;
  const int ctas = P.total_tiles < num_sms() ? P.total_tiles : num_sms();
  if (P.aux && P.stats) MRA_CHECK_CUDA(launch_pdl(gather_tc_kernel<2>, dim3(ctas), dim3(kThreadsGather), smem, st, 1, tmA, tmB, P));
  else if (P.stats) MRA_CHECK_CUDA(launch_pdl(gather_tc_kernel<1>, dim3(ctas), dim3(kThreadsGather), smem, st, 1, tmA, tmB, P));
  else MRA_CHECK_CUDA(launch_pdl(gather_tc_kernel<0>, dim3(ctas), dim3(kThreadsGather), smem, st, 1, tmA, tmB, P));
  MRA_LAUNCH_CHECK();
  return 0;
}

// Adds the pieces of every shared work item (blockIdx.x = work, blockIdx.y = slice of its elements) to dw in K order: the pieces are recomputed with the
// stream-K arithmetic of wseg_begin / wseg_next, so that each is read from the slot its CTA stored it in.
__global__ void __launch_bounds__(256) wgrad_fixup_kernel(const __grid_constant__ WgradP P, int nunits, int kctas) {
  __shared__ int cta[160], which[160];
  __shared__ int npieces;
  const int per_item = P.m_tiles * P.n_tiles;
  const int w = blockIdx.x;
  const int item = w / per_item, rem = w - item * per_item;
  const int g = wg_item_group(P, item);
  const WGroup& G = P.grp[g];
  const int ntap = wg_item_ntap(P, g, item);
  const long long kblocks = (long long)P.tilesW * P.tilesH * P.tilesD * P.N;
  if (threadIdx.x == 0) {
    const long long works_full = (long long)(G.ntaps / G.gpi) * per_item, wl = w - (long long)G.item0 * per_item;
    const long long W0 = G.cost0 + min(wl, works_full) * G.gpi * kblocks + max(wl - works_full, 0ll) * ntap * kblocks;
    const long long W1 = W0 + ntap * kblocks;
    const long long share = (P.total_cost + nunits - 1) / nunits;
    int n = 0;
    bool shared_item = false;
    for (long long u = W0 / share; u * share < W1 && u < nunits && n < 160; ++u) {
      const long long lo = max(W0, u * share), hi = min(W1, min((u + 1) * share, P.total_cost));
      const long long kb0 = (lo - W0) / ntap, kb1 = hi == W1 ? kblocks : (hi - W0) / ntap;
      if (kb1 <= kb0) continue;
      if (kb0 > 0 || kb1 < kblocks) shared_item = true;
      cta[n] = (int)u; which[n] = kb1 < kblocks ? 1 : 0; ++n;
    }
    npieces = shared_item ? n : 0;
  }
  __syncthreads();
  const int np = npieces;
  if (np == 0) return;
  const int mt = rem / P.n_tiles, nt = rem - mt * P.n_tiles;
  const int tap0 = G.tap0 + (item - G.item0) * G.gpi;
  const int ncols = P.ncc * 64, nq = ncols / 4;            // four columns per thread: 16-byte loads
  const int total = kctas * 128 * ntap * nq;
  for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < total; e += gridDim.y * blockDim.x) {
    const int c = (e % nq) * 4;
    int t = e / nq;
    const int gg = t % ntap; t /= ntap;
    const int ml = t % 128, rank = t / 128;
    const int m = (kctas * mt + rank) * 128 + ml;
    if (ml >= 64 * P.m_chunks || m >= P.Km) continue;
    const long long off = (long long)ml * P.part_cols + gg * ncols + c;
    const long long slot = 128ll * P.part_cols;
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int i = 0; i < np; ++i) {                           // K order: the loads may run ahead, the adds keep the order
      const float4 v = __ldcg(reinterpret_cast<const float4*>(P.part + ((long long)(cta[i] * kctas + rank) * 2 + which[i]) * slot + off));
      sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
    }
    float* o = P.dw + (long long)P.twi[tap0 + gg] * P.tap_stride + (long long)m * P.m_stride + (long long)(nt * ncols + c) * P.n_stride;
    if (P.n_stride == 1) {
      float4 d = *reinterpret_cast<float4*>(o);
      d.x += sum.x; d.y += sum.y; d.z += sum.z; d.w += sum.w;
      *reinterpret_cast<float4*>(o) = d;
    } else {
      o[0] += sum.x; o[P.n_stride] += sum.y; o[2 * P.n_stride] += sum.z; o[3 * P.n_stride] += sum.w;
    }
  }
}

// Tile geometry of a wgrad launch (K-block boxes, m / n tiles) and the CTA-pair decision; returns pair.
inline bool wgrad_fill_geometry(const WgradPlan& plan, WgradP& P) {
  const bool sw = plan.m_is_shifted != 0;
  const int Km = sw ? plan.cn : plan.cm, Kn = sw ? plan.cm : plan.cn;
  P.bd = plan.box[0]; P.bh = plan.box[1]; P.bw = plan.box[2];
  P.tilesD = (plan.qdims[0] + P.bd - 1) / P.bd; P.tilesH = (plan.qdims[1] + P.bh - 1) / P.bh;
  P.tilesW = (plan.qdims[2] + P.bw - 1) / P.bw;
  P.N = plan.n; P.sstep = plan.sstep;
  P.Km = Km; P.Kn = Kn;
  P.m_chunks = Km >= 128 ? 2 : 1;
  P.ncc = plan.ncc;
  // CTA pairs (cta_group::2): 256 dense channels per unit, each CTA loads half of the shifted chunks.  Needs whole
  // 256-channel m tiles and one tap per MMA (ncc == 4), and enough K-blocks to feed 74 pairs.
  long long pair_min = 64ll * 64 * 8;                       // K positions (MRA_WGRAD_PAIR_MIN: test hook)
  { const char* e = getenv("MRA_WGRAD_PAIR_MIN"); if (e) pair_min = atoll(e); }
  const bool pair = Km % 256 == 0 && plan.ncc == 4 && (num_sms() % 2) == 0 && getenv("MRA_WGRAD_NOPAIR") == nullptr &&
                    (long long)plan.qdims[0] * plan.qdims[1] * plan.qdims[2] * plan.n >= pair_min;
  P.m_tiles = pair ? Km / 256 : (Km + 127) / 128;
  P.n_tiles = Kn / (64 * P.ncc);
  return pair;
}
// The stream-K side of a wgrad launch: tap groups -> work items -> cost prefixes (needs P.m_tiles / P.n_tiles).  Kept apart
// from the tensor maps so that mra_debug_schedule can walk the schedule on the CPU with the code the kernel runs.
inline bool wgrad_fill_schedule(const WgradPlan& plan, long long kblocks, WgradP& P) {
  P.n_groups = (int)plan.launches.size();
  if (P.n_groups > kMaxWGroups) return false;
  int tapc = 0, itemc = 0;
  P.total_cost = 0;
  for (int gi = 0; gi < P.n_groups; ++gi) {
    const WgradLaunch& L = plan.launches[gi];
    WGroup& G = P.grp[gi];
    G.tap0 = tapc; G.ntaps = (int)L.taps.size();
    G.gpi = L.gpi; G.share = L.share;
    G.item0 = itemc; G.n_items = (G.ntaps + G.gpi - 1) / G.gpi;
    G.cost0 = P.total_cost;
    for (int it = 0; it < G.n_items; ++it) {
      const int nt = G.ntaps - it * G.gpi < G.gpi ? G.ntaps - it * G.gpi : G.gpi;
      P.total_cost += (long long)nt * kblocks * P.m_tiles * P.n_tiles;
    }
    tapc += G.ntaps; itemc += G.n_items;
  }
  P.n_items = itemc;
  return tapc <= kMaxTaps;
}
inline int run_wgrad_tc(const WgradPlan& plan, const void* x, const void* dy, float* dw, cudaStream_t st) {
  int* err = tc_err_flag();
  MRA_REQUIRE(plan.cm % 64 == 0 && plan.cn % 64 == 0 && (int)plan.taps.size() <= kMaxTaps,
              "shape not eligible for the tensor-core wgrad path");
  MRA_REQUIRE(!plan.launches.empty() && (int)plan.launches.size() <= kMaxWGroups, "wgrad plan: bad group count");
  static bool attr_set = false;
  if (!attr_set) {
    MRA_CHECK_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    MRA_CHECK_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit));
    attr_set = true;
  }
  // dense operand on the M side of the MMA, shifted operand on the N side
  const bool sw = plan.m_is_shifted != 0;                  // ConvTranspose3d: dense = x, shifted = dy
  const void* dense = sw ? x : dy;
  const void* shifted = sw ? dy : x;
  const int* ddims = sw ? plan.ndims : plan.mdims;
  const int* sdims = sw ? plan.mdims : plan.ndims;
  const int Km = sw ? plan.cn : plan.cm, Kn = sw ? plan.cm : plan.cn;
  CUtensorMap tmM;
  if (int rc = make_act_map(&tmM, dense, plan.n, ddims[0], ddims[1], ddims[2], Km, plan.box[2], plan.box[1], plan.box[0], 1))
    return rc;
  WMaps maps;
  memset(&maps, 0, sizeof(maps));
  WgradP P;
  memset(&P, 0, sizeof(P));
  const bool pair = wgrad_fill_geometry(plan, P);
  P.dw = dw; P.err = err;
  { const char* e = getenv("MRA_WGRAD_DEBUG"); P.debug = e ? atoi(e) : 0; }
  P.dbg = tc_dbg_counters();
  // dw memory is [taps][cm][cn] (cm = cout, cn = cin); kernel rows m index the dense operand's channels
  P.tap_stride = (long long)plan.cm * plan.cn;
  if (!sw) { P.m_stride = plan.cn; P.n_stride = 1; }
  else     { P.m_stride = 1; P.n_stride = plan.cn; }
  const long long kblocks = (long long)P.tilesW * P.tilesH * P.tilesD * plan.n;
  MRA_REQUIRE(wgrad_fill_schedule(plan, kblocks, P), "wgrad plan: too many taps or tap groups");
  int max_cols = 0;
  for (int gi = 0; gi < P.n_groups; ++gi) {
    const WgradLaunch& L = plan.launches[gi];
    WGroup& G = P.grp[gi];
    const int xd = P.bd + L.ext[0], xh = P.bh + L.ext[1], xw = P.bw + L.ext[2];
    const int tapc = G.tap0;
    G.pitch_w = xw; G.pitch_h = xh * xw;
    G.box_tx = xd * xh * xw * 128;
    const int slot = (G.box_tx + 1023) / 1024 * 1024;
    if (slot > P.box_bytes) P.box_bytes = slot;
    if (G.gpi / G.share > P.sets_max) P.sets_max = G.gpi / G.share;
    if (G.gpi * P.ncc * 64 > max_cols) max_cols = G.gpi * P.ncc * 64;
    for (int i = 0; i < G.ntaps; ++i) {
      const Tap& t = plan.taps[L.taps[i]];
      const Tap& o = L.origin[i];
      P.odd[tapc + i] = (int8_t)o.dd; P.odh[tapc + i] = (int8_t)o.dh; P.odw[tapc + i] = (int8_t)o.dw;
      const int r = ((t.dd - o.dd) * xh + (t.dh - o.dh)) * xw + (t.dw - o.dw);
      MRA_REQUIRE(r >= 0 && t.dd - o.dd <= L.ext[0] && t.dh - o.dh <= L.ext[1] && t.dw - o.dw <= L.ext[2],
                  "wgrad plan: tap outside its shared box");
      P.rshift[tapc + i] = (int16_t)r;
      P.twi[tapc + i] = (int16_t)t.widx;
    }
    if (int rc = make_act_map(&maps.m[gi], shifted, plan.n, sdims[0], sdims[1], sdims[2], Kn, xw, xh, xd, plan.sstep)) return rc;
  }
  const size_t stage_bytes = 2 * kChunkBytes + (size_t)P.sets_max * (P.ncc / (pair ? 2 : 1)) * P.box_bytes;
  int stages = (int)((kSmemLimit - 2048 - kWgradFlushBytes) / stage_bytes);
  MRA_REQUIRE(stages >= 2, "wgrad plan: stage does not fit shared memory");
  if (stages > 6) stages = 6;
  P.stages = stages;
  P.tmem_cols = pow2_cols(max_cols);
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 256 + kWgradFlushBytes;
  // one wave: a CTA per SM (fewer when there is less than ~4 K-blocks of work per CTA); pairs: one unit per two SMs
  long long ctas = pair ? (num_sms() & ~1) : num_sms();
  if (!pair && P.total_cost < ctas * 4) ctas = (P.total_cost + 3) / 4;
  if (ctas < 1) ctas = 1;
  const int kctas = pair ? 2 : 1, nunits = (int)(ctas / kctas);
  MRA_REQUIRE(nunits <= 160, "wgrad: more stream-K units than the fixup kernel tracks");
  bool shared_items = false;                         // does any work item span more than one unit?
  for (int u = 0; u < nunits && !shared_items; ++u) {
    WSegIter it; WSeg sg;
    wseg_begin(P, kblocks, it, u, nunits);
    while (wseg_next(P, kblocks, it, sg))
      if (sg.kb0 > 0 || sg.kb1 < kblocks) { shared_items = true; break; }
  }
  P.part_cols = max_cols;
  if (shared_items)                                  // stream-ordered: capture-safe, freed after the fixup
    MRA_CHECK_CUDA(cudaMallocAsync((void**)&P.part, (size_t)ctas * 2 * 128 * max_cols * sizeof(float), st));
  if (pair) MRA_CHECK_CUDA(launch_pdl(wgrad_tc_kernel<true>, dim3((unsigned)ctas), dim3(kThreads), smem, st, 2, tmM, maps, P));
  else MRA_CHECK_CUDA(launch_pdl(wgrad_tc_kernel<false>, dim3((unsigned)ctas), dim3(kThreads), smem, st, 1, tmM, maps, P));
  MRA_LAUNCH_CHECK();
  if (!shared_items) return 0;
  // an item's elements are spread over many blocks: a few items may each hold up to one piece per unit
  const unsigned slices = (unsigned)max(1ll, min(256ll, ((long long)kctas * 128 * max_cols / 4 + 255) / 256));
  wgrad_fixup_kernel<<<dim3((unsigned)(P.n_items * P.m_tiles * P.n_tiles), slices), 256, 0, st>>>(P, nunits, kctas);
  MRA_LAUNCH_CHECK();
  MRA_CHECK_CUDA(cudaFreeAsync(P.part, st));
  return 0;
}
inline int run_wgrad_tc(const mra_conv_desc& d, const void* x, const void* dy, float* dw, cudaStream_t st) {
  WgradPlan plan;
  MRA_REQUIRE(build_wgrad_plan(d, plan), "unsupported conv geometry");
  return run_wgrad_tc(plan, x, dy, dw, st);
}

}  // namespace tc
}  // namespace mra
