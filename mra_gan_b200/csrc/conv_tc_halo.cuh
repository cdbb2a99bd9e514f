// Halo-plane implicit-GEMM gather kernel (stride-1 launches of conv_plan.h's GATHER computation).
//
// gather_tc_kernel (conv_tc.cuh) loads one 128-row A tile per filter tap: 27 loads of nearly the same
// input voxels for a 3x3x3 filter.  A convolution can do better than a GEMM here: all (kh, kw) taps of one
// input d-plane read shifted windows of ONE halo tile.  This kernel keeps that halo tile (a "plane": the
// (Hb x Wb) input rows under a 128-position output tile, 64 channels wide) in shared memory and feeds every
// tap from it by moving the UMMA descriptor's start address (row shift) -- the SWIZZLE_128B pattern is a
// function of the absolute shared-memory address, so row-shifted starts and a non-1024-byte group stride
// are legal (verified on B200 by tools/halo_probe.cu).  A traffic drops by ~kh*kw/1.4 (k3: 6.4x); only the
// weights (B) are still streamed per tap.
//
// Output tile (M = 128 positions of one launch-space d-plane) in one of two shapes:
//   2D   : 16 h x 8 w.  MMA row m = (h, w) = (m / 8, m % 8); the 8-row groups are Wb = 8 + kw - 1 plane rows
//          apart (descriptor SBO = Wb * 128 B).  No wasted rows when H % 16 == 0 and W % 8 == 0.
//   flat : 128 consecutive positions f of the plane flattened with pitch Wb = W + kw - 1 (SBO = 1024 B as in a
//          dense tile); the kw - 1 positions per line that wrap around are computed and discarded.  Used when
//          the 2D shape would waste more (e.g. the 34^3 dgrad of the residual blocks: 90 % vs 60 % useful rows).
//
// Warp roles: 0..7 = epilogue (two per TMEM lane quadrant, alternate 32-column chunks), 8 = TMA producer of the weight
// ring, 9 = TMA producer of the plane ring, 10 = TMEM allocator + MMA issuer (highest warp id: scheduler priority).  Persistent over tiles, accumulators double-buffered in TMEM.
#pragma once
#include "conv_tc.cuh"
#include "conv_tc_col.cuh"

namespace mra {
namespace tc {

constexpr int kHaloPlaneWarp = kEpiWarps + 1;
constexpr int kHaloMmaWarp = kEpiWarps + 2;
constexpr int kThreadsHalo = 32 * 12;             // 3 whole warpgroups (setmaxnreg is per warpgroup); warp 11 idles

struct HaloP {
  int Dl, Hl, Wl;                   // launch-space (output) dims
  int N;
  int mode;                         // 0 = 2D tile (16 x 8), 1 = flat
  int tiles_hw, tiles_w;            // tiles per d-plane; 2D: tiles along w
  int Wb, Hb;                       // plane box extents in w / h (rows = Wb * Hb)
  int sbo;                          // descriptor stride between 8-row groups, bytes
  int slot_bytes, plane_tx;         // shared-memory slot / bytes delivered per plane
  int NP, NB;                       // plane ring / weight ring depth
  int kd, kh, kw;                   // tap box extents (taps ordered td, th, tw)
  int dmin, hmin, wmin;             // smallest tap offsets
  int Cn, n_tile, n_tiles, kchunks;
  int total_tiles;                  // full-width work items
  int split_from, total_work;       // work items >= split_from are HALF-width (n_tile / 2): two per tile, so that the
                                    // last, partial round of the persistent schedule costs half a round
  int ostep, od0, oh0, ow0;
  long long osn, osd, osh, osw;     // output strides in elements
  void* out;
  int out_bf16;
  const float* bias;
  int act;
  float slope;
  double* stats;
  const void* aux; float aux_nslope;   // norm-backward statistics (EpiArgs::aux)
  int* err;
  uint32_t tmem_cols;
  int16_t twi[kMaxTaps];            // weight slab of tap (td, th, tw)
  int debug;
  unsigned long long* dbg;
  int pair;                         // 1: cta_group::2 pairs (host-side choice of the kernel instantiation)
  int nsub;                         // position tiles per work item: 1, or 2 = DUAL items (two tiles of one plane, neighbours in
                                    // the tile order, share every weight slab; n_tile = 128, the two accumulators side by side)
  int Da;                           // d extent of the A tensor
  int skip;                         // 1: input planes that lie outside A for every tile of a work item are not loaded and
                                    // their MMAs not issued (halo_plane_live); host-checked: every item keeps >= 1 plane
  int b_tx_dbg;                     // timing experiments: bytes per weight box when the box was shrunk (debug bit 5)
};

__device__ __forceinline__ uint64_t desc_kmajor_sw128_sbo(uint32_t saddr, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) |
         (2ull << 61);
}

struct HaloTile { int n, d, d0, n0, h0, w0, f0, hs, roff, width; int rot_kc0, rot_td0, rot_th0, rot_tw0, rot_t; };
// work index -> coordinates.  Order: n_tile fastest, then the tiles of a plane, then d (pair mode: pairs of
// planes, CTA rank r takes d = 2 * dp + r so both tiles share the weight slab and the in-plane geometry), then n.
__host__ __device__ __forceinline__ HaloTile halo_decode(const HaloP& P, int work, int pair, int rank, int sub = 0) {
  HaloTile t;
  int tile = work, half = 0;
  t.width = P.n_tile;
  if (work >= P.split_from) {
    const int k = work - P.split_from;
    tile = P.split_from + (k >> 1); half = k & 1; t.width = P.n_tile >> 1;
  }
  const int nt = tile % P.n_tiles; tile /= P.n_tiles;
  const int items_hw = P.tiles_hw / P.nsub;       // (dual items: tiles_hw is even)
  const int j0 = (tile % items_hw) * P.nsub;      // first tile of the item: the rotation key, the same for both tiles
  const int j = j0 + sub;
  tile /= items_hw;
  const int dsteps = pair ? (P.Dl + 1) / 2 : P.Dl;
  const int dq = tile % dsteps;
  t.d = pair ? 2 * dq + rank : dq;            // may be == Dl for the odd plane's partner: loads hit zero fill, nothing is stored
  t.d0 = pair ? 2 * dq : dq;                  // the work item's first plane (the same for both CTAs of a pair)
  t.n = tile / dsteps;
  // The (channel chunk, td) planes and the (th, tw) taps of a plane are walked in a ROTATED order (the sum over taps is
  // order-free): CTAs that run side by side work on consecutive tiles, so at any moment the SMs stream different weight
  // slabs instead of all 148 hammering the same 32 KB of L2.  The rotation is a function of the tile's position INSIDE
  // ITS SAMPLE -- not of the CTA that happens to run it -- so the fp32 accumulation order of an output element, and with
  // it every bit of a sample's result, is independent of the batch size and of how the schedule deals tiles to CTAs.
  {
    const int key = dq * P.tiles_hw + j0;
    const int nplanes = P.kchunks * P.kd, taps_hw = P.kh * P.kw;
    const int rot_p = key % nplanes;
    t.rot_t = (key / nplanes) % taps_hw;
    t.rot_kc0 = rot_p / P.kd; t.rot_td0 = rot_p - t.rot_kc0 * P.kd;
    t.rot_th0 = t.rot_t / P.kw; t.rot_tw0 = t.rot_t - t.rot_th0 * P.kw;
  }
  t.n0 = nt * P.n_tile + half * t.width;
  if (P.mode == 0) {
    t.h0 = (j / P.tiles_w) * 16; t.w0 = (j % P.tiles_w) * 8;
    t.f0 = 0; t.hs = t.h0; t.roff = 0;
  } else {
    t.f0 = j * 128; t.hs = t.f0 / P.Wb; t.roff = t.f0 - t.hs * P.Wb;
    t.h0 = 0; t.w0 = 0;
  }
  return t;
}

// Statistics are kept per TILE (channel base tb = nt * n_tile), indexed by the chunk's position inside the full tile: a
// half-width tail item (t.n0 = tb or tb + n_tile / 2) adds into chunks coff .. coff + width / 32 - 1 of the same partials
// as the full-width tiles of that (sample, tile) before it, and a flush covers exactly the tile's n_tile channels
// [tb, tb + n_tile) -- never past Cn.  (Host-callable: mra_debug_schedule walks the same code on the CPU.)
__host__ __device__ __forceinline__ void halo_stats_key(const HaloP& P, const HaloTile& t, int& tb, int& coff) {
  tb = t.n0 - (t.n0 % P.n_tile);
  coff = (t.n0 - tb) >> 5;            // even (n_tile >= 128 when items are split), keeps the warps' chunk parity
}

// Does input plane td of the work item whose first output plane is d0 touch the A tensor at all?  A dgrad computes the
// gradient of the PADDED input (34^3 outputs from a 32^3 gradient for the residual blocks): the outermost output planes
// see kd - 1 (or, for the second and second-to-last, kd - 2) input planes that are pure zero fill.  Such a plane is
// skipped by all three roles -- no plane load, no weight slabs, no MMAs -- when it is dead for EVERY tile of the item
// (both planes of a CTA pair): 2 of the 51 (pair, td) steps of the G.rb dgrad, 6 of 102 without pairs.
__host__ __device__ __forceinline__ bool halo_plane_live(const HaloP& P, int d0, int td, int pair) {
  if (!P.skip) return true;
  const int a0 = d0 + P.dmin + td;
  return pair ? (a0 + 1 >= 0 && a0 < P.Da) : (a0 >= 0 && a0 < P.Da);
}

template <bool kPair, int kMode>
__global__ void __launch_bounds__(kThreadsHalo, 1)
gather_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ HaloP P) {
  pdl_launch_dependents();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kCtas = kPair ? 2 : 1;
  const uint32_t b_rows = (uint32_t)P.n_tile / kCtas;            // weight rows this CTA holds (pair: half the slab)
  const uint32_t b_bytes = b_rows * 128u;
  uint8_t* planes = smem;
  uint8_t* bring = smem + (size_t)P.NP * P.slot_bytes;
  uint64_t* p_full = reinterpret_cast<uint64_t*>(bring + (size_t)P.NB * b_bytes);
  uint64_t* p_empty = p_full + P.NP;
  uint64_t* b_full = p_empty + P.NP;
  uint64_t* b_empty = b_full + P.NB;
  uint64_t* acc_full = b_empty + P.NB;           // [2]
  uint64_t* acc_empty = acc_full + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  __shared__ EpiRed epi_red;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = kPair ? (int)cluster_ctarank() : 0;
  const bool leader = rank == 0;
  const int work0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int wstride = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int taps_hw = P.kh * P.kw;
  const bool prof = (P.debug & 2) != 0;
  const int nplanes = P.kchunks * P.kd;        // walked in a per-tile rotated order: HaloTile::rot_* (halo_decode)

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < P.NP; ++s) { mbar_init(&p_full[s], 1); mbar_init(&p_empty[s], 1); }
    for (int s = 0; s < P.NB; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], kEpiWarps * kCtas); }
    fence_barrier_init();
  }
  if (warp == kHaloMmaWarp) {
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

  const bool dbg_nob = (P.debug & 4) != 0, dbg_nop = (P.debug & 8) != 0;     // timing experiments: no weight / plane traffic
  if (warp >= kEpiWarps) {            // third warpgroup: producers, MMA issuer, idle warps -- one setmaxnreg for all of it
  regs_other();
  if (warp == kHaloPlaneWarp) {
    // ---- plane producer: one halo plane per (work item, channel chunk, td); each CTA loads its own tile's planes
    if (elect_one() && !dbg_nop) {
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      for (int w = work0; w < P.total_work && ok; w += wstride) {
        const HaloTile t = halo_decode(P, w, kPair, rank);
        const HaloTile t1 = halo_decode(P, w, kPair, rank, P.nsub - 1);      // dual items: the second tile (else == t)
        int kc = t.rot_kc0, td = t.rot_td0;
        for (int pi = 0; pi < nplanes && ok; ++pi) {
          if (halo_plane_live(P, t.d0, td, kPair)) {
            for (int sub = 0; sub < P.nsub; ++sub) {                         // one ring slot per tile of the item
              const HaloTile& ts = sub ? t1 : t;
              if (!mbar_wait(&p_empty[s], ph ^ 1u, P.err, 21)) { ok = false; break; }
              if (leader) mbar_expect_tx(&p_full[s], (uint32_t)P.plane_tx * kCtas);
              tma_load_5d_g<kPair>(planes + (size_t)s * P.slot_bytes, &tmA, &p_full[s], kc * 64, ts.w0 + P.wmin, ts.hs + P.hmin,
                                   ts.d + P.dmin + td, ts.n);
              if (++s == P.NP) { s = 0; ph ^= 1u; }
            }
          }
          if (++td == P.kd) { td = 0; if (++kc == P.kchunks) kc = 0; }
        }
      }
    }
  } else if (warp == kProdWarp) {
    // ---- weight producer: one (64 x n_tile) slab per (work item, channel chunk, tap); pair: each CTA its half
    if (elect_one() && !dbg_nob) {
      int s = 0;
      uint32_t ph = 0;
      bool ok = true;
      long long t_wait = 0, t_begin = prof ? clock64() : 0;
      for (int w = work0; w < P.total_work && ok; w += wstride) {
        const HaloTile t = halo_decode(P, w, kPair, 0);
        const int n0 = t.n0 + rank * (t.width / kCtas);      // half-width items use the first rows of the (full-size) box
        int kc = t.rot_kc0, td = t.rot_td0;
        for (int pi = 0; pi < nplanes && ok; ++pi) {
          int tap = t.rot_t;                                 // (th, tw) index inside the plane, rotated start
          const int ntap_p = halo_plane_live(P, t.d0, td, kPair) ? taps_hw : 0;
          for (int i = 0; i < ntap_p; ++i) {
            const long long tw0 = prof ? clock64() : 0;
            if (!((P.debug & 64) ? mbar_wait_poll(&b_empty[s], ph ^ 1u, P.err, 22) : mbar_wait(&b_empty[s], ph ^ 1u, P.err, 22))) { ok = false; break; }
            if (prof) t_wait += clock64() - tw0;
            if (leader) mbar_expect_tx(&b_full[s], (P.b_tx_dbg ? (uint32_t)P.b_tx_dbg : b_bytes) * kCtas);
            tma_load_2d_g<kPair>(bring + (size_t)s * b_bytes, &tmB, &b_full[s], kc * 64,
                                 (int)P.twi[td * taps_hw + tap] * P.Cn + n0);
            if (++s == P.NB) { s = 0; ph ^= 1u; }
            if (++tap == taps_hw) tap = 0;
          }
          if (++td == P.kd) { td = 0; if (++kc == P.kchunks) kc = 0; }
        }
      }
      if (prof) { atomicAdd(P.dbg + 0, (unsigned long long)t_wait); atomicAdd(P.dbg + 1, (unsigned long long)(clock64() - t_begin)); }
    }
  } else if (warp == kHaloMmaWarp) {
    if (elect_one() && leader) {
      // The issue loop is a single thread: keep it to a few dozen instructions per stage (no divisions, the
      // descriptors advance by adding constants to their 16-byte-unit address field).
      const uint32_t idesc_full = make_idesc_m(128 * kCtas, P.n_tile), idesc_half = make_idesc_m(128 * kCtas, P.n_tile >> 1);
      const uint64_t a_desc0 = desc_kmajor_sw128_sbo(0, (uint32_t)P.sbo);      // address field filled per plane
      const uint64_t b_desc0 = desc_kmajor_sw128(0);
      const uint32_t planes_u = smem_u32(planes) >> 4, bring_u = smem_u32(bring) >> 4;
      const uint32_t slot_u = (uint32_t)P.slot_bytes >> 4, bst_u = b_bytes >> 4;
      const uint32_t row_u = 128u >> 4;                                        // one plane row, in 16-byte units
      const int kh = P.kh, kw = P.kw, NP = P.NP, NB = P.NB;
      const bool dual = P.nsub == 2;
      const int acc_cols = P.n_tile * P.nsub;                                  // TMEM columns of one accumulator buffer
      const uint32_t line_step = (uint32_t)(P.Wb - (kw - 1)) * row_u;          // from the last tap of a line to the next line's first
      int ps = 0, bs = 0;
      uint32_t pph = 0, bph = 0;
      bool ok = true, b_ready = false;
      int j = 0;
      long long t_wait = 0, t_waitp = 0, t_wacc = 0, t_begin = (prof || (P.debug & 128)) ? clock64() : 0;
      for (int w = work0; w < P.total_work && ok; w += wstride, ++j) {
        const int buf = j & 1;
        const uint32_t aph = ((uint32_t)j >> 1) & 1u;
        const HaloTile t = halo_decode(P, w, kPair, 0);
        const uint32_t roff_u = (uint32_t)t.roff * row_u;      // flat tiles start inside their first plane line
        const uint32_t roff1_u = dual ? (uint32_t)halo_decode(P, w, kPair, 0, 1).roff * row_u : 0u;   // second tile of a dual item
        const uint32_t idesc = t.width == P.n_tile ? idesc_full : idesc_half;
        const uint32_t rot_a_u = (uint32_t)(t.rot_th0 * P.Wb + t.rot_tw0) * row_u;
        const int rot_th0 = t.rot_th0, rot_tw0 = t.rot_tw0;
        const long long ta0 = prof ? clock64() : 0;
        if (!mbar_wait(&acc_empty[buf], aph ^ 1u, P.err, 24)) { ok = false; break; }
        if (prof) t_wacc += clock64() - ta0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * acc_cols);
        const uint32_t d_tmem1 = d_tmem + (uint32_t)P.n_tile;  // dual items: the second tile's accumulator
        uint32_t acc = 0;
        int td_p = t.rot_td0;                                  // td of plane pi (the producers' walk)
        for (int pi = 0; pi < nplanes && ok; ++pi) {
          const bool live = halo_plane_live(P, t.d0, td_p, kPair);
          if (++td_p == P.kd) td_p = 0;
          if (!live) continue;
          const long long tp0 = prof ? clock64() : 0;
          if (!dbg_nop && !mbar_wait(&p_full[ps], pph, P.err, 25)) { ok = false; break; }
          // dual items: the second tile's plane sits in the next ring slot
          int ps1 = ps;
          uint32_t pph1 = pph;
          if (dual) {
            if (++ps1 == NP) { ps1 = 0; pph1 ^= 1u; }
            if (!dbg_nop && !mbar_wait(&p_full[ps1], pph1, P.err, 25)) { ok = false; break; }
          }
          if (prof) t_waitp += clock64() - tp0;
          const uint32_t base_u = planes_u + (uint32_t)ps * slot_u + roff_u;
          const uint32_t sub1_u = planes_u + (uint32_t)ps1 * slot_u + roff1_u - base_u;   // second tile's plane relative to the first's
          uint32_t a_u = base_u + rot_a_u;
          int th = rot_th0, tw = rot_tw0;
          for (int i = 0; i < taps_hw; ++i) {
            const long long tw0 = prof ? clock64() : 0;
            if (!b_ready && !dbg_nob && !mbar_wait(&b_full[bs], bph, P.err, 26)) { ok = false; break; }
            if (prof) t_wait += clock64() - tw0;
            tc_fence_after();
            const uint64_t ad = a_desc0 | (uint64_t)(a_u & 0x3FFFu);
            const uint64_t bd = b_desc0 | (uint64_t)((bring_u + (uint32_t)bs * bst_u) & 0x3FFFu);
            uint64_t* done_bar = &b_empty[bs];
            if (++bs == NB) { bs = 0; bph ^= 1u; }
            b_ready = mbar_test_wait(&b_full[bs], bph);          // peek at the next stage while this one is issued
            umma_f16_g<kPair>(d_tmem, ad, bd, idesc, acc);
            umma_f16_g<kPair>(d_tmem, ad + 2, bd + 2, idesc, 1u);
            umma_f16_g<kPair>(d_tmem, ad + 4, bd + 4, idesc, 1u);
            umma_f16_g<kPair>(d_tmem, ad + 6, bd + 6, idesc, 1u);
            if (dual) {                                          // the same weight slab against the second tile's plane
              const uint64_t ad1 = a_desc0 | (uint64_t)((a_u + sub1_u) & 0x3FFFu);
              umma_f16_g<kPair>(d_tmem1, ad1, bd, idesc, acc);
              umma_f16_g<kPair>(d_tmem1, ad1 + 2, bd + 2, idesc, 1u);
              umma_f16_g<kPair>(d_tmem1, ad1 + 4, bd + 4, idesc, 1u);
              umma_f16_g<kPair>(d_tmem1, ad1 + 6, bd + 6, idesc, 1u);
            }
            acc = 1u;
            umma_commit_g<kPair>(done_bar);
            if (++tw == kw) {
              tw = 0;
              if (++th == kh) { th = 0; a_u = base_u; } else a_u += line_step;
            } else {
              a_u += row_u;
            }
          }
          if (ok) umma_commit_g<kPair>(&p_empty[ps]);
          if (++ps == NP) { ps = 0; pph ^= 1u; }
          if (dual) {
            if (ok) umma_commit_g<kPair>(&p_empty[ps]);
            if (++ps == NP) { ps = 0; pph ^= 1u; }
          }
        }
        if (ok) umma_commit_g<kPair>(&acc_full[buf]);
      }
      if (prof || (P.debug & 128)) {
        atomicAdd(P.dbg + 2, (unsigned long long)t_wait); atomicAdd(P.dbg + 3, (unsigned long long)(clock64() - t_begin));
        atomicAdd(P.dbg + 6, (unsigned long long)t_wacc); atomicAdd(P.dbg + 7, (unsigned long long)t_waitp);
        atomicAdd(P.dbg + 5, 1ull);
      }
    }
  }
  } else {
    // ---- epilogue warps 0..7 -> TMEM lane quadrant (warp % 4), alternate 32-column chunks
    regs_epilogue();
    const EpiWarp W(warp);
    const int q = W.q;
    const int row = q * 32 + lane;
    const int nch_full = P.n_tile / 32;
    int nchunks = nch_full;                  // of the current work item (half-width tail items: t.width < n_tile)
    const bool defer = kMode != 0 && nch_full <= 2;
    EpiStats st;
    st.clear();
    float d1[32], d2[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) { d1[i] = 0.f; d2[i] = 0.f; }
    int st_n = -1, st_n0 = 0;
    const EpiArgs E{P.out, P.out_bf16, P.bias, P.act, P.slope, P.stats != nullptr, P.aux, P.aux_nslope};
    int j = 0;
    bool ok = true;
    const int acc_cols = P.n_tile * P.nsub;      // TMEM columns of one accumulator buffer (dual items: two tiles side by side)
    for (int w = work0; w < P.total_work && ok; w += wstride, ++j) {
      const int buf = j & 1;
      const uint32_t aph = ((uint32_t)j >> 1) & 1u;
      for (int sub = 0; sub < P.nsub && ok; ++sub) {
      const HaloTile t = halo_decode(P, w, kPair, rank, sub);
      const bool last_sub = sub == P.nsub - 1;
      int lh, lw;
      if (P.mode == 0) { lh = t.h0 + (row >> 3); lw = t.w0 + (row & 7); }
      else { const int f = t.roff + row; const int hh = f / P.Wb; lh = t.hs + hh; lw = f - hh * P.Wb; }
      const bool valid = lw < P.Wl && lh < P.Hl && t.d < P.Dl;
      const long long obase = (long long)t.n * P.osn + (long long)(t.d * P.ostep + P.od0) * P.osd +
                              (long long)(lh * P.ostep + P.oh0) * P.osh + (long long)(lw * P.ostep + P.ow0) * P.osw + t.n0;
      int tb, coff;                             // statistics key of the item (halo_stats_key)
      halo_stats_key(P, t, tb, coff);
      if (kMode != 0 && (t.n != st_n || tb != st_n0)) {
        epilogue_flush_stats(P.stats, st_n, P.Cn, st_n0, W.q, W.c_begin, 2, nch_full, lane, st, defer, d1, d2, epi_red);
        st_n = t.n; st_n0 = tb;
      }
      nchunks = t.width / 32;
      AuxRegs ax;
      epilogue_aux_first<kMode>(E, W.c_begin, nchunks, valid, obase, false, ax);
      if (sub == 0) {                           // one accumulator barrier per work item
        ok = mbar_wait(&acc_full[buf], aph, P.err, 23);
        if (!ok) break;
        tc_fence_after();
      }
      const long long te0 = prof ? clock64() : 0;
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * acc_cols + sub * P.n_tile);
      uint64_t* rel_bar = &acc_empty[buf];
      epilogue_tile<kMode>(E, t_addr, W.c_begin, 2, nchunks, valid, obase, t.n0, lane, st, coff >> 1, defer, d1, d2, ax, [&]() {
        if (!last_sub) return;                  // dual items: the buffer is free once the SECOND tile has been read
        tc_fence_before();                      // accumulator fully read: hand the buffer back to the MMA warp
        __syncwarp();
        if (lane == 0) { if constexpr (kPair) mbar_arrive_leader(rel_bar); else mbar_arrive(rel_bar); }
      });
      if (prof && threadIdx.x == 0) atomicAdd(P.dbg + 4, (unsigned long long)(clock64() - te0));
      }
    }
    if (kMode != 0) epilogue_flush_stats(P.stats, st_n, P.Cn, st_n0, W.q, W.c_begin, 2, nch_full, lane, st, defer, d1, d2, epi_red);
  }
  tc_fence_before();
  if constexpr (kPair) cluster_sync_all(); else __syncthreads();
  if (warp == kHaloMmaWarp) {
    if constexpr (kPair)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(P.tmem_cols) : "memory");
    else
      tmem_dealloc(tmem_base, P.tmem_cols);
  }
}

// ------------------------------------------------------------------ host side
// Can this launch run on the halo kernel?  Needs unit A step, taps forming a full (kd, kh, kw) box and a plane
// that fits the shared-memory budget.  Fills P's geometry fields on success.
inline bool halo_setup(const GatherLaunch& L, int n, int ck, int cn, bool pair, HaloP& P, int units_override = 0) {
  if (L.astep != 1 || L.taps.empty()) return false;
  int lo[3] = {1 << 30, 1 << 30, 1 << 30}, hi[3] = {-(1 << 30), -(1 << 30), -(1 << 30)};
  for (const Tap& t : L.taps) {
    const int o[3] = {t.dd, t.dh, t.dw};
    for (int i = 0; i < 3; ++i) { if (o[i] < lo[i]) lo[i] = o[i]; if (o[i] > hi[i]) hi[i] = o[i]; }
  }
  const int kd = hi[0] - lo[0] + 1, kh = hi[1] - lo[1] + 1, kw = hi[2] - lo[2] + 1;
  if ((long long)kd * kh * kw != (long long)L.taps.size() || (int)L.taps.size() > kMaxTaps) return false;
  P.kd = kd; P.kh = kh; P.kw = kw; P.dmin = lo[0]; P.hmin = lo[1]; P.wmin = lo[2];
  for (int i = 0; i < kMaxTaps; ++i) P.twi[i] = -1;
  for (const Tap& t : L.taps) {
    const int idx = ((t.dd - lo[0]) * kh + (t.dh - lo[1])) * kw + (t.dw - lo[2]);
    if (P.twi[idx] != -1) return false;
    P.twi[idx] = (int16_t)t.widx;
  }
  P.Dl = L.dims[0]; P.Hl = L.dims[1]; P.Wl = L.dims[2]; P.N = n;
  int n_tile = pick_n_tile(cn);
  if (n_tile == 0 || ck % 64 != 0) return false;
  P.Cn = cn; P.n_tile = n_tile; P.n_tiles = cn / n_tile; P.kchunks = ck / 64;
  P.nsub = 1;
  // tile shape: 2D (16 x 8) or flat, whichever wastes fewer MMA rows (and fits)
  const long long hw = (long long)P.Hl * P.Wl;
  const int t2h = (P.Hl + 15) / 16, t2w = (P.Wl + 7) / 8;
  const int Wb2 = 8 + kw - 1, Hb2 = 16 + kh - 1;
  const long long rows2 = (long long)t2h * t2w * 128;
  const int Wbf = P.Wl + kw - 1;
  const long long flat_len = (long long)(P.Hl - 1) * Wbf + P.Wl;          // last valid flat position + 1
  const int tf = (int)((flat_len + 127) / 128);
  const int Hbf = (Wbf - 1 + 128 + (kh - 1) * Wbf + (kw - 1) + Wbf - 1) / Wbf;   // lines covering any 128-run + halo
  const long long rowsf = (long long)tf * 128;
  const size_t budget = kSmemLimit - 2048 - kEpiRedBytes;
  auto fits = [&](int Wb, int Hb) {
    if (Wb > 256 || Hb > 256) return false;
    const size_t slot = ((size_t)Wb * Hb * 128 + 1023) / 1024 * 1024;
    return 2 * slot + 2 * (size_t)n_tile * 128 / (pair ? 2 : 1) <= budget;
  };
  const bool ok2 = fits(Wb2, Hb2), okf = fits(Wbf, Hbf);
  if (!ok2 && !okf) return false;
  const bool use_flat = okf && (!ok2 || rowsf * 100 < rows2 * 97);      // flat only when clearly better
  (void)hw;
  if (!use_flat) {
    P.mode = 0; P.tiles_w = t2w; P.tiles_hw = t2h * t2w; P.Wb = Wb2; P.Hb = Hb2; P.sbo = Wb2 * 128;
  } else {
    P.mode = 1; P.tiles_w = 1; P.tiles_hw = tf; P.Wb = Wbf; P.Hb = Hbf; P.sbo = 1024;
  }
  P.plane_tx = P.Wb * P.Hb * 128;
  P.slot_bytes = (P.plane_tx + 1023) / 1024 * 1024;
  P.pair = pair ? 1 : 0;
  // DUAL items (MRA_HALO_DUAL=1): with 256 output channels per tile the kernel is bound by L2 -> SM bytes, three quarters
  // of them weight slabs (G.rb fprop: 1.19 GB per launch at 7.7 TB/s, tensor pipe 79 %; every CTA pair streams all 3.5 MB
  // of weights for each 256-position tile pair).  A dual item is TWO position tiles x 128 channels instead of one tile x
  // 256: the same MMA work and the same 256 TMEM columns per accumulator buffer, but each weight slab (now half as
  // large) feeds two tiles -- weights 1.77 -> 0.89 MB, planes 0.28 -> 0.55 MB per item and CTA: -30 % of the bytes.
  {
    const char* e = getenv("MRA_HALO_DUAL");
    const size_t bB2 = (size_t)128 * 128 / 2;
    if (e && atoi(e) != 0 && pair && n_tile == 256 && P.tiles_hw % 2 == 0 && 4 * (size_t)P.slot_bytes + 4 * bB2 <= budget) {
      n_tile = 128;
      P.n_tile = 128; P.n_tiles = cn / 128; P.nsub = 2;
    }
  }
  // ring depths: weights get what the planes leave (>= 2 each)
  const size_t bB = (size_t)n_tile * 128 / (pair ? 2 : 1);
  int NP, NB;
  if (P.nsub == 2) {
    NP = 4;                                      // two tiles per (chunk, td) step, two steps in flight (a step is 72 MMAs)
    NB = (int)((budget - (size_t)NP * P.slot_bytes) / bB);
    if (NB > 8) NB = 8;                          // (2 NP + 2 NB + 4 mbarriers must fit the 256 bytes behind the rings)
  } else {
    NP = kd >= 3 ? 3 : 2;
    if (kd * P.kchunks == 1) NP = 2;
    NB = (int)((budget - (size_t)NP * P.slot_bytes) / bB);
    while (NB < 3 && NP > 2) { --NP; NB = (int)((budget - (size_t)NP * P.slot_bytes) / bB); }
    if (NB < 2) return false;
    if (NB > 8) NB = 8;
    // spare room goes to a deeper plane ring (up to 4)
    while (NP < 4 && (size_t)(NP + 1) * P.slot_bytes + (size_t)NB * bB <= budget) ++NP;
    { const char* e = getenv("MRA_HALO_NB"); if (e && atoi(e) >= 2 && atoi(e) <= NB) NB = atoi(e); }
    { const char* e = getenv("MRA_HALO_NP"); if (e && atoi(e) >= 2 && atoi(e) <= NP) NP = atoi(e); }
  }
  P.NP = NP; P.NB = NB;
  const long long total = (long long)n * (pair ? (P.Dl + 1) / 2 : P.Dl) * (P.tiles_hw / P.nsub) * P.n_tiles;
  if (total >= (1ll << 31)) return false;
  P.total_tiles = (int)total;
  // persistent schedule: `units` CTAs (or pairs) take work items round-robin.  When the last round is at most
  // half full, its tiles are split into two half-width items each.
  const int units = units_override > 0 ? units_override : (pair ? num_sms() / 2 : num_sms());
  const int rem = (int)(total % units);
  P.split_from = P.total_tiles; P.total_work = P.total_tiles;
  if (total > units && rem > 0 && 2 * rem <= units && n_tile >= 128 && getenv("MRA_GATHER_NOSPLIT") == nullptr) {
    P.split_from = P.total_tiles - rem;
    P.total_work = P.total_tiles + rem;
  }
  return true;
}

// dead-plane skipping (halo_plane_live): on when some (item, td) lies outside A and every item keeps a live plane
inline void halo_fill_skip(HaloP& P, int Da) {
  P.Da = Da;
  P.skip = 0;
  if (getenv("MRA_HALO_NOSKIP") != nullptr) return;
  const int dsteps = P.pair ? (P.Dl + 1) / 2 : P.Dl;
  bool any_dead = false, all_items_live = true;
  for (int dq = 0; dq < dsteps; ++dq) {
    int live = 0;
    for (int td = 0; td < P.kd; ++td) {
      const int a0 = (P.pair ? 2 * dq : dq) + P.dmin + td;
      const bool lv = P.pair ? (a0 + 1 >= 0 && a0 < Da) : (a0 >= 0 && a0 < Da);
      if (lv) ++live; else any_dead = true;
    }
    if (live == 0) all_items_live = false;
  }
  P.skip = (any_dead && all_items_live) ? 1 : 0;
}

inline int run_gather_halo(const GatherPlan& plan, const GatherLaunch& L, HaloP& P, const GatherRun& R, const CUtensorMap& tmB_in,
                           cudaStream_t st) {
  CUtensorMap tmB = tmB_in;
  if (P.pair) {          // each CTA of a pair loads half of the slab's rows
    if (int rc = make_weight_map(&tmB, R.b, (long long)R.slabs * plan.cn, plan.ck, P.n_tile / 2)) return rc;
  }
  { const char* e = getenv("MRA_GATHER_DEBUG");
    if (e && (atoi(e) & 32)) {     // shrink the weight boxes to 8 rows: same handshakes, ~no bytes (results are garbage)
      if (int rc = make_weight_map(&tmB, R.b, (long long)R.slabs * plan.cn, plan.ck, 8)) return rc;
      P.b_tx_dbg = 8 * 128;
    } }
  static bool attr_set = false;
  if (!attr_set) {
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<false, 0>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<false, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<false, 2>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<true, 0>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<true, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    MRA_CHECK_CUDA(cudaFuncSetAttribute((gather_halo_kernel<true, 2>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmemLimit - kEpiRedBytes)));
    attr_set = true;
  }
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
  P.tmem_cols = pow2_cols(2 * P.n_tile * P.nsub);
  halo_fill_skip(P, plan.adims[0]);
  CUtensorMap tmA;
  if (int rc = make_act_map(&tmA, R.a, plan.n, plan.adims[0], plan.adims[1], plan.adims[2], plan.ck, P.Wb, P.Hb, 1, 1)) return rc;
  const size_t smem = (size_t)P.NP * P.slot_bytes + (size_t)P.NB * P.n_tile * 128 / (P.pair ? 2 : 1) + 1024 + 256;
  if (!P.pair) {
    const int ctas = P.total_work < num_sms() ? P.total_work : num_sms();
    if (P.aux && P.stats) MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<false, 2>, dim3(ctas), dim3(kThreadsHalo), smem, st, 1, tmA, tmB, P));
    else if (P.stats) MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<false, 1>, dim3(ctas), dim3(kThreadsHalo), smem, st, 1, tmA, tmB, P));
    else MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<false, 0>, dim3(ctas), dim3(kThreadsHalo), smem, st, 1, tmA, tmB, P));
  } else {
    int pairs = num_sms() / 2;
    if (P.total_work < pairs) pairs = P.total_work;
    const dim3 grid((unsigned)(2 * pairs));
    if (P.aux && P.stats) MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<true, 2>, grid, dim3(kThreadsHalo), smem, st, 2, tmA, tmB, P));
    else if (P.stats) MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<true, 1>, grid, dim3(kThreadsHalo), smem, st, 2, tmA, tmB, P));
    else MRA_CHECK_CUDA(launch_pdl(gather_halo_kernel<true, 0>, grid, dim3(kThreadsHalo), smem, st, 2, tmA, tmB, P));
  }
  MRA_LAUNCH_CHECK();
  return 0;
}

inline bool phase_try_run(const GatherPlan& plan, const GatherRun& R, cudaStream_t st, int* rc);   // conv_tc_phase.cuh

// Run every launch of a gather plan on the tensor cores: the 8 parity phases of a stride-2 dgrad-form plan on the
// phase-halo kernel, stride-1 launches on the halo-plane kernel, the rest (and anything those cannot host) on the
// per-tap kernel.  Channel counts that are multiples of 32 but not of 64 run on the per-tap kernel only (see
// tc_channels_ok): its K chunks come zero-filled from TMA and its epilogue masks the N tile at Cn.
inline int run_gather_tc(const GatherPlan& plan, const GatherRun& R, cudaStream_t st) {
  const int n_tile = gather_n_tile(plan.cn);
  MRA_REQUIRE(n_tile > 0 && tc_channels_ok(plan.ck), "channel counts not eligible for the tensor-core path");
  const bool c64 = tc_channels_c64(plan.ck) && tc_channels_c64(plan.cn);
  const long long rows = (long long)R.slabs * plan.cn;
  CUtensorMap tmB;
  if (int rc = make_weight_map(&tmB, R.b, rows, plan.ck, n_tile)) return rc;
  // MRA_GATHER_MODE (experiments): v1 = per-tap kernel only, single = halo kernel without CTA pairs
  const char* gm = getenv("MRA_GATHER_MODE");
  const bool force_v1 = gm && !strcmp(gm, "v1");
  const bool no_pair = gm && !strcmp(gm, "single");
  const bool no_col = gm && !strcmp(gm, "nocol");
  const bool plane_kernels = !force_v1 && c64;             // phase, column and halo kernels
  if (!force_v1 && gather_mergeable(plan)) {
    int prc = 0;
    if (c64 && !(gm && !strcmp(gm, "nophase")) && phase_try_run(plan, R, st, &prc)) return prc;
    bool slabs_ok = true;
    for (const GatherLaunch& L : plan.launches)
      for (const Tap& t : L.taps) if (t.widx >= R.slabs) slabs_ok = false;
    if (slabs_ok) return run_gather_v1_launch(plan, plan.launches.data(), 8, R, tmB, n_tile, st);
  }
  for (const GatherLaunch& L : plan.launches) {
    bool slabs_ok = true;
    for (const Tap& t : L.taps) if (t.widx >= R.slabs) slabs_ok = false;
    ColP CP;
    memset(&CP, 0, sizeof(CP));
    if (plane_kernels && !no_col && slabs_ok && col_setup(L, plan.n, plan.ck, plan.cn, CP)) {
      if (int rc = run_gather_col(plan, L, CP, R, tmB, st)) return rc;
      continue;
    }
    HaloP P;
    memset(&P, 0, sizeof(P));
    // the halo kernel pays off when several taps share a plane (kh * kw >= 4)
    int lo[2] = {1 << 30, 1 << 30}, hi[2] = {-(1 << 30), -(1 << 30)};
    for (const Tap& t : L.taps) {
      if (t.dh < lo[0]) lo[0] = t.dh; if (t.dh > hi[0]) hi[0] = t.dh;
      if (t.dw < lo[1]) lo[1] = t.dw; if (t.dw > hi[1]) hi[1] = t.dw;
    }
    const bool reuse = !L.taps.empty() && (hi[0] - lo[0] + 1) * (hi[1] - lo[1] + 1) >= 4;
    bool halo = plane_kernels && reuse && halo_setup(L, plan.n, plan.ck, plan.cn, !no_pair, P);
    if (halo) for (const Tap& t : L.taps) if (t.widx >= R.slabs) halo = false;
    if (halo) { if (int rc = run_gather_halo(plan, L, P, R, tmB, st)) return rc; }
    else      { if (int rc = run_gather_v1_launch(plan, &L, 1, R, tmB, n_tile, st)) return rc; }
  }
  return 0;
}

// ------------------------------------------------------------------ split-K for launches that cannot fill the GPU
// The deep layers of the 7-down UNet (512 -> 512 k4 s2 at 8^3 -> 4^3 ... 2^3 -> 1^3, and the dgrads of the matching
// transposed convs) have a handful of output tiles but K = 64 taps x 8..16 channel chunks: two to eight CTAs each streamed
// the whole 33 - 67 MB weight tensor through one TMA producer (0.157 ms per launch whatever the spatial size, 1 - 55
// TFLOP/s).  Such a launch is split into 8 tap ranges that run as the 8 "phases" of the merged launch of gather_tc_kernel
// -- (tile, range) work items, each range writing its fp32 partial sums to its own slice of a scratch tensor shaped
// [N][8 * Do][Ho][Wo][Cn] (the output d offset of range s is s * Do) -- and ksplit_finish_kernel adds the 8 slices, the
// bias and the activation and writes the bf16 result.  8x the CTAs stream the weights in parallel.
constexpr int kSplitParts = 8;
inline bool ksplit_eligible(const GatherPlan& plan) {
  if (getenv("MRA_GATHER_NOKSPLIT") != nullptr || plan.launches.size() != 1) return false;
  const GatherLaunch& L = plan.launches[0];
  const int n_tile = pick_n_tile(plan.cn);
  if (L.astep != 2 || L.ostep != 1 || n_tile == 0 || plan.ck % 64 != 0) return false;
  const int taps = (int)L.taps.size();
  if (taps < 2 * kSplitParts || taps > kMaxTaps || (long long)taps * (plan.ck / 64) < 64) return false;
  if (L.o0[0] != 0 || L.o0[1] != 0 || L.o0[2] != 0 || (kSplitParts - 1) * plan.odims[0] > 127) return false;
  long long tiles = (long long)plan.n * (plan.cn / n_tile);
  for (int i = 0; i < 3; ++i) tiles *= (L.dims[i] + L.box[i] - 1) / L.box[i];
  return tiles * 4 <= num_sms();                 // under a quarter of a wave
}
inline size_t ksplit_workspace_bytes(const mra_conv_desc& d, int which) {
  if (d.dtype != MRA_BF16 || (d.flags & MRA_CONV_FORCE_NAIVE) || !gather_eligible(d, which)) return 0;
  GatherPlan plan;
  if (!build_gather_plan(d, which, plan) || !ksplit_eligible(plan)) return 0;
  return (size_t)plan.n * kSplitParts * plan.odims[0] * plan.odims[1] * plan.odims[2] * plan.cn * sizeof(float);
}
// out[n][pos][c] = act(sum_s part[n][s][pos][c] + bias[c]);  4 channels per thread
__global__ void __launch_bounds__(256) ksplit_finish_kernel(const float* __restrict__ part, bf16* __restrict__ out, int N,
                                                             long long npos, int Cn, const float* __restrict__ bias, int act,
                                                             float slope) {
  const long long c4n = Cn / 4;
  const long long total = (long long)N * npos * c4n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long c4 = i % c4n, r = i / c4n;
    const long long n = r / npos, pos = r - n * npos;
    const float4* p = reinterpret_cast<const float4*>(part + ((n * kSplitParts) * npos + pos) * Cn) + c4;
    float4 a = __ldg(p);
#pragma unroll
    for (int s = 1; s < kSplitParts; ++s) {
      const float4 b = __ldg(p + (long long)s * npos * c4n);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (bias) { const float4 b = __ldg(reinterpret_cast<const float4*>(bias) + c4); a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
    float v[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (act == MRA_ACT_RELU) v[k] = fmaxf(v[k], 0.f);
      else if (act == MRA_ACT_LRELU) v[k] = v[k] > 0.f ? v[k] : v[k] * slope;
      else if (act == MRA_ACT_TANH) v[k] = tanhf(v[k]);
      else if (act == MRA_ACT_SIGMOID) v[k] = 1.f / (1.f + expf(-v[k]));
    }
    __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&lo); o.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(out + (r * Cn + c4 * 4)) = o;
  }
}
inline int run_gather_ksplit(const GatherPlan& plan, const GatherRun& R, float* scratch, cudaStream_t st) {
  const GatherLaunch& L0 = plan.launches[0];
  GatherPlan sp = plan;
  sp.launches.clear();
  sp.odims[0] = plan.odims[0] * kSplitParts;
  const int taps = (int)L0.taps.size();
  for (int s = 0; s < kSplitParts; ++s) {
    GatherLaunch L = L0;
    L.taps.assign(L0.taps.begin() + (long long)taps * s / kSplitParts, L0.taps.begin() + (long long)taps * (s + 1) / kSplitParts);
    L.o0[0] = s * plan.odims[0];
    sp.launches.push_back(L);
  }
  const int n_tile = pick_n_tile(plan.cn);
  CUtensorMap tmB;
  if (int rc = make_weight_map(&tmB, R.b, (long long)R.slabs * plan.cn, plan.ck, n_tile)) return rc;
  GatherRun P{R.a, R.b, R.slabs, nullptr, scratch, 0, MRA_ACT_NONE, 0.f, nullptr};
  if (int rc = run_gather_v1_launch(sp, sp.launches.data(), kSplitParts, P, tmB, n_tile, st)) return rc;
  const long long npos = (long long)plan.odims[0] * plan.odims[1] * plan.odims[2];
  const long long total = (long long)plan.n * npos * (plan.cn / 4);
  long long blocks = (total + 255) / 256;
  if (blocks > 4 * num_sms()) blocks = 4 * num_sms();
  ksplit_finish_kernel<<<(unsigned)blocks, 256, 0, st>>>(scratch, reinterpret_cast<bf16*>(R.out), plan.n, npos, plan.cn, R.bias, R.act,
                                                         R.slope);
  MRA_LAUNCH_CHECK();
  return 0;
}

// `split_done` (optional) tells the caller that the split-K path ran: it does not produce InstanceNorm statistics.
inline int run_gather_tc(const mra_conv_desc& d, int which, const void* a, const void* b, const float* bias, void* out,
                         double* stats, cudaStream_t st, const void* aux = nullptr, float aux_nslope = 0.f,
                         void* workspace = nullptr, size_t workspace_bytes = 0, bool* split_done = nullptr) {
  GatherPlan plan;
  MRA_REQUIRE(build_gather_plan(d, which, plan), "unsupported conv geometry");
  GatherRun R{a, b, d.k * d.k * d.k, bias, out, 1, which == 0 ? d.act : MRA_ACT_NONE, d.slope, stats};
  R.aux = aux; R.aux_nslope = aux_nslope;
  if (split_done) *split_done = false;
  if (aux == nullptr && split_done != nullptr && workspace != nullptr && ksplit_eligible(plan)) {
    const size_t need = (size_t)plan.n * kSplitParts * plan.odims[0] * plan.odims[1] * plan.odims[2] * plan.cn * sizeof(float);
    bool slabs_ok = true;
    for (const Tap& t : plan.launches[0].taps) if (t.widx >= R.slabs) slabs_ok = false;
    if (slabs_ok && workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0) {
      *split_done = true;
      return run_gather_ksplit(plan, R, reinterpret_cast<float*>(workspace), st);
    }
  }
  return run_gather_tc(plan, R, st);
}

}  // namespace tc
}  // namespace mra
