// CUDA kernels (sm_100a) and the C ABI of libpriblast_acc.so.
//
// Kernel set (DESIGN.md §4):
//   k_inside_tile / k_outside_tile   tile-persistent, time-tiled span march (acc_tile.h): one CTA per column
//                                    tile, stencil source rows in shared-memory rings, halo recomputed,
//                                    one deep step (kTT spans' long-range sums) per kTT shallow steps
//   k_outer_scans_warp               the two outer arrays, one warp per sequence
//   k_biloop_tile<LEFT/RIGHT> (the left one also forms the hairpin suffix sums), k_finalize   accessibility
// Every kernel exists for float and double band arithmetic.  The float engine (span-scaled, range
// guarded) is the fast path (spans up to kFp32MaxSpan); sequences whose stored values leave the safe range
// are flagged on the device and re-run by the double engine inside the same prib_acc_compute call, on
// the GPU.  Spans above kMaxSpan run the wide-span FP64 engine (acc_wide.cu), whose flagged sequences are
// re-run by the exact engine (acc_exact.cu) the same way.  There is no CPU path.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges show up in Nsight Systems / ncu --nvtx, cost nothing otherwise

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/priblast_acc.h"
#include "acc_core.h"
#include "acc_exact.h"
#include "acc_tables.h"
#include "acc_tile.h"
#include "acc_wide.h"

using namespace prib;

namespace {

// NVTX range over a host-side scope (one per C-ABI call and per phase of a device batch; SURVEY §5)
struct NvtxRange {
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

constexpr int kThreads = 128;
constexpr int kScanWarps = 4;
constexpr int kFp32MaxSpan = kMaxSpan;  // always try FP32 first: at W = 150 a quarter of random 2 kb sequences
                                         // is flagged and re-run in FP64, still 1.7x faster than FP64 for all (profiles/r1/sweep.json)
// widest CTA of the tile kernels per precision (227 KB of rings / 80 rows): bounds the register budget
#ifndef PRIB_TC32
#define PRIB_TC32 640
#endif
#ifndef PRIB_TC64
#define PRIB_TC64 288
#endif
template <typename real> struct TileChain { static constexpr bool value = sizeof(real) == 4 && PRIB_CHAIN != 0; };
template <typename real> struct TileMaxThreads { static constexpr int value = sizeof(real) == 4 ? PRIB_TC32 : PRIB_TC64; };

// ---------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------
// grid = resident CTAs (one per SM: the rings take ~all shared memory), blockDim = TC, tiles round-robin.
// dynamic smem: (kTilePad + kTileRows * TC) reals + hot tables + (TC + 16) base codes.
constexpr int kProgBytes = 128 + 16;  // 32 per-warp progress counters (warp-to-warp synchronisation of the tile kernels) + the
                                      // transaction barrier of the table copy
template <typename real>
__host__ __device__ constexpr size_t tile_smem_bytes() {
  return ((size_t)kTilePad + (size_t)kTileRows * TileMaxThreads<real>::value) * sizeof(real) +
         (Core<real>::kHotBytes + TileMaxThreads<real>::value + kMaxSpan + 16 + 15) / 16 * 16  // + base codes (outside: TC + W + 8)
         + kProgBytes;                                                                           // + the per-warp progress counters
}

// ---- TMA (bulk asynchronous copy) staging of a band tile -------------------------------------------------
// The start-indexed tile of the left-strand kernel is `rows` contiguous, 16-byte aligned segments of a span-major
// array (row r = columns g0 .. g0 + cols - 1 of span r + 5), so ONE thread hands the whole tile to the copy engine
// (cp.async.bulk.shared.global, SASS UBLKCP) and every thread waits on the transaction barrier; no registers and no
// LSU instructions carry the data.  Cells that do not exist (the DP state is not cleared between batches) are masked
// in shared memory afterwards, each thread its own column.  The end-indexed tile of the right-strand kernel is skewed
// (row r starts at column g0 - 31 - r: not 16-byte aligned) and keeps the LDG -> STS path.
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tma_bar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_bar_expect(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bar_wait(unsigned long long *bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "TMA_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra TMA_DONE;\n"
      "bra TMA_WAIT;\n"
      "TMA_DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_copy_g2s(void *smem_dst, const void *gsrc, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Warp-to-warp synchronisation of the tile kernels (acc_tile.h, "Synchronisation"): one progress counter per warp in
// shared memory.  A warp publishes the number of events it has completed (per group of kTT spans: 1 for the deep step,
// 1 per shallow step) with release semantics and polls its neighbours' counters with acquire semantics.
// Slack (in events) a warp may run ahead of the neighbour that READS its columns, from the ring sizes of acc_tile.h:
// inside: the 4-row multi rings are read one row back (3 steps); outside: the 8-row Beta_stem ring is read up to 6
// rows back (2 steps).  Both also cover the 32/34-row stencil rings (the deep step of a group reads 30/32 rows back).
enum { kEvPerGroup = kTT + 1, kEvSlackIn = 3, kEvSlackOut = 2 };
__device__ __forceinline__ void prog_signal(int *prog, int warp, int lane, int value) {
  __syncwarp();  // every lane's ring / scratch stores (and ring reads) are ordered before lane 0's release
  if (lane == 0)
    asm volatile("st.release.cta.shared.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(prog + warp)), "r"(value) : "memory");
}
__device__ __forceinline__ void prog_wait(const int *prog, int warp, int need) {
  const unsigned addr = (unsigned)__cvta_generic_to_shared(prog + warp);
  int v;
  do {
    asm volatile("ld.acquire.cta.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  } while (v < need);
}
#if defined(PRIB_RELAXED_SYNC)
// Shared-memory-only hand-over: the ring rows and the counter live in the same shared memory, whose accesses are
// performed in the order the SM issues them (STS of the data, then — after __syncwarp — the STS of the counter; the
// reader's LDS of the data are issued after its LDS of the counter returned).  No fence, hence no wait for the global
// stores in flight.  The scratch rows in GLOBAL memory are covered by the release/acquire pair of the last step of
// each group (prog_signal / prog_wait), which is the event the deep steps wait for.
__device__ __forceinline__ void prog_signal_smem(int *prog, int warp, int lane, int value) {
  __syncwarp();
  if (lane == 0)
    asm volatile("st.volatile.shared.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(prog + warp)), "r"(value) : "memory");
}
__device__ __forceinline__ void prog_wait_smem(const int *prog, int warp, int need) {
  const unsigned addr = (unsigned)__cvta_generic_to_shared(prog + warp);
  int v;
  do {
    asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  } while (v < need);
}
#else
__device__ __forceinline__ void prog_signal_smem(int *prog, int warp, int lane, int value) { prog_signal(prog, warp, lane, value); }
__device__ __forceinline__ void prog_wait_smem(const int *prog, int warp, int need) { prog_wait(prog, warp, need); }
#endif
struct StepSignal {  // the hook of Tile::inside_shallow / outside_shallow: runs right after the ring / scratch stores
  int *prog;
  int warp, lane, value;
  bool release;  // last step of a group: release semantics (covers the scratch rows in global memory)
  __device__ __forceinline__ void operator()() const {
    if (release) prog_signal(prog, warp, lane, value);
    else prog_signal_smem(prog, warp, lane, value);
  }
};

template <typename real, int PAR /* parity of the first span of every group (chain formulation) */>
__global__ void __launch_bounds__(TileMaxThreads<real>::value, 1)
k_inside_tile(typename Core<real>::Ctx c, int TX, long long ntiles, real *scratch) {
  constexpr bool CH = TileChain<real>::value;
  typedef Tile<real> TL;
  constexpr int TC = TileMaxThreads<real>::value;  // compile-time row stride
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int t = threadIdx.x, W = c.W, warp = t >> 5, lane = t & 31;
  constexpr int NW = TC / 32;
  real *base = reinterpret_cast<real *>(smem_raw) + kTilePad;
  unsigned char *stab = smem_raw + ((size_t)kTilePad + (size_t)kTileRows * TC) * sizeof(real);  // 16-byte aligned
  uint8_t *sS = stab + Core<real>::kHotBytes;
  const typename Core<real>::SmallTables &T = *reinterpret_cast<const typename Core<real>::SmallTables *>(stab);
  real *scrM1 = scratch + (size_t)blockIdx.x * 2 * (W + 4) * TC;
  real *scrM2 = scrM1 + (size_t)(W + 4) * TC;
  const typename TL::InSmem sm = TL::carve_in(base, TC, sS);
  const int dfirst = TL::first_group(W);
  int *prog = reinterpret_cast<int *>(smem_raw + tile_smem_bytes<real>() - kProgBytes);
  if (t < 32) prog[t] = 0;
  {  // the hot Boltzmann tables (SmallTables up to hot_end) come in as ONE bulk asynchronous copy (TMA engine)
    unsigned long long *tbar = reinterpret_cast<unsigned long long *>(prog + 32);
    if (t == 0) {
      tma_bar_init(tbar, 1);
      tma_bar_expect(tbar, (unsigned)Core<real>::kHotBytes);
      tma_copy_g2s(stab, c.T, (unsigned)Core<real>::kHotBytes, tbar);
    }
    __syncthreads();  // the barrier is initialised before anybody polls it
    tma_bar_wait(tbar, 0);
  }
  int ebase = 0;  // events completed by every warp before this tile
  __syncthreads();
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    typename TL::Geo ge;
    ge.g0 = tile * TX;
    ge.TC = TC;
    ge.TX = TX;
    ge.H = W + 1;
    __syncthreads();  // previous tile fully consumed
    for (int k = t; k < kTileRows * TC; k += TC) base[k] = 0;
    for (int k = t; k < TC + 8; k += TC) sS[k] = (ge.g0 + k < c.NC) ? c.S[ge.g0 + k] : 0;
    typename TL::ColState cs;
    TL::col_state(c, ge.g0 + t, cs);
    __syncthreads();
    // Inside: a cell reads columns t .. t + 29 -> forward neighbour = warp + 1, back-pressure from warp - 1.
    // Chain formulation: the generic sums of column x come from the centre-line threads x .. x + (W + 1) / 2 (warps
    // w .. w + 2) through the double-buffered exchange rows.
    int ev = ebase, grp = 0;
    typename TL::Chain ch;
    if constexpr (CH) TL::clear(ch);
    for (int d0 = dfirst; d0 <= W + 1; d0 += kTT, ++grp) {
      real gs[kTT], mb[kTT], bs[kTT];
      real *xch = sm.xch + (grp & 1) * kTT * TC;
      if (warp + 1 < NW) prog_wait(prog, warp + 1, ev);  // the neighbour has finished the previous group
      if constexpr (CH) {
        if (warp >= 2) prog_wait(prog, warp - 2, ev - kEvPerGroup);  // readers of this exchange buffer (group - 2) are done
        TL::template inside_deep_chain<PAR, TC>(T, ge, sm, scrM1, scrM2, t, d0, ch, xch, mb, bs);
      } else {
        TL::template inside_deep<TC>(T, ge, sm, scrM1, scrM2, t, d0, gs, mb, bs);
      }
      prog_signal_smem(prog, warp, lane, ++ev);
#pragma unroll
      for (int k = 0; k < kTT; ++k) {
        ++ev;  // this step's event
        if (d0 + k >= kTurn) {  // uniform
          if ((k > 0 || CH) && warp + 1 < NW) prog_wait_smem(prog, warp + 1, ev - 1);
          if (CH && warp + 2 < NW) prog_wait_smem(prog, warp + 2, ev - 1 - k);  // its deep step of this group wrote my columns
          if (warp > 0) prog_wait_smem(prog, warp - 1, ev - kEvSlackIn);
          TL::template inside_shallow<TC>(c, T, ge, sm, scrM1, scrM2, t, cs, d0 + k, CH ? xch[k * TC + t] : gs[k], mb[k],
                                          bs[k], StepSignal{prog, warp, lane, ev, k == kTT - 1});
        } else {
          prog_signal(prog, warp, lane, ev);
        }
      }
    }
    ebase = ev;
  }
}

template <typename real>
__global__ void __launch_bounds__(TileMaxThreads<real>::value, 1)
k_outside_tile(typename Core<real>::Ctx c, int TX, long long ntiles, real *scratch) {
  constexpr bool CH = TileChain<real>::value;
  typedef Tile<real> TL;
  constexpr int TC = TileMaxThreads<real>::value;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int t = threadIdx.x, W = c.W, warp = t >> 5, lane = t & 31;
  constexpr int NW = TC / 32;
  real *pad = reinterpret_cast<real *>(smem_raw);
  real *base = pad + kTilePad;
  unsigned char *stab = smem_raw + ((size_t)kTilePad + (size_t)kTileRows * TC) * sizeof(real);
  const typename Core<real>::SmallTables &T = *reinterpret_cast<const typename Core<real>::SmallTables *>(stab);
  uint8_t *sS = stab + Core<real>::kHotBytes;
  real *scrBif = scratch + (size_t)blockIdx.x * 2 * (W + 4) * TC;
  const typename TL::OutSmem sm = TL::carve_out(base, TC, sS);
  const int dlast = TL::first_group(W);  // the groups of the inside pass, walked downwards
  int *prog = reinterpret_cast<int *>(smem_raw + tile_smem_bytes<real>() - kProgBytes);
  if (t < 32) prog[t] = 0;
  {  // the hot Boltzmann tables (SmallTables up to hot_end) come in as ONE bulk asynchronous copy (TMA engine)
    unsigned long long *tbar = reinterpret_cast<unsigned long long *>(prog + 32);
    if (t == 0) {
      tma_bar_init(tbar, 1);
      tma_bar_expect(tbar, (unsigned)Core<real>::kHotBytes);
      tma_copy_g2s(stab, c.T, (unsigned)Core<real>::kHotBytes, tbar);
    }
    __syncthreads();  // the barrier is initialised before anybody polls it
    tma_bar_wait(tbar, 0);
  }
  int ebase = 0;
  __syncthreads();
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    typename TL::Geo ge;
    ge.g0 = tile * TX;
    ge.TC = TC;
    ge.TX = TX;
    ge.H = W + 1;
    __syncthreads();
    for (int k = t; k < kTilePad + kTileRows * TC; k += TC) pad[k] = 0;
    for (int k = t; k < TC + W + kOutBaseTail; k += TC) {
      const long long col = ge.g0 - ge.H - kOutBaseLead + k;
      sS[k] = (col >= 0 && col < c.NC) ? c.S[col] : 0;
    }
    typename TL::ColState cs;
    TL::col_state(c, ge.g0 - ge.H + t, cs);
    __syncthreads();
    // Outside: a cell reads columns t - 30 .. t -> forward neighbour = warp - 1, back-pressure from warp + 1.
    // Chain formulation: the generic sums of column x come from the centre-line threads x - (W + 1) / 2 .. x (warps
    // w - 2 .. w).
    int slot = (W + 1) % kRingOut;
    int ev = ebase, grp = 0;
    typename TL::Chain ch;
    if constexpr (CH) TL::clear(ch);
    for (int d0 = W + 1; d0 >= dlast + kTT - 1; d0 -= kTT, ++grp) {
      typename TL::OutDeep o;
      real *xch = sm.xch + (grp & 1) * kTT * TC;
      if (warp > 0) prog_wait(prog, warp - 1, ev);
      if constexpr (CH) {
        if (warp + 2 < NW) prog_wait(prog, warp + 2, ev - kEvPerGroup);
        TL::template outside_deep_chain<TC>(c, T, ge, sm, scrBif, t, cs, d0, slot, ch, xch, o);
      } else {
        TL::template outside_deep<TC>(c, T, ge, sm, scrBif, t, cs, d0, slot, o);
      }
      prog_signal_smem(prog, warp, lane, ++ev);
#pragma unroll
      for (int k = 0; k < kTT; ++k) {
        ++ev;
        if (d0 - k >= kTurn) {  // uniform
          if ((k > 0 || CH) && warp > 0) prog_wait_smem(prog, warp - 1, ev - 1);
          if (CH && warp >= 2) prog_wait_smem(prog, warp - 2, ev - 1 - k);
          if (warp + 1 < NW) prog_wait_smem(prog, warp + 1, ev - kEvSlackOut);
          TL::template outside_shallow<TC>(c, T, ge, sm, scrBif, t, cs, d0 - k, slot, CH ? xch[k * TC + t] : o.gs[k],
                                           o.bs[k], o.bm1[k], o.ks[k], StepSignal{prog, warp, lane, ev, k == kTT - 1});
        } else {
          prog_signal(prog, warp, lane, ev);
        }
        slot = slot == 0 ? kRingOut - 1 : slot - 1;
      }
    }
    ebase = ev;
  }
}

// Outer arrays (raccess.cpp:230-241, 260-271): serial in the position.  Values stay linear with an exact
// power-of-two rescale; the window of scaled values lives in shared memory; logs are taken 32 positions
// at a time.
// Blocked scan: 32 consecutive positions per round, lane = position.  In "step" coordinates (step = i for
// Alpha_outer, L - i for Beta_outer) both recurrences read  v[st] = v[st-1] + sum_d w(st,d) v[st-d].
//  (0) the weights of the NEXT block stream into the other half of a double buffer with cp.async while
//      this block is computed (the loads are HBM-latency bound, the chain below is shuffle-latency bound);
//  (1) partners before the block: every lane sums its own <= W terms, no communication;
//  (2) partners inside the block: 32 sequential sub-steps, each = one 64-bit broadcast + one FMA on the
//      lanes at distance >= 5; the critical chain is  v[s] = v[s-1] + ext[s]  (ext[s] is final 5 sub-steps
//      earlier), i.e. one shuffle + one add per position.
// wbuf: per-warp 2 x [W + 2][32] weights (each lane only touches its own column), usm: us[] in shared memory.
template <int BYTES>
__device__ __forceinline__ void cp_async_or_zero(void *smem_dst, const void *gsrc, bool pred) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  const int src_bytes = pred ? BYTES : 0;  // 0: nothing is read, the destination is zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;" ::"r"(dst), "l"(gsrc), "n"(BYTES), "r"(src_bytes) : "memory");
}

template <typename real, bool ALPHA>
__device__ void warp_scan(const typename Core<real>::Ctx &c, int sq, double *ring, real *wbuf, const double *usm,
                          int lane) {
  const int L = c.seq_len[sq], W = c.W;
  const long long off = c.seq_off[sq];
  const double kBig = Core<real>::kScanBig, kLn2 = 0.6931471805599453094;  // see scan_alpha_outer (acc_core.h)
  double *dst = ALPHA ? c.lao : c.lbo;
  const real *src = c.arr[A_STEMD];  // cell (st - d, st) sits at column st - d: row stride NC - 1 for Alpha_outer
  const int half = (W + 2) * 32;
  long long e2 = 0;
  if (lane == 0) {
    ring[0] = 1.0;
    dst[off + (ALPHA ? 0 : L)] = 0.0;
  }
  auto stage = [&](int st0, real *buf) {  // this lane's weights of block st0: w(st, d), d = 5 .. W + 1
    const int st = st0 + lane;
    const int dhi = st <= L ? imin(W + 1, st) : 0;
    const long long stride = c.NC - (ALPHA ? 1 : 0);
    const real *p = src + off + (ALPHA ? st : L - st) + 5 * stride;  // running pointers: the address arithmetic of this
    real *q = buf + lane;                                             // loop was 27 % of the kernel's instructions
    for (int d = 5; d <= W + 1; ++d, p += stride, q += 32) cp_async_or_zero<(int)sizeof(real)>(q, d <= dhi ? p : src, d <= dhi);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int cur = 0;
  stage(1, wbuf);
  __syncwarp();
  for (int st0 = 1; st0 <= L; st0 += 32) {
    const int st = st0 + lane;
    const bool ok = st <= L;
    const int i = ALPHA ? st : L - st;
    const int dhi = ok ? imin(W + 1, st) : 0;  // partner step st - d >= 0
    if (st0 + 32 <= L) {
      stage(st0 + 32, wbuf + (cur ^ 1) * half);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    const real *wb = wbuf + cur * half;
    double ext = 0;
    {  // partners before the block: four independent partial sums (the DFMA chain is the latency here)
      double e0 = 0, e1 = 0, e2s = 0, e3 = 0;
      int d = imax(5, lane + 1);
      const real *wp = wb + (d - 5) * 32 + lane;
      for (; d + 3 <= dhi; d += 4, wp += 128) {
        const double w0 = (double)wp[0] * usm[d], w1 = (double)wp[32] * usm[d + 1];
        const double w2 = (double)wp[64] * usm[d + 2], w3 = (double)wp[96] * usm[d + 3];
        e0 += w0 * ring[(st - d) & 255];
        e1 += w1 * ring[(st - d - 1) & 255];
        e2s += w2 * ring[(st - d - 2) & 255];
        e3 += w3 * ring[(st - d - 3) & 255];
      }
      for (; d <= dhi; ++d) e0 += (double)wb[(d - 5) * 32 + lane] * usm[d] * ring[(st - d) & 255];
      ext = (e0 + e1) + (e2s + e3);
    }
    double vprev = ring[(st0 - 1) & 255];
    double myv = 0;
    const int nsub = imin(32, L - st0 + 1);
#pragma unroll 4
    for (int s = 0; s < nsub; ++s) {
      const double vs = __shfl_sync(0xffffffffu, vprev + ext, s);  // lane s holds v[s-1] + ext[s]
      if (lane == s) myv = vs;
      vprev = vs;
      const int dd = lane - s;
      if (dd >= 5 && dd <= dhi) ext += (double)wb[(dd - 5) * 32 + lane] * usm[dd] * vs;
    }
    if (ok) {
      ring[st & 255] = myv;
      dst[off + i] = log(myv) + (double)e2 * kLn2;
    }
    __syncwarp();
    for (int it = 0; it < 4 && vprev > kBig; ++it) {  // uniform (vprev was broadcast): exact power-of-two rescale of the live window
      const int hi = imin(L, st0 + 31), lo = imax(0, hi - W - 2);
      for (int k = lo + lane; k <= hi; k += 32) ring[k & 255] *= 1.0 / kBig;
      vprev *= 1.0 / kBig;
      e2 += Core<real>::kScanBigLog2;
      __syncwarp();
    }
    cur ^= 1;
  }
}

// One warp per (sequence, direction): the two outer arrays of a sequence are independent chains.
template <typename real>
__global__ void __launch_bounds__(32 * kScanWarps) k_outer_scans_warp(typename Core<real>::Ctx c) {
  __shared__ double rings[kScanWarps][256];
  __shared__ double usm[kMaxSpan + 8];
  extern __shared__ __align__(16) unsigned char scan_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int k = threadIdx.x; k < kMaxSpan + 8; k += blockDim.x) usm[k] = c.T->us[k];
  __syncthreads();
  const int job = blockIdx.x * (blockDim.x >> 5) + warp;  // job = 2 * sequence + direction
  const int sq = job >> 1;
  if (sq >= c.nseq) return;
  real *wbuf = reinterpret_cast<real *>(scan_smem) + (size_t)warp * 2 * (c.W + 2) * 32;
  if ((job & 1) == 0) warp_scan<real, true>(c, sq, rings[warp], wbuf, usm, lane);
  else warp_scan<real, false>(c, sq, rings[warp], wbuf, usm, lane);
}

// One band-array tile (rows = spans 5..W-1) into shared memory through the bulk-copy engine: one row = one copy,
// issued by one thread, completion on a transaction barrier; cells that do not exist are zeroed afterwards.
// lim: this thread's column limit, lim_halo[32]: limits of the halo columns.
template <typename real, bool LEFT>
__device__ __forceinline__ void load_band_tile_tma(const typename Core<real>::Ctx &c, const typename BiTile<real>::Geo &ge,
                                                   int arr, real *tile, int lim, const int *lim_halo,
                                                   unsigned long long *bar, unsigned parity) {
  typedef BiTile<real> BT;
  const int tid = threadIdx.x, rows = ge.rows, cols = ge.cols;
  if (rows <= 0) return;
  if (tid == 0) {
    // generic-proxy accesses of the tile (the previous pass) are ordered before the copy engine's writes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const unsigned row_bytes = (unsigned)(cols * sizeof(real));
    tma_bar_expect(bar, (unsigned)rows * row_bytes);
    // left: row r starts at column g0.  right (end-indexed): at column g0 - 31 - r, fetched from the aligned address
    // below it (BiTile::row_off); for the first CTAs that is a few elements before the row, inside the array (r >= 5)
    const real *src = c.arr[arr] + 5 * c.NC + ge.g0;
    for (int r = 0; r < rows; ++r)
      tma_copy_g2s(tile + (size_t)r * cols, src + (long long)r * c.NC - (LEFT ? 0 : 31 + r + 5 + BT::row_off(ge, false, r + 5)),
                   row_bytes, bar);
  }
  tma_bar_wait(bar, parity);
  // mask: a cell of span r exists iff r <= limit of its column (own column, then the 32 halo columns)
  for (int r = lim + 1 > 5 ? lim + 1 : 5; r < rows + 5; ++r) tile[(size_t)(r - 5) * cols + tid + BT::row_off(ge, LEFT, r)] = 0;
  if (tid < 32) {
    const int lh = lim_halo[tid];
    for (int r = lh + 1 > 5 ? lh + 1 : 5; r < rows + 5; ++r)
      tile[(size_t)(r - 5) * cols + ge.TXb + tid + BT::row_off(ge, LEFT, r)] = 0;
  }
}

template <typename real, bool LEFT, int ULO, int TXB>
__global__ void __launch_bounds__(TXB > 0 ? TXB : 512, TXB == 256 ? 2 : TXB == 192 ? 3 : TXB == 128 ? 4 : 1) k_biloop_tile(typename Core<real>::Ctx c) {
  typedef BiTile<real> BT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typename BT::Geo ge;
  ge.TXb = blockDim.x;
  ge.g0 = (long long)blockIdx.x * ge.TXb;
  ge.cols = BT::tile_cols(LEFT, ge.TXb);
  ge.rows = c.W - 5 > 0 ? c.W - 5 : 0;
  real *tile = reinterpret_cast<real *>(smem_raw);
  uint8_t *list = reinterpret_cast<uint8_t *>(tile + (size_t)ge.rows * ge.cols);
  int *lim_halo = reinterpret_cast<int *>(list + (size_t)(c.W + 1) * ge.TXb);  // (W + 1) * TXb is a multiple of 4
  unsigned long long *bar = reinterpret_cast<unsigned long long *>(
      (reinterpret_cast<uintptr_t>(lim_halo + 32) + 7) & ~(uintptr_t)7);  // inside the 64 spare bytes of bi_bytes()
  constexpr int COLS = TXB > 0 ? TXB + 32 + (LEFT ? 0 : BT::kAl) : 0;  // TXB > 0: the tile row stride is known at compile time
  typename BT::Strand st;
  const int lim = BT::tile_col_limit(c, ge, LEFT, threadIdx.x);
  if (threadIdx.x < 32) lim_halo[threadIdx.x] = BT::tile_col_limit(c, ge, LEFT, ge.TXb + threadIdx.x);
  if (threadIdx.x == 0) tma_bar_init(bar, 1);
  __syncthreads();
  // generic loops out of the Alpha_stemI tile
  load_band_tile_tma<real, LEFT>(c, ge, A_STEMI, tile, lim, lim_halo, bar, 0);
  __syncthreads();
  if (LEFT) BT::template left<COLS, ULO>(c, ge, tile, list, threadIdx.x, st);
  else BT::template right<COLS, ULO>(c, ge, tile, list, threadIdx.x, st);
  __syncthreads();
  // bulges out of the Alpha_stemB tile (same buffer)
  load_band_tile_tma<real, LEFT>(c, ge, A_STEMB, tile, lim, lim_halo, bar, 1);
  __syncthreads();
  if (LEFT) BT::template left_bulge<COLS, ULO>(c, ge, tile, list, threadIdx.x, st);
  else BT::template right_bulge<COLS, ULO>(c, ge, tile, list, threadIdx.x, st);
}

template <typename real, bool LEFT>
void launch_biloop(const typename Core<real>::Ctx &k, unsigned grid, int TXb, size_t smem, cudaStream_t st) {
  const bool d5 = k.delta >= 5;
#define PRIB_BI_LAUNCH(X)                                                         \
  do {                                                                            \
    if (d5) k_biloop_tile<real, LEFT, 5, X><<<grid, TXb, smem, st>>>(k);          \
    else k_biloop_tile<real, LEFT, 2, X><<<grid, TXb, smem, st>>>(k);             \
  } while (0)
  // the tuned widths have the tile row stride (and the CTAs per SM) fixed at compile time
  if (TXb == 256) PRIB_BI_LAUNCH(256);
  else if (TXb == 192) PRIB_BI_LAUNCH(192);
  else if (TXb == 128) PRIB_BI_LAUNCH(128);
  else PRIB_BI_LAUNCH(0);
#undef PRIB_BI_LAUNCH
}

#ifndef PRIB_FIN_CTAS
#define PRIB_FIN_CTAS 8
#endif
template <typename real>
__global__ void __launch_bounds__(kThreads, PRIB_FIN_CTAS) k_finalize(typename Core<real>::Ctx c) {
  const long long g = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (g < c.NC) Core<real>::finalize_position(c, g);
}

// Device-side batch layout (what build_layout() of acc_tables.cpp does on the host for the tests): the host
// only ships the raw sequence bytes; base coding (raccess.cpp:55-68) and the column -> sequence map are
// produced here, one thread per column.
__device__ __forceinline__ uint8_t encode_base_dev(unsigned char ch) {
  ch |= 0x20;  // fold case
  return ch == 'a' ? 1 : ch == 'c' ? 2 : ch == 'g' ? 3 : (ch == 'u' || ch == 't') ? 4 : 0;
}
__global__ void __launch_bounds__(256) k_build_layout(long long NC, int nseq, const long long *seq_off,
                                                       const int32_t *seq_len, const long long *raw_off,
                                                       const unsigned char *raw, uint8_t *S, int32_t *col_seq) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= NC) return;
  int lo = 0, hi = nseq;  // last sequence with seq_off <= g
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (seq_off[mid] <= g) lo = mid + 1;
    else hi = mid;
  }
  const int sq = lo - 1;
  int32_t cs = -1;
  uint8_t b = 0;
  if (sq >= 0) {
    const long long i = g - seq_off[sq];
    if (i <= seq_len[sq]) {
      cs = sq;
      if (i >= 1) b = encode_base_dev(raw[raw_off[sq] + i - 1]);
    }
  }
  S[g] = b;
  col_seq[g] = cs;
}

// Issue-rate probes for the roofline denominators (SURVEY §8d: MEASURED_PEAKS.json has no SFU / FP32 /
// FP64 figure, so they are measured here): 8 independent dependency chains per thread.
template <int OP>
__global__ void __launch_bounds__(256) k_probe(float *sink_f, double *sink_d, int iters) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (OP == 2) {
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = 1.0 + 1e-9 * (tid + k);
    const double m = 1.0000001, b = 1e-7;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int k = 0; k < 8; k++) a[k] = fma(a[k], m, b);
    }
    double t = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) t += a[k];
    if (t == 123.456) sink_d[tid] = t;
  } else {
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = 0.5f + 1e-6f * (float)(tid + k);
    const float m = 1.0000001f, b = 1e-7f;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        if (OP == 0) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(a[k]));
        else a[k] = fmaf(a[k], m, b);
      }
    }
    float t = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) t += a[k];
    if (t == 123.456f) sink_f[tid] = t;
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
thread_local std::string g_err;

int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(PRIB_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));            \
  } while (0)

int rows_of(int a, int W) { return (a == X_ML || a == X_MR || a == X_MLS || a == X_MRS) ? 32 : W + 4; }

long long state_bytes_per_column(int W, size_t real_size) {
  long long r = 0;
  for (int a = 0; a < kNumArr; a++) r += rows_of(a, W);
  return r * (long long)real_size + 2 * (long long)sizeof(double);
}

struct Batch {
  int n = 0;
  long long NC = 0, nt = 0;
  std::vector<int> ids;                      // caller's sequence indices, batch order
  std::vector<long long> acc_off, cond_off;  // absolute float offsets into d_out
  uint8_t *d_S = nullptr;
  int32_t *d_col_seq = nullptr, *d_seq_len = nullptr, *d_flags = nullptr;
  long long *d_seq_off = nullptr, *d_acc_off = nullptr, *d_cond_off = nullptr, *d_raw_off = nullptr;
  unsigned char *d_raw = nullptr;
  long long cap_cols = 0, cap_seqs = 0, cap_raw = 0;  // device buffers are grow-only and reused from stage to stage
};

template <typename real>
struct Engine {
  typedef typename Core<real>::SmallTables ST;
  std::vector<ST *> d_small;  // one per minimum accessible length (they differ in kmul only)
  real *d_int11 = nullptr, *d_int21 = nullptr, *d_int22 = nullptr;
  int TC = 0;
  size_t tile_smem = 0;
  int TXb = 0;            // biloop tile width
  int scan_warps = kScanWarps;  // warps (= scan jobs) per CTA of k_outer_scans_warp
  size_t bi_smem = 0;
  long long max_cols = 0;

  void release() {
    for (ST *t : d_small) cudaFree(t);
    cudaFree(d_int11);
    cudaFree(d_int21);
    cudaFree(d_int22);
    d_small.clear();
    d_int11 = d_int21 = d_int22 = nullptr;
  }
};

}  // namespace

struct prib_ctx {
  prib_acc_params prm{};
  int W = 70;
  // Minimum accessible lengths, increasing.  The inside and outside passes, the outer scans and the range flags do not
  // depend on delta, so they run once per batch; the strand weights and the finalize run once per length.
  std::vector<int> lengths;
  bool use_fp32 = true;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
  // phase events: evp[0..4] open the first five phases; length l closes biloop_left, biloop_right and
  // hairpin_finalize with evp[5 + 3 l], evp[6 + 3 l] and evp[7 + 3 l] (PRIB_NUM_PHASES + 1 events for one length)
  std::vector<cudaEvent_t> evp;
  bool phases_pending = false, kernel_timed = true, stage_timed = true;
  // prib_acc_run: the stage fills the arena batch by batch and launches each batch as soon as it is staged, so the
  // host copy of batch k + 1 runs under the kernels of batch k (prib_acc_stage / _compute on their own do not)
  struct Pipelined {
    bool on = false, launched = false;
    const char *const *seq = nullptr;
    long long fpos = 0;
  } pipe;
  Engine<float> e32;
  Engine<double> e64;
  ExactEngine *ex = nullptr;  // mode 2, and the re-run of the wide engine: the reference's own arithmetic (acc_exact.h)
  long long ex_max_cols = 0;
  WideEngine *wide = nullptr;  // spans above kMaxSpan in modes 0 and 1 (acc_wide.h)
  float *d_log = nullptr;
  int grid_tiles = 0;
  char *d_tile_scratch = nullptr;
  char *d_state = nullptr;
  long long state_cap_bytes = 0;  // current size of d_state (grow-only)
  long long state_budget = 0;     // upper bound of the current stage (batches are sized for it)
  long long budget_default = 0, budget_long = 0;
  void set_budget(long long budget) {
    e64.max_cols = budget / state_bytes_per_column(W, 8) / 32 * 32;
    e32.max_cols = budget / state_bytes_per_column(W, 4) / 32 * 32;
    ex_max_cols = budget / exact_state_bytes_per_column(W) / 32 * 32;
    state_budget = budget;  // the block itself is allocated by the first batch (ensure_state)
  }
  // staged work
  std::vector<Batch> batches;
  std::vector<int32_t> seq_len;     // staged sequences, caller order
  std::vector<long long> seq_pos;   // offset of each sequence's bytes in h_arena
  // One page-locked arena holds the raw bytes of every staged sequence in BATCH order (longest first), so each batch
  // goes to the device straight from it: one host copy per sequence, no per-batch staging buffer and hence no stream
  // synchronisation between batches.  Copies for the FP64 re-run of flagged sequences are appended behind.
  unsigned char *h_arena = nullptr;
  size_t h_arena_cap = 0, h_arena_used = 0;
  unsigned char *h_meta = nullptr;  // page-locked per-batch offset arrays (bump-allocated per stage)
  size_t h_meta_cap = 0, h_meta_used = 0;
  size_t n_batches = 0;           // batches[0..n_batches) are live; the rest keep their buffers for reuse
  float *d_out = nullptr;  // length-major: the packed image of length l starts at l * out_floats
  long long out_floats = 0, out_cap = 0;  // out_floats: one length's image; out_cap: the whole allocation
  long long image_floats() const { return out_floats * (long long)lengths.size(); }
  bool staged = false, computed = false;
  float *h_stage = nullptr;
  long long h_stage_floats = 0;
  int32_t *h_flags = nullptr;
  long long h_flags_cap = 0;
  int32_t *d_bad = nullptr;       // number of non-finite outputs of the current compute (finalize_position)
  int32_t *h_bad = nullptr;
  prib_acc_counters cnt{};
};

namespace {

void free_batch(Batch &b) {
  if (!b.d_S && !b.d_seq_len) {
    b = Batch();
    return;
  }
  cudaFree(b.d_S);
  cudaFree(b.d_col_seq);
  cudaFree(b.d_seq_len);
  cudaFree(b.d_flags);
  cudaFree(b.d_seq_off);
  cudaFree(b.d_acc_off);
  cudaFree(b.d_cond_off);
  cudaFree(b.d_raw_off);
  cudaFree(b.d_raw);
  b = Batch();
}

void free_batches(prib_ctx *c) {
  for (auto &b : c->batches) free_batch(b);
  c->batches.clear();
  c->n_batches = 0;
  if (c->d_out) cudaFree(c->d_out);
  c->d_out = nullptr;
  c->out_cap = 0;
  c->out_floats = 0;
  c->seq_len.clear();
  c->seq_pos.clear();
  c->staged = c->computed = false;
}

template <typename real> Engine<real> &engine(prib_ctx *c);
template <> Engine<float> &engine<float>(prib_ctx *c) { return c->e32; }
template <> Engine<double> &engine<double>(prib_ctx *c) { return c->e64; }

template <typename real>
typename Core<real>::Ctx make_ctx(prib_ctx *c, const Batch &b) {
  Engine<real> &e = engine<real>(c);
  typename Core<real>::Ctx k;
  std::memset(&k, 0, sizeof(k));
  k.NC = b.NC;
  k.W = c->W;
  k.delta = c->lengths[0];  // the inside pass stores A_STEM when 2 is one of the lengths
  k.rows = c->W + 4;
  k.nseq = b.n;
  k.S = b.d_S;
  k.col_seq = b.d_col_seq;
  k.seq_len = b.d_seq_len;
  k.seq_off = b.d_seq_off;
  k.T = e.d_small[0];
  k.e_int11 = e.d_int11;
  k.e_int21 = e.d_int21;
  k.e_int22 = e.d_int22;
  k.log_tbl = c->d_log;
  char *p = c->d_state;
  for (int a = 0; a < kNumArr; a++) {
    k.arr[a] = (real *)p;
    p += (long long)rows_of(a, c->W) * b.NC * (long long)sizeof(real);
  }
  k.lao = (double *)p;
  p += b.NC * (long long)sizeof(double);
  k.lbo = (double *)p;
  k.acc_off = b.d_acc_off;
  k.cond_off = b.d_cond_off;
  k.out = c->d_out;
  k.flags = b.d_flags;
  k.bad = c->d_bad;
  return k;
}

int settle_phases(prib_ctx *c) {
  if (!c->phases_pending) return PRIB_OK;
  CU(cudaEventSynchronize(c->evp.back()));
  for (size_t e = 0; e + 1 < c->evp.size(); e++) {  // the last three phases come once per length
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->evp[e], c->evp[e + 1]));
    c->cnt.phase_ms[e < 4 ? e : 4 + (e - 4) % 3] += ms;
  }
  c->phases_pending = false;
  return PRIB_OK;
}

// The DP state is allocated on first use and only grows (up to the budget fixed at create time): a small job
// does not pay for allocating and freeing 100 GB.
int ensure_state(prib_ctx *c, long long bytes) {
  if (bytes <= c->state_cap_bytes) return PRIB_OK;
  if (bytes > c->state_budget) return fail(PRIB_ECUDA, "internal: batch exceeds the DP state budget");
  CU(cudaStreamSynchronize(c->stream));  // nothing may still be using the old block
  cudaFree(c->d_state);
  c->d_state = nullptr;
  c->state_cap_bytes = 0;
  // batches are built longest-first and filled greedily, so the first one is (nearly) the largest: round up a
  // little to avoid a second allocation for a slightly larger later batch
  long long want = std::min(c->state_budget, bytes + bytes / 16);
  if (cudaMalloc(&c->d_state, (size_t)want) != cudaSuccess) {
    cudaGetLastError();
    want = bytes;
    CU(cudaMalloc(&c->d_state, (size_t)want));
  }
  c->state_cap_bytes = want;
  c->cnt.dp_state_bytes = want;
  return PRIB_OK;
}

// Grows a page-locked buffer, keeping the first `keep` bytes.  The stream is drained first: an asynchronous copy may
// still read the old block.
int grow_pinned(prib_ctx *c, unsigned char **buf, size_t *cap, size_t keep, size_t need) {
  if (need <= *cap) return PRIB_OK;
  CU(cudaStreamSynchronize(c->stream));
  unsigned char *nb = nullptr;
  const size_t want = need + need / 8 + 4096;
  CU(cudaMallocHost(&nb, want));
  if (*buf && keep) std::memcpy(nb, *buf, keep);
  if (*buf) cudaFreeHost(*buf);
  *buf = nb;
  *cap = want;
  return PRIB_OK;
}

// Builds the device-side layout of one batch.  ids: caller's indices (their bytes lie back to back in the arena,
// starting at raw_begin); offsets absolute into d_out.  Everything is enqueued on the stream; nothing waits.
int make_batch(prib_ctx *c, const std::vector<int> &ids, const std::vector<long long> &acc_off,
               const std::vector<long long> &cond_off, Batch &b, size_t raw_begin) {
  b.ids = ids;
  b.acc_off = acc_off;
  b.cond_off = cond_off;
  b.n = (int)ids.size();
  // host side: offsets only; the raw bytes go up as they are, the device builds the layout
  const size_t n1 = (size_t)std::max(b.n, 1);
  // page-locked block of this batch: [seq_off | raw_off (n + 1) | acc_off | cond_off | seq_len]
  const size_t need = (n1 * 4 + 1) * 8 + n1 * 4 + 16;
  if (c->h_meta_used + need > c->h_meta_cap)
    return fail(PRIB_ECUDA, "internal: batch metadata arena too small");
  long long *h_so = reinterpret_cast<long long *>(c->h_meta + c->h_meta_used);
  c->h_meta_used += (need + 15) / 16 * 16;
  long long *h_ro = h_so + n1, *h_ao = h_ro + n1 + 1, *h_co = h_ao + n1;
  int32_t *h_sl = reinterpret_cast<int32_t *>(h_co + n1);
  b.nt = 0;
  long long g = kPad;
  for (int k = 0; k < b.n; k++) {
    const int32_t L = c->seq_len[ids[k]];
    h_sl[k] = L;
    h_so[k] = g;
    h_ro[k] = b.nt;
    h_ao[k] = acc_off[k];
    h_co[k] = cond_off[k];
    g += layout_columns(L);
    b.nt += L;
  }
  h_ro[b.n] = b.nt;
  b.NC = (g + kPad + 31) / 32 * 32;
  const long long raw_bytes = std::max<long long>(b.nt, 1);
  if (b.NC > b.cap_cols) {
    cudaFree(b.d_S);
    cudaFree(b.d_col_seq);
    b.d_S = nullptr;
    b.d_col_seq = nullptr;
    b.cap_cols = 0;
    CU(cudaMalloc(&b.d_S, (size_t)b.NC));
    CU(cudaMalloc(&b.d_col_seq, (size_t)b.NC * sizeof(int32_t)));
    b.cap_cols = b.NC;
  }
  if (raw_bytes > b.cap_raw) {
    cudaFree(b.d_raw);
    b.d_raw = nullptr;
    b.cap_raw = 0;
    CU(cudaMalloc(&b.d_raw, (size_t)raw_bytes));
    b.cap_raw = raw_bytes;
  }
  if ((long long)n1 > b.cap_seqs) {
    cudaFree(b.d_seq_len);
    cudaFree(b.d_flags);
    cudaFree(b.d_seq_off);
    cudaFree(b.d_acc_off);
    cudaFree(b.d_cond_off);
    cudaFree(b.d_raw_off);
    b.d_seq_len = b.d_flags = nullptr;
    b.d_seq_off = b.d_acc_off = b.d_cond_off = b.d_raw_off = nullptr;
    b.cap_seqs = 0;
    CU(cudaMalloc(&b.d_seq_len, n1 * sizeof(int32_t)));
    CU(cudaMalloc(&b.d_flags, n1 * sizeof(int32_t)));
    CU(cudaMalloc(&b.d_seq_off, n1 * sizeof(long long)));
    CU(cudaMalloc(&b.d_acc_off, n1 * sizeof(long long)));
    CU(cudaMalloc(&b.d_cond_off, n1 * sizeof(long long)));
    CU(cudaMalloc(&b.d_raw_off, (n1 + 1) * sizeof(long long)));
    b.cap_seqs = (long long)n1;
  }
  if (b.nt > 0)
    CU(cudaMemcpyAsync(b.d_raw, c->h_arena + raw_begin, (size_t)b.nt, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(b.d_seq_len, h_sl, (size_t)b.n * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(b.d_seq_off, h_so, (size_t)b.n * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(b.d_raw_off, h_ro, (size_t)(b.n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(b.d_acc_off, h_ao, (size_t)b.n * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(b.d_cond_off, h_co, (size_t)b.n * 8, cudaMemcpyHostToDevice, c->stream));
  k_build_layout<<<(unsigned)((b.NC + 255) / 256), 256, 0, c->stream>>>(b.NC, b.n, b.d_seq_off, b.d_seq_len,
                                                                         b.d_raw_off, b.d_raw, b.d_S, b.d_col_seq);
  CU(cudaGetLastError());
  c->cnt.h2d_bytes += b.nt + (long long)b.n * 36 + 8;
  c->cnt.kernel_launches += 1;
  return PRIB_OK;
}

int launch_staged_batch(prib_ctx *c, const Batch &b);

// Greedy partition of `order` (already longest-first; the bytes of order[k] lie in the arena in this order, starting
// at raw_begin) into batches that fit `max_cols` columns.
int partition(prib_ctx *c, const std::vector<int> &order, long long max_cols, const std::vector<long long> &acc_abs,
              const std::vector<long long> &cond_abs, std::vector<Batch> &out, size_t *n_live, size_t raw_begin) {
  size_t pos = 0, used = 0;
  {  // metadata arena for all batches of this partition (a bound: every batch pads to 16 bytes and has n + 1 offsets)
    const size_t need = c->h_meta_used + order.size() * 100 + 4096;
    int rc = grow_pinned(c, &c->h_meta, &c->h_meta_cap, c->h_meta_used, need);
    if (rc != PRIB_OK) return rc;
  }
  while (pos < order.size()) {
    std::vector<int> ids;
    std::vector<long long> ao, co;
    long long cols = 2 * kPad;
    size_t bytes = 0;
    while (pos < order.size() && cols + layout_columns(c->seq_len[order[pos]]) <= max_cols) {
      cols += layout_columns(c->seq_len[order[pos]]);
      bytes += (size_t)c->seq_len[order[pos]];
      ids.push_back(order[pos]);
      ao.push_back(acc_abs[order[pos]]);
      co.push_back(cond_abs[order[pos]]);
      pos++;
    }
    if (ids.empty())
      return fail(PRIB_ECUDA, "sequence " + std::to_string(order[pos]) + " does not fit the device DP budget");
    if (used == out.size()) out.emplace_back();
    if (c->pipe.on)  // the bytes of this batch, into their place in the arena
      for (int q : ids) std::memcpy(c->h_arena + c->seq_pos[q], c->pipe.seq[q], (size_t)c->seq_len[q]);
    int rc = make_batch(c, ids, ao, co, out[used], raw_begin);
    if (rc != PRIB_OK) return rc;
    if (c->pipe.on) {
      rc = launch_staged_batch(c, out[used]);
      if (rc != PRIB_OK) return rc;
    }
    raw_begin += bytes;
    ++used;
  }
  *n_live = used;
  return PRIB_OK;
}

template <typename real>
int run_batch(prib_ctx *c, const Batch &b, bool timed) {
  Engine<real> &e = engine<real>(c);
  if (timed && settle_phases(c) != PRIB_OK) return PRIB_ECUDA;
  const long long used = state_bytes_per_column(c->W, sizeof(real)) * b.NC;
  if (ensure_state(c, used) != PRIB_OK) return PRIB_ECUDA;
  const typename Core<real>::Ctx k = make_ctx<real>(c, b);
  cudaStream_t st = c->stream;
  if (used > c->cnt.dp_state_bytes_used) c->cnt.dp_state_bytes_used = used;
  if (timed) CU(cudaEventRecord(c->evp[0], st));
  // the DP state is NOT cleared: every kernel only reads cells written earlier in the same batch
  // (tests/test_hostemu.py::test_no_kernel_reads_a_cell_it_did_not_write poisons the state with NaN)
  CU(cudaMemsetAsync(b.d_flags, 0, sizeof(int32_t) * (size_t)std::max(b.n, 1), st));
  const unsigned grid = (unsigned)((b.NC + kThreads - 1) / kThreads);
  if (timed) CU(cudaEventRecord(c->evp[1], st));
  NvtxRange nvtx_batch("prib:device_batch");
  nvtxRangePushA("prib:inside");
  const int TX = e.TC - (c->W + 1);
  const long long ntiles = (b.NC + TX - 1) / TX;
  const int tgrid = (int)std::min<long long>(ntiles, c->grid_tiles);
  real *scratch = reinterpret_cast<real *>(c->d_tile_scratch);
  if (Tile<real>::first_group(c->W) & 1) k_inside_tile<real, 1><<<tgrid, e.TC, e.tile_smem, st>>>(k, TX, ntiles, scratch);
  else k_inside_tile<real, 0><<<tgrid, e.TC, e.tile_smem, st>>>(k, TX, ntiles, scratch);
  if (timed) CU(cudaEventRecord(c->evp[2], st));
  nvtxRangePop();
  nvtxRangePushA("prib:outer_scans");
  k_outer_scans_warp<real><<<(2 * b.n + e.scan_warps - 1) / e.scan_warps, 32 * e.scan_warps,
                             (size_t)e.scan_warps * 2 * (c->W + 2) * 32 * sizeof(real), st>>>(k);
  if (timed) CU(cudaEventRecord(c->evp[3], st));
  nvtxRangePop();
  nvtxRangePushA("prib:outside");
  k_outside_tile<real><<<tgrid, e.TC, e.tile_smem, st>>>(k, TX, ntiles, scratch);
  if (timed) CU(cudaEventRecord(c->evp[4], st));
  nvtxRangePop();
  // per length: its delta, its tables and its slice of the output image; the strand-weight arrays are overwritten
  const unsigned bgrid = (unsigned)((b.NC + e.TXb - 1) / e.TXb);
  for (size_t l = 0; l < c->lengths.size(); ++l) {
    typename Core<real>::Ctx kl = k;
    kl.delta = c->lengths[l];
    kl.T = e.d_small[l];
    kl.out = c->d_out + (long long)l * c->out_floats;
    nvtxRangePushA("prib:strand_weights");
    launch_biloop<real, true>(kl, bgrid, e.TXb, e.bi_smem, st);
    if (timed) CU(cudaEventRecord(c->evp[5 + 3 * l], st));
    launch_biloop<real, false>(kl, bgrid, e.TXb, e.bi_smem, st);
    if (timed) CU(cudaEventRecord(c->evp[6 + 3 * l], st));
    nvtxRangePop();
    nvtxRangePushA("prib:finalize");  // the hairpin suffix sums come out of the left strand-weight kernel
    k_finalize<real><<<grid, kThreads, 0, st>>>(kl);
    if (timed) CU(cudaEventRecord(c->evp[7 + 3 * l], st));
    nvtxRangePop();
  }
  CU(cudaGetLastError());
  if (timed) c->phases_pending = true;
  c->cnt.kernel_launches += 3 + 3 * (long long)c->lengths.size();
  c->cnt.batches += 1;
  return PRIB_OK;
}

ExactBatch exact_batch(prib_ctx *c, const Batch &b) {
  ExactBatch eb;
  eb.NC = b.NC;
  eb.n = b.n;
  eb.S = b.d_S;
  eb.col_seq = b.d_col_seq;
  eb.seq_len = b.d_seq_len;
  eb.seq_off = b.d_seq_off;
  eb.acc_off = b.d_acc_off;
  eb.cond_off = b.d_cond_off;
  eb.out = c->d_out;
  eb.out_stride = c->out_floats;
  return eb;
}

// mode 2 and the re-run of the wide engine's flagged sequences: every kernel of acc_exact.cu for one batch (phase
// events in the same slots as the fast engines)
int run_batch_exact(prib_ctx *c, const Batch &b, bool timed) {
  if (timed && settle_phases(c) != PRIB_OK) return PRIB_ECUDA;
  const long long used = exact_state_bytes_per_column(c->W) * b.NC;
  if (ensure_state(c, used) != PRIB_OK) return PRIB_ECUDA;
  if (used > c->cnt.dp_state_bytes_used) c->cnt.dp_state_bytes_used = used;
  int launches = 0;
  const int e = exact_run(c->ex, exact_batch(c, b), c->d_state, c->stream, timed ? c->evp.data() : nullptr, &launches);
  if (e != 0) return fail(PRIB_ECUDA, std::string("exact engine: ") + cudaGetErrorString((cudaError_t)e));
  if (timed) c->phases_pending = true;
  c->cnt.kernel_launches += launches;
  c->cnt.batches += 1;
  return PRIB_OK;
}

// spans above kMaxSpan (modes 0 and 1): every kernel of acc_wide.cu for one batch; flags come back like the FP32
// engine's
int run_batch_wide(prib_ctx *c, const Batch &b) {
  if (settle_phases(c) != PRIB_OK) return PRIB_ECUDA;
  const long long used = wide_state_bytes_per_column(c->W) * b.NC;
  if (ensure_state(c, used) != PRIB_OK) return PRIB_ECUDA;
  if (used > c->cnt.dp_state_bytes_used) c->cnt.dp_state_bytes_used = used;
  int launches = 0;
  const int e = wide_run(c->wide, exact_batch(c, b), b.d_flags, c->d_bad, c->d_state, c->stream, c->evp.data(), &launches);
  if (e != 0) return fail(PRIB_ECUDA, std::string("wide-span engine: ") + cudaGetErrorString((cudaError_t)e));
  c->phases_pending = true;
  c->cnt.kernel_launches += launches;
  c->cnt.batches += 1;
  return PRIB_OK;
}

template <typename real>
int setup_engine(prib_ctx *c, const ScaleSpec &spec, size_t smem_max, std::string &err) {
  Engine<real> &e = engine<real>(c);
  HostTablesT<real> tab;
  typedef typename Core<real>::SmallTables ST;
  for (int delta : c->lengths) {  // the small tables per length; everything uploaded below depends on no delta
    if (!build_tables(c->W, delta, spec, tab, err)) return PRIB_EINVAL;
    e.d_small.push_back(nullptr);
    CU(cudaMalloc(&e.d_small.back(), sizeof(ST)));
    CU(cudaMemcpy(e.d_small.back(), &tab.small, sizeof(ST), cudaMemcpyHostToDevice));
  }
  CU(cudaMalloc(&e.d_int11, tab.e_int11.size() * sizeof(real)));
  CU(cudaMemcpy(e.d_int11, tab.e_int11.data(), tab.e_int11.size() * sizeof(real), cudaMemcpyHostToDevice));
  CU(cudaMalloc(&e.d_int21, tab.e_int21.size() * sizeof(real)));
  CU(cudaMemcpy(e.d_int21, tab.e_int21.data(), tab.e_int21.size() * sizeof(real), cudaMemcpyHostToDevice));
  CU(cudaMalloc(&e.d_int22, tab.e_int22.size() * sizeof(real)));
  CU(cudaMemcpy(e.d_int22, tab.e_int22.data(), tab.e_int22.size() * sizeof(real), cudaMemcpyHostToDevice));
  if (sizeof(real) == 8) {
    CU(cudaMemcpyToSymbol(g_conv_d, &tab.small.conv[0][0], sizeof(real) * 32 * 32));
    CU(cudaMemcpyToSymbol(g_bulge_d, tab.small.e_bulge, sizeof(real) * 32));
    CU(cudaMemcpyToSymbol(g_cf_d, tab.small.cf, sizeof(real) * 32));
    CU(cudaMemcpyToSymbol(g_cg_d, tab.small.cg, sizeof(real) * 8));
    {
      const real sc[8] = {tab.small.k2, tab.small.inv_cA, tab.small.e_mlbase, tab.small.e_mlintern, tab.small.e_mlclose, 0, 0, 0};
      CU(cudaMemcpyToSymbol(g_scal_d, sc, sizeof(sc)));
    }
  } else {
    CU(cudaMemcpyToSymbol(g_conv_f, &tab.small.conv[0][0], sizeof(real) * 32 * 32));
    CU(cudaMemcpyToSymbol(g_bulge_f, tab.small.e_bulge, sizeof(real) * 32));
    CU(cudaMemcpyToSymbol(g_cf_f, tab.small.cf, sizeof(real) * 32));
    CU(cudaMemcpyToSymbol(g_cg_f, tab.small.cg, sizeof(real) * 8));
    {
      const real sc[8] = {tab.small.k2, tab.small.inv_cA, tab.small.e_mlbase, tab.small.e_mlintern, tab.small.e_mlclose, 0, 0, 0};
      CU(cudaMemcpyToSymbol(g_scal_f, sc, sizeof(sc)));
    }
    float2 pairs[64];
    for (int a = 0; a < 8; a++)
      for (int b = 0; b < 8; b++)
        pairs[a * 8 + b] = make_float2(a < 7 ? (float)tab.small.cg[a] : 0.f, b < 7 ? (float)tab.small.cg[b] : 0.f);
    CU(cudaMemcpyToSymbol(g_cgpair_f, pairs, sizeof(pairs)));
    std::vector<float2> cp(32 * 32, make_float2(0.f, 0.f));
    for (int u = 0; u < 32; u++)
      for (int sum = 0; sum < 32; sum++) {
        const int u2a = sum - u, u2b = sum - u - 1;
        const float a = (u2a >= 0 && u2a < 32) ? (float)tab.small.conv[u][u2a] : 0.f;
        const float b = (u + 1 < 32 && u2b >= 0 && u2b < 32) ? (float)tab.small.conv[u + 1][u2b] : 0.f;
        cp[u * 32 + sum] = make_float2(a, b);
      }
    CU(cudaMemcpyToSymbol(g_convpair_f, cp.data(), sizeof(float2) * cp.size()));
  }
  if (c->d_log == nullptr) {
    CU(cudaMalloc(&c->d_log, tab.log_tbl.size() * sizeof(float)));
    CU(cudaMemcpy(c->d_log, tab.log_tbl.data(), tab.log_tbl.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  // (function attributes are per device, not per context: always opt in to the device maximum so that
  //  contexts with different spans can coexist)
  // the widest CTA whose rings fit the opt-in shared memory of this device
  // tile width is a compile-time constant of the kernels (row strides become immediates); it is sized
  // for the 227 KB opt-in shared memory of sm_100
  const int TC = TileMaxThreads<real>::value;
  if (tile_smem_bytes<real>() > smem_max)
    return fail(PRIB_ECUDA, "this GPU has less opt-in shared memory than the sm_100a tile kernels need");
  if (TC < c->W + 34) return fail(PRIB_ECUDA, "tile narrower than the span halo");
  e.TC = TC;
  e.tile_smem = tile_smem_bytes<real>();
  CU(cudaFuncSetAttribute((k_inside_tile<real, 0>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
  CU(cudaFuncSetAttribute((k_inside_tile<real, 1>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
  CU(cudaFuncSetAttribute(k_outside_tile<real>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
  // interior-loop tiles: the widest block (<= 512 threads) whose Alpha_stemI tile + span lists fit
  const int rows = c->W - 5 > 0 ? c->W - 5 : 0;
  int TXb = 256;  // two CTAs per SM: one loads its tile while the other computes (measured: 256 beats 512)
  if (const char *te = getenv("PRIB_TXB")) TXb = std::max(32, std::min(512, atoi(te) / 32 * 32));  // tuning knob
  auto bi_bytes = [&](int txb) {
    return (size_t)rows * (txb + 32 + 4) * sizeof(real) + (size_t)(c->W + 1) * txb + 32 * sizeof(int) + 64;  // + 4: right tile's alignment slack
  };
  while (TXb > 32 && bi_bytes(TXb) > smem_max) TXb -= 32;
  e.TXb = TXb;
  e.bi_smem = bi_bytes(TXb);
  if (e.bi_smem > smem_max) return fail(PRIB_ECUDA, "shared memory too small for the interior-loop tiles");
  CU(cudaFuncSetAttribute(k_outer_scans_warp<real>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                          (int)(smem_max - 16 * 1024)));
  {  // double-buffered weights per warp: as many warps per CTA as fit (wide spans in FP64 take > 100 KB each)
    const size_t per_warp = (size_t)2 * (c->W + 2) * 32 * sizeof(real);
    e.scan_warps = (int)std::max<size_t>(1, std::min<size_t>(kScanWarps, (smem_max - 16 * 1024) / per_warp));
    if (per_warp > smem_max - 16 * 1024) return fail(PRIB_ECUDA, "shared memory too small for the outer-array scans");
  }
#define PRIB_BI_ATTR(L, U, X) \
  CU(cudaFuncSetAttribute((k_biloop_tile<real, L, U, X>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max))
  PRIB_BI_ATTR(true, 5, 256); PRIB_BI_ATTR(true, 2, 256); PRIB_BI_ATTR(false, 5, 256); PRIB_BI_ATTR(false, 2, 256);
  PRIB_BI_ATTR(true, 5, 192); PRIB_BI_ATTR(true, 2, 192); PRIB_BI_ATTR(false, 5, 192); PRIB_BI_ATTR(false, 2, 192);
  PRIB_BI_ATTR(true, 5, 128); PRIB_BI_ATTR(true, 2, 128); PRIB_BI_ATTR(false, 5, 128); PRIB_BI_ATTR(false, 2, 128);
  PRIB_BI_ATTR(true, 5, 0); PRIB_BI_ATTR(true, 2, 0); PRIB_BI_ATTR(false, 5, 0); PRIB_BI_ATTR(false, 2, 0);
#undef PRIB_BI_ATTR
  return PRIB_OK;
}

int settle_kernel_time(prib_ctx *c) {
  if (settle_phases(c) != PRIB_OK) return PRIB_ECUDA;
  if (!c->stage_timed) {  // host-to-device copies + layout kernels of the last stage (events on the stream)
    float ms = 0;
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) c->cnt.h2d_ms += ms;
    else cudaGetLastError();
    c->stage_timed = true;
  }
  if (!c->kernel_timed) {
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->evk0, c->evk1));
    c->cnt.kernel_ms += ms;
    c->kernel_timed = true;
  }
  return PRIB_OK;
}

// What has to be on the stream before the first batch of a compute pass: start-of-pass event, the zeroed output image
// (entries the kernels never write -- acc tail, cond head -- must read 0: raccess.cpp:487-488) and the page-locked
// buffer the range flags of all batches come back to.
int compute_prologue(prib_ctx *c) {
  if (settle_kernel_time(c) != PRIB_OK) return PRIB_ECUDA;
  CU(cudaEventRecord(c->evk0, c->stream));
  CU(cudaMemsetAsync(c->d_out, 0, (size_t)std::max<long long>(c->image_floats(), 1) * sizeof(float), c->stream));
  CU(cudaMemsetAsync(c->d_bad, 0, sizeof(int32_t), c->stream));
  const long long nflags = (long long)c->seq_len.size();
  if ((c->use_fp32 || c->wide) && c->h_flags_cap < nflags) {
    CU(cudaStreamSynchronize(c->stream));
    if (c->h_flags) cudaFreeHost(c->h_flags);
    c->h_flags = nullptr;
    c->h_flags_cap = 0;
    CU(cudaMallocHost(&c->h_flags, sizeof(int32_t) * (size_t)std::max<long long>(nflags, 1)));
    c->h_flags_cap = std::max<long long>(nflags, 1);
  }
  c->pipe.fpos = 0;
  return PRIB_OK;
}

// All kernels of one staged batch, and the copy of its range flags behind them (no wait).
int launch_staged_batch(prib_ctx *c, const Batch &b) {
  if (b.n == 0) return PRIB_OK;
  int rc = c->prm.mode == 2 ? run_batch_exact(c, b, true)
           : c->wide        ? run_batch_wide(c, b)
           : c->use_fp32    ? run_batch<float>(c, b, true)
                            : run_batch<double>(c, b, true);
  if (rc != PRIB_OK) return rc;
  c->cnt.sequences += b.n;
  c->cnt.nucleotides += b.nt;
  if (c->use_fp32 || c->wide) {
    CU(cudaMemcpyAsync(c->h_flags + c->pipe.fpos, b.d_flags, sizeof(int32_t) * (size_t)b.n, cudaMemcpyDeviceToHost, c->stream));
    c->pipe.fpos += b.n;
  }
  return PRIB_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

const char *prib_last_error(void) { return g_err.c_str(); }
void prib_internal_set_error(const char *msg) { g_err = msg ? msg : ""; }  // for the other translation units
const char *prib_version(void) { return "priblast-b200 0.2 (sm_100a; fp32 span-scaled tiles + fp64 re-run)"; }

int prib_acc_create(prib_ctx **out, const prib_acc_params *params) {
  if (!out || !params) return fail(PRIB_EINVAL, "null argument");
  return prib_acc_create_lengths(out, params, 1, &params->min_accessible_length);
}

int prib_acc_create_lengths(prib_ctx **out, const prib_acc_params *params, int32_t n_lengths, const int32_t *lengths) {
  if (!out || !params || !lengths) return fail(PRIB_EINVAL, "null argument");
  *out = nullptr;
  if (n_lengths < 1 || n_lengths > PRIB_MAX_LENGTHS)
    return fail(PRIB_EINVAL, "number of minimum accessible lengths must be in 1.." + std::to_string(PRIB_MAX_LENGTHS));
  // a list names the offending entry; a single length keeps the messages of the reference's one -d value
  auto bad_length = [&](int l, const std::string &msg) {
    return fail(PRIB_EINVAL, n_lengths == 1 ? msg : "lengths[" + std::to_string(l) + "] = " + std::to_string(lengths[l]) + ": " + msg);
  };
  for (int l = 0; l < n_lengths; l++)
    if (lengths[l] <= 1) return bad_length(l, "Error: -d option must be greater than 1");  // raccess.hpp:47-50
  if (params->maximal_span < 1 || params->maximal_span > kWideSpan)
    return fail(PRIB_EINVAL, "maximal span must be in 1.." + std::to_string((int)kWideSpan));
  for (int l = 0; l < n_lengths; l++)
    if (lengths[l] > kWideSpan)
      return bad_length(l, "minimum accessible length must be in 2.." + std::to_string((int)kWideSpan));
  for (int l = 1; l < n_lengths; l++)
    if (lengths[l] <= lengths[l - 1]) return bad_length(l, "minimum accessible lengths must be strictly increasing");
  if (params->mode < 0 || params->mode > 2)
    return fail(PRIB_EINVAL, "mode must be 0 (auto), 1 (fp64 only) or 2 (exact: reference arithmetic)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(PRIB_ECUDA, "no CUDA device available (this library has no CPU fallback)");
  if (params->device < 0 || params->device >= ndev) return fail(PRIB_EINVAL, "device ordinal out of range");
  CU(cudaSetDevice(params->device));

  prib_ctx *c = new (std::nothrow) prib_ctx();
  if (!c) return fail(PRIB_ENOMEM, "out of host memory");
  c->prm = *params;
  c->W = params->maximal_span;
  c->lengths.assign(lengths, lengths + n_lengths);
  c->evp.assign(PRIB_NUM_PHASES + 1 + 3 * (n_lengths - 1), nullptr);
  const char *pe = getenv("PRIB_PRECISION");
  int fp32_max_span = kFp32MaxSpan;
  if (const char *me = getenv("PRIB_FP32_MAXSPAN")) fp32_max_span = atoi(me);  // tuning knob
  c->use_fp32 = params->mode == 0 && c->W <= fp32_max_span && c->W <= kMaxSpan && !(pe && strcmp(pe, "fp64") == 0);
  const bool wide = c->W > kMaxSpan && params->mode != 2;  // the tile kernels stop at kMaxSpan
  auto bail = [&](int code) {
    std::string keep = g_err;
    prib_acc_destroy(c);
    g_err = keep;
    return code;
  };
#define CUB(call)                                                                             \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return bail(fail(PRIB_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_)));      \
  } while (0)
  CUB(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  c->stream = c->own_stream;
  CUB(cudaEventCreate(&c->ev0));
  CUB(cudaEventCreate(&c->ev1));
  CUB(cudaEventCreate(&c->evk0));
  CUB(cudaEventCreate(&c->evk1));
  for (auto &e : c->evp) CUB(cudaEventCreate(&e));
  CUB(cudaMalloc(&c->d_bad, sizeof(int32_t)));
  CUB(cudaMallocHost(&c->h_bad, sizeof(int32_t)));
  *c->h_bad = 0;
  cudaDeviceProp prop;
  CUB(cudaGetDeviceProperties(&prop, params->device));
  c->grid_tiles = prop.multiProcessorCount;
  std::string err;
  int rc = PRIB_OK;
  if (c->W <= kMaxSpan) {
    rc = setup_engine<double>(c, ScaleSpec(), prop.sharedMemPerBlockOptin, err);
    if (rc != PRIB_OK) return bail(rc == PRIB_EINVAL ? fail(rc, err) : rc);
  }
  if (wide) {
    double klog2 = default_scale_wide().klog2;
    if (const char *e = getenv("PRIB_WIDE_KLOG2")) klog2 = atof(e);  // tuning knob (profiles/scale_scan.py <W> <n> wide)
    c->wide = wide_create(c->W, c->lengths, klog2, err);
    if (!c->wide) return bail(fail(PRIB_ECUDA, err));
  }
  if (c->use_fp32) {
    ScaleSpec sp32 = default_scale_fp32();
    if (const char *e = getenv("PRIB_KLOG2")) sp32.klog2 = atof(e);  // tuning knobs (profiles/scale_scan.py)
    if (const char *e = getenv("PRIB_ALOG2")) sp32.alog2 = atof(e);
    if (const char *e = getenv("PRIB_BLOG2")) sp32.blog2 = atof(e);
    rc = setup_engine<float>(c, sp32, prop.sharedMemPerBlockOptin, err);
    if (rc != PRIB_OK) return bail(rc == PRIB_EINVAL ? fail(rc, err) : rc);
  }
  if (params->mode == 2 || wide) {
    c->ex = exact_create(c->W, c->lengths, err);
    if (!c->ex) return bail(fail(PRIB_ECUDA, err));
  }
  const size_t scr64 = (size_t)2 * (c->W + 4) * c->e64.TC * sizeof(double);
  const size_t scr32 = (size_t)2 * (c->W + 4) * c->e32.TC * sizeof(float);
  if (!wide) CUB(cudaMalloc(&c->d_tile_scratch, (size_t)c->grid_tiles * std::max(scr64, scr32)));

  size_t free_b = 0, total_b = 0;
  CUB(cudaMemGetInfo(&free_b, &total_b));
  // Default DP budget: 32 GiB per device batch (~6 M nt at W = 70: thousands of tiles per launch, so nothing is lost
  // against one huge batch) instead of most of the HBM — allocating and tearing down a 100 GB block costs ~0.5 s per
  // process, more than the whole accessibility step of a 25 M nt shard.  Long sequences need more: a caller (or the
  // stage call, below) raises it up to 90 % of the free memory.
  long long budget = params->max_batch_bytes > 0 ? params->max_batch_bytes
                                                 : std::min<long long>((long long)(free_b * 0.6), 32LL << 30);
  if (budget > (long long)(free_b * 0.9)) budget = (long long)(free_b * 0.9);
  // Long sequences (mean > 8 kb, e.g. lncRNA sets) get the large budget when no explicit one was given: the two
  // outer-array chains of a 100 kb sequence are a fixed ~16 ms per BATCH, so fewer, larger batches keep the scans
  // below a tenth of the step (prib_acc_stage decides per call).
  c->budget_long = params->max_batch_bytes > 0 ? budget : std::max<long long>(budget, (long long)(free_b * 0.6));
  c->budget_default = budget;
  c->e64.max_cols = budget / state_bytes_per_column(c->W, 8) / 32 * 32;
  if (c->e64.max_cols < 4096) return bail(fail(PRIB_ECUDA, "device memory budget too small for the DP state"));
  c->set_budget(budget);
#undef CUB
  *out = c;
  return PRIB_OK;
}

void prib_acc_destroy(prib_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->prm.device);
  free_batches(c);
  cudaFree(c->d_state);
  cudaFree(c->d_tile_scratch);
  c->e32.release();
  c->e64.release();
  exact_destroy(c->ex);
  wide_destroy(c->wide);
  cudaFree(c->d_log);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  if (c->h_arena) cudaFreeHost(c->h_arena);
  if (c->h_meta) cudaFreeHost(c->h_meta);
  if (c->h_flags) cudaFreeHost(c->h_flags);
  if (c->h_bad) cudaFreeHost(c->h_bad);
  cudaFree(c->d_bad);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->evk0) cudaEventDestroy(c->evk0);
  if (c->evk1) cudaEventDestroy(c->evk1);
  for (auto &e : c->evp)
    if (e) cudaEventDestroy(e);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int prib_acc_set_stream(prib_ctx *c, void *cuda_stream) {
  if (!c) return fail(PRIB_EINVAL, "null context");
  c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
  return PRIB_OK;
}

int prib_acc_stage(prib_ctx *c, int32_t n, const char *const *seq, const int32_t *len) {
  NvtxRange nvtx_call("prib_acc_stage");
  if (!c || n < 0 || (n > 0 && (!seq || !len))) return fail(PRIB_EINVAL, "bad argument");
  CU(cudaSetDevice(c->prm.device));
  c->staged = c->computed = false;
  c->n_batches = 0;
  {
    long long total_len = 0;
    for (int k = 0; k < n; k++) total_len += len[k] > 0 ? len[k] : 0;
    c->set_budget(n > 0 && total_len / n > 8192 ? c->budget_long : c->budget_default);
  }
  const long long max_cols = c->prm.mode == 2 ? c->ex_max_cols : c->use_fp32 ? c->e32.max_cols : c->e64.max_cols;
  for (int k = 0; k < n; k++) {
    if (len[k] < 0) return fail(PRIB_EINVAL, "negative sequence length");
    if (layout_columns(len[k]) + 2 * kPad > std::min(max_cols, c->e64.max_cols))
      return fail(PRIB_ECUDA, "sequence " + std::to_string(k) + " does not fit the device DP budget");
  }
  // packed device output image: [acc L | cond L] per sequence in caller order, one image per length
  std::vector<long long> acc_abs(n), cond_abs(n);
  long long o = 0, total = 0;
  c->seq_len.assign(len, len + n);
  for (int k = 0; k < n; k++) {
    acc_abs[k] = o;
    cond_abs[k] = o + len[k];
    o += 2LL * len[k];
    total += len[k];
  }
  c->out_floats = o;
  // longest first (the order of SortSequences, utils.cpp:53-60), then greedy fill of column budgets:
  // neighbours in a batch have similar lengths, which keeps the per-sequence scan warps balanced.
  std::vector<int> order(n);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return len[a] > len[b]; });
  // the one host copy of the input: into the page-locked arena, in batch order
  c->h_arena_used = c->h_meta_used = 0;
  {
    int rc = grow_pinned(c, &c->h_arena, &c->h_arena_cap, 0, (size_t)total + 64);
    if (rc != PRIB_OK) return rc;
    CU(cudaStreamSynchronize(c->stream));  // a previous stage's copies out of the arena / metadata must be done
  }
  c->seq_pos.resize(n);
  {
    size_t p = 0;
    for (int k = 0; k < n; k++) {
      const int q = order[k];
      c->seq_pos[q] = (long long)p;
      if (!c->pipe.on) std::memcpy(c->h_arena + p, seq[q], (size_t)len[q]);  // (pipelined: batch by batch, in partition)
      p += (size_t)len[q];
    }
    c->h_arena_used = p;
  }
  if (c->image_floats() > c->out_cap || !c->d_out) {
    if (c->d_out) cudaFree(c->d_out);
    c->d_out = nullptr;
    c->out_cap = 0;
    CU(cudaMalloc(&c->d_out, (size_t)std::max<long long>(c->image_floats(), 1) * sizeof(float)));
    c->out_cap = std::max<long long>(c->image_floats(), 1);
  }
  if (c->pipe.on) {
    c->pipe.seq = seq;
    int rc = compute_prologue(c);
    if (rc != PRIB_OK) return rc;
  }
  CU(cudaEventRecord(c->ev0, c->stream));
  if (c->pipe.on) CU(cudaEventRecord(c->ev1, c->stream));  // copies and kernels interleave: no separate copy time
  int rc = partition(c, order, max_cols, acc_abs, cond_abs, c->batches, &c->n_batches, 0);
  c->pipe.seq = nullptr;
  if (rc != PRIB_OK) return rc;
  if (!c->pipe.on) CU(cudaEventRecord(c->ev1, c->stream));
  c->stage_timed = false;
  c->pipe.launched = c->pipe.on;
  c->staged = true;
  return PRIB_OK;
}

int prib_acc_compute(prib_ctx *c) {
  NvtxRange nvtx_call("prib_acc_compute");
  if (!c) return fail(PRIB_EINVAL, "null context");
  if (!c->staged) return fail(PRIB_ESTATE, "prib_acc_compute called before prib_acc_stage");
  CU(cudaSetDevice(c->prm.device));
  if (c->pipe.launched) {
    c->pipe.launched = false;  // prib_acc_run: the stage has launched every batch already
  } else {
    int rc = compute_prologue(c);
    if (rc != PRIB_OK) return rc;
    for (size_t bi = 0; bi < c->n_batches; ++bi) {
      rc = launch_staged_batch(c, c->batches[bi]);
      if (rc != PRIB_OK) return rc;
    }
  }
  // range flags of all batches come back with ONE wait after the last batch (each batch has its own flag array)
  long long fpos = 0;
  std::vector<int> flagged;
  if (c->use_fp32 || c->wide) {
    CU(cudaStreamSynchronize(c->stream));
    fpos = 0;
    for (size_t bi = 0; bi < c->n_batches; ++bi) {
      const Batch &b = c->batches[bi];
      for (int k = 0; k < b.n; k++)
        if (const int bits = c->h_flags[fpos + k]) {
          flagged.push_back(b.ids[k]);
          for (int q = 0; q < 4 && c->use_fp32; q++)
            if (bits & (1 << q)) c->cnt.fp32_flagged[q] += 1;
        }
      fpos += b.n;
    }
  }
  if (!flagged.empty()) {
    // re-run in double (FP32 engine) or in the exact engine (wide engine), on the GPU, writing to the same places of
    // the output image
    const size_t nall = c->seq_len.size();
    std::vector<long long> acc_abs(nall), cond_abs(nall);
    long long o = 0;
    for (size_t k = 0; k < nall; k++) {
      acc_abs[k] = o;
      cond_abs[k] = o + (long long)c->seq_len[k];
      o += 2LL * (long long)c->seq_len[k];
    }
    std::stable_sort(flagged.begin(), flagged.end(), [&](int a, int b) { return c->seq_len[a] > c->seq_len[b]; });
    // their bytes, back to back behind the staged ones
    size_t extra = 0;
    for (int q : flagged) extra += (size_t)c->seq_len[q];
    const size_t rerun_begin = c->h_arena_used;
    int rc = grow_pinned(c, &c->h_arena, &c->h_arena_cap, c->h_arena_used, c->h_arena_used + extra + 64);
    if (rc != PRIB_OK) return rc;
    {
      size_t p = rerun_begin;
      for (int q : flagged) {
        std::memcpy(c->h_arena + p, c->h_arena + c->seq_pos[q], (size_t)c->seq_len[q]);
        p += (size_t)c->seq_len[q];
      }
    }
    const size_t meta_keep = c->h_meta_used;
    std::vector<Batch> fb;
    size_t nfb = 0;
    rc = partition(c, flagged, c->wide ? c->ex_max_cols : c->e64.max_cols, acc_abs, cond_abs, fb, &nfb, rerun_begin);
    for (Batch &b : fb) {
      if (rc == PRIB_OK) rc = c->wide ? run_batch_exact(c, b, false) : run_batch<double>(c, b, false);
      if (rc == PRIB_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = fail(PRIB_ECUDA, "re-run failed");
      free_batch(b);
    }
    c->h_meta_used = meta_keep;  // (compute may be called again on the same staged batches)
    if (rc != PRIB_OK) return rc;
    (c->wide ? c->cnt.exact_rerun_sequences : c->cnt.fp64_rerun_sequences) += (long long)flagged.size();
  }
  CU(cudaEventRecord(c->evk1, c->stream));
  c->kernel_timed = false;
  c->computed = true;
  return PRIB_OK;
}

int prib_acc_sync(prib_ctx *c) {
  if (!c) return fail(PRIB_EINVAL, "null context");
  CU(cudaSetDevice(c->prm.device));
  CU(cudaStreamSynchronize(c->stream));
  return settle_kernel_time(c);
}

int prib_acc_fetch(prib_ctx *c, float *out, const int64_t *acc_off, const int64_t *cond_off) {
  NvtxRange nvtx_call("prib_acc_fetch");
  if (!c || !out || !acc_off || !cond_off) return fail(PRIB_EINVAL, "null argument");
  if (!c->computed) return fail(PRIB_ESTATE, "prib_acc_fetch called before prib_acc_compute");
  CU(cudaSetDevice(c->prm.device));
  // Fast path: the caller's buffer is page-locked (prib_host_alloc / cudaHostRegister) and uses the packed
  // [acc L | cond L] layout in caller order, the images of the lengths back to back: the device image is copied
  // straight into it.
  const size_t n = c->seq_len.size();
  const long long total = c->image_floats();
  bool direct = total > 0;
  {
    long long o = 0;
    for (size_t l = 0; l < c->lengths.size(); l++)
      for (size_t k = 0; k < n && direct; k++) {
        const long long L = (long long)c->seq_len[k];
        direct = acc_off[l * n + k] == o && cond_off[l * n + k] == o + L;
        o += 2 * L;
      }
    if (direct) {
      cudaPointerAttributes at;
      direct = cudaPointerGetAttributes(&at, out) == cudaSuccess && at.type == cudaMemoryTypeHost;
      cudaGetLastError();  // an unregistered pointer is not an error for us
    }
  }
  float *dst = out;
  if (!direct) {
    if (c->h_stage_floats < total) {
      if (c->h_stage) cudaFreeHost(c->h_stage);
      c->h_stage = nullptr;
      c->h_stage_floats = 0;
      CU(cudaMallocHost(&c->h_stage, (size_t)total * sizeof(float)));
      c->h_stage_floats = total;
    }
    dst = c->h_stage;
  }
  if (total > 0) {
    CU(cudaEventRecord(c->ev0, c->stream));
    CU(cudaMemcpyAsync(dst, c->d_out, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaEventRecord(c->ev1, c->stream));
  }
  CU(cudaMemcpyAsync(c->h_bad, c->d_bad, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  if (settle_kernel_time(c) != PRIB_OK) return PRIB_ECUDA;
  if (*c->h_bad != 0)
    return fail(PRIB_ENUMERIC, std::to_string(*c->h_bad) + " accessibility value(s) are not finite: the partition function "
                               "left the double range (span too wide for this sequence); nothing was written");
  if (total > 0) {
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    c->cnt.d2h_ms += ms;
    c->cnt.d2h_bytes += total * (long long)sizeof(float);
  }
  if (!direct) {
    long long o = 0;
    for (size_t l = 0; l < c->lengths.size(); l++)
      for (size_t k = 0; k < n; k++) {
        const size_t L = (size_t)c->seq_len[k];
        std::memcpy(out + acc_off[l * n + k], c->h_stage + o, sizeof(float) * L);
        std::memcpy(out + cond_off[l * n + k], c->h_stage + o + L, sizeof(float) * L);
        o += 2LL * (long long)L;
      }
  }
  return PRIB_OK;
}

int prib_acc_run(prib_ctx *c, int32_t n, const char *const *seq, const int32_t *len, float *out,
                 const int64_t *acc_off, const int64_t *cond_off) {
  if (!c) return fail(PRIB_EINVAL, "null context");
  c->pipe.on = true;  // stage and launch batch by batch
  int rc = prib_acc_stage(c, n, seq, len);
  c->pipe.on = false;
  if (rc != PRIB_OK) {
    c->pipe.launched = false;
    return rc;
  }
  rc = prib_acc_compute(c);
  if (rc != PRIB_OK) return rc;
  return prib_acc_fetch(c, out, acc_off, cond_off);
}

int prib_acc_get_counters(prib_ctx *c, prib_acc_counters *out) {
  if (!c || !out) return fail(PRIB_EINVAL, "null argument");
  *out = c->cnt;
  return PRIB_OK;
}

int prib_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

void *prib_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
    g_err = "cudaMallocHost failed";
    return nullptr;
  }
  return p;
}

void prib_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int prib_peak_probe(int32_t device, double *mufu_gops, double *ffma_gops, double *dfma_gops) {
  if (!mufu_gops || !ffma_gops || !dfma_gops) return fail(PRIB_EINVAL, "null argument");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  float *sf = nullptr;
  double *sd = nullptr;
  CU(cudaMalloc(&sf, (size_t)blocks * threads * sizeof(float)));
  CU(cudaMalloc(&sd, (size_t)blocks * threads * sizeof(double)));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  double *outs[3] = {mufu_gops, ffma_gops, dfma_gops};
  for (int op = 0; op < 3; op++) {
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
      CU(cudaEventRecord(e0));
      if (op == 0) k_probe<0><<<blocks, threads>>>(sf, sd, iters);
      if (op == 1) k_probe<1><<<blocks, threads>>>(sf, sd, iters);
      if (op == 2) k_probe<2><<<blocks, threads>>>(sf, sd, iters);
      CU(cudaEventRecord(e1));
      CU(cudaEventSynchronize(e1));
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, e0, e1));
      const double gops = (double)blocks * threads * iters * 8.0 / (ms * 1e6);
      if (rep > 0 && gops > best) best = gops;
    }
    *outs[op] = best;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sf);
  cudaFree(sd);
  return PRIB_OK;
}

int64_t prib_acc_record_bytes(int32_t len, int32_t delta) {
  if (len < delta || delta < 1) return PRIB_EINVAL;
  return 8 + 4 * (2LL * len - delta + 1);
}

int64_t prib_acc_write_record(const float *acc, const float *cond, int32_t len, int32_t delta, void *dst) {
  // raccess.cpp:447-481: count, acc[0..count), L, delta zeros, cond[delta..L)
  if (!acc || !cond || !dst || len < delta || delta < 1) return PRIB_EINVAL;
  char *p = (char *)dst;
  const int32_t n1 = len - delta + 1;
  std::memcpy(p, &n1, 4);
  p += 4;
  std::memcpy(p, acc, 4 * (size_t)n1);
  p += 4 * (size_t)n1;
  std::memcpy(p, &len, 4);
  p += 4;
  std::memset(p, 0, 4 * (size_t)delta);
  std::memcpy(p + 4 * (size_t)delta, cond + delta, 4 * (size_t)(len - delta));
  p += 4 * (size_t)len;
  return (int64_t)(p - (char *)dst);
}

}  // extern "C"
