// Per-cell mathematics of the B200 accessibility path, written once for device code (acc_kernels.cu)
// and for the host emulation harness used by the CPU-side tests (tests/hostemu/).
//
// Formulation (DESIGN.md §2): the reference keeps every DP variable as a natural-log value in double and
// combines terms with a float-precision logsumexp (raccess.cpp:414-419).  Here every band variable is a
// plain Boltzmann weight (linear domain, FP64), so a recurrence term is one multiply-add and the
// reference's "-INF" sentinel is the number 0:
//   * Alpha (inside) band values are local to the span window and stay far inside the FP64 range for
//     W <= kMaxSpan; the two outer arrays grow like exp(0.25 L) and are kept as logs (lao/lbo).
//   * Beta (outside) band values are carried divided by the partition function Z from the start
//     (the recurrences are linear in Beta), so no exp(-Z) is ever applied to a band value.
//   * LoopEnergy for a generic interior loop (raccess.cpp:808-812) factorises into
//     (outer mismatch) x (inner mismatch) x conv[u1][u2]; the two mismatch factors are folded into
//     per-cell copies of the source arrays (…I / …O below), which turns the 496-term inner loops of
//     raccess.cpp:201-215 / 373-386 / 631-662 into a fixed-coefficient 2-D stencil.
// Layout: every band array is span-major, arr[d * NC + g], g = global column = seq_off + left index,
// so that all threads of a warp (consecutive g, same span d) touch consecutive addresses for every
// source offset of every recurrence.  Columns between sequences are zero padding (>= 32), which makes
// all out-of-range neighbours read as 0 and removes the boundary tests of the reference loops.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define PRIB_HD __host__ __device__ __forceinline__
#else
#define PRIB_HD inline
#endif

namespace prib {

enum { kTurn = 3, kMaxLoop = 30, kMaxSpan = 200, kPad = 32 };
// Widest span of the library (the wide-span FP64 engine, acc_wide.cu, and the exact engine); the tile kernels
// stop at kMaxSpan.
enum { kWideSpan = 1000 };

// Band arrays (see DESIGN.md §3 for who reads what).
enum Arr {
  A_STEM = 0,  // Alpha_stem(i,j)                                   raccess.cpp:103-129
  A_STEMI,     // A_STEM * exp(mismatchI[rt t][s[j+1]][s[i]])       inner-pair factor of :810-811
  A_STEMB,     // A_STEM * tau[t]                                   inner-pair TermAU of :789-794
  A_STEMD,     // A_STEM * exp(Dangle(t,i,j))                       :151, :236, :266
  A_STEMEND,   // Alpha_stemend                                     :193-226
  A_MULTI,     // Alpha_multi                                       :177-191
  A_MULTI1,    // Alpha_multi1                                      :164-175
  A_MULTI2,    // Alpha_multi2                                      :145-162
  B_STEM,      // Beta_stem / Z                                     :367-409
  B_STEMO,     // B_STEM * exp(mismatchI[t][s[i+2]][s[j-1]])        outer-pair factor of :810
  B_STEMB,     // B_STEM * tau[t]
  B_MULTI,     // Beta_multi / Z                                    :281-308
  B_MULTI2,    // Beta_multi2 / Z                                   :326-352
  B_MULTIBIF,  // Beta_multibif / Z                                 :354-364
  X_ML,        // rows 0..30: left-strand loop weight  ML[u1][i]    (restructured :644-650)
  X_MR,        // rows 0..30: right-strand loop weight MR[u2][j']   (restructured :652-658)
  X_SUFH,      // suffix sums over span of hairpin-loop weights     (restructured :546-561)
  X_MLS,       // X_MLS[m][i] = sum over u1 >= m of ML[u1][i] (strands LONGER than the window)
  X_MRS,       // same for MR
  kNumArr
};

PRIB_HD int imin(int a, int b) { return a < b ? a : b; }
PRIB_HD int imax(int a, int b) { return a > b ? a : b; }

PRIB_HD int idx11(int t, int t2, int a, int b) { return ((t * 8 + t2) * 5 + a) * 5 + b; }
PRIB_HD int idx21(int t, int t2, int a, int b, int c) { return (((t * 8 + t2) * 5 + a) * 5 + b) * 5 + c; }
PRIB_HD int idx22(int t, int t2, int a, int b, int c, int d) {
  return ((((t * 8 + t2) * 5 + a) * 5 + b) * 5 + c) * 5 + d;
}


// Uniformly indexed stencil coefficients live in __constant__ memory on the device (one LDC broadcast
// per warp instead of a load through L1); filled by the host at context creation.
#if defined(__CUDACC__)
static __constant__ double g_conv_d[32 * 32];
static __constant__ float g_conv_f[32 * 32];
static __constant__ double g_bulge_d[32];
static __constant__ float g_bulge_f[32];
static __constant__ double g_cf_d[32];
static __constant__ float g_cf_f[32];
// (cg[a], cg[b]) for a, b = 0..7 (index 7 = 0): coefficient pairs of the packed FP32 stencils (FFMA2 takes the pair
// as a 64-bit uniform-register operand, so the coefficients cost no vector registers)
static __constant__ float2 g_cgpair_f[64];
// (conv[u][sum - u], conv[u + 1][sum - u - 1]) at [u * 32 + sum]: the coefficient pairs of the packed strand-weight
// pass (two strand lengths per FFMA2; a 64-bit constant operand instead of two LDC + a MOV per pair)
static __constant__ float2 g_convpair_f[32 * 32];
// scalar factors of the shallow steps (k2, inv_cA, e_mlbase, e_mlintern, e_mlclose): constant-bank operands of the
// FMAs instead of shared-memory loads
static __constant__ double g_scal_d[8];
static __constant__ float g_scal_f[8];
// cg[0..6] for the centre-line chain of the tile kernels (acc_tile.h)
static __constant__ double g_cg_d[8];
static __constant__ float g_cg_f[8];
template <typename real> struct ConstTab;
template <> struct ConstTab<double> {
  static __device__ __forceinline__ const double *conv() { return g_conv_d; }
  static __device__ __forceinline__ const double *bulge() { return g_bulge_d; }
  static __device__ __forceinline__ const double *cf() { return g_cf_d; }
  static __device__ __forceinline__ const double *cg() { return g_cg_d; }
  static __device__ __forceinline__ const double *scal() { return g_scal_d; }
};
template <> struct ConstTab<float> {
  static __device__ __forceinline__ const float *conv() { return g_conv_f; }
  static __device__ __forceinline__ const float *bulge() { return g_bulge_f; }
  static __device__ __forceinline__ const float *cf() { return g_cf_f; }
  static __device__ __forceinline__ const float *cg() { return g_cg_f; }
  static __device__ __forceinline__ const float *scal() { return g_scal_f; }
};
#endif

// Everything below is generic in the scalar type of the band arithmetic: Core<double> is the reference
// precision path, Core<float> the fast path (DESIGN.md §2).  CAP is the widest span the span-indexed tables
// hold: kMaxSpan for the tile kernels, kWideSpan for the wide-span engine (acc_wide.cu).
template <typename real, int CAP = kMaxSpan>
struct Core {
// ring of the outer-array scans: a power of two holding the W + 2 live values
static constexpr int kRing = CAP + 8 <= 256 ? 256 : CAP + 8 <= 1024 ? 1024 : 2048;
// Boltzmann factors exp(-E/kT) of the scaled tables of raccess.hpp:105-158 (built on the host).
struct SmallTables {
  // ---- hot part: everything the tile kernels index per cell; the kernels keep a copy of this prefix
  // (kHotBytes) in shared memory so that a lookup is a 30-cycle LDS instead of a trip through L1/L2 ----
  real e_hairpin[CAP + 8];  // [loop size], incl. the lxc37 extrapolation of raccess.cpp:823 (x cA kappa^d)
  real sB[CAP + 8];         // cB * kappa^-d
  real e_mmH[7][5][5];
  real e_mmI[7][5][5];
  real e_stack[7][7];
  real e_d5[8][5];
  real e_d3[8][5];               // includes TermAU for types > 2 (raccess.hpp:132-134)
  real tau[8];                   // exp(TermAU) for types > 2, else 1
  real cg[8];                    // exp(ninio[k]) for k = 0..6 (ninio saturates at 6: energy_par.hpp:173-174)
  real e_mlbase, e_mlintern, e_mlclose;  // e_mlclose = exp(MLclosing + MLintern)
  // Span scaling (DESIGN.md §2.6): stored Alpha-type values are cA * kappa^d * (true value), stored
  // Beta-type values are cB * kappa^-d * (true value / Z).  kappa = cA = cB = 1 in the FP64 build; the
  // FP32 build uses them to centre the dynamic range.  kappa^(u1+u2) is folded into conv / e_bulge /
  // e_int11 / e_int21 / e_int22, kappa into e_mlbase, cA * kappa^d into e_hairpin[d].
  real k2;                       // kappa^2
  real inv_cA;                   // 1 / cA
  int8_t bp[5][5];
  int8_t rt[8];
  int8_t bpr[5][5];              // rt[bp[a][b]]: the reversed pair type in ONE look-up (the shallow steps chain bp -> rt -> table)
  int8_t hot_end[6];             // marks the end of the hot prefix
  // ---- cold part ----
  real e_bulge[32];              // [u] (device copy in __constant__)
  real conv[32][32];             // generic interior loop: cf[u1+u2] * cg[min(|u1-u2|, 6)], else 0
  real cf[32];                   // exp(internal[sum]) (x kappa^sum), 0 below 4
  real kacc;                     // kappa^2 / (cA cB): un-scales Beta_stemend * loop * Alpha_stem products
  real kmul[2];                  // kappa^w / (cA cB) for w = delta, delta + 1 (CalcMultiProbability)
  real hpB[CAP + 8];        // [dd]: kappa^(dd+1) / cB * exp(hairpin length term of loop size dd-1)
  double us[CAP + 8];       // kappa^-d / cA (outer-array scans run un-scaled in double)
  double kT;
  float log_c_log2;              // fmath LogVar::c_log2
};
static_assert(CAP >= kMaxSpan, "the tables of the tile kernels hold kMaxSpan spans");
static constexpr int kHotBytes = (int)((offsetof(SmallTables, hot_end) + 15) / 16 * 16);

struct Ctx {
  long long NC;            // padded number of columns of this batch
  int W, delta, rows;      // rows = W + 4 (spans 0..W+3; W+2, W+3 stay zero)
  int nseq;
  const uint8_t *S;        // base code per column (0 for column of left index 0 and for padding)
  const int32_t *col_seq;  // sequence id per column, -1 for padding
  const int32_t *seq_len;
  const long long *seq_off;
  const SmallTables *T;
  const real *e_int11;     // [8][8][5][5]
  const real *e_int21;     // [8][8][5][5][5]
  const real *e_int22;     // [8][8][5][5][5][5]
  const float *log_tbl;    // fmath log table, 2048 x (app, rev)
  real *arr[kNumArr];
  double *lao, *lbo;       // log Alpha_outer / log Beta_outer per column
  const long long *acc_off, *cond_off;  // float offsets per sequence into out
  float *out;
  int32_t *flags;          // per sequence: set when a stored value leaves the safe range (FP32 build)
  int32_t *bad;            // one counter per batch: outputs that are not finite (0 = all good); may be null

  PRIB_HD real &at(int a, int d, long long g) const { return arr[a][(long long)d * NC + g]; }
  // persistent result of a tile kernel (streaming stores, st.global.cs, were measured here: no difference)
  PRIB_HD void put(int a, int d, long long g, real v) const { arr[a][(long long)d * NC + g] = v; }
  PRIB_HD real ld(int a, int d, long long g) const { return arr[a][(long long)d * NC + g]; }
};


// exp(CalcDangleEnergy(type,a,b)), raccess.cpp:244-256.  sa = s[a], sb1 = s[b+1].
// stencil coefficient tables: constant memory on the device, the SmallTables copy on the host
static PRIB_HD const real *conv_tab(const SmallTables &T) {
#if defined(__CUDA_ARCH__)
  return ConstTab<real>::conv();
#else
  return &T.conv[0][0];
#endif
}
static PRIB_HD const real *cf_tab(const SmallTables &T) {
#if defined(__CUDA_ARCH__)
  return ConstTab<real>::cf();
#else
  return T.cf;
#endif
}
// scalar factors: I = 0 k2, 1 inv_cA, 2 e_mlbase, 3 e_mlintern, 4 e_mlclose
enum { kScK2 = 0, kScInvCA, kScMlBase, kScMlIntern, kScMlClose };
template <int I>
static PRIB_HD real scal(const SmallTables &T) {
#if defined(__CUDA_ARCH__)
  return ConstTab<real>::scal()[I];
#else
  return I == kScK2 ? T.k2 : I == kScInvCA ? T.inv_cA : I == kScMlBase ? T.e_mlbase : I == kScMlIntern ? T.e_mlintern : T.e_mlclose;
#endif
}
static PRIB_HD const real *cg_tab(const SmallTables &T) {
#if defined(__CUDA_ARCH__)
  return ConstTab<real>::cg();
#else
  return T.cg;
#endif
}
// ninio step of a generic loop, compile-time after unrolling
static PRIB_HD int gidx(int u1, int sum) {
  const int k = 2 * u1 - sum;
  const int a = k < 0 ? -k : k;
  return a > 6 ? 6 : a;
}
static PRIB_HD const real *bulge_tab(const SmallTables &T) {
#if defined(__CUDA_ARCH__)
  return ConstTab<real>::bulge();
#else
  return T.e_bulge;
#endif
}

// Range guard of the FP32 build: stored band values must stay in [2^-55, 2^55] (or be exactly 0) so that
// every product of two of them with a table factor, and every sum of a few hundred such products, stays
// a normal float.  NaN and inf fail the first comparison.  Always true for double.
static PRIB_HD bool in_safe_range(real v) {
  if (sizeof(real) == 8) return true;
  const real hi = (real)3.6028797018963968e16, lo = (real)2.7755575615628914e-17;
  return (v <= hi) && (v == 0 || v >= lo);
}
// which side a value left the safe range on: 1 = too large (or NaN), 2 = too small; the host uses it to pick the scale
// of the second FP32 attempt (prib_acc_compute)
static PRIB_HD int range_bits(real v) {
  if (sizeof(real) == 8) return 0;
  const real hi = (real)3.6028797018963968e16, lo = (real)2.7755575615628914e-17;
  return !(v <= hi) ? 1 : (v != 0 && v < lo) ? 2 : 0;
}
static PRIB_HD void raise_flag(int32_t *flag, int bits) {
#if defined(__CUDA_ARCH__)
  atomicOr(flag, bits);
#else
  *flag |= bits;
#endif
}

static PRIB_HD real e_dangle(const SmallTables &T, int t, bool a_gt0, int sa, bool b_lt_L, int sb1) {
  real x = 1;
  if (a_gt0) x *= T.e_d5[t][sa];
  if (b_lt_L) x *= T.e_d3[t][sb1];
  else x *= T.tau[t];
  return x;
}

struct ColInfo {
  int sq, L, i;
};
static PRIB_HD bool col_info(const Ctx &c, long long g, ColInfo &ci) {
  int sq = c.col_seq[g];
  if (sq < 0) return false;
  ci.sq = sq;
  ci.L = c.seq_len[sq];
  ci.i = (int)(g - c.seq_off[sq]);
  return true;
}

// ------------------------------------------------------------------------------------------------
// Inside: one cell (i, j = i + d) of CalcInsideVariable (raccess.cpp:99-228), span-wavefront order.
// Every source lies at a smaller span (SURVEY §7, validated bit-identical for the reference).
// ------------------------------------------------------------------------------------------------
static PRIB_HD void inside_cell(const Ctx &c, long long g, int d) {
  ColInfo ci;
  if (!col_info(c, g, ci)) return;
  const int L = ci.L, i = ci.i, j = i + d;
  if (j > L) return;
  const SmallTables &T = *c.T;
  const uint8_t *s = c.S + g;  // s[k] = code of base i + k
  const int si = s[0], si1 = s[1], sj = s[d], sj1 = s[d + 1];
  const int t = T.bp[si1][sj];

  // Alpha_stem :103-129
  real stem = 0;
  if (t) {
    const int t2 = T.bp[s[2]][s[d - 1]];
    stem = T.k2 * (c.ld(A_STEMEND, d - 2, g + 1) + c.ld(A_STEM, d - 2, g + 1) * T.e_stack[t][T.rt[t2]]);
  }
  // Alpha_multibif :131-143  (multi1 / multi2 are zero below span 5)
  real mb = 0;
  for (int m = 5; m <= d - 5; ++m) mb += c.ld(A_MULTI1, m, g) * c.ld(A_MULTI2, d - m, g + m);
  mb *= T.inv_cA;
  // Alpha_multi2 :145-162, multi1 :164-175, multi :177-191
  const real stemD = t ? stem * e_dangle(T, t, i > 0, si, j < L, sj1) : 0;
  const real m2 = stemD * T.e_mlintern + c.ld(A_MULTI2, d - 1, g) * T.e_mlbase;
  const real m1 = m2 + mb;
  const real mu = c.ld(A_MULTI, d - 1, g + 1) * T.e_mlbase + mb;

  // Alpha_stemend :193-226, closing pair (i, j+1)
  real se = 0;
  const int te = (j != L) ? T.bp[si][sj1] : 0;
  if (te) {
    real acc = T.e_hairpin[d] * (d != 3 ? T.e_mmH[te][si1][sj] : T.tau[te]);  // HairpinEnergy :819-832
    const int smax = imin(kMaxLoop, d - 5);  // u1 + u2 <= smax keeps the inner span >= 5
    if (smax >= 1) {  // 1-nt bulges :786-787
      acc += T.e_bulge[1] * (c.ld(A_STEM, d - 1, g + 1) * T.e_stack[te][T.rt[T.bp[s[2]][sj]]] +
                             c.ld(A_STEM, d - 1, g) * T.e_stack[te][T.rt[T.bp[si1][s[d - 1]]]]);
    }
    if (smax >= 2) {
      const int t2 = T.rt[T.bp[s[2]][s[d - 1]]];  // 1x1 :797-798
      acc += c.ld(A_STEM, d - 2, g + 1) * c.e_int11[idx11(te, t2, si1, sj)];
      real bs = 0;  // longer bulges :788-795; lengths >= 4 first, then 2 and 3 (the order of the tile kernels)
      for (int u = 4; u <= smax; ++u) bs += T.e_bulge[u] * (c.ld(A_STEMB, d - u, g + u) + c.ld(A_STEMB, d - u, g));
      for (int u = 2; u <= imin(3, smax); ++u) bs += T.e_bulge[u] * (c.ld(A_STEMB, d - u, g + u) + c.ld(A_STEMB, d - u, g));
      acc += T.tau[te] * bs;
    }
    if (smax >= 3) {  // 1x2 and 2x1 :799-804
      const int ta = T.rt[T.bp[s[2]][s[d - 2]]];
      acc += c.ld(A_STEM, d - 3, g + 1) * c.e_int21[idx21(te, ta, si1, s[d - 1], sj)];
      const int tb = T.rt[T.bp[s[3]][s[d - 1]]];
      acc += c.ld(A_STEM, d - 3, g + 2) * c.e_int21[idx21(tb, te, sj, si1, s[2])];
    }
    if (smax >= 4) {
      const int tc = T.rt[T.bp[s[3]][s[d - 2]]];  // 2x2 :805-807
      acc += c.ld(A_STEM, d - 4, g + 2) * c.e_int22[idx22(te, tc, si1, s[2], s[d - 1], sj)];
      real gs = 0;  // generic interior loops :808-812 as a fixed stencil over A_STEMI
      for (int sum = 4; sum <= smax; ++sum) {
        const real *row = c.arr[A_STEMI] + (long long)(d - sum) * c.NC + g;
        real rs = 0;
        for (int u1 = 1; u1 < sum; ++u1)
          if (!(sum == 4 && u1 == 2)) rs += T.cg[gidx(u1, sum)] * row[u1];
        gs += T.cf[sum] * rs;
      }
      acc += T.e_mmI[te][si1][sj] * gs;
    }
    const int tt = T.rt[te];  // multiloop closure :217-221
    acc += mu * T.e_mlclose * T.e_d3[tt][si1] * T.e_d5[tt][sj];
    se = acc;
  }

  c.at(A_STEM, d, g) = stem;
  c.at(A_STEMI, d, g) = t ? stem * T.e_mmI[T.rt[t]][sj1][si] : 0;
  c.at(A_STEMB, d, g) = stem * T.tau[t];
  c.at(A_STEMD, d, g) = stemD;
  c.at(A_STEMEND, d, g) = se;
  c.at(A_MULTI, d, g) = mu;
  c.at(A_MULTI1, d, g) = m1;
  c.at(A_MULTI2, d, g) = m2;
}

// ------------------------------------------------------------------------------------------------
// Outer arrays (raccess.cpp:230-241 and :260-271) as scaled linear recurrences; results stored as logs.
// ring: kRing doubles of scratch.  One caller per sequence.
// ------------------------------------------------------------------------------------------------
// Rescaling: the scaled values stay below kScanBig = 2^256 at every check; between two checks a value can grow by at
// most one un-normalised Alpha_stem weight (<= e^405 ~ 2^584 for a perfect 75-bp GC helix at W <= 200, DESIGN.md
// §2.1) times the weight of a short structure, so nothing overflows 2^1024; the rescale repeats until the value is
// back under the threshold.
static constexpr double kScanBig = 1.157920892373162e77;  // 2^256
static constexpr int kScanBigLog2 = 256;

static PRIB_HD void scan_alpha_outer(const Ctx &c, int sq, double *ring) {
  const int L = c.seq_len[sq], W = c.W;
  const long long off = c.seq_off[sq];
  long long e2 = 0;  // true value = ring value * 2^e2
  ring[0] = 1.0;
  c.lao[off] = 0.0;
  for (int i = 1; i <= L; ++i) {
    double v = ring[(i - 1) & (kRing - 1)];
    const int dmax = imin(W + 1, i);
    for (int d = 5; d <= dmax; ++d) v += (double)c.ld(A_STEMD, d, off + i - d) * c.T->us[d] * ring[(i - d) & (kRing - 1)];
    for (int it = 0; it < 4 && v > kScanBig; ++it) {  // bounded: an infinite v (overflowed FP32 weights of a flagged sequence) must not spin
      for (int k = imax(0, i - W - 2); k < i; ++k) ring[k & (kRing - 1)] *= 1.0 / kScanBig;
      v *= 1.0 / kScanBig;
      e2 += kScanBigLog2;
    }
    ring[i & (kRing - 1)] = v;
    c.lao[off + i] = log(v) + (double)e2 * 0.6931471805599453094;
  }
}

static PRIB_HD void scan_beta_outer(const Ctx &c, int sq, double *ring) {
  const int L = c.seq_len[sq], W = c.W;
  const long long off = c.seq_off[sq];
  long long e2 = 0;
  ring[L & (kRing - 1)] = 1.0;
  c.lbo[off + L] = 0.0;
  for (int i = L - 1; i >= 0; --i) {
    double v = ring[(i + 1) & (kRing - 1)];
    const int dmax = imin(W + 1, L - i);
    for (int d = 5; d <= dmax; ++d) v += (double)c.ld(A_STEMD, d, off + i) * c.T->us[d] * ring[(i + d) & (kRing - 1)];
    for (int it = 0; it < 4 && v > kScanBig; ++it) {  // bounded: an infinite v (overflowed FP32 weights of a flagged sequence) must not spin
      for (int k = i + 1; k <= imin(L, i + W + 2); ++k) ring[k & (kRing - 1)] *= 1.0 / kScanBig;
      v *= 1.0 / kScanBig;
      e2 += kScanBigLog2;
    }
    ring[i & (kRing - 1)] = v;
    c.lbo[off + i] = log(v) + (double)e2 * 0.6931471805599453094;
  }
}

// ------------------------------------------------------------------------------------------------
// Outside: one cell (p, q = p + d) of CalcOutsideVariable (raccess.cpp:273-411), descending span.
// All values are Beta / Z.  Beta_stemend(i,j) == B_STEM[d+2][g-1] (rows above W+1 are zero, which is
// the `q - p >= W ? -INF` of :278-279).
// ------------------------------------------------------------------------------------------------
static PRIB_HD void outside_cell(const Ctx &c, long long g, int d) {
  ColInfo ci;
  if (!col_info(c, g, ci)) return;
  const int L = ci.L, p = ci.i, q = p + d, W = c.W;
  if (q > L) return;
  const SmallTables &T = *c.T;
  const uint8_t *s = c.S + g;
  const int sp = s[0], sp1 = s[1], sq_ = s[d], sq1 = s[d + 1];
  const bool inner = (p != 0 && q != L);
  const int te = inner ? T.bp[sp][sq1] : 0;  // pair (p, q+1)
  const real bse = inner ? c.ld(B_STEM, d + 2, g - 1) : 0;

  real bmulti = 0, bmulti2 = 0, bmbif = 0;
  if (inner) {
    // Beta_multi :281-308
    const int tt = T.rt[te];
    bmulti = c.ld(B_MULTI, d + 1, g - 1) * T.e_mlbase + T.k2 * bse * T.e_mlclose * T.e_d3[tt][sp1] * T.e_d5[tt][sq_];
    // Beta_multi1 :310-324   k = q + m
    real bm1 = 0;
    const int m1max = imin(L - q, W - d);
    for (int m = 5; m <= m1max; ++m) bm1 += c.ld(B_MULTIBIF, d + m, g) * c.ld(A_MULTI2, m, g + d);
    bm1 *= T.inv_cA;
    // Beta_multi2 :326-352   k = p - m
    real ks = 0;
    const int m2max = imin(p, W - d);
    for (int m = 5; m <= m2max; ++m) ks += c.ld(B_MULTIBIF, d + m, g - m) * c.ld(A_MULTI1, m, g - m);
    bmulti2 = bm1 + c.ld(B_MULTI2, d + 1, g) * T.e_mlbase + ks * T.inv_cA;
    // Beta_multibif :354-364
    bmbif = bm1 + bmulti;
  }

  // Beta_stem :367-409, inner pair (p+1, q)
  real bstem = 0;
  const int t2 = T.bp[sp1][sq_];
  if (t2) {
    const int t2r = T.rt[t2];
    const real dang = e_dangle(T, t2, p > 0, sp, q < L, sq1);
    const real base = (real)exp(c.lao[g] + c.lbo[g + d] - c.lao[c.seq_off[ci.sq] + L]) * dang * T.sB[d];  // :370
    real ls = 0;  // sum over enclosing loops; sources sit two spans further out than in the inside pass
    const int smax = imin(kMaxLoop, W - 1 - d);  // source row d + sum + 2 <= W + 1
    // stacking on (p, q+1) :388-398
    if (smax >= 0) ls += bse * T.e_stack[te][t2r];
    if (smax >= 1) {  // 1-nt bulges: outer pairs (p-1, q+1) and (p, q+2)
      const int ta = T.bp[s[-1]][sq1];
      const int tb = T.bp[sp][s[d + 2]];
      ls += T.e_bulge[1] * (c.ld(B_STEM, d + 3, g - 2) * T.e_stack[ta][t2r] +
                               c.ld(B_STEM, d + 3, g - 1) * T.e_stack[tb][t2r]);
    }
    if (smax >= 2) {
      const int to = T.bp[s[-1]][s[d + 2]];  // 1x1: outer (p-1, q+2)
      ls += c.ld(B_STEM, d + 4, g - 2) * c.e_int11[idx11(to, t2r, sp, sq1)];
      real bs = 0;
      for (int u = 2; u <= smax; ++u)
        bs += T.e_bulge[u] * (c.ld(B_STEMB, d + u + 2, g - u - 1) + c.ld(B_STEMB, d + u + 2, g - 1));
      ls += T.tau[t2r] * bs;
    }
    if (smax >= 3) {
      const int ta = T.bp[s[-1]][s[d + 3]];  // 1x2: outer (p-1, q+3)
      ls += c.ld(B_STEM, d + 5, g - 2) * c.e_int21[idx21(ta, t2r, sp, sq1, s[d + 2])];
      const int tb = T.bp[s[-2]][s[d + 2]];  // 2x1: outer (p-2, q+2)
      ls += c.ld(B_STEM, d + 5, g - 3) * c.e_int21[idx21(t2r, tb, sq1, s[-1], sp)];
    }
    if (smax >= 4) {
      const int tc = T.bp[s[-2]][s[d + 3]];  // 2x2: outer (p-2, q+3)
      ls += c.ld(B_STEM, d + 6, g - 3) * c.e_int22[idx22(tc, t2r, s[-1], sp, sq1, s[d + 2])];
      real gs = 0;
      for (int sum = 4; sum <= smax; ++sum) {
        const real *row = c.arr[B_STEMO] + (long long)(d + sum + 2) * c.NC + g - 1;
        real rs = 0;
        for (int u1 = 1; u1 < sum; ++u1)
          if (!(sum == 4 && u1 == 2)) rs += T.cg[gidx(u1, sum)] * row[-u1];
        gs += T.cf[sum] * rs;
      }
      ls += T.e_mmI[t2r][sq1][sp] * gs;
    }
    bstem = base + T.k2 * ls + bmulti2 * T.e_mlintern * dang;  // :401-406
  }

  c.at(B_STEM, d, g) = bstem;
  // factors of the pair (p+1, q) seen as an OUTER pair by cells further in
  c.at(B_STEMO, d, g) = t2 ? bstem * T.e_mmI[t2][s[2]][s[d - 1]] : 0;
  c.at(B_STEMB, d, g) = bstem * T.tau[t2];
  c.at(B_MULTI, d, g) = bmulti;
  c.at(B_MULTI2, d, g) = bmulti2;
  c.at(B_MULTIBIF, d, g) = bmbif;
}

// ------------------------------------------------------------------------------------------------
// Accessibility (raccess.cpp:421-771), restructured.
//   T(i,j',u1,u2) = Beta_stemend(i,j') * exp(LoopEnergy) * Alpha_stem(i+u1, j'-u2)
//   ML[u1][i]  = sum over (j',u2) of T      left strand  = bases i+1 .. i+u1
//   MR[u2][j'] = sum over (i ,u1) of T      right strand = bases j'-u2+1 .. j'
// The reference's k-loops (:644-658) add T to every window start k inside a strand; summing the strand
// weights first and gathering per k afterwards gives the same sums.
// ------------------------------------------------------------------------------------------------
static PRIB_HD real loop_weight(const Ctx &c, const SmallTables &T, const uint8_t *s, long long g, int dp, int te,
                         real bse, real bseO, real bseB, int u1, int u2) {
  // s = S + column of i; outer pair (i, j'+1) with j' = i + dp; inner cell (i+u1, j'-u2).
  const int sum = u1 + u2;
  const int dd = dp - sum;  // inner span
  const long long gi = g + u1;
  if (u1 >= 1 && u2 >= 1) {
    if (sum >= 4 && !(u1 == 2 && u2 == 2)) return bseO * T.conv[u1][u2] * c.ld(A_STEMI, dd, gi);
    const real st = c.ld(A_STEM, dd, gi);
    if (st == 0) return 0;
    const int t2r = T.rt[T.bp[s[u1 + 1]][s[dp - u2]]];
    const int si1 = s[1], sj = s[dp];
    if (sum == 2) return bse * st * c.e_int11[idx11(te, t2r, si1, sj)];
    if (u1 == 1 && u2 == 2) return bse * st * c.e_int21[idx21(te, t2r, si1, s[dp - 1], sj)];
    if (u1 == 2 && u2 == 1) return bse * st * c.e_int21[idx21(t2r, te, sj, si1, s[2])];
    return bse * st * c.e_int22[idx22(te, t2r, si1, s[2], s[dp - 1], sj)];
  }
  const int u = u1 + u2;  // bulge
  if (u == 1) {
    const real st = c.ld(A_STEM, dd, gi);
    if (st == 0) return 0;
    const int t2r = T.rt[T.bp[s[u1 + 1]][s[dp - u2]]];
    return bse * st * T.e_bulge[1] * T.e_stack[te][t2r];
  }
  return bseB * T.e_bulge[u] * c.ld(A_STEMB, dd, gi);
}

// thread = left index i; writes ML[u1][g] for u1 in [delta, 30]
static PRIB_HD void biloop_left(const Ctx &c, long long g) {
  ColInfo ci;
  if (!col_info(c, g, ci)) return;
  const int L = ci.L, i = ci.i, W = c.W;
  const SmallTables &T = *c.T;
  const uint8_t *s = c.S + g;
  const int dpmax = imin(W - 1, L - 1 - i);
  for (int u1 = c.delta; u1 <= kMaxLoop; ++u1) {
    real acc = 0;
    if (i >= 1) {
      for (int dp = u1 + 5; dp <= dpmax; ++dp) {
        const real bse = c.ld(B_STEM, dp + 2, g - 1);
        if (bse == 0) continue;
        const int te = T.bp[s[0]][s[dp + 1]];
        const real bseO = c.ld(B_STEMO, dp + 2, g - 1), bseB = c.ld(B_STEMB, dp + 2, g - 1);
        const int u2max = imin(kMaxLoop, dp - 5) - u1;
        for (int u2 = 0; u2 <= u2max; ++u2) acc += loop_weight(c, T, s, g, dp, te, bse, bseO, bseB, u1, u2);
      }
    }
    c.at(X_ML, u1, g) = acc;
  }
  real suf = 0;
  for (int u1 = kMaxLoop; u1 >= c.delta; --u1) {
    suf += c.ld(X_ML, u1, g);
    c.at(X_MLS, u1, g) = suf;
  }
}

// thread = right end j' of the outer cell; writes MR[u2][g'] for u2 in [delta, 30]
static PRIB_HD void biloop_right(const Ctx &c, long long g2) {
  ColInfo ci;
  if (!col_info(c, g2, ci)) return;
  const int L = ci.L, jp = ci.i, W = c.W;
  const SmallTables &T = *c.T;
  for (int u2 = c.delta; u2 <= kMaxLoop; ++u2) {
    real acc = 0;
    if (jp <= L - 1) {
      const int dpmax = imin(W - 1, jp - 1);  // i = jp - dp >= 1
      for (int dp = u2 + 5; dp <= dpmax; ++dp) {
        const long long g = g2 - dp;
        const real bse = c.ld(B_STEM, dp + 2, g - 1);
        if (bse == 0) continue;
        const uint8_t *s = c.S + g;
        const int te = T.bp[s[0]][s[dp + 1]];
        const real bseO = c.ld(B_STEMO, dp + 2, g - 1), bseB = c.ld(B_STEMB, dp + 2, g - 1);
        const int u1max = imin(kMaxLoop, dp - 5) - u2;
        for (int u1 = 0; u1 <= u1max; ++u1) acc += loop_weight(c, T, s, g, dp, te, bse, bseO, bseB, u1, u2);
      }
    }
    c.at(X_MR, u2, g2) = acc;
  }
  real suf = 0;
  for (int u2 = kMaxLoop; u2 >= c.delta; --u2) {
    suf += c.ld(X_MR, u2, g2);
    c.at(X_MRS, u2, g2) = suf;
  }
}

// thread = i; X_SUFH[dd][g] = sum over j >= i+dd of Beta_stemend(i,j-1) * exp(Hairpin(i,j))   (:546-561)
static PRIB_HD void hairpin_suffix(const Ctx &c, long long g) {
  ColInfo ci;
  if (!col_info(c, g, ci)) return;
  const int L = ci.L, i = ci.i, W = c.W;
  const SmallTables &T = *c.T;
  const uint8_t *s = c.S + g;
  real suf = 0;
#pragma unroll 4
  for (int dd = W; dd >= 4; --dd) {
    if (i >= 1 && i + dd <= L) {
      const real bse = c.ld(B_STEM, dd + 1, g - 1);
      if (bse != 0) {
        const int t = T.bp[s[0]][s[dd]];
        suf += bse * T.hpB[dd] * (dd - 1 != 3 ? T.e_mmH[t][s[1]][s[dd - 1]] : T.tau[t]);
      }
    }
    c.at(X_SUFH, dd, g) = suf;
  }
}

// fmath::log(float), fmath.hpp:738-752, with the host-built table (SURVEY Q2).  No FMA contraction.
static PRIB_HD float fmath_logf(const Ctx &c, float x) {
  union { float f; uint32_t u; } v;
  v.f = x;
  const int a = (int)(v.u & (0xFFu << 23));
  const uint32_t idx = (v.u >> 12) & 2047u;
  const uint32_t b2 = v.u & 4095u;
  const float app = c.log_tbl[2 * idx], rev = c.log_tbl[2 * idx + 1];
#if defined(__CUDA_ARCH__)
  const float t1 = __fmul_rn((float)(a - (127 << 23)), c.T->log_c_log2);
  const float t2 = __fadd_rn(t1, app);
  const float t3 = __fmul_rn((float)b2, rev);
  return __fadd_rn(t2, t3);
#else
  volatile float t1 = (float)(a - (127 << 23)) * c.T->log_c_log2;
  volatile float t2 = t1 + app;
  volatile float t3 = (float)b2 * rev;
  return t2 + t3;
#endif
}

// unpaired-window probabilities of one start position x for window lengths w = delta and delta + 1
struct WindowProb {
  real ext, hp, multi, loop_b, loop_c;
};

static PRIB_HD double multi_prob(const Ctx &c, long long off, int L, int x, int w) {  // :581-612
  const int W = c.W;
  double v = 0;
  const int hi = imin(x + W, L);
  for (int e = x + w - 1 + 5; e <= hi; ++e)  // Alpha_multi below span 5 is zero
    v += (double)c.ld(B_MULTI, e - x + 1, off + x - 1) * (double)c.ld(A_MULTI, e - x - w + 1, off + x + w - 1);
  const int lo = imax(0, x + w - 1 - W);
  for (int b = lo; b <= x - 1 - 5; ++b)
    v += (double)c.ld(B_MULTI2, x + w - 1 - b, off + b) * (double)c.ld(A_MULTI2, x - b - 1, off + b);
  return v * (double)c.T->kmul[w - c.delta];
}

// CalcMultiProbability for w = delta and w + 1 in one walk: the two window lengths share every Beta_multi
// element of the first sum and every Alpha_multi2 element of the second (6 loads per step instead of 8); each
// accumulator sees the terms of its own multi_prob() call in the same order, so the results are bit-identical.
static PRIB_HD void multi_prob_pair(const Ctx &c, long long off, int L, int x, int w, double &p0, double &p1) {
  const int W = c.W;
  double v0 = 0, v1 = 0;
  const int hi = imin(x + W, L);
  {
    const int e0 = x + w - 1 + 5;  // first term of the w sum; the w + 1 sum starts one later
    if (e0 <= hi)
      v0 += (double)c.ld(B_MULTI, e0 - x + 1, off + x - 1) * (double)c.ld(A_MULTI, e0 - x - w + 1, off + x + w - 1);
#pragma unroll 4
    for (int e = e0 + 1; e <= hi; ++e) {
      const double b = (double)c.ld(B_MULTI, e - x + 1, off + x - 1);
      v0 += b * (double)c.ld(A_MULTI, e - x - w + 1, off + x + w - 1);
      v1 += b * (double)c.ld(A_MULTI, e - x - w, off + x + w);
    }
  }
  {
    const int lo0 = imax(0, x + w - 1 - W), lo1 = imax(0, x + w - W);
    if (lo1 > lo0 && lo0 <= x - 1 - 5)  // the w sum reaches one column further to the left
      v0 += (double)c.ld(B_MULTI2, x + w - 1 - lo0, off + lo0) * (double)c.ld(A_MULTI2, x - lo0 - 1, off + lo0);
#pragma unroll 4
    for (int b = lo1; b <= x - 1 - 5; ++b) {
      const double a = (double)c.ld(A_MULTI2, x - b - 1, off + b);
      v0 += (double)c.ld(B_MULTI2, x + w - 1 - b, off + b) * a;
      v1 += (double)c.ld(B_MULTI2, x + w - b, off + b) * a;
    }
  }
  p0 = v0 * (double)c.T->kmul[w - c.delta];
  p1 = v1 * (double)c.T->kmul[w + 1 - c.delta];
}

static PRIB_HD double hairpin_prob(const Ctx &c, long long off, int x, int w) {  // :536-579
  double v = 0;
#pragma unroll 4
  for (int i = imax(1, x - c.W); i < x; ++i) {
    const int dd = x + w - i;
    if (dd <= c.W) v += c.ld(X_SUFH, dd < 4 ? 4 : dd, off + i);
  }
  return v;
}

// b[k]: strands that end exactly at the window end; c[k]: strands that extend beyond it (:644-658)
static PRIB_HD void biloop_gather(const Ctx &c, long long off, int L, int k, double &b, double &cc) {
  const int w = c.delta;
  b = 0;
  cc = 0;
#pragma unroll 4
  for (int i = imax(1, k + w - 1 - kMaxLoop); i <= k - 1; ++i) {
    const int ub = k + w - 1 - i;  // strand length whose last base is the window end
    b += c.ld(X_ML, ub, off + i);
    if (ub + 1 <= kMaxLoop) cc += c.ld(X_MLS, ub + 1, off + i);
  }
#pragma unroll 4
  for (int jp = k + w - 1; jp <= imin(L - 1, k + kMaxLoop - 1); ++jp) {
    const int umin = jp - k + 1;  // strand must start before k
    if (jp == k + w - 1) b += c.ld(X_MRS, umin, off + jp);
    else cc += c.ld(X_MRS, umin, off + jp);
  }
  b *= (double)c.T->kacc;
  cc *= (double)c.T->kacc;
}

// Final per-position step: CalcAccessibility :484-528 incl. the finalisation quirks of :667-680 (Q1, Q3)
// and :754-770 (Q4).  thread = x (1-based start position) = left index of column g.
static PRIB_HD void finalize_position(const Ctx &c, long long g) {
  ColInfo ci;
  if (!col_info(c, g, ci)) return;
  const int L = ci.L, x = ci.i, w = c.delta;
  if (x < 1 || x + w - 1 > L) return;
  const long long off = c.seq_off[ci.sq];
  const double Z = c.lao[off + L];
  const double kT = c.T->kT;

  double b, cc;
  biloop_gather(c, off, L, x, b, cc);
  double bp = 0, cbp = 0;
  if (Z >= -690 && Z <= 690) {  // direct path :667-680 — the float cast of the UN-normalised sum is emulated
    const double eZ = exp(Z);
    if (b != 0) bp = exp((double)fmath_logf(c, (float)((b + cc) * eZ)) - Z);
    if (cc != 0) cbp = exp((double)fmath_logf(c, (float)(cc * eZ)) - Z);
  } else {  // log path :754-770
    if (b != 0) bp = b + cc;
    else if (cc != 0) bp = log(cc) + Z;  // Q4: the log-domain value is never exponentiated
    cbp = cc;
  }

  float *acc = c.out + c.acc_off[ci.sq];
  float *cond = c.out + c.cond_off[ci.sq];
  double prob = 0.0;
  prob += exp(c.lao[off + x - 1] + c.lbo[off + x + w - 1] - Z);
  prob += hairpin_prob(c, off, x, w);
  prob += bp;
  const bool has_cond = x + w - 1 < L;
  double mp0, mp1 = 0;
  if (has_cond) multi_prob_pair(c, off, L, x, w, mp0, mp1);
  else mp0 = multi_prob(c, off, L, x, w);
  prob += mp0;
  const float a = (float)((-(double)fmath_logf(c, (float)prob) * kT) / 1000);
  acc[x - 1] = a;
  bool finite = a == a && a - a == 0.f;  // neither NaN nor inf
  if (has_cond) {
    double pc = 0.0;
    pc += exp(c.lao[off + x - 1] + c.lbo[off + x + w] - Z);
    pc += hairpin_prob(c, off, x, w + 1);
    pc += cbp;
    pc += mp1;
    const float cv = (float)((-(double)fmath_logf(c, (float)pc) * kT) / 1000 - a);
    cond[x + w - 1] = cv;
    finite = finite && cv == cv && cv - cv == 0.f;
  }
  // The reference cannot produce a non-finite value here (its log-domain sums saturate); if this path ever does
  // (overflowed partition function), the caller must hear about it instead of finding NaN in <db>.acc.
  if (!finite && c.bad) {
#if defined(__CUDA_ARCH__)
    atomicAdd(c.bad, 1);
#else
    ++*c.bad;
#endif
  }
}

};  // struct Core

}  // namespace prib
