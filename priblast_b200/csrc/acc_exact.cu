// Exact engine: see acc_exact.h.  Compiled with -fmad=false (no FMA contraction anywhere in this file).
//
// Every device function below follows one function of the reference (file:line under /root/reference/src)
// operation by operation; what is re-designed is the execution order ACROSS cells (span wavefront, one thread
// per cell / per position, whole batches of sequences per launch) and the storage (span-major band arrays,
// column = batch-wide left index, so the 32 lanes of a warp touch consecutive addresses).
#include "acc_exact.h"

#include <math.h>
#include <string.h>

#include <new>
#include <vector>

#include "acc_core.h"  // kTurn, kMaxLoop, kWideSpan, kPad
#include "turner_params.h"

namespace prib {
namespace {

#define EX_NEG (-1000000.0) /* the reference's "-INF", energy_par.hpp:8 */

enum ExArr {
  EA_STEM, EA_STEMEND, EA_MULTI, EA_MULTIBIF, EA_MULTI1, EA_MULTI2,
  EB_STEM, EB_STEMEND, EB_MULTI, EB_MULTIBIF, EB_MULTI1, EB_MULTI2,
  kExArr
};
enum { kExVec = 6 };  // ao, bo, hp, chp, bp, cbp: one double per column

constexpr int kExpdBits = 11;              // fmath.hpp:81
constexpr int kExpdN = 1 << kExpdBits;
constexpr int kLogBits = 11;               // fmath.hpp:82,182
constexpr int kLogN = 1 << kLogBits;

struct ExTab {
  double hairpin[kWideSpan + 8];  // by loop size, with the lxc37 extrapolation of raccess.cpp:823 precomputed
  double bulge[31], internal[31], ninio[kMaxLoop + 1];
  double mmH[7][5][5], mmI[7][5][5], stack[7][7], d5[8][5], d3[8][5];
  double MLclosing, MLintern, MLbase, TermAU, kT;
  double expd_a, expd_ra;
  float c_log2;
  int bp[5][5], rt[8];
  double int11[8 * 8 * 5 * 5];
  unsigned long long expd_tbl[kExpdN];
  float log_tbl[2 * kLogN];
};

struct ExCtx {
  long long NC;
  int W, delta, nseq;
  const uint8_t *S;
  const int32_t *col_seq, *seq_len;
  const long long *seq_off, *acc_off, *cond_off;
  const ExTab *T;
  const double *int21, *int22;
  double *band;  // [kExArr][W + 2][NC]
  double *vec;   // [kExVec][NC]
  float *out;
};

// ---- fmath primitives (fmath.hpp:439-462 expd, SSE2 branch; :738-752 log) ------------------------------
__device__ __forceinline__ double ex_expd(const ExTab &T, double x) {
  if (x <= -708.39641853226408) return 0;
  if (x >= 709.78271289338397) return __longlong_as_double(0x7ff0000000000000LL);
  const double b = (double)(3ULL << 51);
  const double d = x * T.expd_a + b;  // -fmad=false: a multiply, then an add
  const unsigned long long di =
      (unsigned long long)(long long)(int)(unsigned int)(unsigned long long)__double_as_longlong(d);  // low 32 bits, sign-extended
  const unsigned long long iax = __ldg(&T.expd_tbl[di & (kExpdN - 1)]);
  const double t = (d - b) * T.expd_ra - x;
  const unsigned long long adj = (1ULL << (kExpdBits + 10)) - (1ULL << kExpdBits);
  unsigned long long u = ((di + adj) >> kExpdBits) << 52;
  double y = (3.0000000027955394 - t) * (t * t) * 0.16666666685227835064 - t + 1.0;
  u |= iax;
  return y * __longlong_as_double((long long)u);
}

__device__ __forceinline__ float ex_logf(const ExTab &T, float x) {
  const unsigned int bits = __float_as_uint(x);
  const int a = (int)(bits & (0xFFu << 23));
  const unsigned int b1 = bits & (((1u << kLogBits) - 1) << (23 - kLogBits));
  const unsigned int b2 = bits & ((1u << (23 - kLogBits)) - 1);
  const unsigned int idx = b1 >> (23 - kLogBits);
  const float2 tb = __ldg(reinterpret_cast<const float2 *>(T.log_tbl) + idx);
  const float f = (float)(a - (127 << 23)) * T.c_log2 + tb.x;
  return f + (float)b2 * tb.y;
}

// raccess.cpp:414-419
__device__ __forceinline__ double ex_lse(const ExTab &T, double x, double y) {
  return x > y ? x + (double)ex_logf(T, (float)(ex_expd(T, y - x) + 1.0))
               : y + (double)ex_logf(T, (float)(ex_expd(T, x - y) + 1.0));
}

// Per-thread view of one sequence: s[k] = base code of position k (1-based; s[0] = s[L+1] = 0), and the
// band arrays addressed by (left index, span).
struct Seq {
  const uint8_t *s;
  long long off;  // seq_off
  int L;
};

__device__ __forceinline__ double &AT(const ExCtx &c, const Seq &q, int arr, int i, int d) {
  return c.band[((long long)arr * (c.W + 2) + d) * c.NC + q.off + i];
}

// raccess.cpp:773-817 (t2 already reversed by the caller)
__device__ __forceinline__ double ex_loop(const ExCtx &c, const Seq &sq, int t, int t2, int i, int j, int p, int q) {
  const ExTab &T = *c.T;
  const uint8_t *s = sq.s;
  const int u1 = p - i - 1, u2 = j - q - 1;
  if (u1 == 0 && u2 == 0) return T.stack[t][t2];
  if (u1 == 0 || u2 == 0) {
    const int u = u1 == 0 ? u2 : u1;
    double z = T.bulge[u];  // u <= 30 on every call site (loop bounds), the log branch of :784 is dead
    if (u == 1) return z + T.stack[t][t2];
    if (t > 2) z += T.TermAU;
    if (t2 > 2) z += T.TermAU;
    return z;
  }
  if (u1 + u2 == 2) return T.int11[idx11(t, t2, s[i + 1], s[j - 1])];
  if (u1 == 1 && u2 == 2) return __ldg(&c.int21[idx21(t, t2, s[i + 1], s[q + 1], s[j - 1])]);
  if (u1 == 2 && u2 == 1) return __ldg(&c.int21[idx21(t2, t, s[q + 1], s[i + 1], s[p - 1])]);
  if (u1 == 2 && u2 == 2) return __ldg(&c.int22[idx22(t, t2, s[i + 1], s[p - 1], s[q + 1], s[j - 1])]);
  double z = T.internal[u1 + u2] + T.mmI[t][s[i + 1]][s[j - 1]] + T.mmI[t2][s[q + 1]][s[p - 1]];
  const int du = u1 > u2 ? u1 - u2 : u2 - u1;
  z += T.ninio[du];
  return z;
}

// raccess.cpp:819-832
__device__ __forceinline__ double ex_hairpin(const ExCtx &c, const Seq &sq, int t, int i, int j) {
  const ExTab &T = *c.T;
  const int d = j - i - 1;
  double q = T.hairpin[d];
  if (d != 3) q += T.mmH[t][sq.s[i + 1]][sq.s[j - 1]];
  else if (t > 2) q += T.TermAU;
  return q;
}

// raccess.cpp:244-256
__device__ __forceinline__ double ex_dangle(const ExCtx &c, const Seq &sq, int t, int a, int b) {
  const ExTab &T = *c.T;
  double x = 0;
  if (t != 0) {
    if (a > 0) x += T.d5[t][sq.s[a]];
    if (b < sq.L) x += T.d3[t][sq.s[b + 1]];
    if (b == sq.L && t > 2) x += T.TermAU;
  }
  return x;
}

__device__ __forceinline__ bool seq_of_column(const ExCtx &c, long long g, Seq &sq, int &i) {
  if (g >= c.NC) return false;
  const int id = c.col_seq[g];
  if (id < 0) return false;
  sq.off = c.seq_off[id];
  sq.L = c.seq_len[id];
  sq.s = c.S + sq.off;
  i = (int)(g - sq.off);
  return true;
}

// ---- state initialisation (raccess.cpp:70-96: band arrays = -INF, outer arrays and probability vectors = 0) ----
__global__ void k_ex_fill(double *band, long long nband, double *vec, long long nvec) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nband; k += stride) band[k] = EX_NEG;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nvec; k += stride) vec[k] = 0;
}

// ---- inside, one span: raccess.cpp:99-228 for the cells (i, i + d) of every sequence -------------------------
__global__ void __launch_bounds__(128) k_ex_inside(ExCtx c, int d) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  Seq sq;
  int i;
  if (!seq_of_column(c, g, sq, i)) return;
  const int j = i + d, L = sq.L;
  if (j > L || j < kTurn + 1) return;
  const ExTab &T = *c.T;
  const uint8_t *s = sq.s;
  // stem :103-129
  const int t = T.bp[s[i + 1]][s[j]];
  double stem = EX_NEG;
  if (t != 0) {
    const int t2 = T.rt[T.bp[s[i + 2]][s[j - 1]]];
    double v = 0;
    bool have = false;
    const double inner_stem = AT(c, sq, EA_STEM, i + 1, d - 2);
    const double inner_end = AT(c, sq, EA_STEMEND, i + 1, d - 2);
    if (inner_stem != EX_NEG) {
      if (t2 != 0) v = inner_stem + ex_loop(c, sq, t, t2, i + 1, j, i + 2, j - 1);
      have = true;
    }
    if (inner_end != EX_NEG) {
      v = have ? ex_lse(T, v, inner_end) : inner_end;
      have = true;
    }
    if (have) stem = v;
  }
  AT(c, sq, EA_STEM, i, d) = stem;
  // multibif :131-143
  double mb = EX_NEG;
  {
    double v = 0;
    bool have = false;
    for (int k = i + 1; k <= j - 1; k++) {
      const double a = AT(c, sq, EA_MULTI1, i, k - i), b = AT(c, sq, EA_MULTI2, k, j - k);
      if (a != EX_NEG && b != EX_NEG) {
        v = have ? ex_lse(T, v, a + b) : a + b;
        have = true;
      }
    }
    if (have) mb = v;
  }
  AT(c, sq, EA_MULTIBIF, i, d) = mb;
  // multi2 :145-162
  double m2;
  {
    double v = 0;
    bool have = false;
    if (t != 0 && stem != EX_NEG) {
      v = stem + T.MLintern + ex_dangle(c, sq, t, i, j);
      have = true;
    }
    const double prev = AT(c, sq, EA_MULTI2, i, d - 1);
    if (prev != EX_NEG) {
      const double w = prev + T.MLbase;
      m2 = have ? ex_lse(T, v, w) : w;
    } else {
      m2 = have ? v : EX_NEG;
    }
  }
  AT(c, sq, EA_MULTI2, i, d) = m2;
  // multi1 :164-175
  double m1;
  if (m2 != EX_NEG && mb != EX_NEG) m1 = ex_lse(T, m2, mb);
  else if (m2 == EX_NEG) m1 = mb;
  else m1 = m2;
  AT(c, sq, EA_MULTI1, i, d) = m1;
  // multi :177-191
  double mu;
  {
    const double prev = AT(c, sq, EA_MULTI, i + 1, d - 1);
    if (prev != EX_NEG) {
      const double v = prev + T.MLbase;
      mu = mb != EX_NEG ? ex_lse(T, v, mb) : v;
    } else {
      mu = mb;
    }
  }
  AT(c, sq, EA_MULTI, i, d) = mu;
  // stemend :193-226
  if (j != L) {
    const int te = T.bp[s[i]][s[j + 1]];
    double se = EX_NEG;
    if (te != 0) {
      double v = ex_hairpin(c, sq, te, i, j + 1);
      const int pmax = i + kMaxLoop < j - kTurn - 2 ? i + kMaxLoop : j - kTurn - 2;
      for (int p = i; p <= pmax; p++) {
        const int u1 = p - i;
        const int q0 = p + kTurn + 2 > j - kMaxLoop + u1 ? p + kTurn + 2 : j - kMaxLoop + u1;
        for (int q = q0; q <= j; q++) {
          const double st = (p == i && q == j) ? stem : AT(c, sq, EA_STEM, p, q - p);
          if (st == EX_NEG) continue;
          const int t2 = T.bp[s[p + 1]][s[q]];
          if (t2 != 0 && !(p == i && q == j)) v = ex_lse(T, v, st + ex_loop(c, sq, te, T.rt[t2], i, j + 1, p + 1, q));
        }
      }
      const int tt = T.rt[te];
      v = ex_lse(T, v, mu + T.MLclosing + T.MLintern + T.d3[tt][s[i + 1]] + T.d5[tt][s[j]]);
      se = v;
    }
    AT(c, sq, EA_STEMEND, i, d) = se;
  }
}

// ---- outer arrays: raccess.cpp:230-241 (forward = Alpha_outer) and :260-271 (Beta_outer) ---------------------
// One warp per (sequence, direction).  The chain over positions is serial; for one position the lanes gather
// the candidate terms (Alpha_stem + Dangle) in parallel, then lane 0 folds them in the reference's order.
// Dynamic shared memory, per warp: W + 2 terms, then a ring of ex_ring(W) values of the outer array (a power of
// two >= W + 2: the values a position reads lie at most W + 1 behind it).
__host__ __device__ constexpr int ex_ring(int W) { return W + 2 <= 256 ? 256 : W + 2 <= 1024 ? 1024 : 2048; }
constexpr int kExOuterWarps = 4;
size_t ex_outer_smem(int W) { return (size_t)kExOuterWarps * ((W + 2) + ex_ring(W)) * sizeof(double); }

__global__ void __launch_bounds__(32 * kExOuterWarps) k_ex_outer(ExCtx c) {
  extern __shared__ double ex_outer_smem_raw[];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int job = blockIdx.x * kExOuterWarps + wib;
  if (job >= 2 * c.nseq) return;
  const int id = job >> 1;
  const bool fwd = (job & 1) == 0;
  const ExTab &T = *c.T;
  Seq sq;
  sq.off = c.seq_off[id];
  sq.L = c.seq_len[id];
  sq.s = c.S + sq.off;
  const int L = sq.L, W = c.W;
  const int rmask = ex_ring(W) - 1;
  double *term = ex_outer_smem_raw + (size_t)wib * ((W + 2) + ex_ring(W)), *ring = term + (W + 2);
  double *ao = c.vec + 0 * c.NC + sq.off, *bo = c.vec + 1 * c.NC + sq.off;
  const double kSkip = __longlong_as_double(0x7ff0000000000000LL);  // +inf never is a legitimate term
  if (fwd) {
    if (lane == 0) ring[0] = 0;  // Alpha_outer[0] = 0
    __syncwarp();
    for (int i = 1; i <= L; i++) {
      const int lo = i - W - 1 > 0 ? i - W - 1 : 0;
      for (int p = lo + lane; p < i; p += 32) {
        const double st = AT(c, sq, EA_STEM, p, i - p);
        double e = kSkip;
        if (st != EX_NEG) {
          const int t = T.bp[sq.s[p + 1]][sq.s[i]];
          e = st + ex_dangle(c, sq, t, p, i);
        }
        term[p - lo] = e;
      }
      __syncwarp();
      if (lane == 0) {
        double v = ring[(i - 1) & rmask];
        for (int p = lo; p < i; p++) {
          const double e = term[p - lo];
          if (e != kSkip) v = ex_lse(T, v, e + ring[p & rmask]);
        }
        ring[i & rmask] = v;
        ao[i] = v;
      }
      __syncwarp();
    }
  } else {
    if (lane == 0) ring[L & rmask] = 0;  // Beta_outer[L] = 0
    __syncwarp();
    for (int i = L - 1; i >= 0; i--) {
      const int hi = i + W + 1 < L ? i + W + 1 : L;
      for (int p = i + 1 + lane; p <= hi; p += 32) {
        const double st = AT(c, sq, EA_STEM, i, p - i);
        double e = kSkip;
        if (st != EX_NEG) {
          const int t = T.bp[sq.s[i + 1]][sq.s[p]];
          e = st + ex_dangle(c, sq, t, i, p);
        }
        term[p - i - 1] = e;
      }
      __syncwarp();
      if (lane == 0) {
        double v = ring[(i + 1) & rmask];
        for (int p = i + 1; p <= hi; p++) {
          const double e = term[p - i - 1];
          if (e != kSkip) v = ex_lse(T, v, e + ring[p & rmask]);
        }
        ring[i & rmask] = v;
        bo[i] = v;
      }
      __syncwarp();
    }
  }
}

// ---- outside, one span: raccess.cpp:273-411 for the cells (p, p + d) ------------------------------------------
__global__ void __launch_bounds__(128) k_ex_outside(ExCtx c, int d) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  Seq sq;
  int p;
  if (!seq_of_column(c, g, sq, p)) return;
  const int q = p + d, L = sq.L, W = c.W;
  if (q > L || q < kTurn + 1) return;
  const ExTab &T = *c.T;
  const uint8_t *s = sq.s;
  const double *ao = c.vec + 0 * c.NC + sq.off, *bo = c.vec + 1 * c.NC + sq.off;
  double bm2 = EX_NEG;  // Beta_multi2(p, d): stays -INF for p == 0 or q == L
  if (p != 0 && q != L) {
    // stemend :277-279
    const double se = d >= W ? EX_NEG : AT(c, sq, EB_STEM, p - 1, d + 2);
    AT(c, sq, EB_STEMEND, p, d) = se;
    // multi :281-308
    double v = 0;
    bool have = false;
    if (d + 1 <= W + 1) {
      const double prev = AT(c, sq, EB_MULTI, p - 1, d + 1);
      if (prev != EX_NEG) {
        v = prev + T.MLbase;
        have = true;
      }
    }
    const int t = T.bp[s[p]][s[q + 1]];
    const int tt = T.rt[t];
    if (se != EX_NEG) {
      const double w = se + T.MLclosing + T.MLintern + T.d3[tt][s[p + 1]] + T.d5[tt][s[q]];
      v = have ? ex_lse(T, v, w) : w;
    } else if (!have) {
      v = EX_NEG;
    }
    const double bmu = v;
    AT(c, sq, EB_MULTI, p, d) = bmu;
    // multi1 :310-324
    v = 0;
    have = false;
    const int kmax = L < p + W ? L : p + W;
    for (int k = q + 1; k <= kmax; k++) {
      const double a = AT(c, sq, EB_MULTIBIF, p, k - p), b = AT(c, sq, EA_MULTI2, q, k - q);
      if (a != EX_NEG && b != EX_NEG) {
        v = have ? ex_lse(T, v, a + b) : a + b;
        have = true;
      }
    }
    const double bm1 = have ? v : EX_NEG;
    AT(c, sq, EB_MULTI1, p, d) = bm1;
    // multi2 :326-352
    v = 0;
    have = false;
    if (bm1 != EX_NEG) {
      v = bm1;
      have = true;
    }
    if (d <= W) {
      const double nx = AT(c, sq, EB_MULTI2, p, d + 1);
      if (nx != EX_NEG) {
        const double w = nx + T.MLbase;
        v = have ? ex_lse(T, v, w) : w;
        have = true;
      }
    }
    const int klo = q - W > 0 ? q - W : 0;
    for (int k = klo; k < p; k++) {
      const double a = AT(c, sq, EB_MULTIBIF, k, q - k), b = AT(c, sq, EA_MULTI1, k, p - k);
      if (a != EX_NEG && b != EX_NEG) {
        v = have ? ex_lse(T, v, a + b) : a + b;
        have = true;
      }
    }
    bm2 = have ? v : EX_NEG;
    AT(c, sq, EB_MULTI2, p, d) = bm2;
    // multibif :354-364
    double bif;
    if (bm1 != EX_NEG && bmu != EX_NEG) bif = ex_lse(T, bm1, bmu);
    else if (bmu == EX_NEG) bif = bm1;
    else bif = bmu;
    AT(c, sq, EB_MULTIBIF, p, d) = bif;
  }
  // stem :367-409
  const int t2 = T.bp[s[p + 1]][s[q]];
  double bstem = EX_NEG;
  if (t2 != 0) {
    double v = ao[p] + bo[q] + ex_dangle(c, sq, t2, p, q);
    const int t2r = T.rt[t2];
    const int ilo = p - kMaxLoop > 1 ? p - kMaxLoop : 1;
    for (int i = ilo; i <= p; i++) {
      const int jhi = q + kMaxLoop - p + i < L - 1 ? q + kMaxLoop - p + i : L - 1;
      for (int j = q; j <= jhi; j++) {
        const int t = T.bp[s[i]][s[j + 1]];
        if (t != 0 && !(i == p && j == q) && j - i <= W + 1) {
          const double se = AT(c, sq, EB_STEMEND, i, j - i);
          if (se != EX_NEG) v = ex_lse(T, v, se + ex_loop(c, sq, t, t2r, i, j + 1, p + 1, q));
        }
      }
    }
    if (p != 0 && q != L) {
      const int t = T.bp[s[p]][s[q + 1]];
      if (t != 0 && d + 2 <= W + 1) {
        const double up = AT(c, sq, EB_STEM, p - 1, d + 2);
        if (up != EX_NEG) v = ex_lse(T, v, up + ex_loop(c, sq, t, t2r, p, q + 1, p + 1, q));
      }
    }
    bstem = v;
    if (bm2 != EX_NEG) {
      const double w = bm2 + T.MLintern + ex_dangle(c, sq, t2, p, q);
      bstem = ex_lse(T, w, bstem);
    }
  }
  AT(c, sq, EB_STEM, p, d) = bstem;
}

// ---- hairpin probabilities: raccess.cpp:536-579, one thread per window start x -----------------------------
__global__ void __launch_bounds__(128) k_ex_hairpin(ExCtx c) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  Seq sq;
  int x;
  if (!seq_of_column(c, g, sq, x)) return;
  const int L = sq.L, W = c.W, w = c.delta;
  if (x < 1 || x + w - 1 > L) return;
  const ExTab &T = *c.T;
  const double Z = c.vec[0 * c.NC + sq.off + L];
  double v = 0, cv = 0;
  bool have = false, chave = false;
  const int ilo = x - W > 1 ? x - W : 1;
  for (int i = ilo; i < x; i++) {
    const int jhi = i + W < L ? i + W : L;
    for (int j = x + w; j <= jhi; j++) {
      const double be = AT(c, sq, EB_STEMEND, i, j - i - 1);
      if (be == EX_NEG) continue;
      const int t = T.bp[sq.s[i]][sq.s[j]];
      const double h = be + ex_hairpin(c, sq, t, i, j);
      if (j == x + w) {
        v = have ? ex_lse(T, v, h) : h;
        have = true;
      } else {
        cv = chave ? ex_lse(T, cv, h) : h;
        chave = true;
      }
    }
  }
  if (have && chave) v = ex_lse(T, v, cv);
  if (!have && chave) {
    v = cv;
    have = true;
  }
  if (have) c.vec[2 * c.NC + g] = ex_expd(T, v - Z);
  if (chave) c.vec[3 * c.NC + g] = ex_expd(T, cv - Z);
}

// ---- bulge / interior-loop probabilities: raccess.cpp:614-681 (direct) and :683-771 (log-sum) ----------------
// The reference walks the loops (i, j, p, q) once and adds each term to every window start k inside the two
// unpaired strands.  Floating-point addition is not associative, so to get its bits each position k must fold
// the terms of the loops whose strands contain it in the reference's order (i, j, p, q ascending):
//   left strand : i + 1 <= k <= p - w   (k == p - w feeds bp, otherwise cbp)      :644-650 / :713-729
//   right strand: q + 1 <= k <= j - w   (k == j - w feeds bp, otherwise cbp)      :652-658 / :731-745
// (the two cases exclude each other: left needs p > k, right q < k, and q > p).
// One CTA owns kBiB (64) consecutive columns.  It walks the outer pairs (i, j) that can reach any of its positions;
// for each pair the threads evaluate the <= 496 inner pairs ONCE, in parallel (flat index n -> (u1, u2) in the
// order of the reference's p, q loops), compact the existing terms in order into shared memory, and then each
// position folds its own sub-sequence of them: first the right-strand prefixes of the rows p < k + w, then the
// row p == k + w (bp) and all later rows (cbp) — contiguous ranges of the compacted list.
#ifndef PRIB_EX_BIB
#define PRIB_EX_BIB 64  // measured on B200 (direct / log-sum sets of profiles/exact_split.py): 256 -> 246 / 919 ms,
#endif                  // 64 -> 160 / 485 ms, 32 -> 302 / 606 ms
constexpr int kBiB = PRIB_EX_BIB;  // positions (= threads) per CTA
constexpr int kTri = 496;          // (u1, u2) with u1 + u2 <= 30
constexpr int kBiRounds = (kTri + kBiB - 1) / kBiB;
static_assert(kBiB % 32 == 0 && kBiRounds * (kBiB / 32) <= 16, "s_mask holds 16 ballot words");

__device__ __forceinline__ int tri_row_start(int u1) { return 31 * u1 - (u1 * (u1 - 1)) / 2; }

__global__ void __launch_bounds__(kBiB) k_ex_biloop(ExCtx c) {
  __shared__ double s_T[kTri];
  __shared__ unsigned char s_u1[kTri + 16], s_u2[kTri + 16], s_cu2[kTri + 16];
  __shared__ unsigned int s_mask[16];
  __shared__ short s_cstart[34];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long g0 = (long long)blockIdx.x * kBiB;
  const ExTab &T = *c.T;
  const int W = c.W, w = c.delta;
  for (int r = tid; r < 31; r += kBiB) {  // row u1 = r: u2 = 30 - u1 .. 0 (q ascending)
    int n = tri_row_start(r);
    for (int u2 = 30 - r; u2 >= 0; --u2, ++n) {
      s_u1[n] = (unsigned char)r;
      s_u2[n] = (unsigned char)u2;
    }
  }
  __syncthreads();
  // first sequence that can overlap [g0, g0 + kBiB): the last one starting at or before g0
  int lo = 0, hi = c.nseq;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (c.seq_off[mid] <= g0) lo = mid + 1;
    else hi = mid;
  }
  for (int id = lo > 0 ? lo - 1 : 0; id < c.nseq && c.seq_off[id] < g0 + kBiB; ++id) {
    Seq sq;
    sq.off = c.seq_off[id];
    sq.L = c.seq_len[id];
    sq.s = c.S + sq.off;
    const uint8_t *s = sq.s;
    const int L = sq.L;
    const long long rel0 = g0 - sq.off;  // position of thread 0 in this sequence (may be negative)
    const int klo = rel0 > 1 ? (int)rel0 : 1;
    const int khi = (long long)(L - w + 1) < rel0 + kBiB - 1 ? L - w + 1 : (int)(rel0 + kBiB - 1);
    if (klo > khi) continue;  // uniform
    const int k = (int)(rel0 + tid);
    const bool mine = k >= klo && k <= khi;
    const double Z = c.vec[0 * c.NC + sq.off + L];
    const bool direct = Z >= -690 && Z <= 690;  // raccess.cpp:436-443
    double b = 0, cc = 0;
    bool bf = false, cf = false;
    auto add = [&](bool to_b, double v) {
      if (direct) {
        if (to_b) b += v;
        else cc += v;
      } else if (to_b) {
        b = bf ? ex_lse(T, b, v) : v;
        bf = true;
      } else {
        cc = cf ? ex_lse(T, cc, v) : v;
        cf = true;
      }
    };
    int ilo = klo + w - W;
    if (ilo < 1) ilo = 1;
    int ihi = khi - 1;
    if (ihi > L - kTurn - 3) ihi = L - kTurn - 3;  // i < L - TURN - 2
    for (int i = ilo; i <= ihi; i++) {
      const int jhi = i + W < L ? i + W : L;
      int jlo = i + kTurn + 3;
      if (jlo < klo + w) jlo = klo + w;
      for (int j = jlo; j <= jhi; j++) {
        // everything up to the barriers is uniform over the CTA
        const int t = T.bp[s[i]][s[j]];
        if (t == 0) continue;
        {  // can a strand of this pair contain one of our positions?
          int lhi = i + kMaxLoop + 1 - w < j - w ? i + kMaxLoop + 1 - w : j - w;
          if (lhi > khi) lhi = khi;
          const bool left_ok = (klo > i + 1 ? klo : i + 1) <= lhi;
          int rlo = j - kMaxLoop > i + 1 ? j - kMaxLoop : i + 1;
          if (rlo < klo) rlo = klo;
          const bool right_ok = rlo <= (khi < j - w ? khi : j - w);
          if (!left_ok && !right_ok) continue;
        }
        const double be = AT(c, sq, EB_STEMEND, i, j - i - 1);
        if (be == EX_NEG) continue;
        const int u1max = (j - i - 6 < kMaxLoop) ? j - i - 6 : kMaxLoop;  // p <= min(i + 31, j - 5)
        const int nflat = tri_row_start(u1max + 1);
        // 1. evaluate the inner pairs (kBiRounds rounds of kBiB), note which exist
        double tv[kBiRounds];
        int wi[kBiRounds];
        unsigned int mk[kBiRounds];
        bool ok[kBiRounds];
#pragma unroll
        for (int r = 0; r < kBiRounds; ++r) {
          const int n = r * kBiB + tid;
          ok[r] = false;
          tv[r] = 0;
          if (n < nflat) {
            const int u1 = s_u1[n], u2 = s_u2[n];
            const int p = i + 1 + u1, q = j - 1 - u2;
            if (q >= p + kTurn + 1 && (u1 | u2) != 0) {
              const int t2 = T.bp[s[p]][s[q]];
              if (t2 != 0) {
                const double as = AT(c, sq, EA_STEM, p - 1, q - p + 1);
                if (as != EX_NEG) {
                  const double e = be + ex_loop(c, sq, t, T.rt[t2], i, j, p, q) + as;
                  tv[r] = direct ? ex_expd(T, e) : e;
                  ok[r] = true;
                }
              }
            }
          }
          mk[r] = __ballot_sync(0xffffffffu, ok[r]);
          wi[r] = r * (kBiB / 32) + warp;
          if (lane == 0) s_mask[wi[r]] = mk[r];
        }
        __syncthreads();
        // 2. compact in order; start of every row in the compacted list
#pragma unroll
        for (int r = 0; r < kBiRounds; ++r) {
          if (ok[r]) {
            int pos = __popc(mk[r] & ((1u << lane) - 1));
            for (int x = 0; x < wi[r]; ++x) pos += __popc(s_mask[x]);
            s_T[pos] = tv[r];
            s_cu2[pos] = s_u2[r * kBiB + tid];
          }
        }
        for (int r = tid; r <= u1max + 1; r += kBiB) {
          const int bit = tri_row_start(r);
          int pos = 0;
          for (int x = 0; x < (bit >> 5); ++x) pos += __popc(s_mask[x]);
          if ((bit & 31) != 0) pos += __popc(s_mask[bit >> 5] & ((1u << (bit & 31)) - 1));
          s_cstart[r] = (short)pos;
        }
        __syncthreads();
        // 3. every position folds its terms
        if (mine && i <= k - 1 && j >= k + w) {
          const int u1min = k + w - i - 1;  // the row with p - w == k
          const int thr = j - k;            // right strand: q <= k - 1  <=>  u2 >= j - k
          int rmax = u1min < u1max + 1 ? u1min : u1max + 1;
          if (rmax > kMaxLoop + 1 - thr) rmax = kMaxLoop + 1 - thr;
          const bool to_b_r = (k == j - w);
          for (int u1 = 0; u1 < rmax; ++u1) {
            const int xe = s_cstart[u1 + 1];
            for (int x = s_cstart[u1]; x < xe; ++x) {
              if ((int)s_cu2[x] < thr) break;
              add(to_b_r, s_T[x]);
            }
          }
          if (u1min <= u1max) {
            const int x1 = s_cstart[u1min + 1], x2 = s_cstart[u1max + 1];
            for (int x = s_cstart[u1min]; x < x1; ++x) add(true, s_T[x]);
            for (int x = x1; x < x2; ++x) add(false, s_T[x]);
          }
        }
        // no barrier here: the next pair only writes s_mask before its first barrier, and nobody reads
        // s_mask in step 3; s_T / s_cu2 / s_cstart are rewritten after that barrier
      }
    }
    if (mine) {
      if (direct) {  // :667-680
        if (b != 0) b = ex_expd(T, (double)ex_logf(T, (float)(b + cc)) - Z);
        if (cc != 0) cc = ex_expd(T, (double)ex_logf(T, (float)cc) - Z);
      } else {  // :754-770
        if (bf && cf) b = ex_lse(T, b, cc);
        if (!bf && cf) b = cc;
        if (bf) b = ex_expd(T, b - Z);
        if (cf) cc = ex_expd(T, cc - Z);
      }
      c.vec[4 * c.NC + g0 + tid] = b;
      c.vec[5 * c.NC + g0 + tid] = cc;
    }
  }
}

// raccess.cpp:581-612
__device__ __forceinline__ double ex_multi_prob(const ExCtx &c, const Seq &sq, int x, int w, double Z) {
  const ExTab &T = *c.T;
  const int L = sq.L, W = c.W;
  double v = 0;
  bool have = false;
  const int hi = x + W < L ? x + W : L;
  for (int i = x + w - 1; i <= hi; i++) {
    const double b = AT(c, sq, EB_MULTI, x - 1, i - x + 1), a = AT(c, sq, EA_MULTI, x + w - 1, i - x - w + 1);
    if (b != EX_NEG && a != EX_NEG) {
      v = have ? ex_lse(T, v, b + a) : b + a;
      have = true;
    }
  }
  const int lo = x + w - 1 - W > 0 ? x + w - 1 - W : 0;
  for (int i = lo; i < x; i++) {
    const double b = AT(c, sq, EB_MULTI2, i, x + w - 1 - i), a = AT(c, sq, EA_MULTI2, i, x - i - 1);
    if (b != EX_NEG && a != EX_NEG) {
      v = have ? ex_lse(T, v, b + a) : b + a;
      have = true;
    }
  }
  if (!have) return 0.0;
  return ex_expd(T, v - Z);
}

// ---- accessibility and conditional accessibility: raccess.cpp:484-528 -----------------------------------------
__global__ void __launch_bounds__(128) k_ex_finalize(ExCtx c) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  Seq sq;
  int x;
  if (!seq_of_column(c, g, sq, x)) return;
  const int L = sq.L, w = c.delta;
  if (x < 1 || x + w - 1 > L) return;
  const ExTab &T = *c.T;
  const int id = c.col_seq[g];
  const double *ao = c.vec + 0 * c.NC + sq.off, *bo = c.vec + 1 * c.NC + sq.off;
  const double Z = ao[L];
  double prob = 0.0;
  prob += ex_expd(T, ao[x - 1] + bo[x + w - 1] - Z);  // :530-534
  prob += c.vec[2 * c.NC + g];
  prob += c.vec[4 * c.NC + g];
  prob += ex_multi_prob(c, sq, x, w, Z);
  const double lg = (double)ex_logf(T, (float)prob);
  const float acc = (float)((-lg * T.kT) / 1000);
  c.out[c.acc_off[id] + x - 1] = acc;
  if (x + w - 1 < L) {
    double pc = 0.0;
    pc += ex_expd(T, ao[x - 1] + bo[x + w] - Z);
    pc += c.vec[3 * c.NC + g];
    pc += c.vec[5 * c.NC + g];
    pc += ex_multi_prob(c, sq, x, w + 1, Z);
    const double lc = (double)ex_logf(T, (float)pc);
    c.out[c.cond_off[id] + x + w - 1] = (float)((-lc * T.kT) / 1000 - acc);
  }
}

}  // namespace

struct ExactEngine {
  int W = 0;
  std::vector<int> lengths;
  ExTab *d_tab = nullptr;
  double *d_int21 = nullptr, *d_int22 = nullptr;
};

long long exact_state_bytes_per_column(int W) { return ((long long)kExArr * (W + 2) + kExVec) * 8; }

ExactEngine *exact_create(int W, const std::vector<int> &lengths, std::string &err) {
  const prib_turner_params *p = prib_turner_embedded();
  if (!p) {
    err = "embedded Turner parameter blob missing or corrupt";
    return nullptr;
  }
  ExTab *h = new (std::nothrow) ExTab();
  std::vector<double> i21(8 * 8 * 5 * 5 * 5), i22(8 * 8 * 5 * 5 * 5 * 5);
  if (!h) {
    err = "out of host memory";
    return nullptr;
  }
  ExTab &T = *h;
  // Raccess::set_energy_parameters, raccess.hpp:105-158: -E * 10 / kT with E an int (exact product, one
  // rounding in the divide)
  const double kT = (p->temperature_c + p->k0) * p->gasconst;  // energy_par.hpp:12-13
  T.kT = kT;
  T.MLclosing = -p->ml_closing * 10 / kT;
  T.MLintern = -p->ml_intern * 10. / kT;
  T.MLbase = -p->ml_base * 10. / kT;
  T.TermAU = -p->terminal_au * 10 / kT;
  double hairpin[31];
  for (int i = 0; i <= 30; i++) {
    hairpin[i] = -p->hairpin[i] * 10. / kT;
    T.bulge[i] = -p->bulge[i] * 10. / kT;
    T.internal[i] = -p->internal_loop[i] * 10. / kT;
  }
  for (int d = 0; d < kWideSpan + 8; d++)  // HairpinEnergy, raccess.cpp:821-824
    T.hairpin[d] = d <= 30 ? hairpin[d] : hairpin[30] - p->lxc37 * log(d / 30.) * 10. / kT;
  for (int i = 0; i < 7; i++) {
    for (int j = 0; j < 5; j++)
      for (int k = 0; k < 5; k++) {
        T.mmI[i][j][k] = -p->mismatch_i[i][j][k] * 10.0 / kT;
        T.mmH[i][j][k] = -p->mismatch_h[i][j][k] * 10.0 / kT;
      }
    for (int j = 0; j < 7; j++) T.stack[i][j] = -p->stack[i][j] * 10. / kT;
    for (int j = 0; j <= 4; j++) {
      T.d5[i][j] = -p->dangle5[i][j] * 10. / kT;
      T.d3[i][j] = -p->dangle3[i][j] * 10. / kT;
      if (i > 2) T.d3[i][j] += T.TermAU;
    }
  }
  for (int j = 0; j <= 4; j++) T.d5[7][j] = T.d3[7][j] = 0;  // never indexed (pair types are 0..6)
  for (int i = 0; i <= 7; i++)
    for (int j = 0; j <= 7; j++)
      for (int k = 0; k < 5; k++)
        for (int l = 0; l < 5; l++) {
          T.int11[idx11(i, j, k, l)] = -p->int11[i][j][k][l] * 10. / kT;
          for (int m = 0; m < 5; m++) {
            i21[idx21(i, j, k, l, m)] = -p->int21[i][j][k][l][m] * 10. / kT;
            for (int n = 0; n < 5; n++) i22[idx22(i, j, k, l, m, n)] = -p->int22[i][j][k][l][m][n] * 10. / kT;
          }
        }
  for (int i = 0; i <= kMaxLoop; i++) {
    const int v = i * p->f_ninio < p->max_ninio ? i * p->f_ninio : p->max_ninio;
    T.ninio[i] = -v * 10 / kT;
  }
  for (int i = 0; i < 5; i++)
    for (int j = 0; j < 5; j++) T.bp[i][j] = p->bp_pair[i][j];
  for (int i = 0; i < 7; i++) T.rt[i] = p->rtype[i];
  T.rt[7] = 0;
  // fmath ExpdVar, fmath.hpp:161-177
  T.expd_a = (double)kExpdN / log(2.0);
  T.expd_ra = 1 / T.expd_a;
  for (int i = 0; i < kExpdN; i++) {
    const double v = pow(2.0, i * (1.0 / kExpdN));
    unsigned long long bits;
    memcpy(&bits, &v, 8);
    T.expd_tbl[i] = bits & ((1ULL << 52) - 1);
  }
  // fmath LogVar, fmath.hpp:193-207
  T.c_log2 = logf(2.0f) / (1 << 23);
  {
    const double e = 1 / (double)(1 << 24);
    const double hh = 1 / (double)(1 << kLogBits);
    for (int i = 0; i < kLogN; i++) {
      const double x = 1 + (double)i / kLogN;
      const double a = log(x);
      T.log_tbl[2 * i] = (float)a;
      if (i < kLogN - 1) {
        const double b = log(x + hh - e);
        T.log_tbl[2 * i + 1] = (float)((b - a) / ((hh - e) * (1 << 23)));
      } else {
        T.log_tbl[2 * i + 1] = (float)(1 / (x * (1 << 23)));
      }
    }
  }
  ExactEngine *eng = new (std::nothrow) ExactEngine();
  bool ok = eng != nullptr;
  // above W = 254 the outer-array scans need more than the 48 KB of default shared memory (W = 1,000: 64 KB)
  if (ok && ex_outer_smem(W) > 48 * 1024)
    ok = cudaFuncSetAttribute(k_ex_outer, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ex_outer_smem(W)) == cudaSuccess;
  if (ok) {
    eng->W = W;
    eng->lengths = lengths;
    ok = cudaMalloc(&eng->d_tab, sizeof(ExTab)) == cudaSuccess &&
         cudaMalloc(&eng->d_int21, i21.size() * 8) == cudaSuccess &&
         cudaMalloc(&eng->d_int22, i22.size() * 8) == cudaSuccess &&
         cudaMemcpy(eng->d_tab, h, sizeof(ExTab), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(eng->d_int21, i21.data(), i21.size() * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(eng->d_int22, i22.data(), i22.size() * 8, cudaMemcpyHostToDevice) == cudaSuccess;
  }
  delete h;
  if (!ok) {
    err = std::string("exact engine tables: ") + cudaGetErrorString(cudaGetLastError());
    exact_destroy(eng);
    return nullptr;
  }
  return eng;
}

void exact_destroy(ExactEngine *e) {
  if (!e) return;
  cudaFree(e->d_tab);
  cudaFree(e->d_int21);
  cudaFree(e->d_int22);
  delete e;
}

int exact_run(ExactEngine *e, const ExactBatch &b, char *d_state, cudaStream_t st, cudaEvent_t *ev, int *launches) {
  ExCtx c;
  c.NC = b.NC;
  c.W = e->W;
  c.delta = e->lengths[0];
  c.nseq = b.n;
  c.S = b.S;
  c.col_seq = b.col_seq;
  c.seq_len = b.seq_len;
  c.seq_off = b.seq_off;
  c.acc_off = b.acc_off;
  c.cond_off = b.cond_off;
  c.T = e->d_tab;
  c.int21 = e->d_int21;
  c.int22 = e->d_int22;
  c.band = reinterpret_cast<double *>(d_state);
  const long long nband = (long long)kExArr * (c.W + 2) * c.NC;
  c.vec = c.band + nband;
  c.out = b.out;
  const int W = c.W;
  const unsigned grid = (unsigned)((b.NC + 127) / 128);
  int nl = 0;
#define EX_EV(k) \
  if (ev && cudaEventRecord(ev[k], st) != cudaSuccess) return (int)cudaGetLastError()
  EX_EV(0);
  k_ex_fill<<<148 * 8, 256, 0, st>>>(c.band, nband, c.vec, (long long)kExVec * c.NC);
  ++nl;
  EX_EV(1);
  for (int d = kTurn; d <= W + 1; d++, ++nl) k_ex_inside<<<grid, 128, 0, st>>>(c, d);
  EX_EV(2);
  k_ex_outer<<<(unsigned)((2 * b.n + kExOuterWarps - 1) / kExOuterWarps), 32 * kExOuterWarps, ex_outer_smem(W), st>>>(c);
  ++nl;
  EX_EV(3);
  for (int d = W + 1; d >= kTurn; d--, ++nl) k_ex_outside<<<grid, 128, 0, st>>>(c, d);
  EX_EV(4);
  for (size_t l = 0; l < e->lengths.size(); ++l) {
    c.delta = e->lengths[l];
    c.out = b.out + (long long)l * b.out_stride;
    // k_ex_hairpin writes only the positions that have a hairpin term: clear the previous length's
    if (l > 0) {
      const cudaError_t r = cudaMemsetAsync(c.vec + 2 * c.NC, 0, (size_t)(2 * c.NC) * sizeof(double), st);
      if (r != cudaSuccess) return (int)r;
    }
    k_ex_biloop<<<(unsigned)((b.NC + kBiB - 1) / kBiB), kBiB, 0, st>>>(c);
    ++nl;
    EX_EV(5 + 3 * l);
    EX_EV(6 + 3 * l);
    k_ex_hairpin<<<grid, 128, 0, st>>>(c);
    k_ex_finalize<<<grid, 128, 0, st>>>(c);
    nl += 2;
    EX_EV(7 + 3 * l);
  }
#undef EX_EV
  if (launches) *launches = nl;
  return (int)cudaGetLastError();
}

}  // namespace prib
