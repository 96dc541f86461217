// Wide-span engine: spans kMaxSpan < W <= kWideSpan in modes 0 and 1 (DESIGN.md §2.9).
//
// The tile kernels keep their span-indexed tables and stencil rings in shared memory, which bounds them to
// W <= kMaxSpan.  This engine runs the one-cell-at-a-time functions of acc_core.h instead, instantiated with tables
// of kWideSpan spans (Core<double, kWideSpan>), in the schedule of the host emulation (tests/hostemu):
//   inside   one launch per span d = 3 .. W + 1, one thread per column          (inside_cell)
//   scans    one thread per (sequence, direction), ring in global memory     (scan_alpha_outer / scan_beta_outer)
//   outside  one launch per span d = W + 1 .. 3, one thread per column          (outside_cell)
//   strands  one thread per column                                    (biloop_left / _right, hairpin_suffix)
//   finalize one thread per column                                               (finalize_position)
// Every band value is FP64, span-scaled with kappa (default_scale_wide()).  The inside / outside values a cell
// stores are checked against [2^-480, 2^480]; a sequence with a value outside that window (or an outer-array
// scan that overflowed) is flagged, skipped by the finalize kernel and re-run by the caller in the exact engine,
// which works in the log domain and has no range limit.
#include "acc_wide.h"

#include <math.h>
#include <string.h>

#include <memory>
#include <new>

#include "acc_core.h"
#include "acc_tables.h"

namespace prib {
namespace {

typedef Core<double, kWideSpan> KW;
constexpr int kWideThreads = 128;

// Range of the stored band values: every product of two of them with a table factor, and every sum of a few
// thousand such products, stays a normal double.  NaN and inf fail the first comparison.  Bits as in the FP32
// engine: 1 = too large, 2 = too small (inside); x4 for the outside pass; 16 = an outer-array scan overflowed.
__device__ __forceinline__ int wide_bits(double v) { return !(v <= 0x1p480) ? 1 : (v != 0 && v < 0x1p-480) ? 2 : 0; }

__device__ __forceinline__ bool cell_exists(const KW::Ctx &c, long long g, int d, int &sq) {
  sq = c.col_seq[g];
  return sq >= 0 && g - c.seq_off[sq] + d <= c.seq_len[sq];
}

__global__ void __launch_bounds__(kWideThreads) k_wide_inside(KW::Ctx c, int d) {
  const long long g = (long long)blockIdx.x * kWideThreads + threadIdx.x;
  if (g >= c.NC) return;
  KW::inside_cell(c, g, d);
  int sq;
  if (!cell_exists(c, g, d, sq)) return;
  const int bits = wide_bits(c.ld(A_STEM, d, g)) | wide_bits(c.ld(A_STEMEND, d, g)) | wide_bits(c.ld(A_MULTI, d, g)) |
                   wide_bits(c.ld(A_MULTI1, d, g)) | wide_bits(c.ld(A_MULTI2, d, g));
  if (bits) KW::raise_flag(&c.flags[sq], bits);
}

__global__ void __launch_bounds__(kWideThreads) k_wide_scans(KW::Ctx c, double *rings) {
  const int job = blockIdx.x * kWideThreads + threadIdx.x;  // job = 2 * sequence + direction
  if (job >= 2 * c.nseq) return;
  const int sq = job >> 1;
  double *ring = rings + (size_t)job * KW::kRing;
  const long long off = c.seq_off[sq];
  double end;
  if ((job & 1) == 0) {
    KW::scan_alpha_outer(c, sq, ring);
    end = c.lao[off + c.seq_len[sq]];
  } else {
    KW::scan_beta_outer(c, sq, ring);
    end = c.lbo[off];
  }
  if (!isfinite(end)) KW::raise_flag(&c.flags[sq], 16);
}

__global__ void __launch_bounds__(kWideThreads) k_wide_outside(KW::Ctx c, int d) {
  const long long g = (long long)blockIdx.x * kWideThreads + threadIdx.x;
  if (g >= c.NC) return;
  KW::outside_cell(c, g, d);
  int sq;
  if (!cell_exists(c, g, d, sq)) return;
  const int bits = wide_bits(c.ld(B_STEM, d, g)) | wide_bits(c.ld(B_MULTI, d, g)) | wide_bits(c.ld(B_MULTI2, d, g)) |
                   wide_bits(c.ld(B_MULTIBIF, d, g));
  if (bits) KW::raise_flag(&c.flags[sq], 4 * bits);
}

__global__ void __launch_bounds__(kWideThreads) k_wide_strands(KW::Ctx c) {
  const long long g = (long long)blockIdx.x * kWideThreads + threadIdx.x;
  if (g >= c.NC) return;
  KW::biloop_left(c, g);
  KW::biloop_right(c, g);
  KW::hairpin_suffix(c, g);
}

// flagged sequences are left to the exact re-run: their values may be inf / NaN and must not reach the output or
// the non-finite counter
__global__ void __launch_bounds__(kWideThreads) k_wide_finalize(KW::Ctx c) {
  const long long g = (long long)blockIdx.x * kWideThreads + threadIdx.x;
  if (g >= c.NC) return;
  const int sq = c.col_seq[g];
  if (sq < 0 || c.flags[sq] != 0) return;
  KW::finalize_position(c, g);
}

int rows_of(int a, int W) { return (a == X_ML || a == X_MR || a == X_MLS || a == X_MRS) ? kMaxLoop + 2 : W + 4; }

}  // namespace

struct WideEngine {
  int W = 0;
  std::vector<int> lengths;
  std::vector<KW::SmallTables *> d_small;  // one per length (they differ in kmul only)
  double *d_int11 = nullptr, *d_int21 = nullptr, *d_int22 = nullptr;
  float *d_log = nullptr;
  double *d_ring = nullptr;  // scan rings, KW::kRing doubles per (sequence, direction); grow-only
  long long ring_jobs = 0;
};

long long wide_state_bytes_per_column(int W) {
  long long r = 0;
  for (int a = 0; a < kNumArr; a++) r += rows_of(a, W);
  return r * (long long)sizeof(double) + 2 * (long long)sizeof(double);
}

WideEngine *wide_create(int W, const std::vector<int> &lengths, double klog2, std::string &err) {
  std::unique_ptr<HostTablesT<double, kWideSpan>> tab(new (std::nothrow) HostTablesT<double, kWideSpan>());
  if (!tab) {
    err = "out of host memory";
    return nullptr;
  }
  ScaleSpec spec = default_scale_wide();
  spec.klog2 = klog2;
  WideEngine *e = new (std::nothrow) WideEngine();
  if (!e) {
    err = "out of host memory";
    return nullptr;
  }
  e->W = W;
  e->lengths = lengths;
  auto up = [&](auto **dst, const auto *src, size_t bytes) {
    return cudaMalloc(dst, bytes) == cudaSuccess && cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  e->d_small.assign(lengths.size(), nullptr);
  for (size_t l = 0; l < lengths.size(); ++l) {  // everything uploaded after the loop depends on no delta
    if (!build_tables(W, lengths[l], spec, *tab, err)) {
      wide_destroy(e);
      return nullptr;
    }
    if (!up(&e->d_small[l], &tab->small, sizeof(KW::SmallTables))) {
      err = std::string("wide-span engine tables: ") + cudaGetErrorString(cudaGetLastError());
      wide_destroy(e);
      return nullptr;
    }
  }
  const bool ok = up(&e->d_int11, tab->e_int11.data(), tab->e_int11.size() * sizeof(double)) &&
                  up(&e->d_int21, tab->e_int21.data(), tab->e_int21.size() * sizeof(double)) &&
                  up(&e->d_int22, tab->e_int22.data(), tab->e_int22.size() * sizeof(double)) &&
                  up(&e->d_log, tab->log_tbl.data(), tab->log_tbl.size() * sizeof(float));
  if (!ok) {
    err = std::string("wide-span engine tables: ") + cudaGetErrorString(cudaGetLastError());
    wide_destroy(e);
    return nullptr;
  }
  return e;
}

void wide_destroy(WideEngine *e) {
  if (!e) return;
  for (KW::SmallTables *t : e->d_small) cudaFree(t);
  cudaFree(e->d_int11);
  cudaFree(e->d_int21);
  cudaFree(e->d_int22);
  cudaFree(e->d_log);
  cudaFree(e->d_ring);
  delete e;
}

int wide_run(WideEngine *e, const ExactBatch &b, int32_t *flags, int32_t *bad, char *d_state, cudaStream_t st,
             cudaEvent_t *ev, int *launches) {
  const int W = e->W;
  if (2LL * b.n > e->ring_jobs) {
    cudaError_t r = cudaStreamSynchronize(st);  // the old rings may still be in use
    if (r != cudaSuccess) return (int)r;
    cudaFree(e->d_ring);
    e->d_ring = nullptr;
    e->ring_jobs = 0;
    r = cudaMalloc(&e->d_ring, (size_t)2 * b.n * KW::kRing * sizeof(double));
    if (r != cudaSuccess) return (int)r;
    e->ring_jobs = 2LL * b.n;
  }
  KW::Ctx c;
  memset(&c, 0, sizeof(c));
  c.NC = b.NC;
  c.W = W;
  c.delta = e->lengths[0];
  c.rows = W + 4;
  c.nseq = b.n;
  c.S = b.S;
  c.col_seq = b.col_seq;
  c.seq_len = b.seq_len;
  c.seq_off = b.seq_off;
  c.T = e->d_small[0];
  c.e_int11 = e->d_int11;
  c.e_int21 = e->d_int21;
  c.e_int22 = e->d_int22;
  c.log_tbl = e->d_log;
  char *p = d_state;
  for (int a = 0; a < kNumArr; a++) {
    c.arr[a] = (double *)p;
    p += (long long)rows_of(a, W) * b.NC * (long long)sizeof(double);
  }
  c.lao = (double *)p;
  p += b.NC * (long long)sizeof(double);
  c.lbo = (double *)p;
  c.acc_off = b.acc_off;
  c.cond_off = b.cond_off;
  c.out = b.out;
  c.flags = flags;
  c.bad = bad;
  const unsigned grid = (unsigned)((b.NC + kWideThreads - 1) / kWideThreads);
  int nl = 0;
#define WD_EV(k) \
  if (ev && cudaEventRecord(ev[k], st) != cudaSuccess) return (int)cudaGetLastError()
  WD_EV(0);
  // cells that are never written (spans below 3, j > L, padding columns) must read as 0
  cudaError_t r = cudaMemsetAsync(d_state, 0, (size_t)(wide_state_bytes_per_column(W) * b.NC), st);
  if (r == cudaSuccess) r = cudaMemsetAsync(flags, 0, sizeof(int32_t) * (size_t)(b.n > 0 ? b.n : 1), st);
  if (r != cudaSuccess) return (int)r;
  WD_EV(1);
  for (int d = kTurn; d <= W + 1; d++, ++nl) k_wide_inside<<<grid, kWideThreads, 0, st>>>(c, d);
  WD_EV(2);
  k_wide_scans<<<(unsigned)((2 * b.n + kWideThreads - 1) / kWideThreads), kWideThreads, 0, st>>>(c, e->d_ring);
  ++nl;
  WD_EV(3);
  for (int d = W + 1; d >= kTurn; d--, ++nl) k_wide_outside<<<grid, kWideThreads, 0, st>>>(c, d);
  WD_EV(4);
  for (size_t l = 0; l < e->lengths.size(); ++l) {  // the strand arrays are overwritten from one length to the next
    c.delta = e->lengths[l];
    c.T = e->d_small[l];
    c.out = b.out + (long long)l * b.out_stride;
    k_wide_strands<<<grid, kWideThreads, 0, st>>>(c);
    ++nl;
    WD_EV(5 + 3 * l);
    WD_EV(6 + 3 * l);
    k_wide_finalize<<<grid, kWideThreads, 0, st>>>(c);
    ++nl;
    WD_EV(7 + 3 * l);
  }
#undef WD_EV
  if (launches) *launches = nl;
  return (int)cudaGetLastError();
}

}  // namespace prib
