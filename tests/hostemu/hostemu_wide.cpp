// TEST INFRASTRUCTURE — CPU emulation of the wide-span engine (priblast_b200/csrc/acc_wide.cu): the per-cell
// functions of acc_core.h with tables of kWideSpan spans and the engine's span scaling, run in plain loops in the
// kernels' launch order on a zeroed state (what the engine's memset leaves).  The device range check is not
// emulated.  Not linked into libpriblast_acc.so and not a fallback; built by tests/test_wide_params.py.
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../priblast_b200/csrc/acc_core.h"
#include "../../priblast_b200/csrc/acc_tables.h"

using namespace prib;
typedef Core<double, kWideSpan> KW;

extern "C" int hostemu_wide_run_batch(int n, const char *const *seqs, const int32_t *lens, int W, int delta,
                                      float *out, const int64_t *acc_off, const int64_t *cond_off) {
  std::unique_ptr<HostTablesT<double, kWideSpan>> tab(new HostTablesT<double, kWideSpan>());
  std::string err;
  if (!build_tables(W, delta, default_scale_wide(), *tab, err)) return -1;
  BatchLayout lay;
  build_layout(n, seqs, lens, lay);
  for (int k = 0; k < n; k++) {
    std::memset(out + acc_off[k], 0, sizeof(float) * (size_t)lens[k]);
    std::memset(out + cond_off[k], 0, sizeof(float) * (size_t)lens[k]);
  }
  KW::Ctx c;
  std::memset(&c, 0, sizeof(c));
  c.NC = lay.NC;
  c.W = W;
  c.delta = delta;
  c.rows = W + 4;
  c.nseq = n;
  c.S = lay.S.data();
  c.col_seq = lay.col_seq.data();
  c.seq_len = lay.seq_len.data();
  c.seq_off = lay.seq_off.data();
  c.T = &tab->small;
  c.e_int11 = tab->e_int11.data();
  c.e_int21 = tab->e_int21.data();
  c.e_int22 = tab->e_int22.data();
  c.log_tbl = tab->log_tbl.data();
  std::vector<std::vector<double>> arr(kNumArr);
  for (int a = 0; a < kNumArr; a++) {
    const int rows = (a == X_ML || a == X_MR || a == X_MLS || a == X_MRS) ? kMaxLoop + 2 : W + 4;
    arr[a].assign((size_t)rows * (size_t)c.NC, 0.0);
    c.arr[a] = arr[a].data();
  }
  std::vector<double> lao((size_t)c.NC, 0.0), lbo((size_t)c.NC, 0.0), ring(KW::kRing);
  std::vector<int32_t> flags((size_t)n + 1, 0);
  c.lao = lao.data();
  c.lbo = lbo.data();
  c.acc_off = (const long long *)acc_off;
  c.cond_off = (const long long *)cond_off;
  c.out = out;
  c.flags = flags.data();
  for (int d = kTurn; d <= W + 1; d++)
    for (long long g = 0; g < c.NC; g++) KW::inside_cell(c, g, d);
  for (int k = 0; k < n; k++) {
    KW::scan_alpha_outer(c, k, ring.data());
    KW::scan_beta_outer(c, k, ring.data());
  }
  for (int d = W + 1; d >= kTurn; d--)
    for (long long g = 0; g < c.NC; g++) KW::outside_cell(c, g, d);
  for (long long g = 0; g < c.NC; g++) {
    KW::biloop_left(c, g);
    KW::biloop_right(c, g);
    KW::hairpin_suffix(c, g);
  }
  for (long long g = 0; g < c.NC; g++) KW::finalize_position(c, g);
  return 1;
}
