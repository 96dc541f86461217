// Host-side construction of the Boltzmann-factor tables and of the batch column layout.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

#include "acc_core.h"

namespace prib {

template <typename real, int CAP = kMaxSpan>
struct HostTablesT {
  typename Core<real, CAP>::SmallTables small;
  std::vector<real> e_int11, e_int21, e_int22;
  std::vector<float> log_tbl;  // 2048 x (app, rev)
};
typedef HostTablesT<double> HostTables;

// Scales the embedded Turner parameters exactly like Raccess::set_energy_parameters
// (raccess.hpp:105-158) and exponentiates them (always in double; cast to `real` at the end).
// Returns false if the blob is missing.  Instantiated for float and double.
// Span scaling of the stored band values (see SmallTables): kappa = 2^-klog2, cA = 2^alog2, cB = 2^blog2.
struct ScaleSpec {
  double klog2 = 0, alog2 = 0, blog2 = 0;
};
inline ScaleSpec default_scale_fp32() {
  ScaleSpec s;
  // kappa = 2^-0.45 per unit of span: measured on B200 over 1,000 uniform 2 kb sequences per span (profiles/r2/
  // scale_scan.txt): sequences that leave the FP32 safe range and are re-run in FP64 with klog2 = 0.30 / 0.45:
  // W = 70: 1 / 0, W = 100: 12 / 0, W = 150: 227 / 3, W = 200: 802 / 22.  What binds is the OUTSIDE side: Beta / Z of a
  // wide cell is ~1 / Alpha of that cell, i.e. 2^-0.6..-0.7 per nt for well-structured windows, and the stored value
  // cB kappa^-d (Beta / Z) fell under 2^-55 with the round-1 choice of 0.30.
  s.klog2 = 0.45;
  s.alog2 = 4.0;
  s.blog2 = 16.0;
  return s;
}

// Span scaling of the wide-span FP64 engine (acc_wide.cu).  Its stored values are range-checked against 2^+-480,
// so kappa only has to keep Alpha and Beta / Z of the widest cells inside that window: kappa = 2^-klog2 per nt
// (profiles/scale_scan.py <W> <n> wide, DESIGN.md §2.9); cA = cB = 1.
inline ScaleSpec default_scale_wide() {
  ScaleSpec s;
  s.klog2 = 0.45;
  return s;
}

// Instantiated for <float, kMaxSpan>, <double, kMaxSpan> and <double, kWideSpan>.
template <typename real, int CAP>
bool build_tables(int W, int delta, const ScaleSpec &sc, HostTablesT<real, CAP> &out, std::string &err);

// Column layout of one batch (DESIGN.md §3): sequence k occupies columns seq_off[k] .. seq_off[k]+len[k]
// (left indices 0..L), followed by >= kPad zero columns; the first sequence starts at kPad.
struct BatchLayout {
  long long NC = 0;
  std::vector<long long> seq_off;
  std::vector<int32_t> seq_len;
  std::vector<int32_t> col_seq;
  std::vector<uint8_t> S;
};

// Base coding of Raccess::Initiallize (raccess.cpp:55-68).
inline uint8_t encode_base(char ch) {
  switch (ch) {
    case 'A': case 'a': return 1;
    case 'C': case 'c': return 2;
    case 'G': case 'g': return 3;
    case 'T': case 't': case 'U': case 'u': return 4;
    default: return 0;
  }
}

void build_layout(int n, const char *const *seqs, const int32_t *lens, BatchLayout &out);

// Columns a sequence of length L costs in a batch (for batch sizing).
inline long long layout_columns(int L) { return (((long long)L + 1 + kPad) + 31) / 32 * 32; }

}  // namespace prib
