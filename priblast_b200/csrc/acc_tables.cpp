#include "acc_tables.h"

#include <cmath>
#include <cstring>
#include <limits>

#include "turner_params.h"

namespace prib {

template <typename real, int CAP>
bool build_tables(int W, int delta, const ScaleSpec &spec, HostTablesT<real, CAP> &out, std::string &err) {
  const prib_turner_params *p = prib_turner_embedded();
  if (!p) {
    err = "embedded Turner parameter blob missing or corrupt";
    return false;
  }
  if (W < 1 || W > CAP) {
    err = "maximal span out of range (1.." + std::to_string((int)CAP) + ")";
    return false;
  }
  typename Core<real, CAP>::SmallTables &T = out.small;
  std::memset(&T, 0, sizeof(T));
  // energy_par.hpp:12-13; every scaled value is (-E*10)/kT as in raccess.hpp:105-158
  const double kT = (p->temperature_c + p->k0) * p->gasconst;
  T.kT = kT;
  auto sc = [&](int e) { return (double)(-e) * 10. / kT; };
  const double MLclosing = sc(p->ml_closing), MLintern = sc(p->ml_intern), MLbase = sc(p->ml_base);
  const double TermAU = sc(p->terminal_au);
  const double kap = std::exp2(-spec.klog2), cA = std::exp2(spec.alog2), cB = std::exp2(spec.blog2);
  auto kpow = [&](int n) { return std::exp2(-spec.klog2 * n); };
  T.k2 = kap * kap;
  T.inv_cA = 1.0 / cA;
  T.kacc = kap * kap / (cA * cB);
  T.kmul[0] = kpow(delta) / (cA * cB);
  T.kmul[1] = kpow(delta + 1) / (cA * cB);
  // kmul is stored as `real`.  CalcMultiProbability has terms only for windows w <= W - 4 (a multiloop needs a
  // span-5 branch beside the window), so kmul only has to be a normal number up to delta + 1 <= W - 4; for a wider
  // window both sums are empty and an underflowed kmul multiplies 0.  (FP32: kappa^197 / (cA cB) = 2^-109 at
  // W = 200 with the default scale.)
  if (delta + 1 <= W - 4 && !(T.kmul[1] >= std::numeric_limits<real>::min())) {
    err = "span scale too strong for the minimum accessible length (kappa^(delta+1) / (cA cB) underflows)";
    return false;
  }
  T.e_mlbase = kap * std::exp(MLbase);
  T.e_mlintern = std::exp(MLintern);
  T.e_mlclose = std::exp(MLclosing + MLintern);
  for (int t = 0; t < 8; t++) T.tau[t] = t > 2 && t < 7 ? std::exp(TermAU) : 1.0;

  double hairpin[31], bulge[31], internal[31], ninio[kMaxLoop + 1];
  for (int i = 0; i <= 30; i++) {
    hairpin[i] = sc(p->hairpin[i]);
    bulge[i] = sc(p->bulge[i]);
    internal[i] = sc(p->internal_loop[i]);
  }
  for (int i = 0; i <= kMaxLoop; i++) {
    int v = i * p->f_ninio < p->max_ninio ? i * p->f_ninio : p->max_ninio;
    ninio[i] = sc(v);
  }
  // HairpinEnergy length term incl. the logarithmic extrapolation (raccess.cpp:823)
  for (int d = 0; d < CAP + 8; d++) {
    double q = d <= 30 ? hairpin[d] : hairpin[30] - p->lxc37 * std::log(d / 30.) * 10. / kT;
    T.e_hairpin[d] = cA * kpow(d) * std::exp(q);
    T.sB[d] = cB * kpow(-d);
    T.us[d] = kpow(-d) / cA;
    if (d + 1 < CAP + 8) T.hpB[d + 1] = kpow(d + 2) / cB * std::exp(q);  // indexed by dd = loop size + 1
  }
  for (int u = 0; u < 32; u++) T.e_bulge[u] = u <= 30 ? kpow(u) * std::exp(bulge[u]) : 0.0;
  for (int k = 0; k < 8; k++) T.cg[k] = std::exp(ninio[k < 6 ? k : 6]);
  for (int sm = 0; sm < 32; sm++) T.cf[sm] = (sm >= 4 && sm <= 30) ? kpow(sm) * std::exp(internal[sm]) : 0.0;
  // generic interior loops (raccess.cpp:808-812): everything except 1x1, 1x2, 2x1, 2x2 and bulges
  for (int u1 = 1; u1 <= 30; u1++)
    for (int u2 = 1; u1 + u2 <= 30; u2++) {
      if (u1 + u2 < 4 || (u1 == 2 && u2 == 2)) continue;
      T.conv[u1][u2] = T.cf[u1 + u2] * T.cg[std::abs(u1 - u2) < 6 ? std::abs(u1 - u2) : 6];
    }
  for (int i = 0; i < 7; i++) {
    for (int j = 0; j < 5; j++)
      for (int k = 0; k < 5; k++) {
        T.e_mmI[i][j][k] = std::exp(sc(p->mismatch_i[i][j][k]));
        T.e_mmH[i][j][k] = std::exp(sc(p->mismatch_h[i][j][k]));
      }
    for (int j = 0; j < 7; j++) T.e_stack[i][j] = std::exp(sc(p->stack[i][j]));
    for (int j = 0; j < 5; j++) {
      T.e_d5[i][j] = std::exp(sc(p->dangle5[i][j]));
      double d3 = sc(p->dangle3[i][j]);
      if (i > 2) d3 += TermAU;  // raccess.hpp:132-134
      T.e_d3[i][j] = std::exp(d3);
    }
  }
  for (int j = 0; j < 5; j++) T.e_d5[7][j] = T.e_d3[7][j] = 1.0;  // never indexed (types are 0..6)
  for (int a = 0; a < 5; a++)
    for (int b = 0; b < 5; b++) T.bp[a][b] = (int8_t)p->bp_pair[a][b];
  for (int t = 0; t < 7; t++) T.rt[t] = (int8_t)p->rtype[t];
  T.rt[7] = 0;
  for (int a = 0; a < 5; a++)
    for (int b = 0; b < 5; b++) T.bpr[a][b] = T.rt[T.bp[a][b]];

  out.e_int11.resize(8 * 8 * 5 * 5);
  out.e_int21.resize(8 * 8 * 5 * 5 * 5);
  out.e_int22.resize(8 * 8 * 5 * 5 * 5 * 5);
  const int32_t *i11 = &p->int11[0][0][0][0], *i21 = &p->int21[0][0][0][0][0], *i22 = &p->int22[0][0][0][0][0][0];
  for (size_t k = 0; k < out.e_int11.size(); k++) out.e_int11[k] = kpow(2) * std::exp(sc(i11[k]));
  for (size_t k = 0; k < out.e_int21.size(); k++) out.e_int21[k] = kpow(3) * std::exp(sc(i21[k]));
  for (size_t k = 0; k < out.e_int22.size(); k++) out.e_int22[k] = kpow(4) * std::exp(sc(i22[k]));

  // fmath::log(float) table, built from the host libm like fmath's LogVar ctor (fmath.hpp:181-207) so the
  // final -kT*log(P) reproduces the reference's edge values (log(0f) = -88.03, log(inf) = 88.72; SURVEY Q2)
  const int LEN = 11, n = 1 << LEN;
  out.log_tbl.resize(2 * n);
  T.log_c_log2 = ::logf(2.0f) / (1 << 23);
  const double e = 1 / double(1 << 24), h = 1 / double(1 << LEN);
  for (int i = 0; i < n; i++) {
    double x = 1 + double(i) / n;
    double a = std::log(x);
    out.log_tbl[2 * i] = (float)a;
    if (i < n - 1) {
      double b = std::log(x + h - e);
      out.log_tbl[2 * i + 1] = (float)((b - a) / ((h - e) * (1 << 23)));
    } else {
      out.log_tbl[2 * i + 1] = (float)(1 / (x * (1 << 23)));
    }
  }
  return true;
}

template bool build_tables<double, kMaxSpan>(int, int, const ScaleSpec &, HostTablesT<double> &, std::string &);
template bool build_tables<float, kMaxSpan>(int, int, const ScaleSpec &, HostTablesT<float> &, std::string &);
template bool build_tables<double, kWideSpan>(int, int, const ScaleSpec &, HostTablesT<double, kWideSpan> &,
                                              std::string &);

void build_layout(int n, const char *const *seqs, const int32_t *lens, BatchLayout &out) {
  out.seq_off.resize(n);
  out.seq_len.assign(lens, lens + n);
  long long g = kPad;
  for (int k = 0; k < n; k++) {
    out.seq_off[k] = g;
    g += layout_columns(lens[k]);
  }
  out.NC = (g + kPad + 31) / 32 * 32;
  out.col_seq.assign((size_t)out.NC, -1);
  out.S.assign((size_t)out.NC, 0);
  for (int k = 0; k < n; k++) {
    const long long off = out.seq_off[k];
    const int L = lens[k];
    for (int i = 0; i <= L; i++) out.col_seq[(size_t)(off + i)] = k;
    for (int i = 0; i < L; i++) out.S[(size_t)(off + i + 1)] = encode_base(seqs[k][i]);
  }
}

}  // namespace prib
