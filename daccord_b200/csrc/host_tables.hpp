// host_tables.hpp -- host-side construction of the read-only tables the window kernel consumes.
// Replaces, for this path, daccord's computeOffsetLikely (reference src/ComputeOffsetLikely.hpp:26-134),
// OffsetLikely::setup (src/OffsetLikely.hpp:59-99), DotProduct::normalise / the intended
// computeShifted (src/DotProduct.hpp:54-60, :128-136) and KmerLimit (src/DebruijnGraph.hpp:28-75,
// created in src/daccord.cpp:1981-1988).  libmaus2's GMP-512 binomials and FFT convolution are
// replaced by direct double arithmetic; the arrays below (not the formulas) are the contract with
// the kernel: dense [NP][MS] matrices, zero outside each row's support.
#pragma once
#include <cstdint>
#include <cmath>
#include <vector>
#include <algorithm>

namespace dcu_host {

struct HostTables {
  int NP = 0, MS = 0, KLIMN = 0, nk = 0;
  std::vector<double> DPn, DPsq;                 // [NP][MS]
  std::vector<unsigned long long> VSq;           // [MS+1][NP] transposed, last row zero (guard for read positions >= MS)
  std::vector<uint16_t> suplo, suphi;            // [MS]
  std::vector<unsigned long long> klim;          // [nk][KLIMN]
};

// Smallest m with Binomial(n, p) CDF(m) >= lim, n if none.  The pmf is walked unnormalised from its mode (term 1) outward by the
// ratio recurrence, so no term underflows for any n (q^n, the usual starting term, is 0 or a denormal once n ln q < -708 and
// then wrecks the limit of deep windows).  A walk stops after its first term below 1e-30: the terms fall monotonically away from
// the mode, so what is dropped is below n * 1e-30 of a total >= 1.  The CDF is the running sum in ascending m against the walk's
// own total.  Same operations in the same order as oracle/tables.hpp binomRowUpperLimit.
inline unsigned long long binom_upper_limit(double p, unsigned long long n, double lim) {
  double q = 1.0 - p;
  if (!(q > 0.0)) return n;                                 // p = 1 (and NaN)
  const double up = p / q, down = q / p;
  const double mf = std::floor((double)(n + 1) * p);
  const unsigned long long M = mf <= 0.0 ? 0 : (mf >= (double)n ? n : (unsigned long long)mf);
  std::vector<double> hi(1, 1.0), lo;                       // hi[i]: term of m = M + i; lo[i]: term of m = M - 1 - i
  for (unsigned long long m = M; m < n && hi.back() >= 1e-30; ++m) hi.push_back(hi.back() * (double)(n - m) / (double)(m + 1) * up);
  for (unsigned long long m = M; m > 0 && (lo.empty() || lo.back() >= 1e-30); --m) lo.push_back((lo.empty() ? 1.0 : lo.back()) * (double)m / (double)(n - m + 1) * down);
  double total = 0.0;
  for (size_t i = lo.size(); i-- > 0;) total += lo[i];
  for (double t : hi) total += t;
  double sum = 0.0;
  for (size_t i = lo.size(); i-- > 0;) { sum += lo[i]; if (sum >= lim * total) return M - 1 - i; }
  for (size_t i = 0; i < hi.size(); ++i) { sum += hi[i]; if (sum >= lim * total) return M + i; }
  return n;
}

// P(read offset = j | true offset = l): (l+1)-fold geometric insertion law convolved with Binomial(l,p_d) deletions
inline void build_tables(int w, double p_i, double p_d, double est_cor, int k_lo, int k_hi, int klimn, HostTables& T) {
  const int NP = w + 1;
  // insertion-count law before/at one base, truncated at 1e-7
  std::vector<double> geo;
  for (double f = 1.0 - p_i; f >= 1e-7; f *= p_i) geo.push_back(f);
  std::vector<std::vector<double>> rows(NP);
  std::vector<int> first(NP, 0);
  std::vector<double> ins(1, 1.0);               // ins[c] = P(c insertions in total so far)
  for (int l = 0; l < NP; ++l) {
    {                                            // ins <- ins (*) geo, ascending index accumulation
      std::vector<double> nx(ins.size() + geo.size() - 1, 0.0);
      for (size_t n = 0; n < nx.size(); ++n) {
        size_t lo = n + 1 > geo.size() ? n + 1 - geo.size() : 0, hi = std::min(n, ins.size() - 1);
        double s = 0.0;
        for (size_t i = lo; i <= hi; ++i) s += ins[i] * geo[n - i];
        nx[n] = s;
      }
      ins.swap(nx);
    }
    // deletion law, index d = number of deleted bases
    std::vector<double> del(l + 1, 0.0);
    {
      double q = 1.0 - p_d;
      if (q == 0.0) del[l] = 1.0;
      else {
        double r = 1.0;
        for (int t = 0; t < l; ++t) r *= q;
        del[0] = r;
        double ratio = p_d / q;
        for (int j = 0; j < l; ++j) del[j + 1] = del[j] * (double)(l - j) / (double)(j + 1) * ratio;
      }
    }
    // offset = l - d + c.  F[j], j = (l - d) + (l + c), is the reference's convolution index; offset = j - l.
    // Accumulate in ascending i = l - d, which is the order the reference's reversed vector is walked in.
    const int nF = (int)(2 * l + ins.size());
    std::vector<double> row; int fs = 0; bool found = false;
    for (int j = 0; j < nF; ++j) {
      double s = 0.0;
      for (int i = 0; i <= l; ++i) {             // i = l - d
        int vi = j - i;                          // index into the l-zero-padded insertion vector
        if (vi < 0) break;
        if (vi < l) { s += del[l - i] * 0.0; continue; }
        int cidx = vi - l;
        if (cidx < (int)ins.size()) s += del[l - i] * ins[cidx];
      }
      if (s >= 1e-5) {
        if (!found) { found = true; fs = j - l; }
        int off = j - l - fs;
        if ((int)row.size() <= off) row.resize(off + 1, 0.0);
        row[off] = s;
      }
    }
    rows[l] = row; first[l] = fs;
  }
  int MS = 0;
  for (int l = 0; l < NP; ++l) MS = std::max(MS, first[l] + (int)rows[l].size());
  T.NP = NP; T.MS = MS;
  T.DPn.assign((size_t)NP * MS, 0.0); T.DPsq.assign((size_t)NP * MS, 0.0); T.VSq.assign((size_t)(MS + 1) * NP, 0ull);
  // column sums over true positions, ascending l (OffsetLikely.hpp:68-77)
  std::vector<double> colsum(MS, 0.0);
  for (int pos = 0; pos < MS; ++pos) {
    double s = 0.0;
    for (int l = 0; l < NP; ++l) { int o = pos - first[l]; s += (o >= 0 && o < (int)rows[l].size()) ? rows[l][o] : 0.0; }
    colsum[pos] = s;
  }
  for (int l = 0; l < NP; ++l) {
    double ss = 0.0;
    for (double v : rows[l]) ss += v * v;
    double cn = std::sqrt(1.0 / ss);
    for (int o = 0; o < (int)rows[l].size(); ++o) {
      int pos = first[l] + o;
      T.DPn[(size_t)l * MS + pos] = rows[l][o] / colsum[pos];
      double v = rows[l][o] * cn;
      T.DPsq[(size_t)l * MS + pos] = v;
      T.VSq[(size_t)pos * NP + l] = (unsigned long long)(4294967296.0 * v);
    }
  }
  // support ranges per read position (OffsetLikely.hpp:81-93)
  T.suplo.assign(MS, 0); T.suphi.assign(MS, 0);
  int j = 0, k = 0;
  for (int pos = 0; pos < MS; ++pos) {
    while (j < NP && pos >= first[j] + (int)rows[j].size()) ++j;
    while (k < NP && first[k] <= pos) ++k;
    T.suplo[pos] = (uint16_t)j; T.suphi[pos] = (uint16_t)k;
  }
  // k-mer frequency limits: smallest m with Binomial(n, est_cor^k) CDF >= 0.99 (README convention C3)
  T.KLIMN = klimn; T.nk = k_hi - k_lo + 1;
  T.klim.assign((size_t)T.nk * klimn, 0ull);
  for (int kk = k_lo; kk <= k_hi; ++kk) {
    double pk = std::pow(est_cor, (double)kk);
    for (int n = 0; n < klimn; ++n)
      T.klim[(size_t)(kk - k_lo) * klimn + n] = pk == 0.0 ? 0ull : binom_upper_limit(pk, (unsigned long long)n, 0.99);
  }
}

}  // namespace dcu_host
