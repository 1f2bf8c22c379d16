// TEST INFRASTRUCTURE (oracle) -- parity unpinned, see oracle/README.md.
// Position-likelihood tables and k-mer frequency limits of daccord, restated.
//   computeOffsetLikely   : reference src/ComputeOffsetLikely.hpp:26-134
//   OffsetLikely::setup   : reference src/OffsetLikely.hpp:59-99
//   DotProduct            : reference src/DotProduct.hpp:29-137
//   KmerLimit             : reference src/DebruijnGraph.hpp:28-75
// Conventions C3, C4, C5 of oracle/README.md apply (libmaus2 Binom / GmpFloat / FFT
// convolution are replaced by direct double arithmetic in the order written here).
#pragma once
#include <cstdint>
#include <cmath>
#include <vector>
#include <utility>
#include <algorithm>

namespace oracle {

// reference src/DotProduct.hpp:29-137
struct DotVec {
  uint64_t firstsign = 0;        // first read position with a coefficient
  std::vector<double> V;         // coefficients for read positions firstsign..
  std::vector<uint64_t> VS;      // C5: floor(2^32 * V[i])
  uint64_t size() const { return firstsign + V.size(); }
  double at(uint64_t i) const {  // DotProduct::operator[] (src/DotProduct.hpp:75-86)
    if (i < firstsign) return 0.0;
    uint64_t j = i - firstsign;
    return j < V.size() ? V[j] : 0.0;
  }
  // DotProduct::dotproduct (src/DotProduct.hpp:100-120)
  double dot(const double* O, uint64_t Os) const {
    double s = 0;
    for (uint64_t i = 0; i < V.size(); ++i) {
      uint64_t j = firstsign + i;
      if (j < Os) s += V[i] * O[j]; else break;
    }
    return s;
  }
};

struct OffsetLikely {
  std::vector<DotVec> DP, DPnorm, DPnormSquare;
  std::vector<std::pair<uint64_t, uint64_t>> Vsupport;
  uint64_t size() const { return DP.size(); }
  // src/OffsetLikely.hpp:34-43
  uint64_t supportLow(int64_t i) const { return i < (int64_t)Vsupport.size() ? Vsupport[i].first : DPnorm.size(); }
  uint64_t supportHigh(int64_t i) const { return i < (int64_t)Vsupport.size() ? Vsupport[i].second : DPnorm.size(); }
};

// C4: direct convolution, ascending i, double accumulation
inline std::vector<double> conv_direct(const std::vector<double>& a, const std::vector<double>& b) {
  if (a.empty() || b.empty()) return {};
  std::vector<double> out(a.size() + b.size() - 1, 0.0);
  for (size_t n = 0; n < out.size(); ++n) {
    size_t lo = n + 1 > b.size() ? n + 1 - b.size() : 0;
    size_t hi = std::min(n, a.size() - 1);
    double s = 0.0;
    for (size_t i = lo; i <= hi; ++i) s += a[i] * b[n - i];
    out[n] = s;
  }
  return out;
}

// C4: P(X=j), j=0..l of Binomial(l,p) by the multiplicative recurrence
inline std::vector<double> binom_vector(double p, uint64_t l) {
  std::vector<double> b(l + 1, 0.0);
  double q = 1.0 - p;
  if (q == 0.0) { b[l] = 1.0; return b; }
  double r = 1.0;
  for (uint64_t t = 0; t < l; ++t) r *= q;
  b[0] = r;
  double ratio = p / q;
  for (uint64_t j = 0; j < l; ++j) b[j + 1] = b[j] * (double)(l - j) / (double)(j + 1) * ratio;
  return b;
}

inline OffsetLikely computeOffsetLikely(uint64_t maxl, double p_i, double p_d) {
  OffsetLikely OL;
  double q_i = 1.0 - p_i, f_i = q_i;
  std::vector<double> P_I;
  while (f_i >= 1e-7) { P_I.push_back(f_i); f_i *= p_i; }   // ComputeOffsetLikely.hpp:44-48
  std::vector<double> C_I(1, 1.0);
  for (uint64_t l = 0; l <= maxl; ++l) {
    C_I = conv_direct(C_I, P_I);                            // :62
    std::vector<double> V_D = binom_vector(p_d, l);         // :69
    std::vector<double> V_I(V_D.size() - 1 + C_I.size(), 0.0);
    std::copy(C_I.begin(), C_I.end(), V_I.begin() + (V_D.size() - 1));
    std::reverse(V_D.begin(), V_D.end());                   // :80
    std::vector<double> F_I = conv_direct(V_D, V_I);        // :91
    bool signfound = false; int64_t firstsign = 0; std::vector<double> VP;
    for (uint64_t j = 0; j < F_I.size(); ++j)
      if (F_I[j] >= 1e-5) {                                 // :100
        if (!signfound) { signfound = true; firstsign = (int64_t)j - (int64_t)l; }
        uint64_t off = (int64_t)j - (int64_t)l - firstsign;
        while (!(off < VP.size())) VP.push_back(0);
        VP[off] = F_I[j];
      }
    DotVec d; d.firstsign = (uint64_t)firstsign; d.V = VP;
    OL.DP.push_back(d);
  }
  // OffsetLikely::setup (src/OffsetLikely.hpp:59-99)
  uint64_t maxsize = 0;
  for (auto& d : OL.DP) maxsize = std::max(maxsize, d.size());
  std::vector<double> dsum;
  for (uint64_t i = 0; i < maxsize; ++i) {
    double sum = 0.0;
    for (uint64_t j = 0; j < OL.DP.size(); ++j) sum += OL.DP[j].at(i);
    dsum.push_back(sum);
  }
  OL.DPnorm = OL.DP;
  for (auto& d : OL.DPnorm)
    for (uint64_t j = 0; j < maxsize; ++j)
      if (j >= d.firstsign && j - d.firstsign < d.V.size()) d.V[j - d.firstsign] /= dsum[j];
  uint64_t j = 0, k = 0;
  for (uint64_t i = 0; i < maxsize; ++i) {
    while (j < OL.DPnorm.size() && i >= OL.DPnorm[j].firstsign + OL.DPnorm[j].V.size()) ++j;
    while (k < OL.DPnorm.size() && OL.DPnorm[k].firstsign <= i) ++k;
    OL.Vsupport.push_back({j, k});
  }
  OL.DPnormSquare = OL.DP;
  for (auto& d : OL.DPnormSquare) {                          // DotProduct::normalise :128-136
    double s = 0.0;
    for (double v : d.V) s += v * v;
    double c = std::sqrt(1.0 / s);
    for (double& v : d.V) v *= c;
    d.VS.resize(d.V.size());                                 // C5 (DotProduct.hpp:54-60 intent)
    for (size_t i = 0; i < d.V.size(); ++i) d.VS[i] = (uint64_t)(4294967296.0 * d.V[i]);
  }
  return OL;
}

// C3.  The pmf is walked unnormalised from its mode (term 1) outward by the ratio recurrence, so no term underflows for any n
// (q^n, the usual starting term, is 0 or a denormal once n ln q < -708).  A walk stops after its first term below 1e-30: the
// terms fall monotonically away from the mode, so what is dropped is below n * 1e-30 of a total >= 1.  The CDF is the running
// sum in ascending m against the walk's own total.
inline uint64_t binomRowUpperLimit(double p, uint64_t n, double lim) {
  double q = 1.0 - p;
  if (!(q > 0.0)) return n;                                 // p = 1 (and NaN)
  const double up = p / q, down = q / p;
  const double mf = std::floor((double)(n + 1) * p);
  const uint64_t M = mf <= 0.0 ? 0 : (mf >= (double)n ? n : (uint64_t)mf);
  std::vector<double> hi(1, 1.0), lo;                       // hi[i]: term of m = M + i; lo[i]: term of m = M - 1 - i
  for (uint64_t m = M; m < n && hi.back() >= 1e-30; ++m) hi.push_back(hi.back() * (double)(n - m) / (double)(m + 1) * up);
  for (uint64_t m = M; m > 0 && (lo.empty() || lo.back() >= 1e-30); --m) lo.push_back((lo.empty() ? 1.0 : lo.back()) * (double)m / (double)(n - m + 1) * down);
  double total = 0.0;
  for (size_t i = lo.size(); i-- > 0;) total += lo[i];
  for (double t : hi) total += t;
  double sum = 0.0;
  for (size_t i = lo.size(); i-- > 0;) { sum += lo[i]; if (sum >= lim * total) return M - 1 - i; }
  for (size_t i = 0; i < hi.size(); ++i) { sum += hi[i]; if (sum >= lim * total) return M + i; }
  return n;
}

// reference src/DebruijnGraph.hpp:28-75
struct KmerLimit {
  double p_k;
  std::vector<uint64_t> Vlim;
  KmerLimit(double rp_k = 0.0, uint64_t preload = 0) : p_k(rp_k) { for (uint64_t i = 0; i < preload; ++i) getLimit(i); }
  double getLimit(uint64_t i) {
    if (p_k) {
      while (!(i < Vlim.size())) Vlim.push_back(binomRowUpperLimit(p_k, Vlim.size(), 0.99));
      return (double)Vlim[i];
    }
    return 0;
  }
};

}  // namespace oracle
