// Plan compiler, tone-reservation PAPR reduction (EN 302 755 9.6.2, peak-cancellation form): the reserved-carrier
// sets of the symbols, the peak-cancellation kernel of each set and the tone-check twiddles.  Beyond the reference,
// which sends the reserved carriers as zeros (lib/pilotgenp1insert_cc_impl.cc).  Host only, built from
// OfdmPlan::carrier_type when the chain's stage is switched on.
#include "t2_plan.h"

#include <cmath>
#include <map>

namespace t2 {

namespace {
enum { P2PAPR_CARRIER = 3, TRPAPR_CARRIER = 4 };      // dvbt2_carrier_type_t values, as in t2_plan_ofdm.cc
}

bool build_papr_tr_plan(const OfdmPlan &op, PaprTrPlan *p, std::string *err)
{
  const int N = op.dims.fft_n, L = op.dims.num_symbols, cps = op.dims.c_ps;
  p->sym_set.assign(L, 0);
  p->bins.clear();
  p->tones = 0;
  std::map<std::vector<int32_t>, int> index;
  std::vector<std::vector<int32_t> > sets;
  for (int l = 0; l < L; l++) {
    // reserved carriers of the symbol in carrier order, as FFT bins (the bin k_ofdm fills for carrier k)
    std::vector<int32_t> b;
    for (int k = 0; k < cps; k++) {
      const uint8_t t = op.carrier_type[(size_t)l * cps + k];
      if (t == P2PAPR_CARRIER || t == TRPAPR_CARRIER) b.push_back((k + op.left_nulls + N / 2) & (N - 1));
    }
    if (b.empty() || (p->tones && (int)b.size() != p->tones)) {
      if (err) *err = "chain: tone reservation needs the same number of reserved carriers in every symbol";
      return false;
    }
    p->tones = (int)b.size();
    auto it = index.find(b);
    if (it == index.end()) {
      it = index.insert(std::make_pair(b, (int)sets.size())).first;
      sets.push_back(b);
    }
    p->sym_set[l] = it->second;
  }
  p->sets = (int)sets.size();
  const int S = p->tones;
  const double kPi2 = 6.283185307179586476925286766559;
  std::vector<double> cs(N), sn(N);
  for (int i = 0; i < N; i++) { cs[i] = std::cos(kPi2 * i / N); sn[i] = std::sin(kPi2 * i / N); }
  // p_n = (1/|S|) sum_{b in S} exp(+j 2 pi b n / N) in double, rounded to float.  A set that is another set shifted by
  // D bins (the data symbols' sets: one base set shifted by dx * s) has the kernel exp(+j 2 pi D n / N) p_n.
  p->kernel.assign((size_t)p->sets * N, cfloat());
  std::vector<std::vector<double> > kre, kim;
  std::vector<int> direct;          // sets computed term by term
  for (int s = 0; s < p->sets; s++) {
    const std::vector<int32_t> &b = sets[s];
    p->bins.insert(p->bins.end(), b.begin(), b.end());
    int base = -1, shift = 0;
    for (int d : direct) {
      const int D = (b[0] - sets[d][0]) & (N - 1);
      bool same = true;
      for (int i = 0; i < S && same; i++) same = b[i] == ((sets[d][i] + D) & (N - 1));
      if (same) { base = d; shift = D; break; }
    }
    std::vector<double> re(N), im(N);
    if (base < 0) {
      for (int n = 0; n < N; n++) {
        double r = 0.0, q = 0.0;
        for (int i = 0; i < S; i++) {
          const int a = (int)(((long long)b[i] * n) & (N - 1));
          r += cs[a]; q += sn[a];
        }
        re[n] = r / S; im[n] = q / S;
      }
      direct.push_back(s);
    }
    else
      for (int n = 0; n < N; n++) {
        const int a = (int)(((long long)shift * n) & (N - 1));
        re[n] = cs[a] * kre[base][n] - sn[a] * kim[base][n];
        im[n] = cs[a] * kim[base][n] + sn[a] * kre[base][n];
      }
    for (int n = 0; n < N; n++) { p->kernel[(size_t)s * N + n].re = (float)re[n]; p->kernel[(size_t)s * N + n].im = (float)im[n]; }
    kre.push_back(std::move(re)); kim.push_back(std::move(im));
  }
  p->tone_tw.resize(N);
  for (int i = 0; i < N; i++) { p->tone_tw[i].re = (float)cs[i]; p->tone_tw[i].im = (float)-sn[i]; }
  return true;
}

} // namespace t2
