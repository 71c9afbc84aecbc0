// Plan compiler, OFDM side: per-symbol carrier tables (P2 / scattered / continual / edge pilots,
// reserved tones, data), pilot reference sequence, P1 preamble, inverse-sinc table.
// Block 5 of the reference (lib/pilotgenp1insert_cc_impl.cc).  Host only, runs once per make().
#include "t2_plan.h"

#include <algorithm>
#include <cmath>
#include <complex>
#include <cstring>

#include "t2_std_tables.inc"

namespace t2 {

namespace {

// carrier classes, numbered like the reference's dvbt2_carrier_type_t (pilotgenp1insert_cc_impl.h:30-40)
enum { DATA_CARRIER = 1, P2PILOT_CARRIER, P2PAPR_CARRIER, TRPAPR_CARRIER, SCATTERED_CARRIER,
       CONTINUAL_CARRIER, P2PILOT_CARRIER_INVERTED, SCATTERED_CARRIER_INVERTED, CONTINUAL_CARRIER_INVERTED };

struct ReservedTones { const uint16_t *p2; const uint16_t *tr; int n; };

ReservedTones reserved_tones(int fi)
{
  static const ReservedTones t[6] = {
    { kP2Reserved_1k, kTrReserved_1k, 10 },   { kP2Reserved_2k, kTrReserved_2k, 18 },
    { kP2Reserved_4k, kTrReserved_4k, 36 },   { kP2Reserved_8k, kTrReserved_8k, 72 },
    { kP2Reserved_16k, kTrReserved_16k, 144 }, { kP2Reserved_32k, kTrReserved_32k, 288 } };
  return t[fi];
}

// Continual-pilot groups used per FFT size (EN 302 755 Annex G: CP groups nest with the FFT size;
// positions are taken modulo K_mod below 32K).  SURVEY Appendix C / reference :1292-2705.
const int kCpGroupsUsed[6] = { 1, 2, 3, 4, 5, 6 };
const int kCpModulo[6] = { 1632, 1632, 3264, 6528, 13056, 0 };
// MISO group 2 inverts continual pilots that coincide with inverted scattered-pilot positions
// (EN 302 755 9.2.8).  The reference implements that inversion only for the (FFT size, pilot pattern)
// pairs it considers usable with MISO; for the pairs below init_pilots() has no MISO branch
// (lib/pilotgenp1insert_cc_impl.cc:1292-2705) and continual pilots stay non-inverted.  Bit (pp-1).
const unsigned kCpNoMisoInversion[6] = {
  (1u << 1) | (1u << 3) | (1u << 4) | (1u << 6),   // 1K : PP2 PP4 PP5 PP7
  (1u << 1) | (1u << 6),                           // 2K : PP2 PP7
  (1u << 1) | (1u << 6),                           // 4K : PP2 PP7
  (1u << 1) | (1u << 6),                           // 8K : PP2 PP7
  (1u << 1) | (1u << 5) | (1u << 6),               // 16K: PP2 PP6 PP7
  (1u << 0) | (1u << 2) | (1u << 4) | (1u << 6) }; // 32K: PP1 PP3 PP5 PP7

} // namespace

bool build_ofdm_plan(const OfdmParams &prm, OfdmPlan *p, std::string *err)
{
  p->prm = prm;
  if (!ofdm_dims(prm.carriermode, prm.fftsize, prm.pilotpattern, prm.guardinterval, prm.numdatasyms,
                 prm.paprmode, prm.preamble, &p->dims, err)) return false;
  OfdmDims &d = p->dims;
  if (prm.vlength != d.fft_n) {
    if (err) *err = "pilotgenp1insert_cc: vlength must equal the FFT size";
    return false;
  }
  const int N = d.fft_n, CPS = d.c_ps, fi = d.fft_index, dx = d.dx, dy = d.dy, KEXT = d.k_ext;
  const int pp = prm.pilotpattern;
  const bool tx2 = d.miso && prm.misogroup == MISO_TX2;
  const bool tr = prm.paprmode == PAPR_TR || prm.paprmode == PAPR_BOTH;
  const bool ext = prm.carriermode == CARRIERS_EXTENDED;
  const ReservedTones rt = reserved_tones(fi);
  const int rt_off = fi >= 3 ? KEXT : 0;   // reference adds K_EXT to the P2 reserved set only for >= 8K
  const int L = d.num_symbols;
  p->left_nulls = (N - CPS) / 2 + 1;
  p->normalization = (float)(5.0 / std::sqrt(27.0 * CPS));
  p->samples_per_frame = L * (N + d.gi) + 2048;

  // ---- pilot reference sequence: PRBS x^11 + x^2 + 1 per carrier, PN chip per symbol (9.2.2)
  std::vector<uint8_t> prbs(CPS + d.k_offset + 1);
  {
    unsigned sr = 0x7ff;
    for (size_t i = 0; i < prbs.size(); i++) {
      const unsigned b = (sr ^ (sr >> 2)) & 1u;
      prbs[i] = (uint8_t)(sr & 1u);
      sr >>= 1;
      if (b) sr |= 0x400;
    }
  }
  auto pn = [](int l) { return (kPnSequencePacked[l >> 3] >> (7 - (l & 7))) & 1; };
  if (L > 2624) { if (err) *err = "pilotgenp1insert_cc: too many symbols"; return false; }

  // ---- carrier classes
  std::vector<uint8_t> p2map(CPS, DATA_CARRIER), fcmap(CPS, DATA_CARRIER);
  {
    const int step = (fi == 5 && !d.miso) ? 6 : 3;
    auto p2type = [&](int i) -> uint8_t {
      return (tx2 && ((i / 3) % 2) && (i % 3 == 0)) ? P2PILOT_CARRIER_INVERTED : P2PILOT_CARRIER;
    };
    for (int i = 0; i < CPS; i += step) p2map[i] = p2type(i);
    if (ext)
      for (int i = 0; i < KEXT; i++) {
        p2map[i] = p2type(i);
        p2map[i + (CPS - KEXT)] = p2type(i + (CPS - KEXT));
      }
    if (d.miso) {
      p2map[KEXT + 1] = P2PILOT_CARRIER; p2map[KEXT + 2] = P2PILOT_CARRIER;
      p2map[CPS - KEXT - 2] = P2PILOT_CARRIER; p2map[CPS - KEXT - 3] = P2PILOT_CARRIER;
    }
    for (int i = 0; i < rt.n; i++) p2map[rt.p2[i] + rt_off] = P2PAPR_CARRIER;
    if (d.miso)
      for (int i = 0; i < rt.n; i++) {
        const int ki = rt.p2[i] + KEXT;
        if (ki % 3 == 1 && (i == rt.n - 1 || ki + 1 != rt.p2[i + 1] + KEXT)) p2map[ki + 1] = P2PILOT_CARRIER;
        if (ki % 3 == 2 && (i == 0 || ki - 1 != rt.p2[i - 1] + KEXT)) p2map[ki - 1] = P2PILOT_CARRIER;
      }
    // frame closing symbol (9.2.7)
    for (int i = 0; i < CPS; i += dx)
      fcmap[i] = (tx2 && ((i / dx) % 2)) ? SCATTERED_CARRIER_INVERTED : SCATTERED_CARRIER;
    if ((fi == 0 && (pp == 3 || pp == 4)) || (fi == 1 && pp == 6)) fcmap[CPS - 2] = SCATTERED_CARRIER;
    const uint8_t edge = (tx2 && ((prm.numdatasyms + d.n_p2 - 1) % 2)) ? SCATTERED_CARRIER_INVERTED : SCATTERED_CARRIER;
    fcmap[0] = edge; fcmap[CPS - 1] = edge;
    if (tr) for (int i = 0; i < rt.n; i++) fcmap[rt.p2[i] + rt_off] = TRPAPR_CARRIER;
  }
  // continual pilots of data symbols (static over symbols)
  std::vector<uint8_t> cpmap(CPS, DATA_CARRIER);
  {
    const bool cp_inv = tx2 && !((kCpNoMisoInversion[fi] >> pp) & 1u);
    const int ngroups = (int)(sizeof(kCpGroups) / sizeof(kCpGroups[0]));
    for (int gi = 0; gi < ngroups; gi++) {
      const CpGroupDesc &g = kCpGroups[gi];
      if (g.pp != pp + 1 || g.group > kCpGroupsUsed[fi]) continue;
      for (int i = 0; i < g.n; i++) {
        const int k = kCpModulo[fi] ? g.k[i] % kCpModulo[fi] : g.k[i];
        if (k >= CPS) continue;
        cpmap[k] = (cp_inv && ((k / dx) % 2) && (k % dx == 0)) ? CONTINUAL_CARRIER_INVERTED : CONTINUAL_CARRIER;
      }
    }
    if (ext) {
      const int next = (int)(sizeof(kCpExt) / sizeof(kCpExt[0]));
      const int fk = fi == 3 ? 8 : fi == 4 ? 16 : fi == 5 ? 32 : 0;
      for (int e = 0; e < next; e++) {
        const CpExtDesc &g = kCpExt[e];
        if (g.pp != pp + 1 || g.fft_k != fk) continue;
        for (int i = 0; i < g.n; i++) {
          const int k = g.k[i];
          if (k >= CPS) continue;
          cpmap[k] = (cp_inv && ((k / dx) % 2) && (k % dx == 0)) ? CONTINUAL_CARRIER_INVERTED : CONTINUAL_CARRIER;
        }
      }
    }
  }

  // ---- pool of pilot values
  CellPool &pool = p->pool;
  pool.cells.clear();
  pool.l1post_base = 0; pool.l1post_cells = 0; pool.l1post_variants = 1;
  {
    const double a_p2 = (fi == 5 && !d.miso) ? std::sqrt(37.0) / 5.0 : std::sqrt(31.0) / 5.0;
    const double a_cp = fi <= 1 ? 4.0 / 3.0 : fi == 2 ? (4.0 * std::sqrt(2.0)) / 3.0 : 8.0 / 3.0;
    const double a_sp = pp <= 1 ? 4.0 / 3.0 : pp <= 3 ? 7.0 / 4.0 : 7.0 / 3.0;
    const double amps[3] = { a_p2, a_sp, a_cp };
    cfloat z; z.re = 0.0f; z.im = 0.0f;
    pool.cells.push_back(z);
    for (int a = 0; a < 3; a++) {
      cfloat v; v.im = 0.0f;
      v.re = (float)amps[a]; pool.cells.push_back(v);
      v.re = (float)(-amps[a]); pool.cells.push_back(v);
    }
  }
  enum { POOL_ZERO = 0, POOL_P2 = 1, POOL_SP = 3, POOL_CP = 5 };

  // ---- per-symbol carrier codes
  p->code.assign((size_t)L * CPS, 0);
  p->carrier_type.assign((size_t)L * CPS, 0);
  p->sym_data_start.assign(L + 1, 0);
  std::vector<uint8_t> map(CPS);
  int data_index = 0;
  const int fc_symbol = d.n_fc ? L - 1 : -1;
  for (int l = 0; l < L; l++) {
    if (l < d.n_p2) map = p2map;
    else if (l == fc_symbol) map = fcmap;
    else {
      map = cpmap;
      const int target = dx * (l % dy);
      for (int i = 0; i < CPS; i++) {
        int rem = (i - KEXT) % (dx * dy);
        if (rem < 0) rem += dx * dy;
        if (rem == target) map[i] = (tx2 && ((i / dx) % 2)) ? SCATTERED_CARRIER_INVERTED : SCATTERED_CARRIER;
      }
      const uint8_t edge = (tx2 && (l % 2)) ? SCATTERED_CARRIER_INVERTED : SCATTERED_CARRIER;
      map[0] = edge; map[CPS - 1] = edge;
      if (tr) {
        const int shift = ext ? dx * ((l + KEXT / dx) % dy) : dx * (l % dy);
        for (int i = 0; i < rt.n; i++) map[rt.tr[i] + shift] = TRPAPR_CARRIER;
      }
    }
    p->sym_data_start[l] = data_index;
    const int chip = pn(l);
    for (int k = 0; k < CPS; k++) {
      const int neg = prbs[k + d.k_offset] ^ chip;   // 1 -> negative amplitude
      int32_t c;
      switch (map[k]) {
        case DATA_CARRIER: c = data_index++; break;
        case P2PILOT_CARRIER: c = -(1 + POOL_P2 + neg); break;
        case P2PILOT_CARRIER_INVERTED: c = -(1 + POOL_P2 + (neg ^ 1)); break;
        case SCATTERED_CARRIER: c = -(1 + POOL_SP + neg); break;
        case SCATTERED_CARRIER_INVERTED: c = -(1 + POOL_SP + (neg ^ 1)); break;
        case CONTINUAL_CARRIER: c = -(1 + POOL_CP + neg); break;
        case CONTINUAL_CARRIER_INVERTED: c = -(1 + POOL_CP + (neg ^ 1)); break;
        default: c = -(1 + POOL_ZERO); break;
      }
      p->code[(size_t)l * CPS + k] = c;
      p->carrier_type[(size_t)l * CPS + k] = map[k];
    }
  }
  p->sym_data_start[L] = data_index;
  if (data_index != d.active_items) {
    if (err) *err = "pilotgenp1insert_cc: carrier map does not match the cell counts of this mode";
    return false;
  }

  // ---- P1 symbol (EN 302 755 9.8; reference :1119-1178, :2802-2810)
  {
    int seq[385], rnd[384], bits[384];
    {
      unsigned sr = 0x4e46;
      for (int i = 0; i < 384; i++) {
        const unsigned b = (sr ^ (sr >> 1)) & 1u;
        rnd[i] = b ? -1 : 1;
        sr >>= 1;
        if (b) sr |= 0x4000;
      }
    }
    const int s1 = prm.preamble & 7, s2 = ((prm.fftsize & 7) << 1) & 15;
    int n = 0;
    for (int i = 0; i < 8; i++) for (int j = 7; j >= 0; j--) bits[n++] = (kP1S1Patterns[s1 * 8 + i] >> j) & 1;
    for (int i = 0; i < 32; i++) for (int j = 7; j >= 0; j--) bits[n++] = (kP1S2Patterns[s2 * 32 + i] >> j) & 1;
    for (int i = 0; i < 8; i++) for (int j = 7; j >= 0; j--) bits[n++] = (kP1S1Patterns[s1 * 8 + i] >> j) & 1;
    seq[0] = 1;
    for (int i = 1; i < 385; i++) seq[i] = bits[i - 1] ? -seq[i - 1] : seq[i - 1];
    std::vector<double> freq(1024, 0.0);
    for (int i = 0; i < 384; i++) freq[kP1ActiveCarriers[i] + 86] = (double)(seq[i + 1] * rnd[i]);
    const double kPi2 = 6.283185307179586476925286766559;
    const float scale = (float)std::sqrt(384.0);
    std::vector<cfloat> ptime(1024), pshift(1024);
    for (int variant = 0; variant < 2; variant++) {
      // variant 1: spectrum moved up by one carrier (cyclically)
      std::vector<cfloat> &dst = variant ? pshift : ptime;
      for (int t = 0; t < 1024; t++) {
        double re = 0.0, im = 0.0;
        for (int m = 0; m < 1024; m++) {
          const double v = freq[m];
          if (v == 0.0) continue;
          const int mm = (m + variant) & 1023;        // position in the (shifted) spectrum
          const int bin = (mm + 512) & 1023;          // fftshift into FFT bin order
          const double ph = kPi2 * (double)((bin * t) & 1023) / 1024.0;
          re += v * std::cos(ph); im += v * std::sin(ph);
        }
        dst[t].re = (float)re / scale; dst[t].im = (float)im / scale;
      }
    }
    p->p1.clear();
    for (int j = 0; j < 542; j++) p->p1.push_back(pshift[j]);
    for (int j = 0; j < 1024; j++) p->p1.push_back(ptime[j]);
    for (int j = 542; j < 1024; j++) p->p1.push_back(pshift[j]);
  }

  // ---- inverse sinc (reference :1179-1219)
  p->inv_sinc.clear();
  if (prm.equalization) {
    double fs;
    switch (prm.bandwidth) {
      case BANDWIDTH_1_7_MHZ: fs = 131.0 * 1000000.0 / 71.0; break;
      case BANDWIDTH_5_0_MHZ: fs = 5.0 * 8000000.0 / 7.0; break;
      case BANDWIDTH_6_0_MHZ: fs = 6.0 * 8000000.0 / 7.0; break;
      case BANDWIDTH_7_0_MHZ: fs = 7.0 * 8000000.0 / 7.0; break;
      case BANDWIDTH_8_0_MHZ: fs = 8.0 * 8000000.0 / 7.0; break;
      case BANDWIDTH_10_0_MHZ: fs = 10.0 * 8000000.0 / 7.0; break;
      default: fs = 1.0; break;
    }
    const double fstep = fs / N;
    double f = 0.0, rms = 0.0;
    p->inv_sinc.assign(N, 0.0f);
    for (int i = 0; i < N / 2; i++) {
      const double x = 3.14159265358979323846 * f / fs;
      const double sinc = i == 0 ? 1.0 : std::sin(x) / x;
      rms += sinc * sinc;
      p->inv_sinc[i + N / 2] = (float)(1.0 / sinc);
      p->inv_sinc[N / 2 - i - 1] = (float)(1.0 / sinc);
      f += fstep;
    }
    rms = std::sqrt(rms / (N / 2));
    for (int i = 0; i < N; i++) p->inv_sinc[i] *= (float)rms;
  }
  return true;
}

bool compose_chain(const FramePlan &fp, const OfdmPlan &op, bool cells_cell_interleaved, ChainTables *out,
                   std::string *err)
{
  if (fp.mapped_items != op.dims.active_items || fp.dims.c_ps != op.dims.c_ps) {
    if (err) *err = "chain: frame mapper and pilot generator parameters do not describe the same frame";
    return false;
  }
  const int base = (int)op.pool.cells.size();
  out->pool = op.pool;
  out->pool.cells.insert(out->pool.cells.end(), fp.pool.cells.begin(), fp.pool.cells.end());
  out->pool.l1post_base = base + fp.pool.l1post_base;
  out->pool.l1post_cells = fp.pool.l1post_cells;
  out->pool.l1post_variants = fp.pool.l1post_variants;
  out->code.resize(op.code.size());
  for (size_t i = 0; i < op.code.size(); i++) {
    const int32_t c = op.code[i];
    if (c < 0) { out->code[i] = c; continue; }
    const int32_t f = fp.code[c];
    out->code[i] = f >= 0 ? (cells_cell_interleaved ? fp.ci_dst[f] : f) : -(1 + base + (-(f + 1)));
  }
  return true;
}

bool compose_chain16(const FramePlan &fp, const OfdmPlan &op, Chain16Tables *out, std::string *err)
{
  if (fp.mapped_items != op.dims.active_items || fp.dims.c_ps != op.dims.c_ps) {
    if (err) *err = "chain: frame mapper and pilot generator parameters do not describe the same frame";
    return false;
  }
  const int base = (int)op.pool.cells.size();
  out->pool = op.pool;
  out->pool.cells.insert(out->pool.cells.end(), fp.pool.cells.begin(), fp.pool.cells.end());
  out->pool.l1post_base = base + fp.pool.l1post_base;
  out->pool.l1post_cells = fp.pool.l1post_cells;
  out->pool.l1post_variants = fp.pool.l1post_variants;
  const int L = op.dims.num_symbols, cps = op.dims.c_ps;
  out->code.assign(op.code.size(), 0);
  out->run_desc.clear();
  out->run_ptr.assign(L + 1, 0);
  out->stage_bytes.assign(L, 0);
  out->run_cnt.assign(L, 0);
  out->max_slots = 0;
  out->max_runs = 0;
  out->plp.assign(op.code.size(), 0);
  // cell-interleaved index -> (PLP, address in the chain's cell memory: the PLP's region, see FramePlan::plp_chain_off)
  std::vector<uint8_t> plp_of((size_t)fp.stream_items);
  for (int pl = 0; pl < fp.num_plp; pl++)
    std::fill(plp_of.begin() + fp.plp_first_cell[pl], plp_of.begin() + fp.plp_first_cell[pl + 1], (uint8_t)pl);
  auto addr = [&](int32_t x) { return x - fp.plp_first_cell[plp_of[x]] + fp.plp_chain_off[plp_of[x]]; };
  for (int l = 0; l < L; l++) {
    const int s0 = op.sym_data_start[l], s1 = op.sym_data_start[l + 1];     // frame positions of this symbol
    // staging layout: the symbol's source cells sorted by source address, copied run by run with bulk
    // asynchronous copies (cp.async.bulk: 16-byte aligned source, destination and size).  A run is a maximal
    // stretch of consecutive source cells (2 bytes each); its copy is the enclosing 16-byte aligned span of the
    // frame's cell memory, landed at the next 16-byte aligned staging offset, so a cell keeps its position inside
    // its 16-byte unit (up to 7 unused cells at either end of a run).
    std::vector<std::pair<int32_t, int32_t> > ps;      // (source cell, frame-order position - s0)
    for (int pos = s0; pos < s1; pos++) {
      const int32_t f = fp.framed[pos];
      if (f >= 0) ps.push_back(std::make_pair(addr(fp.ci_dst[f]), pos - s0));
    }
    std::sort(ps.begin(), ps.end());
    std::vector<int32_t> slot_of_pos(s1 - s0, -1);
    if ((out->run_desc.size() / 2) & 1) { out->run_desc.push_back(0); out->run_desc.push_back(0); }   // lists start 16-byte aligned
    out->run_ptr[l] = (int32_t)(out->run_desc.size() / 2);
    int32_t next_unit = 0;                              // 16-byte staging units used so far
    size_t i = 0;
    while (i < ps.size()) {
      const int32_t first_unit = ps[i].first >> 3;      // 8 cells per 16-byte unit
      size_t j = i + 1;
      while (j < ps.size() && ps[j].first == ps[j - 1].first + 1) j++;
      const int32_t last_unit = ps[j - 1].first >> 3;
      int32_t u0 = first_unit;
      while (u0 <= last_unit) {                         // a copy carries at most 65535 units (1 MB): split longer runs
        const int32_t n = std::min<int32_t>(last_unit - u0 + 1, 65535);
        if (next_unit + (u0 - first_unit) + n > 8191) {      // staging byte offsets are 17-bit
          if (err) *err = "chain: a symbol's cells do not fit the staging address range";
          return false;
        }
        out->run_desc.push_back(u0);
        out->run_desc.push_back((int32_t)(((uint32_t)(next_unit + (u0 - first_unit)) << 16) | (uint32_t)n));
        u0 += n;
      }
      for (size_t k = i; k < j; k++) slot_of_pos[ps[k].second] = 8 * next_unit + (ps[k].first - 8 * first_unit);
      next_unit += last_unit - first_unit + 1;
      i = j;
    }
    out->stage_bytes[l] = 16 * next_unit;
    out->run_cnt[l] = (int32_t)(out->run_desc.size() / 2) - out->run_ptr[l];
    if (out->run_cnt[l] > out->max_runs) out->max_runs = out->run_cnt[l];
    if (8 * next_unit > out->max_slots) out->max_slots = 8 * next_unit;
    // carrier codes: data carrier -> staging slot of its cell
    for (int k = 0; k < cps; k++) {
      const int32_t c = op.code[(size_t)l * cps + k];
      int32_t v;
      if (c < 0) v = c;
      else {
        const int32_t pos = fp.fi_src[c];
        const int32_t f = fp.framed[pos];
        v = f >= 0 ? slot_of_pos[pos - s0] : -(1 + base + (-(f + 1)));
        if (f >= 0) out->plp[(size_t)l * cps + k] = plp_of[fp.ci_dst[f]];
      }
      out->code[(size_t)l * cps + k] = v;
    }
  }
  out->run_ptr[L] = (int32_t)(out->run_desc.size() / 2);
  out->run_desc.push_back(0); out->run_desc.push_back(0);      // the kernel fetches lists in 16-byte units
  return true;
}

bool compose_miso(const OfdmPlan &op, const Chain16Tables &t, const OfdmPlan &og, bool group2, MisoTables *out,
                  std::string *err)
{
  const int L = op.dims.num_symbols, cps = op.dims.c_ps;
  bool same = og.dims.num_symbols == L && og.dims.c_ps == cps && og.pool.cells.size() == op.pool.cells.size();
  for (size_t i = 0; same && i < og.pool.cells.size(); i++)      // pilot amplitudes (the pool part og's codes index)
    same = og.pool.cells[i].re == t.pool.cells[i].re && og.pool.cells[i].im == t.pool.cells[i].im;
  if (!same) {
    if (err) *err = "chain: the MISO groups' pilot plans do not describe the same frame";
    return false;
  }
  out->code.assign((size_t)L * cps, 0);
  out->plp.assign((size_t)L * cps, 0);
  out->pool = t.pool;
  // per pool cell: 0 = not yet placed, 1 = lands at an even position of group 2 (-conj), 2 = at an odd one (conj)
  std::vector<uint8_t> placed(t.pool.cells.size(), 0);
  std::vector<int32_t> carrier_of;
  for (int l = 0; l < L; l++) {
    const int s = op.sym_data_start[l], n = op.sym_data_start[l + 1] - s;
    if (group2 && (n & 1)) {
      if (err) *err = "chain: MISO processing needs an even number of cells in every symbol; symbol " + std::to_string(l) +
                      " has " + std::to_string(n);
      return false;
    }
    carrier_of.assign(n, -1);
    for (int k = 0; k < cps; k++) {
      const int32_t c = op.code[(size_t)l * cps + k];
      if ((c >= 0) != (og.code[(size_t)l * cps + k] >= 0) || (c >= 0 && c != og.code[(size_t)l * cps + k])) {
        if (err) *err = "chain: the MISO groups' data carriers differ";
        return false;
      }
      if (c >= 0) carrier_of[c - s] = k;
    }
    for (int k = 0; k < cps; k++) {
      const size_t ck = (size_t)l * cps + k;
      const int32_t c = og.code[ck];
      if (c < 0) { out->code[ck] = c; continue; }
      const int i = c - s;
      const size_t src = (size_t)l * cps + carrier_of[group2 ? i ^ 1 : i];
      const int32_t v = t.code[src];
      out->code[ck] = v;
      out->plp[ck] = t.plp[src];
      if (!group2 || v >= 0) continue;
      const int32_t p = ~v;
      const cfloat z = t.pool.cells[p];
      if (z.re == 0.0f && z.im == 0.0f) continue;      // the shared zero cell: -conj(0) = conj(0) = 0
      const uint8_t want = (uint8_t)(1 + (i & 1));
      if (placed[p] && placed[p] != want) {
        if (err) *err = "chain: a pool cell lands at an even and at an odd position of a symbol";
        return false;
      }
      placed[p] = want;
    }
  }
  // a placed L1-post cell of variant 0 stands for the same cell of every variant (same position in every frame)
  const CellPool &q = t.pool;
  for (size_t p = 0; p < placed.size(); p++) {
    if (!placed[p]) continue;
    const bool post = (int)p >= q.l1post_base && (int)p < q.l1post_base + q.l1post_cells;
    for (int v = 0; v < (post ? q.l1post_variants : 1); v++) {
      cfloat &z = out->pool.cells[p + (size_t)v * q.l1post_cells];
      if (placed[p] == 1) z.re = -z.re;
      else z.im = -z.im;
    }
  }
  return true;
}

} // namespace t2
