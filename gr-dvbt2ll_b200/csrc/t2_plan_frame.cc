// Plan compiler, frame side: OFDM dimensions, L1-pre / L1-post signalling cells, cell interleaver,
// time interleaver, frame assembly (incl. the multi-P2 zig-zag) and frequency interleaver, all
// folded into ONE gather table per T2 frame (block 4 of the reference,
// lib/framemapperfint_cc_impl.cc).  Host only, runs once per make().
#include <atomic>
#include <cstdlib>
#include "t2_plan.h"

#include <cmath>
#include <cstring>

#include "t2_std_tables.inc"

namespace t2 {

static std::atomic<int> g_overfull_policy(-1);
void set_overfull_policy(int policy) { g_overfull_policy.store(policy ? 1 : 0); }
bool overfull_warn_policy()
{
  int v = g_overfull_policy.load();
  if (v < 0) {
    const char *e = std::getenv("DVBT2LL_OVERFULL");
    v = (e && (e[0] == 'w' || e[0] == 'W' || e[0] == '1')) ? 1 : 0;
    g_overfull_policy.store(v);
  }
  return v == 1;
}


// ------------------------------------------------------------------------------------------------
// OFDM dimensions (EN 302 755 Tables 47-49, 51, 67; reference framemapper :290-915, pilotgen :56-666)
// ------------------------------------------------------------------------------------------------
static int fft_index_of(int fftsize)
{
  switch (fftsize) {
    case FFTSIZE_1K: return 0;
    case FFTSIZE_2K: return 1;
    case FFTSIZE_4K: return 2;
    case FFTSIZE_8K: case FFTSIZE_8K_T2GI: return 3;
    case FFTSIZE_16K: case FFTSIZE_16K_T2GI: return 4;
    case FFTSIZE_32K: case FFTSIZE_32K_T2GI: return 5;
  }
  return -1;
}

bool ofdm_dims(int carriermode, int fftsize, int pilotpattern, int guardinterval, int numdatasyms,
               int paprmode, int preamble, OfdmDims *d, std::string *err)
{
  static const int n_p2[6] = { 16, 8, 4, 2, 1, 1 };
  static const int c_p2_siso[6] = { 558, 1118, 2236, 4472, 8944, 22432 };
  static const int c_p2_miso[6] = { 546, 1098, 2198, 4398, 8814, 17612 };
  static const int c_ps_norm[6] = { 853, 1705, 3409, 6817, 13633, 27265 };
  static const int c_ps_ext[6] = { 853, 1705, 3409, 6913, 13921, 27841 };
  static const int k_ext[6] = { 0, 0, 0, 48, 144, 288 };
  static const int tr_cells[6] = { 10, 18, 36, 72, 144, 288 };
  static const int dxs[8] = { 3, 6, 6, 12, 12, 24, 24, 6 };
  static const int dys[8] = { 4, 2, 4, 2, 4, 2, 4, 16 };
  const int fi = fft_index_of(fftsize);
  if (fi < 0) { if (err) *err = "unknown FFT size"; return false; }
  if (pilotpattern < 0 || pilotpattern > 7) { if (err) *err = "unknown pilot pattern"; return false; }
  if (guardinterval < GI_1_32 || guardinterval > GI_19_256) { if (err) *err = "unknown guard interval"; return false; }
  const int ext = carriermode == CARRIERS_EXTENDED ? 1 : 0;
  d->fft_index = fi;
  d->fft_n = 1024 << fi;
  d->miso = !(preamble == PREAMBLE_T2_SISO || preamble == PREAMBLE_T2_LITE_SISO);
  d->n_p2 = n_p2[fi];
  d->c_p2 = d->miso ? c_p2_miso[fi] : c_p2_siso[fi];
  d->c_ps = ext ? c_ps_ext[fi] : c_ps_norm[fi];
  d->k_ext = ext ? k_ext[fi] : 0;
  d->k_offset = ext ? 0 : k_ext[fi];
  const uint16_t *cc = &kCellCounts[((fi * 2 + ext) * 8 + pilotpattern) * 3];
  d->c_data = cc[0]; d->n_fc = cc[1]; d->c_fc = cc[2];
  if (paprmode == PAPR_TR || paprmode == PAPR_BOTH) {
    if (d->c_data) d->c_data -= tr_cells[fi];
    if (d->n_fc) d->n_fc -= tr_cells[fi];
    if (d->c_fc) d->c_fc -= tr_cells[fi];
  }
  if (!d->miso) {
    // combinations without a frame closing symbol (EN 302 755 Table 51 / reference :898-915)
    if ((guardinterval == GI_1_128 && pilotpattern == 6) || (guardinterval == GI_1_32 && pilotpattern == 3) ||
        (guardinterval == GI_1_16 && pilotpattern == 1) || (guardinterval == GI_19_256 && pilotpattern == 1)) {
      d->n_fc = 0; d->c_fc = 0;
    }
  }
  d->dx = dxs[pilotpattern];
  d->dy = dys[pilotpattern];
  const int N = d->fft_n;
  switch (guardinterval) {
    case GI_1_32: d->gi = N / 32; break;
    case GI_1_16: d->gi = N / 16; break;
    case GI_1_8: d->gi = N / 8; break;
    case GI_1_4: d->gi = N / 4; break;
    case GI_1_128: d->gi = N / 128; break;
    case GI_19_128: d->gi = (N * 19) / 128; break;
    default: d->gi = (N * 19) / 256; break;
  }
  d->num_symbols = numdatasyms + d->n_p2;
  if (d->n_fc == 0) {
    d->num_data_symbols_no_fc = numdatasyms;
    d->active_items = d->n_p2 * d->c_p2 + numdatasyms * d->c_data;
  }
  else {
    d->num_data_symbols_no_fc = numdatasyms - 1;
    d->active_items = d->n_p2 * d->c_p2 + (numdatasyms - 1) * d->c_data + d->n_fc;
  }
  if (numdatasyms < 1 || d->c_data == 0) {
    if (err) *err = "unsupported (FFT size, pilot pattern) combination or no data symbols";
    return false;
  }
  return true;
}

// ------------------------------------------------------------------------------------------------
// L1 signalling (EN 302 755 clause 7; reference :114-250, :1366-1910)
// ------------------------------------------------------------------------------------------------
namespace {

struct BitWriter {
  std::vector<uint8_t> b;
  void put(unsigned v, int n) { for (int i = n - 1; i >= 0; i--) b.push_back((uint8_t)((v >> i) & 1u)); }
};

void append_crc32(std::vector<uint8_t> &bits)
{
  const uint32_t c = crc32_bits(bits.data(), (int)bits.size());
  for (int n = 31; n >= 0; n--) bits.push_back((uint8_t)((c >> n) & 1u));
}

// systematic BCH(short, t=12) + LDPC(16200, code) of an already padded K_bch-bit word
std::vector<uint8_t> l1_fec(const std::vector<uint8_t> &kbits, int nbch, int ldpc_code)
{
  const std::vector<uint8_t> g = bch_generator(168);
  std::vector<uint8_t> bch(kbits);
  const std::vector<uint8_t> par = bch_parity_bits(kbits.data(), (int)kbits.size(), g);
  bch.insert(bch.end(), par.begin(), par.end());
  std::vector<uint8_t> cw(16200);
  ldpc_encode_host(ldpc_code, bch.data(), nbch, 16200, cw.data());
  return cw;
}

void qam_lut(int bits, std::vector<cfloat> &lut)
{
  // non-rotated Gray-mapped constellations, same arithmetic as the data-cell LUTs
  MapPlan mp;
  std::string e;
  build_map_plan(FECFRAME_SHORT, C1_2, bits / 2 - 1, 0, &mp, &e);
  lut = mp.lut;
}

int l1_ldpc_code(bool pre)
{
  // the two L1 codes are appended to kLdpcCodes with rate = -1: 16K 1/4 (q = 36), 16K 1/2 (q = 25)
  const int n = (int)(sizeof(kLdpcCodes) / sizeof(kLdpcCodes[0]));
  for (int i = 0; i < n; i++)
    if (kLdpcCodes[i].rate == -1 && kLdpcCodes[i].q == (pre ? 36 : 25)) return i;
  return -1;
}

void build_l1pre(const FrameParams &prm, int l1_post_size, int l1_post_info_size, std::vector<cfloat> &cells)
{
  BitWriter w;
  w.put(0, 8);                                   // TYPE: TS only
  w.put(prm.carriermode, 1);                     // BWT_EXT
  w.put(prm.preamble, 3);                        // S1
  w.put(prm.fftsize & 7, 3); w.put(0, 1);        // S2 field 1 + mixed bit
  w.put(0, 1);                                   // L1_REPETITION_FLAG
  w.put(prm.guardinterval, 3);
  w.put(prm.paprmode, 4);
  w.put(prm.l1constellation, 4);                 // L1_MOD
  w.put(0, 2);                                   // L1_COD
  w.put(0, 2);                                   // L1_FEC_TYPE
  w.put(l1_post_size, 18);
  w.put(l1_post_info_size, 18);                  // L1_POST_INFO_SIZE (350 - 32 for one PLP)
  w.put(prm.pilotpattern, 4);
  w.put(0, 8);                                   // TX_ID_AVAILABILITY
  w.put(0, 16);                                  // CELL_ID
  w.put(0x3085, 16);                             // NETWORK_ID
  w.put(0x8001, 16);                             // T2_SYSTEM_ID
  w.put(prm.t2frames, 8);
  w.put(prm.numdatasyms, 12);
  w.put(0, 3);                                   // REGEN_FLAG
  w.put(0, 1);                                   // L1_POST_EXTENSION
  w.put(1, 3);                                   // NUM_RF
  w.put(0, 3);                                   // CURRENT_RF_IDX
  w.put(prm.version, 4);
  w.put(prm.version == VERSION_131 ? prm.l1scrambled : 0, 1);
  w.put(0, 1);                                   // T2_BASE_LITE
  w.put((prm.reservedbiasbits && prm.version == VERSION_131) ? 0xf : 0, 4);
  append_crc32(w.b);                             // 200 bits
  std::vector<uint8_t> k(w.b);
  k.resize(3072, 0);                             // zero padding up to K_bch (16K, rate 1/4)
  const std::vector<uint8_t> cw = l1_fec(k, 3240, l1_ldpc_code(true));
  // puncture parity groups (Table 32): first 31 groups completely, 328 bits of the 32nd
  std::vector<uint8_t> punct(16200, 0);
  for (int c = 0; c < 32; c++) {
    const int g = kL1PrePunctureOrder[c];
    const int cnt = c < 31 ? 360 : 328;
    for (int c2 = 0; c2 < cnt; c2++) punct[3240 + c2 * 36 + g] = 1;
  }
  cells.clear();
  auto bpsk = [&](int bit) { cfloat v; v.re = bit ? -1.0f : 1.0f; v.im = 0.0f; cells.push_back(v); };
  for (int i = 0; i < 200; i++) bpsk(cw[i]);
  for (int i = 0; i < 168; i++) bpsk(cw[3072 + i]);
  for (int i = 3240; i < 16200; i++) if (!punct[i]) bpsk(cw[i]);
}

// what L1-post signals of one PLP
struct PlpL1 { int blocks, cell_size, framesize, rate, constellation, rotation, type, group, start; };

int plp_cod_of(int rate)
{
  switch (rate) {
    case C1_3: return 6; case C2_5: return 7; case C1_2: return 0; case C3_5: return 1;
    case C2_3: return 2; case C3_4: return 3; case C4_5: return 4; case C5_6: return 5;
  }
  return 0;
}

void build_l1post(const FrameParams &prm, const PlpL1 *plps, int num_plp, int subslices, int subslice_interval,
                  int type2_start, int frame_idx, int n_post, int n_punc, int eta, std::vector<cfloat> &cells)
{
  const bool v131 = prm.version == VERSION_131;
  const bool bias = prm.reservedbiasbits && v131;
  BitWriter w;
  w.put(subslices, 15);                          // SUB_SLICES_PER_FRAME
  w.put(num_plp, 8);                             // NUM_PLP
  w.put(0, 4);                                   // NUM_AUX
  w.put(0, 8);                                   // AUX_CONFIG_RFU
  w.put(0, 3);                                   // RF_IDX
  w.put(729833333u, 32);                         // FREQUENCY
  for (int pl = 0; pl < num_plp; pl++) {         // configurable part, 89 bits per PLP
    w.put(pl, 8);                                // PLP_ID
    w.put(plps[pl].type, 3);                     // PLP_TYPE
    w.put(3, 5);                                 // PLP_PAYLOAD_TYPE (TS)
    w.put(0, 1);                                 // FF_FLAG
    w.put(0, 3);                                 // FIRST_RF_IDX
    w.put(0, 8);                                 // FIRST_FRAME_IDX
    w.put(plps[pl].group, 8);                    // PLP_GROUP_ID
    w.put(plp_cod_of(plps[pl].rate), 3);         // PLP_COD
    w.put(plps[pl].constellation, 3);            // PLP_MOD
    w.put(plps[pl].rotation, 1);                 // PLP_ROTATION
    w.put(plps[pl].framesize, 2);                // PLP_FEC_TYPE
    w.put(plps[pl].blocks, 10);                  // PLP_NUM_BLOCKS_MAX
    w.put(1, 8);                                 // FRAME_INTERVAL
    w.put(prm.tiblocks, 8);                      // TIME_IL_LENGTH
    w.put(0, 1);                                 // TIME_IL_TYPE
    w.put(0, 1);                                 // IN_BAND_A_FLAG
    w.put((prm.inband && v131) ? 1 : 0, 1);      // IN_BAND_B_FLAG
    w.put(bias ? 0x7ff : 0, 11);                 // RESERVED_1
    w.put(prm.version == VERSION_111 ? 0 : prm.inputmode + 1, 2);   // PLP_MODE
    w.put(0, 1);                                 // STATIC_FLAG
    w.put(0, 1);                                 // STATIC_PADDING_FLAG
  }
  w.put(0, 2);                                   // FEF_LENGTH_MSB
  w.put(bias ? 0x3fffffff : 0, 30);              // RESERVED_2
  w.put(frame_idx, 8);                           // FRAME_IDX (dynamic)
  w.put(subslice_interval, 22);                  // SUB_SLICE_INTERVAL
  w.put(type2_start, 22);                        // TYPE_2_START
  w.put(0, 8);                                   // L1_CHANGE_COUNTER
  w.put(0, 3);                                   // START_RF_IDX
  w.put(bias ? 0xff : 0, 8);                     // RESERVED_3
  for (int pl = 0; pl < num_plp; pl++) {         // dynamic part, 48 bits per PLP
    w.put(pl, 8);                                // PLP_ID (dynamic; the reference leaves its single one uninitialised = 0)
    w.put(plps[pl].start, 22);                   // PLP_START
    w.put(plps[pl].blocks, 10);                  // PLP_NUM_BLOCKS
    w.put(bias ? 0xff : 0, 8);                   // RESERVED_4
  }
  w.put(bias ? 0xff : 0, 8);                     // RESERVED_5
  append_crc32(w.b);                             // K_sig = 213 + 137 num_plp bits (350 for one PLP)
  std::vector<uint8_t> sig(w.b);
  const int ksig = (int)sig.size();
  if (v131 && prm.l1scrambled) {
    std::vector<uint8_t> pr(ksig);
    bb_prbs_bits(ksig, pr.data());
    for (int i = 0; i < ksig; i++) sig[i] ^= pr[i];
  }
  // zero-padding of BCH information bits by groups of 360 (Table 34 / reference :1698-1756)
  const uint8_t *pad_order, *punct_order;
  switch (prm.l1constellation) {
    case L1_MOD_16QAM: pad_order = kL1PostPadOrder_16qam; punct_order = kL1PostPunctureOrder_16qam; break;
    case L1_MOD_64QAM: pad_order = kL1PostPadOrder_64qam; punct_order = kL1PostPunctureOrder_64qam; break;
    default: pad_order = kL1PostPadOrder_bqpsk; punct_order = kL1PostPunctureOrder_bqpsk; break;
  }
  const int KBCH = 7032, NBCH = 7200;
  std::vector<uint8_t> padded(KBCH, 0), is_pad(KBCH, 0);
  int m, last;
  if (ksig <= 360) { m = 19; last = 360 - ksig; }
  else { m = (KBCH - ksig) / 360; last = KBCH - ksig - 360 * m; }
  for (int n = 0; n < m; n++) {
    const int g = pad_order[n], len = (g == 19) ? 192 : 360;
    for (int i = 0; i < len; i++) is_pad[g * 360 + i] = 1;
  }
  {
    const int g = pad_order[m], len = (g == 19) ? 192 : 360;
    for (int i = 0; i < last; i++) is_pad[g * 360 + len - last + i] = 1;
  }
  {
    int idx = 0;
    for (int n = 0; n < KBCH; n++) padded[n] = is_pad[n] ? 0 : sig[idx++];
  }
  const std::vector<uint8_t> cw = l1_fec(padded, NBCH, l1_ldpc_code(false));
  std::vector<uint8_t> punct(16200, 0);
  {
    const int full = n_punc / 360;
    for (int c = 0; c < full; c++)
      for (int c2 = 0; c2 < 360; c2++) punct[NBCH + c2 * 25 + punct_order[c]] = 1;
    for (int c2 = 0; c2 < n_punc - full * 360; c2++) punct[NBCH + c2 * 25 + punct_order[full]] = 1;
  }
  std::vector<uint8_t> tx;
  for (int i = 0; i < KBCH; i++) if (!is_pad[i]) tx.push_back(cw[i]);
  for (int i = KBCH; i < NBCH; i++) tx.push_back(cw[i]);
  for (int i = NBCH; i < 16200; i++) if (!punct[i]) tx.push_back(cw[i]);
  tx.resize(n_post, 0);

  cells.clear();
  if (prm.l1constellation == L1_MOD_BPSK) {
    for (int i = 0; i < n_post; i++) { cfloat v; v.re = tx[i] ? -1.0f : 1.0f; v.im = 0.0f; cells.push_back(v); }
    return;
  }
  std::vector<cfloat> lut;
  qam_lut(eta, lut);
  if (prm.l1constellation == L1_MOD_QPSK) {
    for (int d = 0; d < n_post / 2; d++) cells.push_back(lut[(tx[2 * d] << 1) | tx[2 * d + 1]]);
    return;
  }
  // 16QAM / 64QAM: column-row bit interleaver without twist, then demux with the map as SOURCE index
  const int ncol = 2 * eta, rows = n_post / ncol;
  const uint8_t *mux = (eta == 4) ? kL1Demux16 : kL1Demux64;
  std::vector<uint8_t> il(n_post);
  for (int k = 0; k < rows; k++)
    for (int c = 0; c < ncol; c++) il[k * ncol + c] = tx[rows * c + k];
  for (int d = 0; d < rows; d++) {
    unsigned pack = 0;
    for (int e = 0; e < ncol; e++) pack = (pack << 1) | il[d * ncol + mux[e]];
    cells.push_back(lut[pack >> eta]);
    cells.push_back(lut[pack & ((1u << eta) - 1)]);
  }
}

// PLP types, groups and sub-slicing (FrameParams::plp_layout): validates them and fills the plan's layout fields and each
// PLP's type, group and PLP_START.  Without plp_layout: type-1 PLPs of group 1, one sub-slice, PLP_START = first cell.
bool plp_layout(const FrameParams &prm, int P, FramePlan *p, PlpL1 *plps, std::string *err)
{
  auto refuse = [&](int pl, const char *why) {
    if (err) *err = "framemapperfint_cc: PLP " + std::to_string(pl) + ": " + why;
    return false;
  };
  const int N = prm.plp_layout ? prm.num_subslices : 1;
  if (N < 1 || N > 32767) {
    if (err) *err = "framemapperfint_cc: sub-slices per frame outside 1..32767";
    return false;
  }
  bool type2 = false;
  for (int pl = 0; pl < P; pl++) {
    const int t = prm.plp_layout ? prm.plp_type[pl] : 1, g = prm.plp_layout ? prm.plp_group[pl] : 1;
    if (t < 0 || t > 2) return refuse(pl, "PLP_TYPE outside 0..2 (common, data type 1, data type 2)");
    if (pl > 0 && t < p->plp_type[pl - 1]) return refuse(pl, "listed out of mapping order (common, then type-1, then type-2 PLPs)");
    if (g < 0 || g > 255) return refuse(pl, "PLP_GROUP_ID outside 0..255");
    const int D = plps[pl].blocks * plps[pl].cell_size;
    if (t == 2 && D % N) return refuse(pl, "type-2 cells per frame are not a multiple of the sub-slices per frame");
    p->plp_type[pl] = plps[pl].type = t;
    p->plp_group[pl] = plps[pl].group = g;
    p->plp_slice_cells[pl] = t == 2 ? D / N : D;
    type2 = type2 || t == 2;
  }
  if (N > 1 && !type2) {
    if (err) *err = "framemapperfint_cc: more than one sub-slice per frame without a type-2 PLP";
    return false;
  }
  for (int pl = 0; pl < P; pl++) {
    if (p->plp_type[pl] != 0) continue;
    int data = 0;
    for (int o = 0; o < P; o++) {
      if (o != pl && p->plp_group[o] == p->plp_group[pl] && p->plp_type[o] == 0) return refuse(pl, "common PLP of a group with another common PLP");
      if (p->plp_group[o] == p->plp_group[pl] && p->plp_type[o] != 0) data++;
    }
    if (!data) return refuse(pl, "common PLP of a group without a data PLP");
  }
  // common and type-1 PLPs one after the other from address 0, then the type-2 PLPs' sub-slices
  p->num_subslices = N;
  p->type2_start = p->subslice_interval = 0;
  int start = 0;
  for (int pl = 0; pl < P; pl++) {
    if (p->plp_type[pl] == 2 && (pl == 0 || p->plp_type[pl - 1] != 2)) p->type2_start = start;
    p->plp_start[pl] = plps[pl].start = start;
    start += p->plp_slice_cells[pl];
    if (p->plp_type[pl] == 2) p->subslice_interval += p->plp_slice_cells[pl];
  }
  return true;
}

// frequency interleaver permutation function H (EN 302 755 8.5; reference :916-977)
void freq_perm(int fft_index, int limit, bool odd, std::vector<int32_t> &H)
{
  static const int taps1k[] = { 0, 4 }, taps2k[] = { 0, 3 }, taps4k[] = { 0, 2 }, taps8k[] = { 0, 1, 4, 6 },
                   taps16k[] = { 0, 1, 4, 5, 9, 11 }, taps32k[] = { 0, 1, 2, 12 };
  static const int *taps[6] = { taps1k, taps2k, taps4k, taps8k, taps16k, taps32k };
  static const int ntaps[6] = { 2, 2, 2, 4, 6, 4 };
  static const uint8_t *pe[6] = { kFreqPermEven_1k, kFreqPermEven_2k, kFreqPermEven_4k, kFreqPermEven_8k, kFreqPermEven_16k, kFreqPerm_32k };
  static const uint8_t *po[6] = { kFreqPermOdd_1k, kFreqPermOdd_2k, kFreqPermOdd_4k, kFreqPermOdd_8k, kFreqPermOdd_16k, kFreqPerm_32k };
  const int nbits = 9 + fft_index;         // N_r - 1
  const int mmax = 1024 << fft_index;
  const uint8_t *perm = odd ? po[fft_index] : pe[fft_index];
  H.clear();
  unsigned reg = 0;
  for (int i = 0; i < mmax; i++) {
    if (i < 2) reg = 0;
    else if (i == 2) reg = 1;
    else {
      unsigned fb = 0;
      for (int k = 0; k < ntaps[fft_index]; k++) fb ^= (reg >> taps[fft_index][k]) & 1u;
      reg = ((reg & ((1u << nbits) - 1)) >> 1) | (fb << (nbits - 1));
    }
    unsigned v = 0;
    for (int n = 0; n < nbits; n++) v |= ((reg >> n) & 1u) << perm[n];
    v += (unsigned)(i & 1) * (unsigned)(mmax / 2);
    if ((int)v < limit) H.push_back((int32_t)v);
  }
}

} // namespace

// ------------------------------------------------------------------------------------------------
bool build_frame_plan(const FrameParams &prm, FramePlan *p, std::string *err)
{
  p->prm = prm;
  FecSpec fs;
  if (!fec_spec(prm.framesize, prm.rate, &fs)) { if (err) *err = "framemapperfint_cc: unsupported (framesize, rate)"; return false; }
  p->cell_size = cells_per_fecframe(prm.framesize, prm.constellation);
  if (!p->cell_size) { if (err) *err = "framemapperfint_cc: unknown constellation"; return false; }
  if (prm.fecblocks < 1 || prm.tiblocks < 0 || prm.t2frames < 1 || prm.t2frames > 255) {
    if (err) *err = "framemapperfint_cc: fecblocks/tiblocks/t2frames out of range";
    return false;
  }
  if (prm.l1constellation < L1_MOD_BPSK || prm.l1constellation > L1_MOD_64QAM) { if (err) *err = "framemapperfint_cc: unknown L1 constellation"; return false; }
  if (!ofdm_dims(prm.carriermode, prm.fftsize, prm.pilotpattern, prm.guardinterval, prm.numdatasyms,
                 prm.paprmode, prm.preamble, &p->dims, err)) return false;
  const OfdmDims &d = p->dims;
  // PLPs: the reference's single one, or several type-1 PLPs one after the other, each with the frame's parameters or
  // (plp_modcod) its own
  const int P = p->num_plp = prm.num_plp > 1 ? prm.num_plp : 1;
  if (P > MAX_PLP) { if (err) *err = "framemapperfint_cc: too many PLPs"; return false; }
  int plp_blocks[MAX_PLP];
  PlpL1 plps[MAX_PLP];
  p->plp_first_block[0] = 0;
  p->plp_first_cell[0] = 0;
  p->plp_sets = 0;
  for (int pl = 0; pl < P; pl++) {
    plp_blocks[pl] = P == 1 ? prm.fecblocks : prm.plp_fecblocks[pl];
    if (plp_blocks[pl] < 1 || plp_blocks[pl] > 1023) { if (err) *err = "framemapperfint_cc: FEC blocks of a PLP out of range"; return false; }
    p->plp_first_block[pl + 1] = p->plp_first_block[pl] + plp_blocks[pl];
    PlpL1 &q = plps[pl];
    q.blocks = plp_blocks[pl];
    q.framesize = prm.plp_modcod ? prm.plp_framesize[pl] : prm.framesize;
    q.rate = prm.plp_modcod ? prm.plp_rate[pl] : prm.rate;
    q.constellation = prm.plp_modcod ? prm.plp_constellation[pl] : prm.constellation;
    q.rotation = prm.plp_modcod ? prm.plp_rotation[pl] : prm.rotation;
    FecSpec qs;
    if (!fec_spec(q.framesize, q.rate, &qs)) { if (err) *err = "framemapperfint_cc: unsupported (framesize, rate) of a PLP"; return false; }
    q.cell_size = p->plp_cell_size[pl] = cells_per_fecframe(q.framesize, q.constellation);
    if (!q.cell_size) { if (err) *err = "framemapperfint_cc: unknown constellation of a PLP"; return false; }
    p->plp_first_cell[pl + 1] = p->plp_first_cell[pl] + q.blocks * q.cell_size;
    int s = 0;
    while (s < pl && !(plps[s].framesize == q.framesize && plps[s].rate == q.rate && plps[s].constellation == q.constellation &&
                       plps[s].rotation == q.rotation)) s++;
    p->plp_set[pl] = s < pl ? p->plp_set[s] : p->plp_sets++;
  }
  if (p->plp_first_block[P] != prm.fecblocks) { if (err) *err = "framemapperfint_cc: fecblocks is not the sum over the PLPs"; return false; }
  if (!plp_layout(prm, P, p, plps, err)) return false;
  p->plp_chain_off[0] = 0;
  for (int pl = 0; pl < P; pl++) {
    const int end = p->plp_chain_off[pl] + plp_blocks[pl] * plps[pl].cell_size;
    p->plp_chain_off[pl + 1] = p->plp_sets > 1 ? (end + 7) & ~7 : end;
  }
  const int F = prm.fecblocks;
  static const int etas[4] = { 1, 2, 4, 6 };
  const int eta = p->eta_mod = etas[prm.l1constellation];

  // N_post / N_punc (EN 302 755 7.3.1.2; reference :978-987 incl. its float ceil) from K_sig = 213 + 137 NUM_PLP bits
  // (configurable 35 + 35 + 89 P + 32, dynamic 71 + 48 P + 8, CRC-32; 350 for the reference's single PLP)
  const int ksig = p->l1post_sig_bits = 213 + 137 * P;
  const int n_punc_temp = (6 * (7032 - ksig)) / 5;
  const int n_post_temp = ksig + 168 + 9000 - n_punc_temp;
  if (d.n_p2 == 1) p->n_post = (int)std::ceil((float)n_post_temp / (2 * (float)eta)) * 2 * eta;
  else p->n_post = (int)std::ceil((float)n_post_temp / ((float)eta * (float)d.n_p2)) * eta * d.n_p2;
  p->n_punc = n_punc_temp - (p->n_post - n_post_temp);
  const int l1post_cells = p->n_post / eta;

  p->stream_items = p->plp_first_cell[P];
  p->mapped_items = d.active_items;
  const int fixed = 1840 + l1post_cells + (d.n_fc - d.c_fc);
  p->overfull = p->mapped_items < p->stream_items + fixed;
  // Length of the linear frame before truncation.  Reference :1138-1141: an over-full frame only logs a warning,
  // grows its private frame buffers to stream_items + fixed "to avoid segfault" and carries on; the frequency
  // interleaver then reads the physical frame only, so the cells that do not fit are dropped.  By default creation
  // fails with the reference's message; with the opt-in policy the same truncated frame is produced.  PLPs with their
  // own parameters have no reference behaviour to reproduce: such a frame is always refused.
  int linear_items = p->mapped_items;
  if (p->overfull) {
    if (!overfull_warn_policy() || prm.plp_modcod || prm.plp_layout) {
      if (err) *err = "Frame Mapper, too many FEC blocks in T2 frame.";
      return false;
    }
    linear_items = p->stream_items + fixed;
  }
  p->dummy_cells = linear_items - p->stream_items - fixed;

  // ---- cell interleaver permutation (EN 302 755 6.4; reference :999-1107), one per PLP
  {
    std::vector<std::vector<int32_t> > perm(P);
    int deg[MAX_PLP];
    p->plp_cell_perm_inv.assign(P, std::vector<uint16_t>());
    for (int pl = 0; pl < P; pl++) {
      const int Nc = plps[pl].cell_size;
      static const int degs_n[4] = { 15, 14, 14, 13 }, degs_s[4] = { 13, 12, 12, 11 };
      deg[pl] = (plps[pl].framesize == FECFRAME_NORMAL ? degs_n : degs_s)[plps[pl].constellation];
      static const int t11[] = { 0, 3 }, t12[] = { 0, 2 }, t13[] = { 0, 1, 4, 6 }, t14[] = { 0, 1, 4, 5, 9, 11 }, t15[] = { 0, 1, 2, 12 };
      const int *taps; int nt;
      switch (deg[pl]) {
        case 11: taps = t11; nt = 2; break; case 12: taps = t12; nt = 2; break; case 13: taps = t13; nt = 4; break;
        case 14: taps = t14; nt = 6; break; default: taps = t15; nt = 4; break;
      }
      unsigned reg = 0;
      const unsigned mask = (1u << (deg[pl] - 1)) - 1;
      for (int i = 0; i < (1 << deg[pl]); i++) {
        if (i < 2) reg = 0;
        else if (i == 2) reg = 1;
        else {
          unsigned fb = 0;
          for (int k = 0; k < nt; k++) fb ^= (reg >> taps[k]) & 1u;
          reg = ((reg & mask) >> 1) | (fb << (deg[pl] - 2));
        }
        reg |= (unsigned)(i & 1) << (deg[pl] - 1);
        if ((int)reg < Nc) perm[pl].push_back((int32_t)reg);
      }
      if ((int)perm[pl].size() != Nc) { if (err) *err = "internal: cell permutation size"; return false; }
      p->plp_cell_perm_inv[pl].assign(Nc, 0);
      for (int w = 0; w < Nc; w++) p->plp_cell_perm_inv[pl][perm[pl][w]] = (uint16_t)w;
    }
    p->cell_perm = perm[0];
    p->cell_perm_inv = p->plp_cell_perm_inv[0];

    // TI block split (reference :1108-1119) and per-FEC-block shifts (restart per TI block, :1974-1992), PLP by PLP
    p->fec_shift.clear();
    std::vector<int> ti_block_sizes, ti_block_rows;
    for (int pl = 0; pl < P; pl++) {
      const int Fp = plp_blocks[pl], Nc = plps[pl].cell_size;
      int small, big, nbig, nsmall;
      if (prm.tiblocks == 0) { small = big = 1; nbig = 0; nsmall = Fp; }
      else {
        small = (int)std::floor((float)Fp / (float)prm.tiblocks);
        big = (int)std::ceil((float)Fp / (float)prm.tiblocks);
        nbig = Fp % prm.tiblocks;
        nsmall = prm.tiblocks - nbig;
      }
      for (int s = 0; s < nsmall + nbig; s++) {
        const int k = s < nsmall ? small : big;
        ti_block_sizes.push_back(k);
        ti_block_rows.push_back(Nc / 5);
        unsigned n = 0;
        for (int r = 0; r < k; r++) {
          int shift = Nc;
          while (shift >= Nc) {
            unsigned t = n, sh = 0;
            for (int b = 0; b < deg[pl]; b++) { sh |= t & 1u; sh <<= 1; t >>= 1; }
            shift = (int)sh;
            n++;
          }
          p->fec_shift.push_back(shift);
        }
      }
    }
    if ((int)p->fec_shift.size() != F) { if (err) *err = "framemapperfint_cc: fecblocks/tiblocks combination leaves FEC blocks unassigned"; return false; }

    // cell-interleaved memory index <-> input index
    std::vector<int32_t> ci_src((size_t)p->stream_items);
    p->ci_dst.assign((size_t)p->stream_items, 0);
    for (int pl = 0; pl < P; pl++) {
      const int Nc = plps[pl].cell_size;
      for (int r = p->plp_first_block[pl]; r < p->plp_first_block[pl + 1]; r++) {
        const int base = p->plp_first_cell[pl] + (r - p->plp_first_block[pl]) * Nc;
        for (int w = 0; w < Nc; w++) {
          const int x = base + (perm[pl][w] + p->fec_shift[r]) % Nc;
          ci_src[x] = base + w;
          p->ci_dst[(size_t)base + w] = x;
        }
      }
    }

    // time interleaver read-out (EN 302 755 6.5; reference :1999-2028)
    p->ti_src.assign((size_t)p->stream_items, 0);
    if (prm.tiblocks == 0) p->ti_src = ci_src;
    else {
      size_t o = 0;
      for (size_t s = 0; s < ti_block_sizes.size(); s++) {
        const int cols = 5 * ti_block_sizes[s], rows = ti_block_rows[s];
        for (int j = 0; j < rows; j++)
          for (int c = 0; c < cols; c++) p->ti_src[o + (size_t)cols * j + c] = ci_src[o + (size_t)rows * c + j];
        o += (size_t)rows * cols;
      }
    }
  }

  // ---- pool: [L1-pre 1840][L1-post x t2frames][dummy][zero]
  CellPool &pool = p->pool;
  pool.cells.clear();
  p->pool_l1pre = 0;
  {
    std::vector<cfloat> c;
    build_l1pre(prm, l1post_cells, ksig - 32, c);
    if ((int)c.size() != 1840) { if (err) *err = "internal: L1-pre size"; return false; }
    pool.cells.insert(pool.cells.end(), c.begin(), c.end());
  }
  pool.l1post_base = (int)pool.cells.size();
  pool.l1post_cells = l1post_cells;
  pool.l1post_variants = prm.t2frames;
  for (int v = 0; v < prm.t2frames; v++) {
    std::vector<cfloat> c;
    build_l1post(prm, plps, P, p->num_subslices, p->subslice_interval, p->type2_start, v, p->n_post, p->n_punc, eta, c);
    if ((int)c.size() != l1post_cells) { if (err) *err = "internal: L1-post size"; return false; }
    pool.cells.insert(pool.cells.end(), c.begin(), c.end());
  }
  p->pool_dummy = (int)pool.cells.size();
  {
    std::vector<uint8_t> pr(p->dummy_cells > 0 ? p->dummy_cells : 1);
    bb_prbs_bits(p->dummy_cells, pr.data());
    for (int i = 0; i < p->dummy_cells; i++) { cfloat v; v.re = pr[i] ? -1.0f : 1.0f; v.im = 0.0f; pool.cells.push_back(v); }
  }
  p->pool_zero = (int)pool.cells.size();
  { cfloat z; z.re = 0.0f; z.im = 0.0f; pool.cells.push_back(z); }

  // ---- linear frame (before zig-zag): [L1-pre][L1-post][data][dummy][unmodulated]
  std::vector<int32_t> linear((size_t)linear_items);
  {
    size_t k = 0;
    for (int i = 0; i < 1840; i++) linear[k++] = -(1 + p->pool_l1pre + i);
    for (int i = 0; i < l1post_cells; i++) linear[k++] = -(1 + pool.l1post_base + i);
    // data cells in mapping order: each PLP's time-interleaver output at its data-cell addresses (FrameParams::plp_layout)
    for (int pl = 0; pl < P; pl++) {
      const int L = p->plp_slice_cells[pl], step = p->plp_type[pl] == 2 ? p->subslice_interval : L;
      for (int i = 0; i < p->plp_first_cell[pl + 1] - p->plp_first_cell[pl]; i++)
        linear[k + p->plp_start[pl] + (size_t)(i / L) * step + i % L] = p->ti_src[(size_t)p->plp_first_cell[pl] + i];
    }
    k += (size_t)p->stream_items;
    for (int i = 0; i < p->dummy_cells; i++) linear[k++] = -(1 + p->pool_dummy + i);
    for (int i = 0; i < d.n_fc - d.c_fc; i++) linear[k++] = -(1 + p->pool_zero);
  }
  // ---- P2 zig-zag when N_P2 > 1 (reference :2047-2103)
  std::vector<int32_t> framed((size_t)linear_items);
  if (d.n_p2 == 1) framed = linear;
  else {
    const int NP = d.n_p2, CP = d.c_p2;
    const int pre_per = 1840 / NP, post_per = l1post_cells / NP;
    for (int n = 0; n < NP; n++)
      for (int j = 0; j < pre_per; j++) framed[(size_t)n * CP + j] = linear[n + (size_t)j * NP];
    for (int n = 0; n < NP; n++)
      for (int j = 0; j < post_per; j++) framed[(size_t)n * CP + pre_per + j] = linear[1840 + n + (size_t)j * NP];
    size_t read = 1840 + (size_t)l1post_cells;
    const int rest = CP - pre_per - post_per;
    for (int n = 0; n < NP; n++)
      for (int j = 0; j < rest; j++) framed[(size_t)n * CP + pre_per + post_per + j] = linear[read++];
    for (size_t i = (size_t)NP * CP; i < (size_t)linear_items; i++) framed[i] = linear[read++];
  }
  // ---- frequency interleaver, symbol parity counted from 0 in every T2 frame (reference :2104-2142)
  std::vector<int32_t> He, Ho, HeP2, HoP2, HeFC, HoFC;
  const int fi = d.fft_index;
  freq_perm(fi, d.c_data, false, He);  freq_perm(fi, d.c_data, true, Ho);
  freq_perm(fi, d.c_p2, false, HeP2);  freq_perm(fi, d.c_p2, true, HoP2);
  freq_perm(fi, d.n_fc, false, HeFC);  freq_perm(fi, d.n_fc, true, HoFC);
  if (fi == 5) {
    // 32K: even symbols use the inverse of the odd permutation (EN 302 755 8.5 / reference :961-977)
    auto invert = [](const std::vector<int32_t> &odd, std::vector<int32_t> &even) {
      even.assign(odd.size(), 0);
      for (size_t j = 0; j < odd.size(); j++) even[odd[j]] = (int32_t)j;
    };
    invert(Ho, He); invert(HoP2, HeP2); invert(HoFC, HeFC);
  }
  p->code.assign((size_t)p->mapped_items, 0);
  p->fi_src.assign((size_t)p->mapped_items, 0);
  {
    size_t off = 0;
    int sym = 0;
    auto emit = [&](const std::vector<int32_t> &H, int n) {
      for (int j = 0; j < n; j++) {
        p->fi_src[off + j] = (int32_t)(off + H[j]);
        p->code[off + j] = framed[off + H[j]];
      }
      off += n; sym++;
    };
    for (int j = 0; j < d.n_p2; j++) emit((sym & 1) ? HoP2 : HeP2, d.c_p2);
    for (int j = 0; j < d.num_data_symbols_no_fc; j++) emit((sym & 1) ? Ho : He, d.c_data);
    if (d.n_fc) emit((sym & 1) ? HoFC : HeFC, d.n_fc);
    if (off != (size_t)p->mapped_items) { if (err) *err = "internal: frame size"; return false; }
  }
  framed.resize((size_t)p->mapped_items);      // over-full: what lies beyond the physical frame is never transmitted
  p->framed.swap(framed);
  return true;
}

} // namespace t2
