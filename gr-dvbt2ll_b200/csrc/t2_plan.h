// Host-side "plan" of the DVB-T2 modulator hot path.
//
// Design: everything irregular in EN 302 755 (rate tables, BCH generator, LDPC address tables,
// column twist / demux, constellation LUTs, PRBS permutations, L1 signalling, pilot patterns, P1)
// is turned into DATA once per make(); the CUDA kernels in t2_kernels.cu are few, table-driven and
// batch many FECFRAMEs / OFDM symbols / T2 frames per launch.  The reference interleaves table
// generation and DSP in the block classes (lib/*_impl.cc); citations below name the code whose
// observable behaviour each plan reproduces.
//
// Bit order convention everywhere on the device: "stream order" = bit i of a stream lives in
// byte i/8 at bit position 7-(i%8) (MSB first), and 32-bit words are big-endian views of those
// bytes, so word bit 31 is the earliest bit.
#ifndef T2_PLAN_H
#define T2_PLAN_H

#include <cstdint>
#include <string>
#include <vector>

namespace t2 {

// ---- enum values: ABI of reference include/dvbt2ll/dvbt2ll_config.h:60-202 -------------------
enum { C1_2 = 0, C3_5, C2_3, C3_4, C4_5, C5_6, C1_3, C2_5 };
enum { MOD_QPSK = 0, MOD_16QAM, MOD_64QAM, MOD_256QAM };
enum { FECFRAME_SHORT = 0, FECFRAME_NORMAL = 1 };
enum { INPUTMODE_NORMAL = 0, INPUTMODE_HIEFF = 1 };
enum { CARRIERS_NORMAL = 0, CARRIERS_EXTENDED = 1 };
enum { PREAMBLE_T2_SISO = 0, PREAMBLE_T2_MISO, PREAMBLE_NON_T2, PREAMBLE_T2_LITE_SISO, PREAMBLE_T2_LITE_MISO };
enum { FFTSIZE_2K = 0, FFTSIZE_8K, FFTSIZE_4K, FFTSIZE_1K, FFTSIZE_16K, FFTSIZE_32K,
       FFTSIZE_8K_T2GI, FFTSIZE_32K_T2GI, FFTSIZE_16K_T2GI = 11 };
enum { GI_1_32 = 0, GI_1_16, GI_1_8, GI_1_4, GI_1_128, GI_19_128, GI_19_256 };
enum { PAPR_OFF = 0, PAPR_ACE, PAPR_TR, PAPR_BOTH };
enum { L1_MOD_BPSK = 0, L1_MOD_QPSK, L1_MOD_16QAM, L1_MOD_64QAM };
enum { VERSION_111 = 0, VERSION_121, VERSION_131 };
enum { MISO_TX1 = 0, MISO_TX2 };
enum { BANDWIDTH_1_7_MHZ = 0, BANDWIDTH_5_0_MHZ, BANDWIDTH_6_0_MHZ, BANDWIDTH_7_0_MHZ,
       BANDWIDTH_8_0_MHZ, BANDWIDTH_10_0_MHZ };

struct cfloat { float re, im; };

// ---- FEC dimensions (reference lib/bbheaderbch_bb_impl.cc:51-165) -----------------------------
struct FecSpec {
  int normal;      // 1 = 64800, 0 = 16200
  int rate;        // dvbt2_code_rate_t
  int nldpc;       // 64800 | 16200
  int kbch, nbch;  // BCH message / codeword bits
  int q;           // LDPC q = (nldpc - nbch) / 360
  int bch_r;       // BCH parity bits: 192 (N12), 160 (N10), 168 (S12)
};
bool fec_spec(int framesize, int rate, FecSpec *out);
int cells_per_fecframe(int framesize, int constellation);   // 0 if invalid

// ---- GF(2) polynomial helpers (host) ----------------------------------------------------------
// Polynomials are vectors of coefficients indexed by power (p[i] = coeff of x^i).
std::vector<uint8_t> bch_generator(int r);   // r = 128/160/192 normal, 168 short
// Remainder of m(x) * x^r mod g(x); message bit 0 = highest-order coefficient; result in
// transmission order (highest-order first), one bit per byte.
std::vector<uint8_t> bch_parity_bits(const uint8_t *msg_bits, int k, const std::vector<uint8_t> &g);

// ---- block 1: BB header + scrambler + BCH (reference lib/bbheaderbch_bb_impl.cc) --------------
struct BbPlan {
  FecSpec fec;
  int mode, inband, fecblocks, tsrate;
  int payload_bytes;                  // (kbch - 80) / 8 when no in-band padding
  std::vector<uint8_t> scramble;      // kbch/8 bytes of the BB PRBS (x^14 + x^15, init 0x4A80 form)
  uint8_t crc8_tab[256];              // CRC-8 poly 0xD5, MSB first (reference :222-240)
  // 192-bit left-aligned remainder registers as 6 big-endian words.
  std::vector<uint32_t> bch_byte_tab; // [2][256][6]: (b(x) x^r) mod g, then (b(x) x^(r+8)) mod g
  int chunk_bytes;                    // message bytes per lane (32 lanes per FECFRAME)
  int lead_zero_bytes;                // zero bytes virtually prepended so 32 * chunk_bytes covers kbch/8
  std::vector<uint32_t> bch_shift_cols; // [6][32][6] column form of "multiply by x^(8*chunk_bytes) mod g"
  std::vector<uint8_t> inband_bytes;  // 13 bytes of in-band type B signalling (reference :327-355)
};
bool build_bb_plan(int framesize, int rate, int mode, int inband, int fecblocks, int tsrate, BbPlan *p,
                   std::string *err);

// ---- LDPC (reference restatement lib/bbheaderbch_bb_impl.cc:533-646; live path = gr-dtv) -------
// Rotation form (SURVEY section 7 fact 3): with parity rows R_t (t = 0..q-1, 360 bits each, bit s of
// row t <-> natural parity index q*s + t), table entry a of info group g contributes
// R_{a mod q} ^= rotate(info_group_g, a div q).  After the accumulator, parity row t equals
// prefix_t(R) ^ E, E = exclusive prefix-XOR over the 360 bit positions of XOR_t R_t.
struct LdpcPlan {
  FecSpec fec;
  int groups;                          // nbch / 360
  std::vector<uint16_t> row_ptr;       // [q + 1]
  std::vector<uint32_t> entries;       // per row: (shift << 16) | group
  int max_row_deg;
};
bool build_ldpc_plan(int framesize, int rate, LdpcPlan *p, std::string *err);
// Generic scatter-form host encoder (used for L1 signalling and by CPU-side self checks):
// info bits (1/byte) of length nbch -> nldpc bits natural order.  code index into kLdpcCodes.
void ldpc_encode_host(int code_index, const uint8_t *info, int nbch, int nldpc, uint8_t *out);
int ldpc_code_index(int normal, int rate);   // -1 if none

// ---- block 3: bit interleaver + demux + constellation mapper (lib/interleavermod_bc_impl.cc) ----
struct MapPlan {
  FecSpec fec;
  int constellation, rotation;
  int mod;                 // bits per cell
  int cell_size;           // cells per FECFRAME
  // For output cell-bit position i (cell = i / mod, MSB first inside the cell) the source bit index
  // inside the parity-interleaved codeword "u" (info bits, then q rows of 360 parity bits).
  std::vector<uint16_t> bit_src;      // [nldpc]
  std::vector<cfloat> lut;            // [1 << mod], rotated if rotation on (reference :169-253)
  int cyclic_delay;                   // 1: out[j] = (Re lut[c_j], Im lut[c_{j-1 mod cell_size}])
  // column-twist geometry for the kernel's word-parallel path (0 columns for QPSK)
  int ncol;
  uint8_t col_of_bit[16];             // twist-matrix column feeding output bit p of the demux word (p = 0 MSB)
  uint8_t twist_of_col[16];
  // single-table form of the constellation: Im lut[w] == Re lut[w~], w~ = (((w << 1) & im_mask_i) | ((w >> 1) & im_mask_q)) ^ im_flip
  int im_from_re;                     // 1 when that identity holds bit for bit for every word (checked at plan time)
  uint32_t im_mask_i, im_mask_q, im_flip;
  // QPSK: cells [0, qpsk_lin_cells) take bits 2c, 2c+1 of the codeword as it arrives (a multiple of 16 cells: the info
  // part, or everything for the parity-interleaved short codes); qpsk_lut[b] = the four cell codes of message byte b
  int qpsk_lin_cells;
  // QPSK without parity interleaving: the parity cells read the natural-order parity bits q s + t <- codeword bit
  // nbch + 360 t + s; when qpsk_par_q > 0 the kernel rebuilds that natural order with 32 x 32 bit transposes (in the
  // shared-memory words of the info part, which is spent by then) and maps it through the same table
  int qpsk_par_q, qpsk_nbch;
  std::vector<uint32_t> qpsk_lut;     // [256][2]: codes of cells 0,1 | 2,3 of the byte (own word | w~ << 8)
};
bool build_map_plan(int framesize, int rate, int constellation, int rotation, MapPlan *p, std::string *err);

// ---- OFDM dimensions shared by blocks 4 and 5 --------------------------------------------------
struct OfdmDims {
  int fft_n;        // 1024..32768
  int fft_index;    // 0..5 for 1K,2K,4K,8K,16K,32K
  int miso;
  int n_p2, c_p2, c_data, n_fc, c_fc, c_ps, k_ext, k_offset;
  int dx, dy;
  int gi;           // guard interval samples
  int num_symbols;  // numdatasyms + n_p2
  int num_data_symbols_no_fc;  // data symbols excluding the frame closing symbol
  int active_items; // cells per T2 frame in carrier order (without pilots)
};
bool ofdm_dims(int carriermode, int fftsize, int pilotpattern, int guardinterval, int numdatasyms,
               int paprmode, int preamble, OfdmDims *d, std::string *err);

// Special-cell pool shared by the frame mapper and the OFDM kernels: negative codes -(1+idx) index it.
struct CellPool {
  std::vector<cfloat> cells;
  int l1post_base;      // first L1-post cell of variant 0
  int l1post_cells;     // cells per variant (N_post / eta_mod)
  int l1post_variants;  // t2_frames
};

// ---- block 4: cell/time interleaver + L1 + frame builder + frequency interleaver ---------------
// (reference lib/framemapperfint_cc_impl.cc).  The whole block is ONE static gather: code[j] >= 0 is
// an input cell index inside the T2 frame's fecblocks*cell_size cells, code[j] < 0 is pool cell
// -(1+code[j]) (L1-post cells additionally offset by (frame_idx % t2_frames) * l1post_cells).
enum { MAX_PLP = 16 };
struct FrameParams {
  int framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize,
      guardinterval, l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version,
      preamble, inputmode, reservedbiasbits, l1scrambled, inband;
  // Beyond the reference (single PLP, lib/framemapperfint_cc_impl.cc:152 num_plp = 1): num_plp > 1 type-1 data PLPs of
  // the same modulation / code / time-interleaving parameters, PLP p carrying plp_fecblocks[p] FEC blocks per T2 frame
  // (fecblocks = their sum), laid one after the other in the frame.  num_plp = 0 or 1 is the reference's case.
  int num_plp;
  int plp_fecblocks[MAX_PLP];
  // plp_modcod = 1: PLP p has its own FEC type, code rate, constellation and rotation (L1-post PLP_FEC_TYPE, PLP_COD,
  // PLP_MOD, PLP_ROTATION); otherwise every PLP takes framesize / rate / constellation / rotation above.  A frame whose
  // PLPs do not fit is then always refused (there is no reference behaviour to reproduce).
  int plp_modcod;
  int plp_framesize[MAX_PLP], plp_rate[MAX_PLP], plp_constellation[MAX_PLP], plp_rotation[MAX_PLP];
};
struct FramePlan {
  FrameParams prm;
  OfdmDims dims;
  int cell_size, stream_items, mapped_items;   // cell_size: PLP 0's cells per FECFRAME
  int eta_mod, n_post, n_punc, dummy_cells;
  bool overfull;                       // reference warns "too many FEC blocks in T2 frame"
  int num_plp;                         // >= 1
  int plp_first_block[MAX_PLP + 1];    // first FEC block of each PLP inside the T2 frame's block list
  int plp_cell_size[MAX_PLP];          // cells per FECFRAME of each PLP
  int plp_first_cell[MAX_PLP + 1];     // first cell of each PLP in the frame's data cells (L1-post PLP_START)
  // Chain mode: PLP p's 16-bit cells start at plp_chain_off[p] of the frame's cell memory.  PLPs of one parameter set
  // follow each other (plp_chain_off = plp_first_cell); with more than one set (plp_sets > 1, one mapper launch per
  // PLP) every PLP starts on an 8-cell (16-byte) boundary.  plp_chain_off[num_plp] = cells of a frame in that memory.
  int plp_chain_off[MAX_PLP + 1];
  int plp_sets;                        // distinct (framesize, rate, constellation, rotation) among the PLPs
  int plp_set[MAX_PLP];                // the set of each PLP (0 = PLP 0's)
  std::vector<std::vector<uint16_t> > plp_cell_perm_inv;   // [num_plp] inverse cell permutation of each PLP
  int l1post_sig_bits;                 // K_sig of L1-post (350 for one PLP)
  std::vector<int32_t> cell_perm;      // cell interleaver permutation (reference :1087-1107)
  std::vector<int32_t> fec_shift;      // per FEC block cyclic shift (reference :1981-1992), with its PLP's cell count
  std::vector<int32_t> ti_src;         // time-interleaver read-out position -> input cell index (cell int. composed)
  std::vector<int32_t> ci_dst;         // input cell index -> index in cell-interleaved memory
  std::vector<uint16_t> cell_perm_inv; // inverse of cell_perm
  std::vector<int32_t> code;           // [mapped_items]  == framed[fi_src[j]]
  std::vector<int32_t> framed;         // [mapped_items] codes in frame order, BEFORE the frequency interleaver
  std::vector<int32_t> fi_src;         // [mapped_items] frequency interleaver: out[j] = framed[fi_src[j]]
  CellPool pool;                       // [L1-pre 1840][L1-post x t2frames][dummy][zero]
  int pool_l1pre, pool_dummy, pool_zero;
};
bool build_frame_plan(const FrameParams &prm, FramePlan *p, std::string *err);
// over-full T2 frames: 0 = refuse at plan time (default), 1 = warn and truncate like the reference (:1138-1141)
void set_overfull_policy(int policy);
bool overfull_warn_policy();

// ---- block 5: pilots + IFFT + guard interval + P1 (reference lib/pilotgenp1insert_cc_impl.cc) ---
struct OfdmParams {
  int carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble,
      misogroup, equalization, bandwidth, vlength;
};
struct OfdmPlan {
  OfdmParams prm;
  OfdmDims dims;
  int left_nulls;
  float normalization;                 // float(5 / sqrt(27 * C_PS))  (reference :1095)
  int samples_per_frame;               // num_symbols * (N + GI) + 2048
  // carrier code per (symbol, carrier k in [0, C_PS)): >= 0 running data-cell index inside the T2
  // frame's active_items input; < 0 pool cell (pilot amplitudes with sign, zero).
  std::vector<int32_t> code;           // [num_symbols * c_ps]
  std::vector<int32_t> sym_data_start; // [num_symbols + 1] running data index at symbol start
  CellPool pool;                       // [zero][+p2,-p2,+sp,-sp,+cp,-cp]
  std::vector<cfloat> p1;              // 2048 samples (reference :1119-1178, :2802-2810)
  std::vector<float> inv_sinc;         // [fft_n] (real) or empty when equalization off
  // carrier class per (symbol, k): the reference's dvbt2_carrier_type_t values, kept for tests
  std::vector<uint8_t> carrier_type;   // [num_symbols * c_ps]
};
bool build_ofdm_plan(const OfdmParams &prm, OfdmPlan *p, std::string *err);

// Tone-reservation PAPR reduction (beyond the reference, which leaves the reserved carriers at zero): the reserved
// carriers of each symbol (P2PAPR_CARRIER / TRPAPR_CARRIER of carrier_type) as FFT bins, one entry per distinct set
// (P2 and frame-closing symbols share one, the data symbols' are one base set shifted by dx * s: at most dy + 1).
struct PaprTrPlan {
  int sets, tones;                     // distinct sets, reserved carriers per set
  std::vector<int32_t> sym_set;        // [num_symbols] set of each symbol
  std::vector<int32_t> bins;           // [sets][tones] FFT bins (k + left_nulls + N/2) mod N, carrier order
  std::vector<cfloat> kernel;          // [sets][N] p_n = (1/tones) sum_b exp(+j 2 pi b n / N), p_0 = 1
  std::vector<cfloat> tone_tw;         // [N] exp(-j 2 pi i / N)
};
bool build_papr_tr_plan(const OfdmPlan &op, PaprTrPlan *p, std::string *err);

// Chain mode: compose frame plan and OFDM plan into one per-carrier code table whose non-negative
// entries index the natural-order cells produced by the mapper kernel, and merge the pools.
struct ChainTables {
  std::vector<int32_t> code;   // [num_symbols * c_ps]
  CellPool pool;
};
// cells_cell_interleaved: the mapper kernel already stored the cells in cell-interleaved order (fused), so
// data codes index that memory instead of the natural-order cells.
bool compose_chain(const FramePlan &fp, const OfdmPlan &op, bool cells_cell_interleaved, ChainTables *out,
                   std::string *err);

// Chain mode with 16-bit cells: the mapper kernel stores every data cell as (own cell word | previous cell
// word << 8) in cell-interleaved order; the OFDM kernel first copies the cells of one symbol into a shared-
// memory staging area with bulk asynchronous copies (TMA, cp.async.bulk): the symbol's source cells are sorted by
// address and grouped into runs of consecutive cells (for a time-interleaved PLP: one run per TI column); each run
// is copied as its enclosing 16-byte aligned span (up to 7 unused cells at either end).  The carriers are then
// filled from the staging area.
struct Chain16Tables {
  std::vector<int32_t> code;        // [num_symbols * c_ps]: >= 0 staging slot of the symbol, < 0 pool cell
  // bulk copies that stage a symbol's cells: 2 words per run = { source 16-byte unit (from the frame's first cell),
  // (staging 16-byte unit << 16) | length in 16-byte units }, symbols back to back
  std::vector<int32_t> run_desc;
  std::vector<int32_t> run_ptr;     // [num_symbols + 1] first run of each symbol (even: lists are 16-byte aligned, padded with a zero entry)
  std::vector<int32_t> run_cnt;     // [num_symbols] runs of each symbol
  int max_runs;                     // longest list
  std::vector<int32_t> stage_bytes; // [num_symbols] bytes the symbol's copies deliver (mbarrier transaction count)
  int max_slots;                    // largest number of staging slots (cells) of any symbol
  std::vector<uint8_t> plp;         // [num_symbols * c_ps]: the PLP whose cell a data carrier takes (0 for the others)
  CellPool pool;
};
bool compose_chain16(const FramePlan &fp, const OfdmPlan &op, Chain16Tables *out, std::string *err);

// MISO processing (EN 302 755 9.1, modified Alamouti; beyond the reference, which sends group 1's cells from both
// transmitter groups).  With g_{l,i} the cells of OFDM symbol l in the order the frequency interleaver emits them
// (i < C_l, L1 / dummy / unmodulated cells included): group 1 sends e = g, group 2 sends e_{l,2i} = -conj(g_{l,2i+1}),
// e_{l,2i+1} = conj(g_{l,2i}) in every P2, data and frame-closing symbol; pilots, nulls and reserved carriers are the
// group's own.  The carrier tables of one group's output over the staging of `t` (whose runs, staging slots and copy
// sizes every group shares): non-data carriers from `og` (the group's pilot plan), data carriers from t.code at the
// carrier of cell i (group 1) or i ^ 1 (group 2, refused if a symbol has an odd cell count).  Group 2's kernel negates
// Re (i even) or Im (i odd) of a data cell; a pool cell (L1, dummy) lands at one position per frame, so the group-2 pool
// holds its transformed value instead (the shared zero cell stays as it is).
struct MisoTables {
  std::vector<int32_t> code;   // [num_symbols * c_ps], Chain16Tables::code's convention
  std::vector<uint8_t> plp;    // [num_symbols * c_ps]
  CellPool pool;
};
// op: the pilot plan `t` was composed with
bool compose_miso(const OfdmPlan &op, const Chain16Tables &t, const OfdmPlan &og, bool group2, MisoTables *out,
                  std::string *err);

// small utilities
void bb_prbs_bits(int n, uint8_t *out);          // 1 bit per byte; reference :357-369
uint32_t crc32_bits(const uint8_t *bits, int n); // CRC-32 MSB first, init all ones (reference framemapper :1205-1224)

} // namespace t2
#endif
