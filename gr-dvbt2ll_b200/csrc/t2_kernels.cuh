// Device-side argument blocks and launch wrappers of the sm_100a kernels (t2_kernels.cu).
#ifndef T2_KERNELS_CUH
#define T2_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace t2k {

// ---- K1: BB header + payload + CRC-8 sync substitution + scrambler + BCH -----------------------
struct BbArgs {
  const uint8_t *ts;          // channel-major TS bytes; ts + c * ts_pitch = first byte of this call
  long long ts_pitch;
  int hist_valid;             // 1: the 187 bytes before ts are valid stream history
  int n_channels, frames;     // FECFRAMEs per channel in this call
  int count0;                 // packet phase (0..187) of ts[0]
  int fec_block0;             // in-band type B phase of the first FECFRAME
  int kbch, nbch, bch_r, payload_bytes, mode, inband, fecblocks;
  int chunk_bytes, lead_zero_bytes;
  const uint8_t *scramble;    // kbch / 8
  const uint8_t *crc8_tab;    // 256: the CRC-8 byte table (BB header)
  // The CRC-8 of a 187-byte packet read as 47 little-endian words (one leading byte, zeroed by the masks) is linear in
  // the data: bit k = parity(XOR_j word_j & crc8_pos_mask[j][k]).  Kernel parameters live in the constant bank, so
  // with the loop unrolled every mask is an instruction operand: one AND-XOR per word and CRC bit, no look-ups.
  uint32_t crc8_pos_mask[47][8];
  const uint32_t *bch_tab;    // 2 * 256 * 6: T0 then T1
  const uint32_t *bch_cols;   // 6 * 32 * 6
  const uint8_t *inband_bytes;// 13
  uint8_t *out;               // packed codewords, pitch out_pitch bytes per FECFRAME
  int out_pitch;
  // FECFRAME job (= channel * frames + j) -> output slot: job itself, or -- several PLPs per T2 frame, one launch per
  // PLP -- (job / out_group) * out_group_stride + out_group_off + job % out_group: the PLP's out_group FEC blocks of
  // every T2 frame land at their place inside the frame's list of out_group_stride blocks
  int out_group, out_group_stride, out_group_off;
  int *sync_errors;           // counter of payload sync bytes != 0x47 (reference logs a warning)
  // buffer extents for the bounds-checking debug build (DVBT2LL_DEBUG_BOUNDS); 0 = unknown, not checked
  long long ts_len;           // valid TS bytes per channel from ts + c * ts_pitch on
  long long out_len;          // bytes behind `out`
};
void launch_bb_bch(const BbArgs &a, cudaStream_t s);

// ---- K2: LDPC (IRA) ------------------------------------------------------------------------------
struct LdpcArgs {
  const uint8_t *in;  int in_pitch;    // packed BCH codewords
  uint8_t *out;       int out_pitch;   // packed: info bits then q rows of 360 parity bits ("u" order)
  int frames;
  int nbch, nldpc, q, groups;
  const uint16_t *row_ptr;   // q + 1
  const uint32_t *entries;   // (shift << 16) | group
  int lane_per_row;          // 1: a lane accumulates all 12 words of a parity row (fewer instructions, more bank conflicts);
                             // 0: a lane per (row, word).  Which is faster depends on the code: set from the plan.
  long long in_len, out_len; // bytes behind in / out (debug build bounds checks; 0 = not checked)
};
void launch_ldpc(const LdpcArgs &a, cudaStream_t s);

// ---- K3: bit interleaver + demux + constellation mapping (+ cyclic Q delay) -----------------------
struct MapArgs {
  const uint8_t *in;  int in_pitch;    // packed "u" codewords
  float2 *out;                         // frames * cell_size cells
  int frames;
  int nldpc, mod, cell_size, cyclic_delay;
  const uint16_t *bit_src;   // nldpc (generic path, used when ncol == 0: QPSK)
  const uint2 *qpsk_lut;     // QPSK: four cell codes per codeword byte, for the first qpsk_lin_cells cells (see MapPlan)
  int qpsk_lin_cells;
  int qpsk_par_q, qpsk_nbch; // > 0: parity cells through in-kernel bit transposes (see MapPlan), q rows of 360 bits behind bit nbch
  const float2 *lut;         // 1 << mod
  // QAM fast path: column-twist geometry; col_of_bit[p] = twist-matrix column feeding output bit p
  // (p = 0 is the MSB of the ncol-bit demux word), twist_of_col[c] = start row of column c
  int ncol;                  // 0 = use bit_src
  uint8_t col_of_bit[16];
  uint8_t twist_of_col[16];
  // the same geometry per output bit (filled by launch_map): first codeword bit and twist of the column feeding bit p --
  // constant-bank operands of the instantiations whose column count is a template parameter
  int base_of_bit[16], twist_of_bit[16];
  // optional fused cell interleaver (chain mode): out[(perm[c] + shift_r) % cell_size] = cell c of FEC block r
  uint16_t *out16;           // chain mode: 16-bit cell codes (own word | imaginary-part word << 8) instead of `out`
  long long out16_frame_stride;   // cells between T2 frames in out16 (multiple of 4: frames stay 8-byte aligned)
  const uint16_t *ci_inv;    // inverse of the cell permutation, or NULL for natural order
  // chain mode, optional: four copies of ci_inv shifted by 0..3 entries (copy k, entry j = ci_inv[j + k] as the PADDED
  // index c + 2 (c / 64) of k_map's code array, copies ci_inv4_stride entries apart, 8-byte aligned) so that any four
  // consecutive entries are one aligned 8-byte load
  const uint16_t *ci_inv4;
  int ci_inv4_stride;
  const int32_t *fec_shift;  // [fecblocks] cyclic shift per FEC block of the T2 frame
  int fecblocks;
  // single-table constellation (MapPlan::im_from_re): the word supplying the imaginary part is stored as
  // w~ = (((w << 1) & im_mask_i) | ((w >> 1) & im_mask_q)) ^ im_flip, and Im = Re lut[w~]
  int im_from_re;
  uint32_t im_mask_i, im_mask_q, im_flip;
  long long in_len, out_len; // bytes behind in, cells behind out / out16 (debug build bounds checks; 0 = not checked)
};
void launch_map(const MapArgs &a, cudaStream_t s);

// ---- bit format helpers for the drop-in blocks (1 bit per byte <-> packed) ------------------------
// pack: in = frames * nbits bytes (0/1) -> out packed with pitch
void launch_pack_bits(const uint8_t *in, int nbits, uint8_t *out, int out_pitch, int frames, cudaStream_t s);
// unpack first nbits of each packed frame
void launch_unpack_bits(const uint8_t *in, int in_pitch, int nbits, uint8_t *out, int frames, cudaStream_t s);
// LDPC drop-in output: packed "u" order -> 1 bit/byte natural order (parity index q*s + t <- row t, bit s)
void launch_unpack_ldpc(const uint8_t *in, int in_pitch, int nbch, int nldpc, int q, uint8_t *out, int frames,
                        cudaStream_t s);
// interleavermod drop-in input: 1 bit/byte natural-order codeword -> packed "u" order
void launch_pack_ldpc(const uint8_t *in, int nbch, int nldpc, int q, uint8_t *out, int out_pitch, int frames,
                      cudaStream_t s);

// ---- K4: frame mapper gather (cell int + time int + L1 + frame + frequency int composed) ----------
struct GatherArgs {
  const float2 *in;  long long in_stride;    // cells per T2 frame in
  float2 *out;       long long out_stride;   // cells per T2 frame out (= n codes)
  const int32_t *code; int n;
  const float2 *pool;
  int l1post_base, l1post_cells, l1post_variants;
  int frames; int frame_idx0;               // t2_frame_num of the first frame
};
void launch_gather(const GatherArgs &a, cudaStream_t s);

// ---- K5: carrier fill + IFFT + normalisation + guard interval + P1 --------------------------------
struct OfdmArgs {
  const float2 *cells; long long cells_stride;   // per T2 frame (stride in cells for both cell formats)
  // chain mode with 16-bit cells: cells16 != NULL selects it; then `code_pos` holds the carrier codes below
  // (OFDM_CODE_*, written by OfdmDevice::init)
  const uint16_t *cells16;   // [frame][fecblocks * cell_size] cell-interleaved 16-bit codes; frames start 16-byte aligned
  // bulk copies (cp.async.bulk) that stage a symbol's cells in shared memory: run i = { source 16-byte unit from the
  // frame's first cell, (staging 16-byte unit << 16) | length in units }, symbols back to back
  const int2 *run_desc;
  const int32_t *run_ptr;    // [num_symbols + 1] first run of each symbol (even)
  const int32_t *run_cnt;    // [num_symbols] number of runs
  int desc_cap;              // run descriptors the shared-memory descriptor buffer holds (even, >= the longest list)
  const int32_t *stage_bytes;// [num_symbols] bytes delivered by the symbol's copies
  const int32_t *sym_flags;  // [num_symbols] bit 0: the symbol has carriers coded 0x80000000 + pool cell
  int stage_cap;             // staging slots (cells) reserved in shared memory (multiple of 8)
  const float2 *lut; int lut_n;   // constellation LUT
  int lut_single;            // 1: imaginary parts come from the real-part table (the cell codes carry w~, see MapArgs)
  int lut_rep_shift;         // set by launch_ofdm: log2 of the number of LUT copies kept in shared memory
  void *out;           long long out_stride;     // samples per T2 frame (complex64, or short2 when out_fmt = 1)
  int out_fmt;               // 0 = complex64, 1 = interleaved 16-bit I/Q (x * 32767, saturated)
  float sink_gain;           // extra gain folded into `norm` and the P1 samples (1 = the reference block's output)
  const int32_t *code_pos;   // [num_symbols][split][M] carrier codes in shared-memory POSITION order
  const float2 *pool;        // special cells, one copy per L1-post variant (copy v holds the L1-post cells of frame index v)
  long long pool_stride;     // cells per copy
  int l1post_base, l1post_cells, l1post_variants;
  const float2 *p1;          // 2048
  const float *sinc_pos;     // [split][M] inverse-sinc factors in position order, or NULL
  const float2 *tw;          // W_M^m, m < M  (M = sub-transform size)
  const float2 *tw_split;    // W_N^n, n < N/2 (only when N = 2 M): recombination of the even/odd-bin halves
  int fft_n, log2_m, split;  // M = 1 << log2_m, split = N / M (1 or 2)
  int c_ps, left_nulls, gi, num_symbols;
  float norm;
  int frames; int frame_idx0;         // t2 frame number of the first frame, reduced mod l1post_variants by the host
  int frames_per_channel;    // frame f -> t2 frame number frame_idx0 + (f % frames_per_channel)
  // extents for the debug build bounds checks (0 = not checked): cells behind cells / cells16, samples behind out,
  // cells in one copy of the pool
  long long cells_len, out_len, pool_len;
  // > 1: `lut` holds that many constellation tables back to back (lut_n entries in all, the largest table first) and the
  // data carrier codes carry their table's first entry (OFDM_CODE_TAB_SHIFT); the k_ofdm instantiations with OFDM_FMT_MT run
  int lut_tables;
  // 1: MISO group-2 carrier codes (OFDM_CODE_MISO_IM); the k_ofdm instantiations with OFDM_FMT_MISO run
  int miso;
};
// Chain-mode carrier codes of k_ofdm (code_pos), one 32-bit word per carrier:
//   data carrier         -> 2 * staging slot                       bits 1..16 (byte offset into the staging area)
//                           | first table entry << 21              bits 21..30, only with several tables (lut_tables > 1)
//                           | OFDM_CODE_MISO_IM                    bit 0, only in the MISO group-2 codes (miso = 1)
//   small pool cell p<8  -> (p + 1) << 17                          bits 17..20 (zero / pilot amplitudes, in shared memory)
//   other pool cell      -> 0x80000000 | pool index                (L1 signalling, dummy cells; their symbols are flagged)
// Non-data carriers look up entry (staging slot 0's code) of the first table, which is the largest: any cell code
// stays inside it.
constexpr int OFDM_CODE_TAB_SHIFT = 21;
// MISO group 2 (EN 302 755 9.1, modified Alamouti): a data carrier's code names the staging slot of the other cell of
// its pair, and the looked-up value has its real part negated (bit 0 clear: -conj) or its imaginary part (bit 0 set:
// conj).  Pool cells come from a pool whose values are already transformed.
constexpr unsigned OFDM_CODE_MISO_IM = 1u;
constexpr unsigned OFDM_CODE_TAB_MAX = 1023;      // largest first-entry index the table bits hold
constexpr unsigned OFDM_CODE_SMALL_POOL = 0x1E0000u;   // bits of a small pool cell
// returns the number of constellation-table copies kept in shared memory (chain mode; 1 otherwise)
int launch_ofdm(const OfdmArgs &a, cudaStream_t s);
// shared-memory position (before swizzle) at which the carrier-fill stage must store bin m of an
// M = 2^log2_m point sub-transform (mixed-radix digit reversal matching the kernel's pass schedule)
int ofdm_position_of_bin(int m, int log2_m);
// index inside the per-(symbol, phase) tables at which the entry of position p is kept
int ofdm_table_index(int p, int log2_m);

// ---- K6: tone-reservation PAPR reduction on the reserved carriers (chain, opt-in) ------------------------------------
// Per OFDM symbol (P1 untouched), with x = the symbol's useful samples, p = the kernel of its reserved set S:
//   c = x; repeat up to `iterations` times: m = argmax |c_m|^2 (lowest index on ties); y = |c_m|; stop if y <= vclip;
//   beta = (y - vclip) c_m / y; stop if a reserved carrier would exceed tone_max; c_n -= beta p[(n - m) mod N].
// Output: [last gi samples of c | c] in the sink format.
struct PaprArgs {
  const float2 *in;          // complex64 samples at gain 1 (k_ofdm's output), T2 frames spf samples apart
  void *out;                 // the same layout in the sink format; == in for the in-place form
  int out_fmt;               // 0 = complex64, 1 = interleaved int16 I/Q (round(gain * c * 32767), saturated)
  float gain;                // sink gain (1 in the in-place form)
  int inplace;               // 1: out == in, complex64, gain 1: symbols without an update and P1 are not rewritten
  long long spf;             // samples per T2 frame
  int fft_n, gi, num_symbols, frames;
  int iterations;            // 1..64
  float vclip, tone_max;     // clip magnitude (units of x), bound of a reserved carrier (bin units)
  float tone_scale;          // 1 / (normalization * tones)
  int tones;                 // |S|
  const int32_t *sym_set;    // [num_symbols] set of each symbol
  const int32_t *bins;       // [sets][tones]
  const float2 *kernel;      // [sets][fft_n]
  const float2 *tone_tw;     // [fft_n] exp(-j 2 pi i / N)
  int16_t *stats;            // [frames][num_symbols]: updates applied | stop reason << 8 (PAPR_STOP_*)
  int sets;
  long long in_len, out_len; // samples behind in / out (debug build bounds checks; 0 = not checked)
};
enum { PAPR_STOP_CLIP = 1, PAPR_STOP_TONE = 2, PAPR_STOP_LIMIT = 3 };
void launch_papr_tr(const PaprArgs &a, cudaStream_t s);

long long kernel_launch_count();

} // namespace t2k
#endif
