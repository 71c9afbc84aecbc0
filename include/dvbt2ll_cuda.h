/*
 * dvbt2ll_cuda.h -- C ABI of libdvbt2ll_cuda.so, the B200 (sm_100a) implementation of the
 * gr-dvbt2ll DVB-T2 modulator hot path.
 *
 * This is the drop-in boundary: each entry point is what a GNU Radio block's constructor /
 * forecast() / general_work() / destructor calls.  Plain pointers and sizes only; buffers handed to
 * *_work() are HOST memory owned by the caller (the GNU Radio scheduler); the call is synchronous.
 * Handles are independent (no global mutable state; one CUDA stream per handle) and may be used
 * from different threads, one thread per handle at a time -- the GNU Radio threading contract.
 *
 * Reference interfaces replaced (paths relative to the gr-dvbt2ll tree):
 *   dvbt2ll_bbheaderbch_*      <- gr::dvbt2ll::bbheaderbch_bb       include/dvbt2ll/bbheaderbch_bb.h:49,
 *                                 lib/bbheaderbch_bb_impl.cc:42-196 (ctor), :207-216 (forecast), :648-742 (work)
 *   dvbt2ll_ldpc_*             <- gr::dtv::dvb_ldpc_bb (GNU Radio in-tree, wired in apps/vv009-4kshort.grc);
 *                                 restated by the reference at lib/bbheaderbch_bb_impl.cc:533-646
 *   dvbt2ll_interleavermod_*   <- gr::dvbt2ll::interleavermod_bc    include/dvbt2ll/interleavermod_bc.h:49,
 *                                 lib/interleavermod_bc_impl.cc:42-255, :264-268, :270-704
 *   dvbt2ll_framemapperfint_*  <- gr::dvbt2ll::framemapperfint_cc   include/dvbt2ll/framemapperfint_cc.h:49,
 *                                 lib/framemapperfint_cc_impl.cc:41-1190, :1942-1946, :1948-2151
 *   dvbt2ll_pilotgenp1insert_* <- gr::dvbt2ll::pilotgenp1insert_cc  include/dvbt2ll/pilotgenp1insert_cc.h:49,
 *                                 lib/pilotgenp1insert_cc_impl.cc:43-1229, :1239-1243, :2784-2907
 *   dvbt2ll_chain_*            <- new, additive: the five stages fused device-resident (what bench.py times)
 *
 * All integer parameters carry the enum VALUES of include/dvbt2ll/dvbt2ll_config.h:60-202.
 *
 * Return conventions: *_create() returns NULL on failure; *_work() returns the number of output
 * items produced (>= 0) or a negative error code; dvbt2ll_last_error() returns a thread-local
 * message for the most recent failure on the calling thread.
 */
#ifndef DVBT2LL_CUDA_H
#define DVBT2LL_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVBT2LL_API_EXPORT __attribute__((visibility("default")))

#define DVBT2LL_ERR_INVALID   (-1)   /* bad argument / unsupported parameter combination */
#define DVBT2LL_ERR_CUDA      (-2)   /* CUDA runtime error or no usable device (there is NO CPU fallback) */
#define DVBT2LL_ERR_SHORT     (-3)   /* not enough input items for the requested output */

typedef struct dvbt2ll_handle dvbt2ll_handle;   /* opaque */

DVBT2LL_API_EXPORT const char *dvbt2ll_last_error(void);
DVBT2LL_API_EXPORT const char *dvbt2ll_version(void);
/* Number of kernel launches issued by this library in the calling process (all handles). */
DVBT2LL_API_EXPORT long long dvbt2ll_kernel_launches(void);
/* 1 when a CUDA device is usable. */
DVBT2LL_API_EXPORT int dvbt2ll_device_available(void);

/* ---- common to all block handles ------------------------------------------------------------- */
/* set_output_multiple() value of the block: items of ONE frame of output. */
DVBT2LL_API_EXPORT int dvbt2ll_output_multiple(const dvbt2ll_handle *h);
/* forecast(): input items needed for noutput output items. */
DVBT2LL_API_EXPORT int dvbt2ll_forecast(const dvbt2ll_handle *h, int noutput);
/* general_work() on HOST buffers.  Processes floor(noutput / output_multiple) frames (any number,
 * unlike the reference which is only correct for one), writes *consumed = input items used
 * (the value the block passes to consume_each) and returns the output items produced. */
DVBT2LL_API_EXPORT int dvbt2ll_work(dvbt2ll_handle *h, const void *in, int ninput, void *out, int noutput,
                                    int *consumed);
/* Same on DEVICE buffers (already resident in HBM), asynchronous on `stream` (a cudaStream_t, NULL =
 * the handle's own stream followed by a synchronize). */
DVBT2LL_API_EXPORT int dvbt2ll_work_device(dvbt2ll_handle *h, const void *d_in, int ninput, void *d_out,
                                           int noutput, int *consumed, void *stream);
/* Number of warnings the reference would have logged so far ("Transport Stream sync error!"). */
DVBT2LL_API_EXPORT int dvbt2ll_warnings(const dvbt2ll_handle *h);
DVBT2LL_API_EXPORT void dvbt2ll_destroy(dvbt2ll_handle *h);
/* Host-side plan introspection (tables the kernels consume), for tests: copies at most cap bytes
 * of the named table to out and returns the table size in bytes, or -1 for an unknown name. */
DVBT2LL_API_EXPORT long long dvbt2ll_plan_get(const dvbt2ll_handle *h, const char *name, void *out, long long cap);

/* ---- bbheaderbch_bb: TS bytes -> BBFRAME -> scrambled -> BCH codeword, 1 bit per output byte --- */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_bbheaderbch_create(int framesize, int rate, int mode, int inband,
                                                              int fecblocks, int tsrate);

/* ---- LDPC: nbch bits -> 64800 | 16200 bits (info then parity, natural order), 1 bit per byte --- */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_ldpc_create(int framesize, int rate);

/* ---- interleavermod_bc: FECFRAME bits (1 per byte) -> cell_size complex64 cells ---------------- */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_interleavermod_create(int framesize, int rate, int constellation,
                                                                 int rotation);

/* ---- framemapperfint_cc: fecblocks*cell_size cells -> mapped_items cells per T2 frame ---------- */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_framemapperfint_create(
    int framesize, int rate, int constellation, int rotation, int fecblocks, int tiblocks, int carriermode,
    int fftsize, int guardinterval, int l1constellation, int pilotpattern, int t2frames, int numdatasyms,
    int paprmode, int version, int preamble, int inputmode, int reservedbiasbits, int l1scrambled, int inband);

/* ---- pilotgenp1insert_cc: active cells -> P1 + num_symbols * (N + GI) time samples ------------- */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_pilotgenp1insert_create(
    int carriermode, int fftsize, int pilotpattern, int guardinterval, int numdatasyms, int paprmode,
    int version, int preamble, int misogroup, int equalization, int bandwidth, int vlength);

/* ---- fused device-resident chain (TS bytes -> baseband), batching channels x T2 frames --------- */
typedef struct dvbt2ll_chain_params {
  int framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize, guardinterval,
      l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble, inputmode,
      reservedbiasbits, l1scrambled, inband, misogroup, equalization, bandwidth, vlength, tsrate;
} dvbt2ll_chain_params;

/* device < 0: current device.  max_frames = largest channels*frames batch a single run will be given. */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_chain_create(const dvbt2ll_chain_params *p, int max_frames, int device);
/* Several PLPs (beyond the reference, which is single-PLP: lib/framemapperfint_cc_impl.cc:152 num_plp = 1): num_plp
 * type-1 data PLPs that share the modulation / code / time-interleaving parameters of `p`, PLP i carrying
 * plp_fecblocks[i] FEC blocks per T2 frame (p->fecblocks is ignored; their sum is used), laid one after the other in the
 * frame and signalled in L1-post (NUM_PLP, the per-PLP configurable and dynamic fields, PLP_START; K_sig = 213 + 137
 * num_plp bits).  Every PLP is its own transport stream: the TS rows handed to dvbt2ll_chain_run_* are then
 * row = channel * num_plp + plp, each dvbt2ll_chain_plp_ts_bytes(h, plp, first_frame, n_frames) bytes long.
 * num_plp = 1 is dvbt2ll_chain_create. */
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_chain_create_multiplp(const dvbt2ll_chain_params *p, int num_plp,
                                                                 const int *plp_fecblocks, int max_frames, int device);
/* PLPs with their own robustness: num_plp (1..16) type-1 data PLPs, PLP i with its own FEC type, code rate,
 * constellation and rotation (enum values of dvbt2ll_config.h, validated as dvbt2ll_chain_create validates them) and
 * plp[i].fecblocks (1..1023) FEC blocks per T2 frame; p->framesize / rate / constellation / rotation / fecblocks are
 * ignored.  L1-post signals PLP_COD, PLP_MOD, PLP_ROTATION and PLP_FEC_TYPE per PLP, PLP_START advances by each PLP's
 * cells.  Time interleaving (tiblocks) stays shared.  Everything else as dvbt2ll_chain_create_multiplp (TS row =
 * channel * num_plp + plp, one stream per PLP).  A frame whose PLPs do not fit is always refused, whatever
 * dvbt2ll_set_overfull_policy says.  Returns NULL and sets dvbt2ll_last_error on any failure. */
typedef struct dvbt2ll_plp_params {
  int fecblocks, framesize, rate, constellation, rotation;
} dvbt2ll_plp_params;
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_chain_create_plps(const dvbt2ll_chain_params *p, int num_plp,
                                                             const dvbt2ll_plp_params *plp, int max_frames, int device);
/* PLP types, groups and sub-slicing (EN 302 755 7.2.3.1 PLP_TYPE / PLP_GROUP_ID, 8.3.6.3; beyond the reference, whose
 * single PLP is a type-1 data PLP).  As dvbt2ll_chain_create_plps, plus per PLP i the L1-post PLP_TYPE type[i] (0 =
 * common, 1 = data type 1, 2 = data type 2) and PLP_GROUP_ID group[i] (0..255), and num_subslices = N (1..32767), the
 * SUB_SLICES_PER_FRAME of the frame's type-2 PLPs.  The PLPs are listed in mapping order -- common PLPs, then type-1, then
 * type-2 -- and PLP_ID is the list index.  In the frame's data cells (L1-post PLP_START addresses):
 *   - common and type-1 PLPs each take one block of their D_i = PLP_NUM_BLOCKS x N_cells cells, one after the other
 *     from address 0; TYPE_2_START is the sum of their cells (0 without type-2 PLPs);
 *   - type-2 PLP i has sub-slices of L_i = D_i / N cells, SUB_SLICE_INTERVAL = sum of L_i over the type-2 PLPs, and
 *     cell k of its time-interleaver output goes to PLP_START_i + (k div L_i) SUB_SLICE_INTERVAL + k mod L_i, with
 *     PLP_START_i = TYPE_2_START + sum of L_j over the type-2 PLPs j before it;
 *   - dummy cells and the frame-closing symbol's unmodulated cells follow the last data cell.
 * BB framing, FEC, cell and time interleaving, FEC groups, taps and TS rows (channel * num_plp + plp) are those of
 * dvbt2ll_chain_create_plps, which is this call with every type 1, every group 1 and N = 1.  Refused, naming the PLP: a
 * type outside 0..2; PLPs out of mapping order; N outside 1..32767; N > 1 without a type-2 PLP; a type-2 PLP whose D_i is
 * not a multiple of N; a group outside 0..255; two common PLPs in one group; a common PLP whose group has no data PLP.
 * dvbt2ll_plan_get "frame.plp_layout": int32 per PLP { type, group, cells per sub-slice (D_i unless type 2) }, then N,
 * SUB_SLICE_INTERVAL, TYPE_2_START; "frame.plp_cells" column 1 is each PLP's PLP_START. */
typedef struct dvbt2ll_plp_layout {
  int num_subslices;
  int type[16], group[16];
} dvbt2ll_plp_layout;
DVBT2LL_API_EXPORT dvbt2ll_handle *dvbt2ll_chain_create_plp_layout(const dvbt2ll_chain_params *p, int num_plp,
                                                                   const dvbt2ll_plp_params *plp,
                                                                   const dvbt2ll_plp_layout *layout, int max_frames,
                                                                   int device);
DVBT2LL_API_EXPORT int dvbt2ll_chain_num_plp(const dvbt2ll_handle *h);
/* Stream bytes that must precede the first TS byte of first_frame in every row handed to dvbt2ll_chain_run_*:
 * 187 in normal input mode once the stream has started (CRC-8 of the packet in flight), else 0. */
DVBT2LL_API_EXPORT long long dvbt2ll_chain_history_bytes(const dvbt2ll_handle *h, long long first_frame);
DVBT2LL_API_EXPORT long long dvbt2ll_chain_plp_ts_bytes(const dvbt2ll_handle *h, int plp, long long first_frame, int n_frames);
DVBT2LL_API_EXPORT long long dvbt2ll_chain_ts_bytes_per_frame(const dvbt2ll_handle *h);
/* TS bytes (per channel) consumed by T2 frames [first_frame, first_frame + n_frames): constant per frame in normal
 * input mode; in high-efficiency mode the dropped sync bytes make it depend on the stream position. */
DVBT2LL_API_EXPORT long long dvbt2ll_chain_ts_bytes(const dvbt2ll_handle *h, long long first_frame, int n_frames);
DVBT2LL_API_EXPORT long long dvbt2ll_chain_samples_per_frame(const dvbt2ll_handle *h);
DVBT2LL_API_EXPORT int dvbt2ll_chain_fecframes_per_frame(const dvbt2ll_handle *h);
/* n_channels independent transport streams, each contributing n_frames consecutive T2 frames starting at
 * its stream frame number first_frame (streams start on a packet boundary at frame 0).  d_ts: channel-major,
 * dvbt2ll_chain_ts_bytes(h, first_frame, n_frames) bytes per channel with pitch ts_pitch.  In normal input mode with
 * first_frame > 0 each channel pointer must be preceded by the 187 stream bytes before it (CRC-8 of the packet in
 * flight), so ts_pitch >= bytes + 187; high-efficiency mode needs no history.
 * d_out: complex64, channel-major, n_frames*samples_per_frame per channel.  Asynchronous on `stream`. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_run_device(dvbt2ll_handle *h, const void *d_ts, long long ts_pitch,
                                                int n_channels, int n_frames, long long first_frame,
                                                void *d_out, void *stream);
/* Same with HOST buffers: H2D copy, run, D2H copy, synchronize. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_run_host(dvbt2ll_handle *h, const void *ts, long long ts_pitch, int n_channels,
                                              int n_frames, long long first_frame, void *out);
/* Optional sink stage of the flowgraph folded into the last kernel (apps/vv009-4kshort.grc: multiply_const 0.2 ->
 * USRP sink, which converts to 16-bit I/Q): gain scales the baseband; format 0 = complex64 (default, identical to
 * pilotgenp1insert_cc's output when gain = 1), format 1 = interleaved int16 I/Q = round(gain * x * 32767), saturated.
 * With format 1 the output buffers of dvbt2ll_chain_run_* hold 4 bytes per sample. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_set_sink(dvbt2ll_handle *h, int format, float gain);
/* Stage taps of the most recent chain run, for parity tests: "bch" (packed bits), "fec" (packed, parity
 * in interleaved-row order), "cells" (uint16 cell codes in cell-interleaved order: own constellation word |
 * word supplying the imaginary part << 8, frame stride padded to a multiple of 4 cells).  "bch.<p>" / "fec.<p>": PLP
 * p's codewords only, [channel][frame][block] at the pitch of its code.  With dvbt2ll_chain_create_plps and more than
 * one (framesize, rate, constellation, rotation) among the PLPs, "bch" and "fec" are refused, and in "cells" PLP p's
 * cells start at an 8-cell boundary of each frame (dvbt2ll_plan_get "frame.plp_cells": per PLP cells per FECFRAME,
 * first cell in the frame, first cell in this memory).  Copies to HOST; returns
 * bytes or negative error. */
DVBT2LL_API_EXPORT long long dvbt2ll_chain_tap(dvbt2ll_handle *h, const char *stage, void *out, long long cap);
/* Tone-reservation PAPR reduction (EN 302 755 9.6.2, peak-cancellation form; beyond the reference, which sends the
 * reserved carriers as zeros).  Needs paprmode PAPR_TR or PAPR_BOTH.  iterations = 0 switches the stage off (the
 * default), 1..64 switches it on; vclip (a sample magnitude in the units of the complex64 output at gain 1) and tone_max
 * (the largest magnitude of a reserved carrier, in the units where data cells have unit mean power) must be finite and
 * > 0.  Per OFDM symbol (P1 untouched), with x the useful samples and p_n = (1/|S|) sum_{b in S} exp(+j 2 pi b n / N)
 * the kernel of its reserved bins S: c = x; up to `iterations` times: m = argmax |c_m| (lowest m on equal float
 * values), y = |c_m|, stop if y <= vclip; beta = (y - vclip) c_m / y; stop, without this update, if a reserved carrier
 * R_b - beta exp(-j 2 pi b m / N) / (normalization |S|) would exceed tone_max; c_n -= beta p_{(n - m) mod N}.  Only
 * the reserved carriers change.  The symbol is then [last GI samples of c | c], through the sink.  Builds the tables
 * on the host (dvbt2ll_plan_get "ofdm.tr_set": int32 set per symbol, "ofdm.tr_bins": int32 [sets][|S|] FFT bins,
 * "ofdm.tr_kernel": complex64 [sets][N]); may be called between runs.  Tap "papr": one int16 per (channel, frame,
 * symbol) of the last run, updates applied | stop reason << 8 (1 = clip reached, 2 = tone_max, 3 = iteration limit);
 * refused while the stage is off. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_set_papr_tr(dvbt2ll_handle *h, int iterations, float vclip, float tone_max);
/* MISO processing (EN 302 755 9.1, modified Alamouti; beyond the reference, whose group-2 output carries group 1's
 * cells with only the pilots changed).  Let g_{l,0..C_l-1} be the cells of OFDM symbol l in the order the frequency
 * interleaver emits them (the order of the data carriers, k rising; L1-pre / L1-post, dummy and the unmodulated cells of
 * the frame-closing symbol included).  Group 1 sends e = g; group 2 sends e_{l,2i} = -conj(g_{l,2i+1}) and
 * e_{l,2i+1} = conj(g_{l,2i}), i < C_l / 2, in every P2, data and frame-closing symbol.  Pilots, nulls, reserved
 * carriers and P1 are not touched: each group keeps its own pilots (misogroup).
 * dvbt2ll_chain_set_miso: needs preamble T2_MISO or T2_LITE_MISO (refused otherwise, and for a frame with an odd cell
 * count in a symbol, naming it); with on = 1 a chain with misogroup TX2 emits group 2 with MISO processing from
 * dvbt2ll_chain_run_* and dvbt2ll_work*, tone reservation still applying after it; with misogroup TX1 the output is
 * unchanged.  Default off.  Once on, dvbt2ll_plan_get "chain.miso_code" (int32 carrier codes of group 2, "chain.code"'s
 * convention) and "chain.miso_pool" (complex64, its pool with the L1 / dummy cells transformed) can be read.
 * dvbt2ll_chain_run_{device,host}_miso: both groups from one pass of BB/BCH, LDPC and mapper -- group 1 to out1, group 2
 * with MISO processing to out2, whatever misogroup says; the arguments are those of dvbt2ll_chain_run_{device,host}, both
 * outputs take the sink, the stage time "ofdm" covers both k_ofdm launches.  Refused without a MISO preamble, with tone
 * reservation on, or with a NULL output. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_set_miso(dvbt2ll_handle *h, int on);
DVBT2LL_API_EXPORT int dvbt2ll_chain_run_device_miso(dvbt2ll_handle *h, const void *d_ts, long long ts_pitch, int n_channels,
                                                     int n_frames, long long first_frame, void *d_out1, void *d_out2,
                                                     void *stream);
DVBT2LL_API_EXPORT int dvbt2ll_chain_run_host_miso(dvbt2ll_handle *h, const void *ts, long long ts_pitch, int n_channels,
                                                   int n_frames, long long first_frame, void *out1, void *out2);
/* Device time in ms of each stage kernel (bb_bch, ldpc, map, ofdm, total), averaged over the chain runs issued since
 * timing was enabled (at most the last 64); events are recorded per run, so the caller's timed loop needs no sync.
 * With tone reservation on, "ofdm" covers k_ofdm and the tone-reservation kernel after it. */
DVBT2LL_API_EXPORT int dvbt2ll_chain_stage_ms(dvbt2ll_handle *h, float *ms5);
DVBT2LL_API_EXPORT void dvbt2ll_chain_enable_timing(dvbt2ll_handle *h, int on);

/* ---- transport-stream ingest helpers (host side): what stands in front of the chain when the TS comes from a file
 * or a socket instead of the flowgraph's ule_source (apps/vv009-4kshort.grc:1663).  dvbt2ll_ts_sync: first offset at which
 * 0x47 repeats every 188 bytes over 5 packets, -1 if none.  dvbt2ll_ts_fill: dst = bytes [pos, pos + dst_bytes) of the
 * packet-aligned stream src, continued with null packets (PID 0x1FFF) past its last whole packet -- rate adaptation when
 * the multiplex runs dry; pos < 0 reads as zeros.  Returns the null-packet bytes written. */
DVBT2LL_API_EXPORT long long dvbt2ll_ts_sync(const unsigned char *ts, size_t n);
DVBT2LL_API_EXPORT long long dvbt2ll_ts_fill(unsigned char *dst, size_t dst_bytes, const unsigned char *src, size_t src_bytes,
                                             long long pos);

/* ---- small device utilities for hosts without a CUDA runtime binding of their own (tests, language bindings):
 * synchronous copies, allocation and device selection for the raw device pointers the *_device entry points take. */
DVBT2LL_API_EXPORT int dvbt2ll_copy_to_host(void *dst, const void *d_src, size_t bytes);
DVBT2LL_API_EXPORT int dvbt2ll_copy_to_device(void *d_dst, const void *src, size_t bytes);
DVBT2LL_API_EXPORT void *dvbt2ll_device_alloc(size_t bytes);
DVBT2LL_API_EXPORT void dvbt2ll_device_free(void *p);
DVBT2LL_API_EXPORT int dvbt2ll_device_count(void);
DVBT2LL_API_EXPORT int dvbt2ll_set_device(int device);
DVBT2LL_API_EXPORT int dvbt2ll_device_synchronize(void);
/* a non-blocking stream on the current device, usable wherever an entry point takes a `stream` */
DVBT2LL_API_EXPORT void *dvbt2ll_stream_create(void);
DVBT2LL_API_EXPORT void dvbt2ll_stream_destroy(void *stream);
DVBT2LL_API_EXPORT int dvbt2ll_stream_synchronize(void *stream);

/* ---- behaviour switches --------------------------------------------------------------------------- */
/* Over-full T2 frame (more FEC blocks than the frame has cells for).  The reference logs "Frame Mapper, too many FEC
 * blocks in T2 frame." and keeps running, dropping the cells that do not fit (lib/framemapperfint_cc_impl.cc:1138-1141).
 * policy 0 (default): *_create() fails with that message; policy 1: reproduce the reference -- the handle is created,
 * dvbt2ll_warnings() reports 1 and the frames carry what the reference's frames carry.  Also settable through the
 * environment (DVBT2LL_OVERFULL=warn).  Process-wide; affects handles created afterwards. */
DVBT2LL_API_EXPORT void dvbt2ll_set_overfull_policy(int policy);
/* dvbt2ll_work() on HOST buffers: when on, the buffers are registered with cudaHostRegister the first time they are
 * seen, so both copies run as DMA at PCIe rate (GNU Radio hands over pageable memory).  Only for callers whose buffers
 * outlive the handle (the scheduler's do); default off, or DVBT2LL_HOST_REGISTER=1 in the environment. */
DVBT2LL_API_EXPORT void dvbt2ll_set_host_register(dvbt2ll_handle *h, int on);
/* Device-resident hand-off between adjacent drop-in blocks of one process: after dvbt2ll_work() the producer keeps
 * its last four outputs in HBM (a thread-per-block scheduler lets it run ahead of its consumer); a consumer linked to
 * it takes its input from there when the host range it is handed lies inside one of them (the scheduler passes the
 * very buffer on), skipping its host-to-device copy.  The blocks may be driven by different threads. */
DVBT2LL_API_EXPORT int dvbt2ll_link(dvbt2ll_handle *producer, dvbt2ll_handle *consumer);
/* Automatic hand-off, process-wide (also DVBT2LL_AUTO_LINK=1 in the environment): every drop-in block keeps its last
 * four outputs resident and a block that was not linked explicitly looks its input range up among the other blocks'
 * resident outputs -- a flowgraph assembled by unchanged Python/GRC code gets the hand-off without calling
 * dvbt2ll_link().  Host buffers are still written (never lazy).  Default off. */
DVBT2LL_API_EXPORT void dvbt2ll_set_auto_link(int on);
/* Number of work() calls of `consumer` that found their input resident in HBM (tests, tuning). */
DVBT2LL_API_EXPORT long long dvbt2ll_link_hits(const dvbt2ll_handle *consumer);
/* Opt-in on top of dvbt2ll_link(): the producer no longer writes its host output buffer on every call; the items stay
 * in HBM for the linked consumer.  Whatever the consumer has not taken from HBM is written to the host buffer late --
 * before the producer reuses that device copy (four calls later, or when it is handed the same host range again), or
 * at once when the consumer asks for the range with a non-matching pointer -- so the linked pair never loses items.  Only for edges whose ONLY reader is the linked
 * consumer: any other reader of that host buffer (a second block on the same output, a probe) sees stale bytes; and the
 * output buffer of a call must stay allocated for the producer's next four calls (the scheduler's buffers do). */
DVBT2LL_API_EXPORT int dvbt2ll_link_lazy_host(dvbt2ll_handle *producer, int on);
/* Number of late host writes `producer` had to do (0 in a flowgraph whose scheduler passes every buffer straight on). */
DVBT2LL_API_EXPORT long long dvbt2ll_link_late_writes(const dvbt2ll_handle *producer);

/* ---- ordered multi-GPU reassembly on one GPU ------------------------------------------------------
 * T2 frames shard across GPUs with no data-path collective; the one exchange is putting the ranks' finished frames
 * back into ONE ordered stream on the root GPU -- the single sink of the reference flowgraph
 * (apps/vv009-4kshort.grc:1696-1697).  A "step" is one batch of every rank; its ordered output is one slot of
 * slot_bytes in a ring of n_slots on the root.  The root's chain writes into the slot in place; the other ranks
 * produce into a local buffer and push it with one peer copy over NVLink (copy engine, side stream), overlapping
 * their next step.  Arrival and slot release are device-side counters waited on with stream memory operations:
 * no host synchronisation anywhere.  Ranks are processes (CUDA IPC) or several handles of one process.
 *   every rank:  g = create(); export(blob); <all ranks' blobs, rank order> -> connect();
 *   every step:  acquire(step, offset, producer, &p); dvbt2ll_chain_run_device(..., p, producer); push(step, offset, bytes, producer);
 *   root only:   wait(step, consumer, &slot); <consume slot on consumer>; release(step, consumer). */
#define DVBT2LL_GATHER_BLOB_BYTES 256
typedef struct dvbt2ll_gather dvbt2ll_gather;
DVBT2LL_API_EXPORT const char *dvbt2ll_gather_last_error(void);
/* local_bytes: largest part this rank pushes per step (ignored on the root). 1 <= n_slots <= 8, world <= 64. */
DVBT2LL_API_EXPORT dvbt2ll_gather *dvbt2ll_gather_create(int rank, int world, int root, int device, size_t slot_bytes,
                                                         size_t local_bytes, int n_slots);
DVBT2LL_API_EXPORT int dvbt2ll_gather_export(dvbt2ll_gather *g, void *blob, size_t cap);
DVBT2LL_API_EXPORT int dvbt2ll_gather_connect(dvbt2ll_gather *g, const void *blobs, size_t bytes);
DVBT2LL_API_EXPORT int dvbt2ll_gather_acquire(dvbt2ll_gather *g, long long step, size_t offset, void *producer_stream, void **ptr);
DVBT2LL_API_EXPORT int dvbt2ll_gather_push(dvbt2ll_gather *g, long long step, size_t offset, size_t bytes, void *producer_stream);
DVBT2LL_API_EXPORT int dvbt2ll_gather_wait(dvbt2ll_gather *g, long long step, void *consumer_stream, void **slot);
DVBT2LL_API_EXPORT int dvbt2ll_gather_release(dvbt2ll_gather *g, long long step, void *consumer_stream);
DVBT2LL_API_EXPORT void *dvbt2ll_gather_side_stream(dvbt2ll_gather *g);
DVBT2LL_API_EXPORT void dvbt2ll_gather_destroy(dvbt2ll_gather *g);

#ifdef __cplusplus
}
#endif
#endif /* DVBT2LL_CUDA_H */
