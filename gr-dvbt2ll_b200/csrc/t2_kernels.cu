// Hand-written sm_100a kernels of the DVB-T2 modulator hot path.
//
//   k_bb_bch   warp per FECFRAME : BB header, TS payload with CRC-8 sync substitution, BB scrambler,
//                                  BCH parity as GF(2) polynomial remainder (per-lane chunk remainders
//                                  from a byte table, combined with a ballot-evaluated x^L multiply)
//   k_ldpc     warp per FECFRAME : IRA parity as XOR of 360-bit cyclic rotations (funnel shifts on a
//                                  wrap-extended copy of each info group), accumulator in closed form
//   k_map      CTA per FECFRAME  : bit interleaver + demux (table driven bit gather from shared
//                                  memory), constellation LUT, cyclic Q delay, coalesced float2 stores
//   k_gather   grid-stride       : frame mapper as one static gather
//   k_ofdm     CTA per OFDM symbol: carrier fill (gather + pilots), in-place shared-memory DIT FFT
//                                  (radix 16/8/4/2 in registers, padded layout), scale, CP, P1
//
// None of the stages is a dense contraction, so no tensor-core MMA is used: the cell-domain kernels are
// HBM/L2 bound, the bit-domain ones integer-pipe bound, the IFFT shared-memory bound.  The 32K k_ofdm
// uses tensor memory as storage only (the parked even-bin half, see the TMEM helpers).
#include "t2_kernels.cuh"

#include <atomic>

// Bounds-checking debug build (make -C gr-dvbt2ll_b200/csrc debug -> libdvbt2ll_cuda_dbg.so, selected with
// DVBT2LL_LIB): every index the kernels derive from tables or stream positions is checked against the extent of
// the buffer it addresses; a violation prints its source line and traps.  compute-sanitizer is closed on the GPU
// pool, so the parity suite is run once under this build instead.
#ifdef DVBT2LL_DEBUG_BOUNDS
#include <cstdio>
#define BND(ok)                                                                                                   \
  do {                                                                                                            \
    if (!(ok)) {                                                                                                  \
      printf("DVBT2LL bounds violation: %s (t2_kernels.cu:%d, block %d thread %d)\n", #ok, __LINE__, (int)blockIdx.x, (int)threadIdx.x); \
      __trap();                                                                                                   \
    }                                                                                                             \
  } while (0)
#else
#define BND(ok) do { } while (0)
#endif

namespace t2k {

static std::atomic<long long> g_launches(0);
long long kernel_launch_count() { return g_launches.load(); }
static inline void count_launch() { g_launches.fetch_add(1); }
void count_extra_launch() { count_launch(); }      // kernels of other translation units (t2_gather.cu)

// Per-device caches: function attributes and the SM count belong to a device, and one process may drive several
// (dvbt2ll_chain_create takes a device index).  Racing writers store the same value.
constexpr int MAX_DEVICES = 64;
static inline int current_device()
{
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev < 0 || dev >= MAX_DEVICES) ? 0 : dev;
}

static inline int sm_count()
{
  static int n[MAX_DEVICES];
  const int dev = current_device();
  if (!n[dev]) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    n[dev] = v > 0 ? v : 148;
  }
  return n[dev];
}

// opt in to `bytes` of dynamic shared memory for kernel `k` once per device
template <class K>
static inline void allow_smem(K k, int bytes, bool (&done)[MAX_DEVICES])
{
  const int dev = current_device();
  if (done[dev]) return;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  done[dev] = true;
}

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }
// 32 stream bits starting at bit position p of a big-endian word array
__device__ __forceinline__ uint32_t window32(const uint32_t *w, int p)
{
  const int k = p >> 5;
  return __funnelshift_l(w[k + 1], w[k], p & 31);
}

// ================================================================================================
// K1  BB framing + scrambler + BCH
// ================================================================================================
constexpr int BB_MAX_WARPS = 32;      // warps (= FECFRAMEs in flight) per CTA; fewer when the frame buffers do not fit

__device__ __forceinline__ int multiples_in(int a, int b, int m)   // multiples of m in [a, b), a,b >= 0
{
  return (b + m - 1) / m - (a + m - 1) / m;
}

// TS index of de-synced payload byte P in high-efficiency mode (sync bytes dropped), c0 = packet phase of ts[0]
__device__ __forceinline__ long long hem_ts_index(long long P, int c0)
{
  const int t0 = (188 - c0) % 188;      // TS index of the first sync byte
  if (P < t0) return P;
  const long long pp = P - t0;
  return t0 + 1 + pp + pp / 187;
}

// W6 = false: remainder register of at most 160 bits (5 words): the sixth word is identically zero and skipped
template <bool W6>
__global__ void __launch_bounds__(BB_MAX_WARPS * 32) k_bb_bch(const BbArgs a)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  // BCH remainder tables, one row per message NIBBLE and one private copy per lane: word w of row n of table k
  // (k = nibble position inside a 16-bit step: n x^(r + 4k) mod g) for lane l sits at ((k*16 + n)*NW + w)*32 + l,
  // i.e. always in bank l -- 32 lanes looking up 32 different rows never conflict (a byte-indexed table shared by
  // the warp costs ~3.3 wavefronts per access instead).
  constexpr int NW = W6 ? 6 : 5;
  uint32_t *s_ntab = reinterpret_cast<uint32_t *>(smem_raw);  // 4 * 16 * NW * 32
  uint32_t *s_cols = s_ntab + 4 * 16 * NW * 32;               // 6 * 32 * 6
  uint8_t *s_crc8 = reinterpret_cast<uint8_t *>(s_cols + 6 * 32 * 6);   // 256: CRC-8 byte table (BB header)
  uint8_t *s_buf = s_crc8 + 256;
  const int nbytes = a.nbch / 8, msg_bytes = a.kbch / 8;
  constexpr int HIST = 192;                                   // stream history kept in front of each frame buffer
  const int buf_pitch = ((nbytes + 15) & ~15) + HIST;

  // (eight table words requested per round trip: with few warps per CTA -- small batches -- this prologue is otherwise a
  // chain of ~30 dependent L2 latencies, a third of the kernel's time at 8 channels per GPU)
#pragma unroll 1
  for (int i0 = threadIdx.x; i0 < 4 * 16 * NW * 32; i0 += 8 * blockDim.x) {
    uint32_t v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int i = i0 + u * blockDim.x;
      const int w = (i >> 5) % NW, kn = (i >> 5) / NW, k = kn >> 4, n = kn & 15;
      // from the byte tables T0 = b x^r, T1 = b x^(r+8): nibble n at position k is byte (n << 4*(k&1)) of table k>>1
      v[u] = i < 4 * 16 * NW * 32 ? __ldg(a.bch_tab + ((k >> 1) * 256 + (n << (4 * (k & 1)))) * 6 + w) : 0u;
    }
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int i = i0 + u * blockDim.x;
      if (i < 4 * 16 * NW * 32) s_ntab[i] = v[u];
    }
  }
#pragma unroll 4
  for (int i = threadIdx.x; i < 6 * 32 * 6; i += blockDim.x) s_cols[i] = __ldg(a.bch_cols + i);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_crc8[i] = a.crc8_tab[i];
  __syncthreads();
  const uint8_t *S1 = s_crc8;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t *buf = s_buf + warp * buf_pitch + HIST;             // buf[10 - k] = TS byte k positions before the frame's payload
  uint32_t *bufw = reinterpret_cast<uint32_t *>(buf);
  const int total = a.n_channels * a.frames;
  const int D = a.payload_bytes;
  const bool hem = a.mode != 0;
  const uint32_t *scr32 = reinterpret_cast<const uint32_t *>(a.scramble);   // zero padded to a word multiple

  const int nwarps = blockDim.x >> 5;
  for (int job = blockIdx.x * nwarps + warp; job < total; job += gridDim.x * nwarps) {
    const int c = job / a.frames, j = job - c * a.frames;
    const uint8_t *ts = a.ts + (long long)c * a.ts_pitch;
    const int nb = a.inband ? multiples_in(a.fec_block0, a.fec_block0 + j, a.fecblocks) : 0;
    const bool ib = a.inband && ((a.fec_block0 + j) % a.fecblocks == 0);
    const long long P0 = (long long)j * D - 13LL * nb;     // payload bytes before this frame
    const int Dj = D - (ib ? 13 : 0);
    // TS index at which the frame's read loop starts, and packet phase there
    long long t_start;
    if (!hem) t_start = P0;
    else t_start = P0 == 0 ? 0 : hem_ts_index(P0 - 1, a.count0) + 1;
    const int count = (int)((a.count0 + t_start) % 188);

    BND(10 + Dj + (ib ? 13 : 0) <= msg_bytes && msg_bytes + a.bch_r / 8 == nbytes && nbytes <= buf_pitch - HIST);
    BND(a.out_len == 0 || a.out_group != 0 || (long long)(job + 1) * a.out_pitch <= a.out_len + (a.out_pitch - nbytes));
    // ---- stage the raw payload in shared memory (buf byte 10 + i = payload byte i)
    if (!hem) {
      const uint8_t *src = ts + P0;
      BND(a.ts_len == 0 || (P0 >= 0 && P0 + Dj <= a.ts_len));
      {
        // the TS is read once, from DRAM: ask L2 for the payload of this warp's NEXT FECFRAME now
        const int nj = job + gridDim.x * nwarps;
        if (nj < total) {
          const int nc = nj / a.frames, njj = nj - nc * a.frames;
          const int nnb = a.inband ? multiples_in(a.fec_block0, a.fec_block0 + njj, a.fecblocks) : 0;
          const uint8_t *nsrc = a.ts + (long long)nc * a.ts_pitch + ((long long)njj * D - 13LL * nnb);
          for (int o = lane * 128; o < D; o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nsrc + o));
        }
      }
      if (lane < 2) buf[10 + lane] = src[lane];
      const int w_end = (10 + Dj) >> 2;                    // words [3, w_end) lie completely inside the payload
      {
        // buffer word w = payload bytes 4 w - 10 .. 4 w - 7: the payload's misalignment is the same for every word of the
        // frame, so a word is a funnel shift of two ALIGNED global words.  All eight loads of a batch are issued
        // unconditionally (indices clamped to the last valid word) before the first is used: as predicated unaligned loads
        // the compiler waited for each pair in turn, and that wait was a quarter of the kernel's stall samples.
        const uintptr_t ad = reinterpret_cast<uintptr_t>(src + 2);            // address of buffer word 3
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(ad & ~(uintptr_t)3);
        const int sh = (int)(ad & 3) * 8;
        const int last = w_end - 4;                                           // index (from word 3) of the last whole word
        if (last >= 0)
        for (int w0 = lane; w0 <= last; w0 += 128) {
          uint32_t lo[4], hi[4];
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const int k = min(w0 + 32 * u, last);
            lo[u] = __ldg(wp + k);
            hi[u] = __ldg(wp + k + (sh ? 1 : 0));
          }
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (w0 + 32 * u <= last) bufw[3 + w0 + 32 * u] = __funnelshift_r(lo[u], hi[u], sh);
        }
      }
      for (int i = 4 * w_end - 10 + lane; i < Dj; i += 32) buf[10 + i] = src[i];
      // the 187 bytes before the frame (previous packet's tail) for the first CRC-8; missing history reads as 0,
      // which leaves a zero CRC state unchanged
      // (kept contiguous with the payload, under the place the BB header is written to afterwards)
      for (int k = 1 + lane; k <= 187; k += 32) buf[10 - k] = (P0 - k >= 0 || a.hist_valid) ? src[-k] : (uint8_t)0;
    }
    else {
      BND(a.ts_len == 0 || hem_ts_index(P0 + Dj - 1, a.count0) < a.ts_len);
      for (int i = lane; i < Dj; i += 32) buf[10 + i] = ts[hem_ts_index(P0 + i, a.count0)];
      // sync bytes skipped by this frame: positions between t_start and the last payload byte
      const long long t_end = hem_ts_index(P0 + Dj - 1, a.count0);
      const int first = (int)((188 - (a.count0 + t_start) % 188) % 188);
      for (long long t = t_start + first + 188LL * lane; t <= t_end; t += 188LL * 32)
        if (ts[t] != 0x47) atomicAdd(a.sync_errors, 1);
    }
    __syncwarp();
    // ---- NORMAL mode: each sync byte is replaced by the CRC-8 of the previous packet's 187 bytes
    // (bytes of this frame come from shared memory, earlier ones from the stream history in global memory)
    uint8_t my_crc[2] = { 0, 0 };
    const int i0 = (188 - count) % 188;
    if (!hem) {
#pragma unroll
      for (int rnd = 0; rnd < 2; rnd++) {
        const int si = i0 + 188 * (lane + 32 * rnd);
        if (si < Dj) {
          if (buf[10 + si] != 0x47) atomicAdd(a.sync_errors, 1);
          // CRC-8 of the 187 bytes before the sync byte: 47 unaligned little-endian words starting one byte early
          // (that byte masked off).  The CRC is GF(2)-linear in the data: each of its bits is the parity of the XOR of
          // (word & position mask) over the words, the masks being constant-bank operands -- no table look-ups, no
          // serial state
          const uint8_t *p = buf + 10 + si - 188;
          BND(10 + si - 188 >= -HIST && si < Dj);
          const uint32_t *pw = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
          const int sh = (int)(reinterpret_cast<uintptr_t>(p) & 3) * 8;
          uint32_t lo = pw[0];
          uint32_t acc[8] = { 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u };
#pragma unroll
          for (int st = 0; st < 47; st++) {
            const uint32_t hi = pw[st + 1];
            const uint32_t t = __funnelshift_r(lo, hi, sh);
            lo = hi;
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] ^= t & a.crc8_pos_mask[st][k];
          }
          uint32_t crc = 0;
#pragma unroll
          for (int k = 0; k < 8; k++) crc |= (__popc(acc[k]) & 1u) << k;
          my_crc[rnd] = (uint8_t)crc;
        }
      }
    }
    __syncwarp();
    if (!hem) {
#pragma unroll
      for (int rnd = 0; rnd < 2; rnd++) {
        const int si = i0 + 188 * (lane + 32 * rnd);
        if (si < Dj) buf[10 + si] = my_crc[rnd];
      }
    }
    // ---- BB header (EN 302 755 5.1.7): MATYPE, UPL, DFL, SYNC, SYNCD, CRC-8 (xor MODE)
    if (lane == 0) {
      uint8_t h[10];
      h[0] = 0xF0;            // TS, SIS, CCM, no ISSY, no NPD, EXT 00
      h[1] = 0x00;
      const int upl = hem ? 0 : 188 * 8, dfl = a.kbch - 80 - (ib ? 104 : 0);
      const int syncd = count ? (188 - count) * 8 : 0;
      h[2] = (uint8_t)(upl >> 8); h[3] = (uint8_t)upl;
      h[4] = (uint8_t)(dfl >> 8); h[5] = (uint8_t)dfl;
      h[6] = hem ? 0x00 : 0x47;
      h[7] = (uint8_t)(syncd >> 8); h[8] = (uint8_t)syncd;
      uint8_t crc = 0;
      for (int i = 0; i < 9; i++) crc = S1[crc ^ h[i]];
      h[9] = hem ? (crc ^ 1) : crc;
      for (int i = 0; i < 10; i++) buf[i] = h[i];
    }
    if (ib)
      for (int i = lane; i < 13; i += 32) buf[10 + Dj + i] = a.inband_bytes[i];
    __syncwarp();
    // ---- BB scrambler, word-wise
    for (int w = lane; w < (msg_bytes + 3) >> 2; w += 32) bufw[w] ^= __ldg(scr32 + w);
    __syncwarp();

    // ---- BCH: per-lane remainder of a chunk of the message (byte-table LFSR on a 192-bit register)
    uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0, r4 = 0, r5 = 0;
    {
      int s = lane * a.chunk_bytes - a.lead_zero_bytes;
      const int e = s + a.chunk_bytes;
      if (s < 0) s = 0;
      int i = s;
      const uint32_t *nt = s_ntab + lane;
      constexpr int ROW = NW * 32;              // words between rows of a table
      // one message byte: two nibble rows
      auto step8 = [&](uint32_t byte) {
        const uint32_t x = (r0 >> 24) ^ byte;
        const uint32_t *t1 = nt + (16 + (x >> 4)) * ROW, *t0 = nt + (x & 15u) * ROW;
        r0 = ((r0 << 8) | (r1 >> 24)) ^ t1[0] ^ t0[0];
        r1 = ((r1 << 8) | (r2 >> 24)) ^ t1[32] ^ t0[32];
        r2 = ((r2 << 8) | (r3 >> 24)) ^ t1[64] ^ t0[64];
        r3 = ((r3 << 8) | (r4 >> 24)) ^ t1[96] ^ t0[96];
        r4 = ((r4 << 8) | (W6 ? r5 >> 24 : 0u)) ^ t1[128] ^ t0[128];
        if (W6) r5 = (r5 << 8) ^ t1[NW * 32 - 32] ^ t0[NW * 32 - 32];
      };
      // two message bytes (big-endian halfword): four nibble rows, all independent of each other
      auto step16 = [&](uint32_t half) {
        const uint32_t x = (r0 >> 16) ^ half;
        const uint32_t *t3 = nt + (48 + (x >> 12)) * ROW, *t2 = nt + (32 + ((x >> 8) & 15u)) * ROW,
                       *t1 = nt + (16 + ((x >> 4) & 15u)) * ROW, *t0 = nt + (x & 15u) * ROW;
        r0 = ((r0 << 16) | (r1 >> 16)) ^ t3[0] ^ t2[0] ^ t1[0] ^ t0[0];
        r1 = ((r1 << 16) | (r2 >> 16)) ^ t3[32] ^ t2[32] ^ t1[32] ^ t0[32];
        r2 = ((r2 << 16) | (r3 >> 16)) ^ t3[64] ^ t2[64] ^ t1[64] ^ t0[64];
        r3 = ((r3 << 16) | (r4 >> 16)) ^ t3[96] ^ t2[96] ^ t1[96] ^ t0[96];
        r4 = ((r4 << 16) | (W6 ? r5 >> 16 : 0u)) ^ t3[128] ^ t2[128] ^ t1[128] ^ t0[128];
        if (W6) r5 = (r5 << 16) ^ t3[NW * 32 - 32] ^ t2[NW * 32 - 32] ^ t1[NW * 32 - 32] ^ t0[NW * 32 - 32];
      };
      // head: single bytes up to a word boundary of the frame buffer (the same 0..3 bytes for every lane: the chunk
      // length is a multiple of 4); body: one conflict-free 32-bit load per four message bytes; tail: single bytes
      for (; (i & 3) && i < e; i++) step8(buf[i]);
      for (; i + 4 <= e; i += 4) {
        const uint32_t mw = bufw[i >> 2];
        step16(__byte_perm(mw, 0u, 0x4401u));
        step16(__byte_perm(mw, 0u, 0x4423u));
      }
      for (; i < e; i++) step8(buf[i]);
    }
    // ---- Horner combine: acc = acc * x^(8*chunk) + R_i, the multiply evaluated column-wise:
    // lane l computes output bit (31 - l) of every word as parity(acc & column) and a ballot
    // assembles the words, so acc stays warp-uniform.
    uint32_t c0 = __shfl_sync(0xffffffffu, r0, 0), c1 = __shfl_sync(0xffffffffu, r1, 0),
             c2 = __shfl_sync(0xffffffffu, r2, 0), c3 = __shfl_sync(0xffffffffu, r3, 0),
             c4 = __shfl_sync(0xffffffffu, r4, 0), c5 = __shfl_sync(0xffffffffu, r5, 0);
    {
      // this lane's six column masks stay in registers for the whole combine
      constexpr int NW = W6 ? 6 : 5;
      uint32_t col[NW][NW];
#pragma unroll
      for (int w = 0; w < NW; w++)
#pragma unroll
        for (int k = 0; k < NW; k++) col[w][k] = s_cols[(w * 32 + lane) * 6 + k];
      for (int i = 1; i < 32; i++) {
        uint32_t n[6];
        n[5] = 0;
#pragma unroll
        for (int w = 0; w < NW; w++) {
          uint32_t x = (c0 & col[w][0]) ^ (c1 & col[w][1]) ^ (c2 & col[w][2]) ^ (c3 & col[w][3]) ^ (c4 & col[w][4]);
          if (W6) x ^= c5 & col[w][NW - 1];
          n[w] = __ballot_sync(0xffffffffu, __popc(x) & 1);
        }
        c0 = n[0] ^ __shfl_sync(0xffffffffu, r0, i);
        c1 = n[1] ^ __shfl_sync(0xffffffffu, r1, i);
        c2 = n[2] ^ __shfl_sync(0xffffffffu, r2, i);
        c3 = n[3] ^ __shfl_sync(0xffffffffu, r3, i);
        c4 = n[4] ^ __shfl_sync(0xffffffffu, r4, i);
        c5 = n[5] ^ __shfl_sync(0xffffffffu, r5, i);
      }
    }
    if (lane < a.bch_r / 8) {
      const int wsel = lane >> 2;
      const uint32_t word = wsel == 0 ? c0 : wsel == 1 ? c1 : wsel == 2 ? c2 : wsel == 3 ? c3 : wsel == 4 ? c4 : c5;
      buf[msg_bytes + lane] = (uint8_t)(word >> (24 - 8 * (lane & 3)));
    }
    __syncwarp();
    // ---- store the packed codeword
    const long long oslot = a.out_group ? (long long)(job / a.out_group) * a.out_group_stride + a.out_group_off + job % a.out_group : job;
    uint8_t *o = a.out + oslot * a.out_pitch;
    const int nw = nbytes >> 2;
    uint32_t *ow = reinterpret_cast<uint32_t *>(o);
    for (int i = lane; i < nw; i += 32) ow[i] = bufw[i];
    for (int i = (nw << 2) + lane; i < nbytes; i += 32) o[i] = buf[i];
    __syncwarp();
  }
}

void launch_bb_bch(const BbArgs &a, cudaStream_t s)
{
  const int nbytes = a.nbch / 8;
  const int buf_pitch = ((nbytes + 15) & ~15) + 192;
  const bool w6 = a.bch_r > 160;
  const size_t fixed = (size_t)4 * 16 * (w6 ? 6 : 5) * 32 * 4 + 6 * 32 * 6 * 4 + 256;
  const int total = a.n_channels * a.frames;
  if (total < 1) return;
  static bool attr6[MAX_DEVICES], attr5[MAX_DEVICES];
  allow_smem(k_bb_bch<true>, 227 * 1024, attr6);
  allow_smem(k_bb_bch<false>, 227 * 1024, attr5);
  // one CTA per SM (the lane-private tables take 40-48 KB), as many warps as frame buffers fit
  int warps = BB_MAX_WARPS;
  while (warps > 4 && fixed + (size_t)warps * buf_pitch > 227 * 1024) warps -= 4;
  // spread the FECFRAMEs evenly: with `spread` FECFRAMEs per SM the warps make ceil(spread / warps) rounds, and a
  // last round that is nearly empty runs latency-bound -- use just enough warps for that many equal rounds
  const int spread = (total + sm_count() - 1) / sm_count();
  if (spread < warps) warps = spread < 1 ? 1 : spread;
  else {
    const int rounds = (spread + warps - 1) / warps;
    warps = (spread + rounds - 1) / rounds;
  }
  const size_t smem = fixed + (size_t)warps * buf_pitch;
  int blocks = (total + warps - 1) / warps;
  const int cap = sm_count();                 // one resident wave; warps loop over the remaining FECFRAMEs
  if (blocks > cap) blocks = cap;
  if (w6) k_bb_bch<true><<<blocks, warps * 32, smem, s>>>(a);
  else k_bb_bch<false><<<blocks, warps * 32, smem, s>>>(a);
  count_launch();
}

// ================================================================================================
// K2  LDPC
// ================================================================================================
constexpr int LDPC_WARPS = 3;

// 32 stream bits starting at bit position p of a packed byte stream held as raw (little-endian loaded) words
__device__ __forceinline__ uint32_t window32_be(const uint32_t *w, int p)
{
  const int k = p >> 5;
  return __funnelshift_l(bswap32(w[k + 1]), bswap32(w[k]), p & 31);
}

// big-endian 32-bit value at byte offset `off` of a byte stream held as raw (little-endian loaded) words
__device__ __forceinline__ uint32_t be32_at(const uint32_t *w, int off)
{
  const int k = off >> 2;
  return __byte_perm(__ldg(w + k), __ldg(w + k + 1), 0x0123u + 0x1111u * (unsigned)(off & 3));
}

__global__ void __launch_bounds__(LDPC_WARPS * 32, 8) k_ldpc(const LdpcArgs a, int warp_words, int cw_words)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint32_t *s_all = reinterpret_cast<uint32_t *>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t *rows = s_all + warp * warp_words;     // [q][12] parity rows
  uint32_t *ext = rows + cw_words;                // [groups][13]
  const int q = a.q, G = a.groups;
  const int info_bytes = a.nbch / 8;

  for (int job = blockIdx.x * LDPC_WARPS + warp; job < a.frames; job += gridDim.x * LDPC_WARPS) {
    const uint8_t *in = a.in + (long long)job * a.in_pitch;
    uint8_t *out = a.out + (long long)job * a.out_pitch;
    const uint32_t *cw = reinterpret_cast<const uint32_t *>(in);      // packed BCH codeword, read through L1
    BND(a.in_len == 0 || (long long)job * a.in_pitch + 45 * G + 8 <= a.in_len);
    BND(a.out_len == 0 || (long long)job * a.out_pitch + a.nldpc / 8 <= a.out_len);
    BND(45 * G == info_bytes && warp_words >= G * 13 + q * 12);
    // ---- info bits pass through to the output
    {
      uint32_t *ow = reinterpret_cast<uint32_t *>(out);
      const int nw = info_bytes >> 2;
      for (int i = lane; i < nw; i += 256) {           // eight loads in flight per lane (their latency was 13 % of the stall samples)
        uint32_t v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = __ldg(cw + min(i + 32 * u, nw - 1));
#pragma unroll
        for (int u = 0; u < 8; u++) if (i + 32 * u < nw) ow[i + 32 * u] = v[u];
      }
      for (int b = (nw << 2) + lane; b < info_bytes; b += 32) out[b] = __ldg(in + b);
    }
    // ---- wrap-extended groups: 13 words = circular bits [0, 416) of each 360-bit group.  A group is 45 bytes, so
    // word w is the big-endian 32-bit value at byte 45 g + 4 w (w <= 10), bytes {44, 0, 1, 2} (w = 11) or bytes 3..6
    // (w = 12): unaligned loads by byte permute (bytes past the group only land in positions that are masked off)
    for (int idx0 = lane; idx0 < G * 13; idx0 += 128) {      // four words (twelve loads) in flight per lane
      uint32_t v[4], h[4];
      int wsel[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int idx = min(idx0 + 32 * u, G * 13 - 1);
        const int g = idx / 13, w = idx - g * 13;
        wsel[u] = w;
        v[u] = be32_at(cw, 45 * g + (w == 12 ? 3 : 4 * w));
        h[u] = be32_at(cw, 45 * g);                          // head of the group: completes word 11
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (idx0 + 32 * u < G * 13) ext[idx0 + 32 * u] = wsel[u] == 11 ? (v[u] & 0xFF000000u) | (h[u] >> 8) : v[u];
    }
    __syncwarp();
    // ---- pre-accumulator parity rows: R_t = XOR of rotated info groups
    if (a.lane_per_row) {
      // a lane per row, all twelve words of it: a table entry is fetched and decoded once per row instead of once
      // per word, and the window position just advances by 32 bits (mod 360) from word to word
      for (int t = lane; t < q; t += 32) {
        uint32_t acc[12];
#pragma unroll
        for (int w = 0; w < 12; w++) acc[w] = 0u;
        const int e1 = a.row_ptr[t + 1];
        for (int e = a.row_ptr[t]; e < e1; e++) {
          const uint32_t en = __ldg(a.entries + e);
          BND((int)(en & 0xffffu) < G && (en >> 16) < 360u);
          const uint32_t *eg = ext + (en & 0xffffu) * 13;
          int p = (en >> 16) ? 360 - (int)(en >> 16) : 0;
#pragma unroll
          for (int w = 0; w < 12; w++) {
            acc[w] ^= window32(eg, p);
            p += 32;
            if (p >= 360) p -= 360;
          }
        }
        acc[11] &= 0xFF000000u;
#pragma unroll
        for (int w = 0; w < 12; w++) rows[t * 12 + w] = acc[w];
      }
    }
    else
    for (int idx = lane; idx < q * 12; idx += 32) {
      const int t = idx / 12, w = idx - t * 12;
      uint32_t acc = 0;
      const int e1 = a.row_ptr[t + 1];
      int e = a.row_ptr[t];
      for (; e + 4 <= e1; e += 4) {                          // four table entries and their windows in flight
        uint32_t en[4];
#pragma unroll
        for (int u = 0; u < 4; u++) en[u] = __ldg(a.entries + e + u);
#pragma unroll
        for (int u = 0; u < 4; u++) {
          int p = 32 * w - (int)(en[u] >> 16);
          if (p < 0) p += 360;
          BND((int)(en[u] & 0xffffu) < G && (en[u] >> 16) < 360u && p >= 0 && p < 360);
          acc ^= window32(ext + (en[u] & 0xffffu) * 13, p);
        }
      }
      for (; e < e1; e++) {
        const uint32_t en = __ldg(a.entries + e);
        int p = 32 * w - (int)(en >> 16);
        if (p < 0) p += 360;
        BND((int)(en & 0xffffu) < G && (en >> 16) < 360u && p >= 0 && p < 360);
        acc ^= window32(ext + (en & 0xffffu) * 13, p);
      }
      if (w == 11) acc &= 0xFF000000u;
      rows[idx] = acc;
    }
    __syncwarp();
    // ---- accumulator, part 1: T_t = XOR_{t' <= t} R_t'  (prefix over rows, word-parallel)
    if (lane < 12) {
      uint32_t run = 0;
      for (int t = 0; t < q; t++) { run ^= rows[t * 12 + lane]; rows[t * 12 + lane] = run; }
    }
    __syncwarp();
    // ---- part 2: E = exclusive prefix-XOR along the 360 bit positions of T_{q-1}
    uint32_t E = 0;
    {
      uint32_t x = lane < 12 ? rows[(q - 1) * 12 + lane] : 0;
      x ^= x >> 1; x ^= x >> 2; x ^= x >> 4; x ^= x >> 8; x ^= x >> 16;   // inclusive, MSB first
      // carry into word w = parity of all earlier words = XOR of their last inclusive bits
      uint32_t par = x & 1u, carry = par;
#pragma unroll
      for (int d = 1; d < 16; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, carry, d);
        if (lane >= d) carry ^= o;
      }
      carry ^= par;     // exclusive over words
      E = (x >> 1) ^ (carry ? 0xFFFFFFFFu : 0u);
      if (lane == 11) E &= 0xFF000000u;
    }
    // ---- apply E, then store the parity rows: rows are 360-bit strings laid end to end after the info bits
    for (int i0 = 0; i0 < q * 12; i0 += 32) {          // warp-uniform trip count (shuffle inside)
      const int idx = i0 + lane;
      const uint32_t ew = __shfl_sync(0xffffffffu, E, idx % 12);
      if (idx < q * 12) rows[idx] ^= ew;
    }
    __syncwarp();
    if ((info_bytes & 3) == 0) {
      // word-wise: output word j holds parity bits [32 j, 32 j + 32) = a window of row t (+ the head of row t + 1)
      uint32_t *pw = reinterpret_cast<uint32_t *>(out + info_bytes);
      const int nwp = (q * 360) >> 5;                  // q * 45 bytes is a multiple of 4 only if q is; tail below
      for (int j = lane; j < nwp; j += 32) {
        const int P = j << 5;
        const int t = P / 360, o = P - t * 360;
        uint32_t v = window32(rows + t * 12, o);
        const int n1 = 360 - o;                        // bits left in row t
        if (n1 < 32) v = (v & ~(0xFFFFFFFFu >> n1)) | (rows[(t + 1) * 12] >> n1);
        pw[j] = bswap32(v);
      }
      for (int b = (nwp << 2) + lane; b < q * 45; b += 32) {
        const int t = b / 45, bb = b - t * 45;
        out[info_bytes + b] = (uint8_t)(rows[t * 12 + (bb >> 2)] >> (24 - 8 * (bb & 3)));
      }
    }
    else {
      for (int b = lane; b < q * 45; b += 32) {
        const int t = b / 45, bb = b - t * 45;
        out[info_bytes + b] = (uint8_t)(rows[t * 12 + (bb >> 2)] >> (24 - 8 * (bb & 3)));
      }
    }
    __syncwarp();
  }
}

void launch_ldpc(const LdpcArgs &a, cudaStream_t s)
{
  // per warp: extended groups + parity rows (the codeword itself is read from global memory / L1)
  const int cw_words = a.q * 12 + 4;
  const int warp_words = (a.groups * 13 + cw_words + 3) & ~3;
  const size_t smem = (size_t)LDPC_WARPS * warp_words * 4;
  if (a.frames < 1) return;
  static bool attr[MAX_DEVICES];
  allow_smem(k_ldpc, 200 * 1024, attr);
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ldpc, LDPC_WARPS * 32, smem);
  if (per_sm < 1) per_sm = 1;
  const int blocks = (a.frames + LDPC_WARPS - 1) / LDPC_WARPS;      // one FECFRAME per warp, no loop: finest tail
  k_ldpc<<<blocks, LDPC_WARPS * 32, smem, s>>>(a, warp_words, cw_words);
  count_launch();
}

// ================================================================================================
// K3  bit interleaver + demux + mapper
// ================================================================================================
// QAM path (column twist + demux): for 32 consecutive rows d of the twist matrix, column c contributes the
// 32 consecutive codeword bits u[rows*c + (d - twist[c]) mod rows] -- one funnel-shifted window of the
// packed codeword per column.  The windows are loaded in OUTPUT-bit order (demux folded into which
// column feeds which row), a 32x32 bit-matrix transpose in registers turns them into 32 cell-pair words,
// and the cells go to shared memory as bytes; the column count is a template parameter (k_map_n).  QPSK (no twist /
// demux: k_map, k_map_qtr) maps the cells whose bits sit in place in the codeword through a byte table, the parity
// cells by in-register bit transposes (k_map_qtr) or, like any other cell, bit by bit through the bit_src table.
constexpr int MAP_THREADS = 128;

template <int J>
__device__ __forceinline__ void transpose32_stage(uint32_t (&A)[32])
{
  constexpr uint32_t m = J == 16 ? 0x0000FFFFu : J == 8 ? 0x00FF00FFu : J == 4 ? 0x0F0F0F0Fu : J == 2 ? 0x33333333u : 0x55555555u;
#pragma unroll
  for (int k = 0; k < 32; k++) {
    if ((k & J) == 0) {
      const uint32_t t = (A[k] ^ (A[k + J] >> J)) & m;
      A[k] ^= t;
      A[k + J] ^= t << J;
    }
  }
}

// in-place 32x32 bit-matrix transpose (recursive block swap) in (row, MSB-first column) coordinates
__device__ __forceinline__ void transpose32(uint32_t (&A)[32])
{
  transpose32_stage<16>(A);
  transpose32_stage<8>(A);
  transpose32_stage<4>(A);
  transpose32_stage<2>(A);
  transpose32_stage<1>(A);
}

// Bit interleaver + demux + cell codes + output of FECFRAME f whose packed "u"-order codeword sits in shared memory
// (raw byte order, zero slack words behind it).  The caller has synchronised the CTA on `u`; ends without a barrier.
// QTR: the instantiation that carries the QPSK transposed-parity path (its 32-register tile would otherwise raise the
// register count of every mapper launch)
// NCOL: the column count of the twist matrix (8, 12 or 16) as a compile-time constant, 0 for QPSK (no twist matrix) --
// which rows of the bit tile are empty is then known to the compiler (the transposes shrink for 8 and 12 columns) and
// the per-bit geometry comes from the kernel-parameter constant bank (a.base_of_bit / a.twist_of_bit, compile-time
// indices).
template <bool QTR, int NCOL = 0>
__device__ __forceinline__ void map_body(const MapArgs &a, const int f, const uint32_t *u, const float2 *lut, uint16_t *cw,
                                         const int shift)
{
  const int mod = a.mod, Nc = a.cell_size;
  // single-table constellation (MapPlan::im_from_re): the byte that supplies the imaginary part is kept as w~
  const bool tilde = a.im_from_re != 0;
  const uint32_t tI = a.im_mask_i * 0x01010101u, tQ = a.im_mask_q * 0x01010101u, tF = a.im_flip * 0x01010101u;
  auto tilde4 = [&](uint32_t w) -> uint32_t { return tilde ? ((((w << 1) & tI) | ((w >> 1) & tQ)) ^ tF) : w; };   // four packed cell words
  auto tilde1 = [&](uint32_t w) -> uint32_t { return tilde4(w) & 0xFFu; };
  if constexpr (NCOL != 0) {
    const int rows = a.nldpc / NCOL;
    const int groups = (rows + 31) >> 5;
    for (int g = threadIdx.x; g < groups; g += blockDim.x) {
      const int d0 = g << 5;
      uint32_t A[32];
#pragma unroll
      for (int y = 0; y < 32; y++) A[y] = 0;
#pragma unroll
      for (int y = 16; y < 32; y++) {
        const int rho = y - (32 - NCOL);       // output bit (0 = MSB of the NCOL-bit demux word) held by row y
        if (rho >= 0) {
          int s0 = d0 - a.twist_of_bit[rho];
          if (s0 < 0) s0 += rows;
          const int base = a.base_of_bit[rho];
          const int n1 = rows - s0;
          uint32_t w = window32_be(u, base + s0);
          if (n1 < 32) w = (w & ~(0xFFFFFFFFu >> n1)) | (window32_be(u, base) >> n1);
          A[y] = w;
        }
      }
      transpose32(A);
      // transpose32 uses (row, MSB-first column) coordinates: window bit i (from the MSB) of row y moves to
      // bit y (from the MSB) of A[i], so A[i] is the NCOL-bit word of row d0 + i of the twist matrix.
      // Emit cells (two per word when NCOL = 2 mod, else one) as packed bytes.
      // Four consecutive cells as bytes w = [c0 c1 c2 c3] (c0 lowest), then their codes by byte permutes: with
      // the Q delay [c0 | prev << 8, c1 | c0 << 8], [c2 | c1 << 8, c3 | c2 << 8] (prev = c3 of the previous
      // four; the first cell of the thread is patched below), without it [c0 | c0 << 8, ...].
      const uint32_t mask = (1u << mod) - 1u;
      // X = the four words supplying the imaginary parts (as w~): the previous cell's under the Q delay, else the own
      const int xs = a.cyclic_delay ? 8 : 0;
      uint32_t wprev = 0;
      if (NCOL == 2 * mod) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(cw + 2 * d0 + 2 * g);      // 64 cells + 1 pad word per thread
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const uint32_t p0 = A[i], p1 = A[i + 1];
          const uint32_t w = (p0 >> mod) | ((p0 & mask) << 8) | ((p1 >> mod) << 16) | ((p1 & mask) << 24);
          const uint32_t wt = tilde4(w), X = __funnelshift_l(wprev, wt, xs);
          dst[i] = __byte_perm(w, X, 0x5140u);
          dst[i + 1] = __byte_perm(w, X, 0x7362u);
          wprev = wt;
        }
      }
      else {
        uint32_t *dst = reinterpret_cast<uint32_t *>(cw + d0 + 2 * (g >> 1));   // 32 cells per thread, pad per 64
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const uint32_t w = (A[i] & mask) | ((A[i + 1] & mask) << 8) | ((A[i + 2] & mask) << 16) | ((A[i + 3] & mask) << 24);
          const uint32_t wt = tilde4(w), X = __funnelshift_l(wprev, wt, xs);
          dst[i >> 1] = __byte_perm(w, X, 0x5140u);
          dst[(i >> 1) + 1] = __byte_perm(w, X, 0x7362u);
          wprev = wt;
        }
      }
    }
    if (a.cyclic_delay) {
      // first cell of every thread's run: the imaginary part comes from the last cell of the previous run
      __syncthreads();
      const int run = NCOL == 2 * mod ? 64 : 32;
      for (int c = threadIdx.x * run; c < Nc; c += blockDim.x * run) {
        const int pc = c == 0 ? Nc - 1 : c - 1;
        reinterpret_cast<uint8_t *>(cw)[2 * (c + 2 * (c >> 6)) + 1] = (uint8_t)tilde1(cw[pc + 2 * (pc >> 6)]);
      }
    }
  }
  else if (mod == 2 && (Nc & 3) == 0) {
    // QPSK: four cells per step -- their eight source bit positions are one 16-byte load
    const uint8_t *ub = reinterpret_cast<const uint8_t *>(u);
    // cells whose bits sit in place in the codeword (the info part; everything for the parity-interleaved codes): a
    // 32-bit word is sixteen cells, each byte's four codes come from one 8-byte table entry
    const int lin = a.qpsk_lin_cells;
    for (int wi = threadIdx.x; wi < (lin >> 4); wi += blockDim.x) {
      const uint32_t W = u[wi];                      // raw byte order: byte k of the stream is bits 8k..8k+7
      uint32_t *dst = reinterpret_cast<uint32_t *>(cw + 16 * wi + 2 * (wi >> 2));
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const uint2 cd = __ldg(a.qpsk_lut + ((W >> (8 * k)) & 255u));
        dst[2 * k] = cd.x;
        dst[2 * k + 1] = cd.y;
      }
    }
    // cells [lin, gen_end) go bit by bit through bit_src; with the transposed parity path that is only the few info
    // cells behind the last whole table word
    const int gen_end = QTR && a.qpsk_par_q > 0 ? (a.qpsk_nbch >> 1) : Nc;
    for (int c = lin + 4 * threadIdx.x; c < gen_end; c += 4 * blockDim.x) {
      const uint4 pp = __ldg(reinterpret_cast<const uint4 *>(a.bit_src) + (c >> 2));
      const uint32_t w[4] = { pp.x, pp.y, pp.z, pp.w };
      uint32_t code[4];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const uint32_t p0 = w[k] & 0xFFFFu, p1 = w[k] >> 16;
        const uint32_t v = (((ub[p0 >> 3] >> (7 - (p0 & 7))) & 1u) << 1) | ((ub[p1 >> 3] >> (7 - (p1 & 7))) & 1u);
        code[k] = v | (tilde1(v) << 8);
      }
      uint32_t *dst = reinterpret_cast<uint32_t *>(cw + c + 2 * (c >> 6));
      dst[0] = code[0] | (code[1] << 16);
      dst[1] = code[2] | (code[3] << 16);
    }
    if (QTR && a.qpsk_par_q > 0) {
      // parity cells: natural parity bit q s + t is codeword bit nbch + 360 t + s, a q x 360 bit-matrix transpose.
      // One thread per 32 x 32 tile: 32 row windows -> register transpose -> 32 column pieces; once every tile is in
      // registers the (spent) info words of `u` become the natural-order parity stream, pieces OR-ed in at their bit
      // offsets, and the byte table maps it like the info part.
      const int q = a.qpsk_par_q, nbch = a.qpsk_nbch, par0 = nbch >> 1;
      const int tr = (q + 31) >> 5;                      // tile rows; 12 tile columns (360 = 11.25 x 32)
      const bool have = (int)threadIdx.x < tr * 12;
      const int t0 = ((int)threadIdx.x / 12) << 5, s0 = ((int)threadIdx.x % 12) << 5;
      uint32_t A[32];
      if (have) {
#pragma unroll
        for (int y = 0; y < 32; y++) A[y] = t0 + y < q ? window32_be(u, nbch + 360 * (t0 + y) + s0) : 0u;
        transpose32(A);                                   // A[i]: column s0 + i, row t0 + y at bit 31 - y
      }
      __syncthreads();                                    // everyone is done with the info words, all tiles are in registers
      uint32_t *nat = const_cast<uint32_t *>(u);          // big-endian bit stream: natural parity bit P at word P / 32, bit 31 - P % 32
      const int nat_words = ((q * 360 + 31) >> 5) + 1;
      for (int i = threadIdx.x; i < nat_words; i += blockDim.x) nat[i] = 0u;
      __syncthreads();
      if (have) {
        const int nv = min(32, q - t0);
        const uint32_t vmask = nv >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu >> nv);
#pragma unroll
        for (int i = 0; i < 32; i++) {
          if (s0 + i < 360) {
            const uint32_t word = A[i] & vmask;
            const int P = q * (s0 + i) + t0, sh = P & 31;
            atomicOr(nat + (P >> 5), word >> sh);
            if (sh) atomicOr(nat + (P >> 5) + 1, word << (32 - sh));
          }
        }
      }
      __syncthreads();
      const int npar = Nc - par0;                          // parity cells
      for (int wi = threadIdx.x; wi < ((npar + 15) >> 4); wi += blockDim.x) {
        const uint32_t W = nat[wi];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int c = par0 + 16 * wi + 4 * k;
          if (c < Nc) {
            const uint2 cd = __ldg(a.qpsk_lut + ((W >> (24 - 8 * k)) & 255u));
            uint32_t *dst = reinterpret_cast<uint32_t *>(cw + c + 2 * (c >> 6));
            dst[0] = cd.x;
            dst[1] = cd.y;
          }
        }
      }
    }
    if (a.cyclic_delay) {
      __syncthreads();
      for (int c = threadIdx.x; c < Nc; c += blockDim.x) {
        const int pc = c == 0 ? Nc - 1 : c - 1;
        reinterpret_cast<uint8_t *>(cw)[2 * (c + 2 * (c >> 6)) + 1] = (uint8_t)tilde1(cw[pc + 2 * (pc >> 6)]);
      }
    }
  }
  else {
    for (int c = threadIdx.x; c < Nc; c += blockDim.x) {
      const uint16_t *src = a.bit_src + c * mod;
      uint32_t v = 0;
      for (int b = 0; b < mod; b++) {
        const int p = __ldg(src + b);
        v = (v << 1) | ((reinterpret_cast<const uint8_t *>(u)[p >> 3] >> (7 - (p & 7))) & 1u);
      }
      cw[c + 2 * (c >> 6)] = (uint16_t)(v | (tilde1(v) << 8));
    }
    if (a.cyclic_delay) {
      __syncthreads();
      // only high bytes are written and only low bytes read: no ordering needed between the threads
      for (int c = threadIdx.x; c < Nc; c += blockDim.x) {
        const int pc = c == 0 ? Nc - 1 : c - 1;
        reinterpret_cast<uint8_t *>(cw)[2 * (c + 2 * (c >> 6)) + 1] = (uint8_t)tilde1(cw[pc + 2 * (pc >> 6)]);
      }
    }
  }
  __syncthreads();
  auto code = [&](int c) -> unsigned { return cw[c + 2 * (c >> 6)]; };     // padded layout, see above
  float2 *out = a.out + (long long)f * Nc;
  if (a.out16) {
    // chain mode: the 16-bit codes in cell-interleaved order: cell ci_inv[y] goes to position (y + shift) mod Nc.
    // Two segments with a constant position - y, so table reads and stores are a base pointer + constant offsets.
    uint16_t *o16 = a.out16 + (long long)(f / a.fecblocks) * a.out16_frame_stride + (long long)(f % a.fecblocks) * Nc;
    if (a.ci_inv4) {
      // four cells per step: destinations taken in aligned groups of four (one 8-byte store); their four permutation
      // entries are one 8-byte load from the copy of the table that is shifted by the group's source phase
      // (ci_inv4[k][j] = ci_inv[j + k]); ragged ends of a segment go cell by cell
      const long long a0 = o16 - a.out16;                     // absolute cell index of destination 0 (a.out16 is 16-byte aligned)
#pragma unroll 1
      for (int seg = 0; seg < 2; seg++) {
        const int y_beg = seg ? Nc - shift : 0, y_end = seg ? Nc : Nc - shift;
        const int dofs = seg ? shift - Nc : shift;            // destination = y + dofs
        if (y_end <= y_beg) continue;
        const int head = (int)((4 - ((a0 + y_beg + dofs) & 3)) & 3);
        const int yv = min(y_end, y_beg + head);              // first y of the aligned part
        const int ngrp = (y_end - yv) >> 2;
        const int k = yv & 3;                                 // source phase of every group
        const uint2 *ci4 = reinterpret_cast<const uint2 *>(a.ci_inv4 + (long long)k * a.ci_inv4_stride + (yv - k));
        uint2 *ov = reinterpret_cast<uint2 *>(o16 + yv + dofs);
        // the shifted copies hold the PADDED index c + 2 (c / 64) of each cell: no index arithmetic per look-up
        auto emit4 = [&](int g, const uint2 ci) {
          const unsigned c0 = ci.x & 0xFFFFu, c1 = ci.x >> 16, c2 = ci.y & 0xFFFFu, c3 = ci.y >> 16;
          BND((int)c0 < Nc + 2 * (Nc >> 6) + 2 && (int)c1 < Nc + 2 * (Nc >> 6) + 2 && (int)c2 < Nc + 2 * (Nc >> 6) + 2 && (int)c3 < Nc + 2 * (Nc >> 6) + 2);
          BND(a.out_len == 0 || (a0 + yv + dofs + 4ll * g >= 0 && a0 + yv + dofs + 4ll * g + 4 <= a.out_len));
          ov[g] = make_uint2((unsigned)cw[c0] | ((unsigned)cw[c1] << 16), (unsigned)cw[c2] | ((unsigned)cw[c3] << 16));
        };
        // the permutation entries come from L2 (the CTAs' shared memory leaves almost no L1).  The QPSK instantiation
        // (three CTAs per SM: little else to hide the round trip behind) keeps four requests in flight per thread
        // (c2: mapper 0.071 -> 0.064 ms); with eight CTAs per SM the same batching is 5 % SLOWER (c3: 0.137 -> 0.144), so
        // the QAM instantiation keeps the two-deep unrolled loop
        int g = threadIdx.x;
        if (QTR)
        for (; g + 3 * MAP_THREADS < ngrp; g += 4 * MAP_THREADS) {
          uint2 ci[4];
#pragma unroll
          for (int k4 = 0; k4 < 4; k4++) ci[k4] = __ldg(ci4 + g + k4 * MAP_THREADS);
#pragma unroll
          for (int k4 = 0; k4 < 4; k4++) emit4(g + k4 * MAP_THREADS, ci[k4]);
        }
#pragma unroll 2
        for (; g < ngrp; g += MAP_THREADS) emit4(g, __ldg(ci4 + g));
        // ragged ends: up to 3 cells before and after the aligned part
        const int tail0 = yv + 4 * ngrp;
        const int nrag = (yv - y_beg) + (y_end - tail0);
        if ((int)threadIdx.x < nrag) {
          const int y = (int)threadIdx.x < yv - y_beg ? y_beg + threadIdx.x : tail0 + (threadIdx.x - (yv - y_beg));
          o16[y + dofs] = (uint16_t)code(__ldg(a.ci_inv + y));
        }
      }
    }
    else {
#pragma unroll 1
    for (int seg = 0; seg < 2; seg++) {
      const int y_end = seg ? Nc : Nc - shift;
      uint16_t *o = o16 + (seg ? shift - Nc : shift);
      // eight permutation look-ups in flight per thread
#pragma unroll 1
      for (int y0 = (seg ? Nc - shift : 0) + threadIdx.x; y0 < y_end; y0 += 8 * MAP_THREADS) {
        const uint16_t *ci = a.ci_inv + y0;
        uint16_t *oy = o + y0;
        const int left = y_end - y0;
        int c[8];
#pragma unroll
        for (int k = 0; k < 8; k++) c[k] = k * MAP_THREADS < left ? __ldg(ci + k * MAP_THREADS) : 0;
#pragma unroll
        for (int k = 0; k < 8; k++)
          if (k * MAP_THREADS < left) oy[k * MAP_THREADS] = (uint16_t)code(c[k]);
      }
    }
    }
  }
  else if (a.ci_inv) {
    // fused cell interleaver with complex output
    for (int xo = threadIdx.x; xo < Nc; xo += blockDim.x) {
      int y = xo - shift;
      if (y < 0) y += Nc;
      const unsigned cd = code(__ldg(a.ci_inv + y));
      out[xo] = make_float2(lut[cd & 255u].x, tilde ? lut[cd >> 8].x : lut[cd >> 8].y);
    }
  }
  else {
    // drop-in block: complex64 cells in natural order, two cells per 16-byte store (the first cell of a FECFRAME that
    // starts on an odd cell and a last odd one go alone)
    auto cell = [&](int c) -> float2 {
      const unsigned cd = code(c);
      return make_float2(lut[cd & 255u].x, tilde ? lut[cd >> 8].x : lut[cd >> 8].y);
    };
    const int head = (int)(((long long)f * Nc) & 1);
    const int npair = (Nc - head) >> 1;
    if ((reinterpret_cast<uintptr_t>(a.out) & 15) == 0) {
      float4 *o4 = reinterpret_cast<float4 *>(out + head);
      for (int pr = threadIdx.x; pr < npair; pr += blockDim.x) {
        const float2 c0 = cell(head + 2 * pr), c1 = cell(head + 2 * pr + 1);
        o4[pr] = make_float4(c0.x, c0.y, c1.x, c1.y);
      }
      if (threadIdx.x == 0 && head) out[0] = cell(0);
      if (threadIdx.x == 32 && head + 2 * npair < Nc) out[Nc - 1] = cell(Nc - 1);
    }
    else
    for (int c = threadIdx.x; c < Nc; c += blockDim.x) out[c] = cell(c);
  }
}

// shared-memory words of the mapper part: codeword (+ slack), constellation table, padded cell codes
__host__ __device__ inline int map_u_words(int nldpc) { return (((nldpc + 31) / 32) + 11) & ~3; }
__host__ __device__ inline int map_cw_halfwords(int cell_size) { return ((cell_size + 127) & ~63) + 2 * (cell_size / 64 + 2); }

template <bool QTR, int NCOL = 0>
__device__ __forceinline__ void k_map_impl(const MapArgs &a)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int nwords = (a.nldpc + 31) / 32;
  uint32_t *u = reinterpret_cast<uint32_t *>(smem_raw);                   // packed codeword, raw byte order, + slack
  float2 *lut = reinterpret_cast<float2 *>(u + map_u_words(a.nldpc));     // [1 << mod]
  // cell codes of the FECFRAME: own cell word | (word supplying the imaginary part << 8), i.e. the previous cell's
  // word under the cyclic Q delay, the cell's own otherwise.  Padded: cell c at index c + 2 (c / 64).
  uint16_t *cw = reinterpret_cast<uint16_t *>(lut + (1 << a.mod));
  // packed codeword into shared memory as raw bytes with 16-byte asynchronous copies (frames are 16-byte pitched)
  const int n16 = (nwords + 3) >> 2;
  auto fetch = [&](int f) {
    const uint8_t *in = a.in + (long long)f * a.in_pitch;
    const unsigned dst0 = (unsigned)__cvta_generic_to_shared(u);
    for (int i = threadIdx.x; i < n16; i += MAP_THREADS)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst0 + 16u * i), "l"(in + 16 * i));
    asm volatile("cp.async.commit_group;\n" ::);
  };
  // the CTA's first codeword is requested before the tables are set up: one exposed global round trip instead of two
  if ((int)blockIdx.x < a.frames) fetch(blockIdx.x);
  // (the constellation table is only read by the complex64 output of the drop-in block: the chain's 16-bit codes skip it)
  if (!a.out16)
    for (int i = threadIdx.x; i < (1 << a.mod); i += blockDim.x) lut[i] = a.lut[i];

  for (int f = blockIdx.x; f < a.frames; f += gridDim.x) {
    const int shift = a.fec_shift ? __ldg(a.fec_shift + f % a.fecblocks) : 0;     // requested early: used by the last stage
    if (f != (int)blockIdx.x) {
      __syncthreads();                    // the previous frame's body has finished with u
      fetch(f);
    }
    asm volatile("cp.async.wait_group 0;\n" ::);
    if (threadIdx.x < 4) u[4 * n16 + threadIdx.x] = 0u;
    __syncthreads();
    map_body<QTR, NCOL>(a, f, u, lut, cw, shift);
  }
}
// QPSK (no twist matrix)
__global__ void __launch_bounds__(MAP_THREADS) k_map(const MapArgs a) { k_map_impl<false>(a); }
// 8, 12 or 16 twist-matrix columns as a compile-time constant (16QAM / short 256QAM, 64QAM, normal 256QAM)
template <int NCOL>
__global__ void __launch_bounds__(MAP_THREADS) k_map_n(const MapArgs a) { k_map_impl<false, NCOL>(a); }
// QPSK with the transposed parity path: three CTAs per SM fit beside the 32400 cell codes of a normal FECFRAME
__global__ void __launch_bounds__(MAP_THREADS, 3) k_map_qtr(const MapArgs a) { k_map_impl<true>(a); }

void launch_map(const MapArgs &a, cudaStream_t s)
{
  const size_t smem = (size_t)map_u_words(a.nldpc) * 4 + (size_t)(1 << a.mod) * 8 + 2 * (size_t)map_cw_halfwords(a.cell_size);
  // one FECFRAME per CTA: the hardware scheduler balances the tail at frame granularity
  const int blocks = a.frames;
  if (blocks < 1) return;
  static bool attr[MAX_DEVICES], attr_q[MAX_DEVICES];
  allow_smem(k_map, 100 * 1024, attr);      // QPSK normal: 32400 cell codes
  allow_smem(k_map_qtr, 100 * 1024, attr_q);
  const bool qtr = a.qpsk_par_q > 0 && a.mod == 2 && a.ncol == 0 && (a.cell_size & 3) == 0;
  if (!qtr && (a.ncol == 8 || a.ncol == 12 || a.ncol == 16)) {
    MapArgs b = a;
    const int rows = a.nldpc / a.ncol;
    for (int rho = 0; rho < 16; rho++) {
      const int col = rho < a.ncol ? a.col_of_bit[rho] : 0;
      b.base_of_bit[rho] = rows * col;
      b.twist_of_bit[rho] = a.twist_of_col[col];
    }
    static bool attr_n[3][MAX_DEVICES];
    if (a.ncol == 8) { allow_smem(k_map_n<8>, 100 * 1024, attr_n[0]); k_map_n<8><<<blocks, MAP_THREADS, smem, s>>>(b); }
    else if (a.ncol == 12) { allow_smem(k_map_n<12>, 100 * 1024, attr_n[1]); k_map_n<12><<<blocks, MAP_THREADS, smem, s>>>(b); }
    else { allow_smem(k_map_n<16>, 100 * 1024, attr_n[2]); k_map_n<16><<<blocks, MAP_THREADS, smem, s>>>(b); }
    count_launch();
    return;
  }
  if (qtr) k_map_qtr<<<blocks, MAP_THREADS, smem, s>>>(a);
  else k_map<<<blocks, MAP_THREADS, smem, s>>>(a);
  count_launch();
}

// ================================================================================================
// bit format helpers
// ================================================================================================
__global__ void k_pack_bits(const uint8_t *in, int nbits, uint8_t *out, int out_pitch, int frames)
{
  const int nbytes = (nbits + 7) / 8;
  const long long total = (long long)frames * nbytes;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i / nbytes), b = (int)(i - (long long)f * nbytes);
    const uint8_t *p = in + (long long)f * nbits + 8 * b;
    uint32_t v = 0;
    for (int k = 0; k < 8; k++) v = (v << 1) | ((8 * b + k < nbits) ? (p[k] & 1u) : 0u);
    out[(long long)f * out_pitch + b] = (uint8_t)v;
  }
}

__global__ void k_unpack_bits(const uint8_t *in, int in_pitch, int nbits, uint8_t *out, int frames)
{
  const long long total = (long long)frames * nbits;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i / nbits), b = (int)(i - (long long)f * nbits);
    out[i] = (in[(long long)f * in_pitch + (b >> 3)] >> (7 - (b & 7))) & 1u;
  }
}

__global__ void k_unpack_ldpc(const uint8_t *in, int in_pitch, int nbch, int nldpc, int q, uint8_t *out, int frames)
{
  const long long total = (long long)frames * nldpc;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i / nldpc), b = (int)(i - (long long)f * nldpc);
    int p = b;
    if (b >= nbch) { const int x = b - nbch; p = nbch + 360 * (x % q) + x / q; }
    out[i] = (in[(long long)f * in_pitch + (p >> 3)] >> (7 - (p & 7))) & 1u;
  }
}

__global__ void k_pack_ldpc(const uint8_t *in, int nbch, int nldpc, int q, uint8_t *out, int out_pitch, int frames)
{
  const int nbytes = nldpc / 8;
  const long long total = (long long)frames * nbytes;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i / nbytes), b = (int)(i - (long long)f * nbytes);
    const uint8_t *fr = in + (long long)f * nldpc;
    uint32_t v = 0;
    for (int k = 0; k < 8; k++) {
      const int p = 8 * b + k;          // position in "u" order
      int n = p;                        // natural index
      if (p >= nbch) { const int x = p - nbch; n = nbch + q * (x % 360) + x / 360; }
      v = (v << 1) | (fr[n] & 1u);
    }
    out[(long long)f * out_pitch + b] = (uint8_t)v;
  }
}

// ---- the same conversions, vectorised (HBM-bound: 1 byte per bit on one side).  Frames are multiples of 8 bits, so with
// 8-byte aligned buffers every 8 one-bit bytes are one aligned 8-byte access; the byte <-> 8 bytes conversion is a
// multiply that moves each bit to its place (no carries: all partial products land on distinct bits).
// eight one-bit bytes (first = most significant) -> one byte
__device__ __forceinline__ uint32_t pack8(uint2 v)
{
  return ((((v.x & 0x01010101u) * 0x08040201u) >> 24) << 4) | (((v.y & 0x01010101u) * 0x08040201u) >> 24);
}
// one byte -> eight one-bit bytes (most significant bit first)
__device__ __forceinline__ uint2 unpack8(uint32_t b)
{
  // nibble n = b0 b1 b2 b3: (n * 0x00204081) & 0x01010101 has b3, b2, b1, b0 in bytes 0..3; the byte permute reverses them
  return make_uint2(__byte_perm(((b >> 4) * 0x00204081u) & 0x01010101u, 0u, 0x0123u),
                    __byte_perm(((b & 15u) * 0x00204081u) & 0x01010101u, 0u, 0x0123u));
}
// pack / unpack of the first nbits (a multiple of 8) of a frame: a thread per packed byte, so that a warp's 8-byte
// accesses on the one-bit side are 256 contiguous bytes (four independent ones in flight per thread)
__device__ __forceinline__ void pack_span(const uint8_t *src, int nbits, uint8_t *dst)
{
  const int nb = nbits >> 3, T = blockDim.x;
  const uint2 *s8 = reinterpret_cast<const uint2 *>(src);
  int b = threadIdx.x;
  for (; b + 3 * T < nb; b += 4 * T) {
    const uint2 v0 = __ldg(s8 + b), v1 = __ldg(s8 + b + T), v2 = __ldg(s8 + b + 2 * T), v3 = __ldg(s8 + b + 3 * T);
    dst[b] = (uint8_t)pack8(v0); dst[b + T] = (uint8_t)pack8(v1); dst[b + 2 * T] = (uint8_t)pack8(v2); dst[b + 3 * T] = (uint8_t)pack8(v3);
  }
  for (; b < nb; b += T) dst[b] = (uint8_t)pack8(__ldg(s8 + b));
}
__device__ __forceinline__ void unpack_span(const uint8_t *src, int nbits, uint8_t *dst)
{
  const int nb = nbits >> 3, T = blockDim.x;
  uint2 *d8 = reinterpret_cast<uint2 *>(dst);
  int b = threadIdx.x;
  for (; b + 3 * T < nb; b += 4 * T) {
    const uint32_t v0 = src[b], v1 = src[b + T], v2 = src[b + 2 * T], v3 = src[b + 3 * T];
    d8[b] = unpack8(v0); d8[b + T] = unpack8(v1); d8[b + 2 * T] = unpack8(v2); d8[b + 3 * T] = unpack8(v3);
  }
  for (; b < nb; b += T) d8[b] = unpack8(src[b]);
}

__global__ void __launch_bounds__(256) k_pack_bits_v(const uint8_t *in, int nbits, uint8_t *out, int out_pitch, int frames)
{
  for (int f = blockIdx.x; f < frames; f += gridDim.x) pack_span(in + (long long)f * nbits, nbits, out + (long long)f * out_pitch);
}

__global__ void __launch_bounds__(256) k_unpack_bits_v(const uint8_t *in, int in_pitch, int nbits, uint8_t *out, int frames)
{
  for (int f = blockIdx.x; f < frames; f += gridDim.x) unpack_span(in + (long long)f * in_pitch, nbits, out + (long long)f * nbits);
}

// LDPC codeword, packed "u" order -> natural order, 1 bit per byte.  The q x 360 parity bit matrix is transposed through
// shared memory: a thread takes one packed byte (row t, columns 8 k .. 8 k + 7), expands it with one multiply per nibble
// and writes the eight one-bit bytes to their natural places q (8 k + j) + t of a shared-memory image of the parity part
// (lanes on consecutive rows: consecutive bytes); the image then leaves with 8-byte stores.
__global__ void __launch_bounds__(256) k_unpack_ldpc_v(const uint8_t *in, int in_pitch, int nbch, int nldpc, int q, uint8_t *out, int frames)
{
  extern __shared__ __align__(16) uint8_t sm_fmt[];
  const int npar = nldpc - nbch, ib = nbch >> 3;
  uint8_t *sp = sm_fmt;                      // npar one-bit bytes, natural order
  for (int f = blockIdx.x; f < frames; f += gridDim.x) {
    const uint8_t *src = in + (long long)f * in_pitch;
    uint8_t *o = out + (long long)f * nldpc;
    for (int i = threadIdx.x; i < q * 45; i += blockDim.x) {
      const int k = i / q, t = i - k * q;
      const uint2 e = unpack8(src[ib + 45 * t + k]);
      uint8_t *d = sp + q * 8 * k + t;
      d[0] = (uint8_t)e.x; d[q] = (uint8_t)(e.x >> 8); d[2 * q] = (uint8_t)(e.x >> 16); d[3 * q] = (uint8_t)(e.x >> 24);
      d[4 * q] = (uint8_t)e.y; d[5 * q] = (uint8_t)(e.y >> 8); d[6 * q] = (uint8_t)(e.y >> 16); d[7 * q] = (uint8_t)(e.y >> 24);
    }
    unpack_span(src, nbch, o);
    __syncthreads();
    uint2 *d8 = reinterpret_cast<uint2 *>(o + nbch);
    for (int i = threadIdx.x; i < (npar >> 3); i += blockDim.x) d8[i] = reinterpret_cast<const uint2 *>(sp)[i];
    __syncthreads();
  }
}

// natural-order codeword, 1 bit per byte -> packed "u" order: parity bytes staged in shared memory by 8-byte loads, a
// thread packs the eight bits of one byte of a parity row (lanes on consecutive rows: consecutive shared-memory bytes)
__global__ void __launch_bounds__(256) k_pack_ldpc_v(const uint8_t *in, int nbch, int nldpc, int q, uint8_t *out, int out_pitch, int frames)
{
  extern __shared__ __align__(16) uint8_t sm_fmt[];
  const int npar = nldpc - nbch, ib = nbch >> 3;
  uint8_t *sp = sm_fmt, *so = sm_fmt + npar;
  for (int f = blockIdx.x; f < frames; f += gridDim.x) {
    const uint8_t *fr = in + (long long)f * nldpc;
    uint8_t *o = out + (long long)f * out_pitch;
    {
      const uint2 *s8 = reinterpret_cast<const uint2 *>(fr + nbch);
      uint2 *d8 = reinterpret_cast<uint2 *>(sp);
      const int n8 = npar >> 3, T = blockDim.x;
      int i = threadIdx.x;
      for (; i + 3 * T < n8; i += 4 * T) {         // four loads in flight per thread
        const uint2 v0 = __ldg(s8 + i), v1 = __ldg(s8 + i + T), v2 = __ldg(s8 + i + 2 * T), v3 = __ldg(s8 + i + 3 * T);
        d8[i] = v0; d8[i + T] = v1; d8[i + 2 * T] = v2; d8[i + 3 * T] = v3;
      }
      for (; i < n8; i += T) d8[i] = __ldg(s8 + i);
    }
    pack_span(fr, nbch, o);
    __syncthreads();
    for (int i = threadIdx.x; i < q * 45; i += blockDim.x) {
      const int k = i / q, t = i - k * q;
      const uint8_t *col = sp + q * 8 * k + t;
      uint32_t v = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) v = (v << 1) | (col[q * j] & 1u);
      so[45 * t + k] = (uint8_t)v;
    }
    __syncthreads();
    for (int b = threadIdx.x; b < q * 45; b += blockDim.x) o[ib + b] = so[b];
    __syncthreads();
  }
}

static inline bool aligned8(const void *a, const void *b) { return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 7) == 0; }
static inline int frame_grid(int frames)
{
  const int cap = sm_count() * 16;
  return frames < cap ? frames : cap;
}

static inline int grid_for(long long total, int threads)
{
  long long b = (total + threads - 1) / threads;
  const long long cap = (long long)sm_count() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

void launch_pack_bits(const uint8_t *in, int nbits, uint8_t *out, int out_pitch, int frames, cudaStream_t s)
{
  if (frames < 1) return;
  if ((nbits & 7) == 0 && (out_pitch & 3) == 0 && aligned8(in, out)) k_pack_bits_v<<<frame_grid(frames), 256, 0, s>>>(in, nbits, out, out_pitch, frames);
  else
  k_pack_bits<<<grid_for((long long)frames * ((nbits + 7) / 8), 256), 256, 0, s>>>(in, nbits, out, out_pitch, frames);
  count_launch();
}
void launch_unpack_bits(const uint8_t *in, int in_pitch, int nbits, uint8_t *out, int frames, cudaStream_t s)
{
  if (frames < 1) return;
  if ((nbits & 7) == 0 && (in_pitch & 3) == 0 && aligned8(in, out)) k_unpack_bits_v<<<frame_grid(frames), 256, 0, s>>>(in, in_pitch, nbits, out, frames);
  else
  k_unpack_bits<<<grid_for((long long)frames * nbits, 256), 256, 0, s>>>(in, in_pitch, nbits, out, frames);
  count_launch();
}
void launch_unpack_ldpc(const uint8_t *in, int in_pitch, int nbch, int nldpc, int q, uint8_t *out, int frames, cudaStream_t s)
{
  if (frames < 1) return;
  const bool shape_ok = (nbch & 7) == 0 && (nldpc & 7) == 0 && nldpc - nbch == 360 * q && nldpc - nbch <= 44 * 1024;
  if (shape_ok && (in_pitch & 3) == 0 && aligned8(in, out))
    k_unpack_ldpc_v<<<frame_grid(frames), 256, (size_t)(nldpc - nbch), s>>>(in, in_pitch, nbch, nldpc, q, out, frames);
  else
  k_unpack_ldpc<<<grid_for((long long)frames * nldpc, 256), 256, 0, s>>>(in, in_pitch, nbch, nldpc, q, out, frames);
  count_launch();
}
void launch_pack_ldpc(const uint8_t *in, int nbch, int nldpc, int q, uint8_t *out, int out_pitch, int frames, cudaStream_t s)
{
  if (frames < 1) return;
  const int npar = nldpc - nbch;
  const bool shape_ok = (nbch & 7) == 0 && (nldpc & 7) == 0 && npar == 360 * q && npar + npar / 8 <= 44 * 1024;
  if (shape_ok && (out_pitch & 3) == 0 && aligned8(in, out))
    k_pack_ldpc_v<<<frame_grid(frames), 256, (size_t)npar + npar / 8, s>>>(in, nbch, nldpc, q, out, out_pitch, frames);
  else
  k_pack_ldpc<<<grid_for((long long)frames * (nldpc / 8), 256), 256, 0, s>>>(in, nbch, nldpc, q, out, out_pitch, frames);
  count_launch();
}

// ================================================================================================
// K4  frame mapper gather
// ================================================================================================
__device__ __forceinline__ float2 fetch_cell(int code, const float2 *__restrict__ cells, const float2 *__restrict__ pool,
                                            int l1post_base, int l1post_cells, int variant)
{
  if (code >= 0) return __ldg(cells + code);
  int idx = -(code + 1);
  if ((unsigned)(idx - l1post_base) < (unsigned)l1post_cells) idx += variant * l1post_cells;
  return __ldg(pool + idx);
}

// address of the cell a code stands for (the load itself is left to the caller, so that a thread's loads are independent)
__device__ __forceinline__ const float2 *cell_ptr(int code, const float2 *__restrict__ cells, const float2 *__restrict__ pool,
                                                 int l1post_base, int l1post_cells, int variant)
{
  if (code >= 0) return cells + code;
  int idx = -(code + 1);
  if ((unsigned)(idx - l1post_base) < (unsigned)l1post_cells) idx += variant * l1post_cells;
  return pool + idx;
}

// One thread: two consecutive output cells of FPB T2 frames.  The code pair is one 8-byte load shared by the FPB frames,
// the 2 * FPB gathers (random 8-byte reads: the composed cell / time / frequency interleavers leave no locality) are all
// in flight before the first store, and a store is 16 bytes (V16: frames start on even cells).  Frames are walked in
// chunks of FPB by blockIdx.y, so the input cells of the chunk in flight (FPB x 13 MB for c3) stay in L2 while their
// four cells per 32-byte sector are picked up.
template <int FPB, bool V16>
__global__ void __launch_bounds__(256) k_gather(const GatherArgs a)
{
  const int npair = a.n >> 1;
  for (int f0 = blockIdx.y * FPB; f0 < a.frames; f0 += gridDim.y * FPB) {
    for (int pr = blockIdx.x * 256 + threadIdx.x; pr < npair; pr += gridDim.x * 256) {
      const int2 cd = __ldg(reinterpret_cast<const int2 *>(a.code) + pr);
      float2 v0[FPB], v1[FPB];
#pragma unroll
      for (int k = 0; k < FPB; k++) {
        const int f = f0 + k;
        if (f < a.frames) {
          const int variant = (a.frame_idx0 + f) % a.l1post_variants;
          const float2 *in = a.in + (long long)f * a.in_stride;
          BND(cd.x < a.in_stride && cd.y < a.in_stride);
          v0[k] = __ldg(cell_ptr(cd.x, in, a.pool, a.l1post_base, a.l1post_cells, variant));
          v1[k] = __ldg(cell_ptr(cd.y, in, a.pool, a.l1post_base, a.l1post_cells, variant));
        }
      }
#pragma unroll
      for (int k = 0; k < FPB; k++) {
        const int f = f0 + k;
        if (f < a.frames) {
          float2 *o = a.out + (long long)f * a.out_stride + 2 * pr;
          if (V16) __stcs(reinterpret_cast<float4 *>(o), make_float4(v0[k].x, v0[k].y, v1[k].x, v1[k].y));
          else { __stcs(o, v0[k]); __stcs(o + 1, v1[k]); }
        }
      }
    }
    // odd cell count: the last cell of each frame of the chunk
    if ((a.n & 1) && blockIdx.x == 0 && (int)threadIdx.x < FPB && f0 + (int)threadIdx.x < a.frames) {
      const int f = f0 + threadIdx.x, j = a.n - 1;
      const int variant = (a.frame_idx0 + f) % a.l1post_variants;
      a.out[(long long)f * a.out_stride + j] =
          fetch_cell(__ldg(a.code + j), a.in + (long long)f * a.in_stride, a.pool, a.l1post_base, a.l1post_cells, variant);
    }
  }
}

void launch_gather(const GatherArgs &a, cudaStream_t s)
{
  if (a.frames < 1 || a.n < 1) return;
  constexpr int FPB = 4;
  const int npair = a.n >> 1;
  int gx = (npair + 255) / 256;
  if (gx < 1) gx = 1;
  int gy = (a.frames + FPB - 1) / FPB;
  if (gy > 65535) gy = 65535;
  const dim3 grid(gx, gy);
  // 16-byte stores need every frame to start on a 16-byte boundary
  const bool v16 = (a.out_stride & 1) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 15) == 0;
  if (v16) k_gather<FPB, true><<<grid, 256, 0, s>>>(a);
  else k_gather<FPB, false><<<grid, 256, 0, s>>>(a);
  count_launch();
}

// ================================================================================================
// K5  OFDM symbol: carrier fill, IFFT, scale, guard interval, P1
// ================================================================================================
// In-place decimation-in-time FFT of M = 2^LOG2M points in shared memory, backward sign
// (x[t] = sum_b X_b e^{+j 2 pi b t / M}).  Pass j multiplies element q of each butterfly by
// W_{n_j}^{i q}, does an R-point DFT in registers and writes back in place; inputs are stored at
// digit-reversed positions so the result comes out in natural order.  The host lays the per-symbol
// carrier code table out in POSITION order (t2k::ofdm_position_of_bin), so the fill stage reads the
// table coalesced, writes shared memory linearly and never computes a digit reversal.
// Shared-memory layout: one spare slot per 16 points (padx below), conflict-free per half-warp for 8-byte
// elements for every access pattern used, with compile-time address offsets inside a butterfly.
//
// N = 32K does not fit (256 KB): it is split by bin parity (decimation in time at the top level):
// phase 0 transforms the even bins and parks E[n] in tensor memory, in the slots of the thread that
// produced it; phase 1 transforms the odd bins and stores E[n] +/- W_N^n O[n] to out[n] and out[n + N/2].
// Each carrier is gathered exactly once and every global store is a full, contiguous line.

// Shared-memory layout of the transform: point p lives at float2 index padx(p) = p + p / 16 (one spare slot per 16).
// Every access pattern of the pass schedule -- 16 consecutive points, stride-4/8/16 groups of a first pass, and the
// stride-NPREV butterflies -- then hits 16 distinct 8-byte bank pairs per half-warp, and because padx(a + b) =
// padx(a) + padx(b) whenever b is a multiple of 16 (or a, b are the block / digit parts of a small-stride butterfly),
// the 16 addresses of a butterfly are ONE base register plus compile-time offsets.
__host__ __device__ constexpr int padx(int p) { return p + (p >> 4); }

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
// complex add / subtract as ONE packed FP32x2 instruction each (sm_100 FADD2 / FFMA2); a - b = fma(b, -1, a) is exact
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }

// multiply by exp(+j 2 pi k / 16); k is a compile-time constant after unrolling
__device__ __forceinline__ float2 tw16(float2 d, int k)
{
  const float h = 0.70710678118654752440f, c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f;
  switch (k) {
    case 0: return d;
    case 1: return cmul(d, make_float2(c1, s1));
    case 2: return make_float2(h * (d.x - d.y), h * (d.x + d.y));
    case 3: return cmul(d, make_float2(s1, c1));
    case 4: return make_float2(-d.y, d.x);
    case 5: return cmul(d, make_float2(-s1, c1));
    case 6: return make_float2(-h * (d.x + d.y), h * (d.x - d.y));
    default: return cmul(d, make_float2(-c1, s1));
  }
}

// R-point backward DFT in registers (radix-2 DIF, fully unrolled); output index k is left in v[bitrev(k)]
template <int R>
__device__ __forceinline__ void dft_reg(float2 (&v)[R])
{
#pragma unroll
  for (int len = R; len >= 2; len >>= 1) {
#pragma unroll
    for (int base = 0; base < R; base += len) {
#pragma unroll
      for (int j = 0; j < len / 2; j++) {
        const float2 p = v[base + j], q = v[base + j + len / 2];
        v[base + j] = cadd(p, q);
        v[base + j + len / 2] = tw16(csub(p, q), (j * 16) / len);
      }
    }
  }
}

__host__ __device__ constexpr int bitrev_c(int k, int r)
{
  int out = 0;
  for (int b = 1; b < r; b <<= 1) { out = (out << 1) | (k & 1); k >>= 1; }
  return out;
}

// twiddles W_{n}^{i q}, q = 1..R-1: w1 from the table, powers by a short product tree; applied to v
template <int R>
__device__ __forceinline__ void apply_twiddles(float2 (&v)[R], float2 w1)
{
  float2 w[R];
  w[1] = w1;
#pragma unroll
  for (int qd = 2; qd < R; qd++) w[qd] = (qd & 1) ? cmul(w[qd - 1], w[1]) : cmul(w[qd >> 1], w[qd >> 1]);
#pragma unroll
  for (int qd = 1; qd < R; qd++) v[qd] = cmul(v[qd], w[qd]);
}

// one in-place DIT pass of radix 16 over M points; NPREV = length of the already transformed sub-blocks
// w1: the twiddle base W^i of the thread's butterflies (i = threadIdx.x mod NPREV, the same for every u because T is a
// multiple of NPREV), loaded once by the caller
template <int M, int NPREV, int T>
__device__ __forceinline__ void fft_pass16(float2 *x, float2 w1)
{
  constexpr int NB = M / 16;
  static_assert(T % NPREV == 0, "the twiddle base needs a thread-constant butterfly index");
#pragma unroll (NB / T == 2 ? 2 : 1)
  for (int u = threadIdx.x; u < NB; u += T) {
    const int i = u & (NPREV - 1);
    float2 *xb = x + padx((u - i) * 16 + i);
    float2 v[16];
#pragma unroll
    for (int qd = 0; qd < 16; qd++) v[qd] = xb[padx(qd * NPREV)];
    apply_twiddles<16>(v, w1);
    dft_reg<16>(v);
#pragma unroll
    for (int k = 0; k < 16; k++) xb[padx(k * NPREV)] = v[bitrev_c(k, 16)];
  }
}

// REGTW form of a radix-16 pass for NB = 2 T butterflies: a thread owns butterflies u = tid and tid + T, which share
// their twiddle base (T is a multiple of NPREV), so every twiddle W^q is generated ONCE -- by the running product
// W^q = W^(q-1) W, three live values instead of a fifteen-entry tree the compiler re-derives per butterfly at the
// 128-register cap -- and applied to both butterflies' element q at once.
template <int M, int NPREV, int T>
__device__ __forceinline__ void fft_pass16x2(float2 *x, float2 w1)
{
  static_assert(M / 16 == 2 * T && T % NPREV == 0, "two butterflies per thread with a common twiddle base");
  const int u = threadIdx.x, i = u & (NPREV - 1);
  float2 *xa = x + padx((u - i) * 16 + i);
  float2 *xc = xa + padx(T * 16);                // butterfly u + T: (u + T - i) * 16 + i, T * 16 a multiple of 16
  float2 va[16], vb[16];
#pragma unroll
  for (int qd = 0; qd < 16; qd++) { va[qd] = xa[padx(qd * NPREV)]; vb[qd] = xc[padx(qd * NPREV)]; }
  float2 w = w1;
#pragma unroll
  for (int qd = 1; qd < 16; qd++) {
    va[qd] = cmul(va[qd], w);
    vb[qd] = cmul(vb[qd], w);
    if (qd < 15) w = cmul(w, w1);
  }
  dft_reg<16>(va);
  dft_reg<16>(vb);
#pragma unroll
  for (int k = 0; k < 16; k++) { xa[padx(k * NPREV)] = va[bitrev_c(k, 16)]; xc[padx(k * NPREV)] = vb[bitrev_c(k, 16)]; }
}

// exp(+j 2 pi k / 32), k compile-time after unrolling
__device__ __forceinline__ float2 w32(int k)
{
  switch (k) {
    case 0: return make_float2(1.f, 0.f);
    case 1: return make_float2(0.98078528040323043f, 0.19509032201612825f);
    case 2: return make_float2(0.92387953251128674f, 0.38268343236508978f);
    case 3: return make_float2(0.83146961230254524f, 0.55557023301960218f);
    case 4: return make_float2(0.70710678118654757f, 0.70710678118654746f);
    case 5: return make_float2(0.55557023301960229f, 0.83146961230254524f);
    case 6: return make_float2(0.38268343236508984f, 0.92387953251128674f);
    case 7: return make_float2(0.19509032201612833f, 0.98078528040323043f);
    case 8: return make_float2(0.f, 1.f);
    case 9: return make_float2(-0.19509032201612819f, 0.98078528040323043f);
    case 10: return make_float2(-0.38268343236508973f, 0.92387953251128674f);
    case 11: return make_float2(-0.55557023301960196f, 0.83146961230254546f);
    case 12: return make_float2(-0.70710678118654746f, 0.70710678118654757f);
    case 13: return make_float2(-0.83146961230254535f, 0.55557023301960218f);
    case 14: return make_float2(-0.92387953251128674f, 0.38268343236508989f);
    default: return make_float2(-0.98078528040323043f, 0.19509032201612861f);
  }
}

// exp(+j 2 pi k / 64), k < 8, compile-time after unrolling
__device__ __forceinline__ float2 w64(int k)
{
  switch (k) {
    case 0: return make_float2(1.f, 0.f);
    case 1: return make_float2(0.99518472667219693f, 0.098017140329560604f);
    case 2: return make_float2(0.98078528040323043f, 0.19509032201612825f);
    case 3: return make_float2(0.95694033573220882f, 0.29028467725446233f);
    case 4: return make_float2(0.92387953251128674f, 0.38268343236508978f);
    case 5: return make_float2(0.88192126434835505f, 0.47139673682599764f);
    case 6: return make_float2(0.83146961230254524f, 0.55557023301960218f);
    default: return make_float2(0.77301045336273699f, 0.63439328416364549f);
  }
}

// where the per-position tables (carrier codes, inverse-sinc factors) keep the entry of shared-memory position p:
// p itself, except for the 16K sub-transform, whose fill reads 16 consecutive positions per thread as four vector
// loads -- stored [quad][group][4] so that each load is contiguous across the warp
int ofdm_table_index(int p, int log2_m)
{
  if (log2_m != 14 && log2_m != 12) return p;       // the transforms whose fill carries a radix-16 first pass
  const int g = p >> 4, q = (p >> 2) & 3, r = p & 3;
  return ((q << (log2_m - 4)) + g) * 4 + r;
}

int ofdm_position_of_bin(int m, int log2_m)
{
  // digits of m taken from the most significant end go to the least significant end of the position
  // pass order: the short radix 2^(log2_m mod 4) first, then radix 16 -- except the 16K sub-transform, which runs
  // 16, 16, 16, 4 (first pass fused with the carrier fill, the cheap radix-4 pass fused with the output)
  const int first = log2_m & 3;
  int lg[4], nr = 0;
  if (first && log2_m != 14) lg[nr++] = first;
  for (int i = 0; i < log2_m / 4; i++) lg[nr++] = 4;
  if (first && log2_m == 14) lg[nr++] = first;
  int p = 0, out_shift = 0, rem = log2_m;
  for (int j = 0; j < nr; j++) {
    rem -= lg[j];
    p |= ((m >> rem) & ((1 << lg[j]) - 1)) << out_shift;
    out_shift += lg[j];
  }
  return p;
}

// one output sample: complex64, or (sink format 1) interleaved 16-bit I/Q = round(x * 32767), saturated
template <int FMT> struct SinkT { typedef float2 type; };
template <> struct SinkT<1> { typedef short2 type; };
__device__ __forceinline__ void store_sample(float2 *p, int idx, float2 v) { __stcs(p + idx, v); }
__device__ __forceinline__ void store_sample(short2 *p, int idx, float2 v)
{
  int xi = __float2int_rn(v.x * 32767.f), yi = __float2int_rn(v.y * 32767.f);
  xi = max(-32768, min(32767, xi)); yi = max(-32768, min(32767, yi));
  p[idx] = make_short2((short)xi, (short)yi);
}

// Kernel schedule per (symbol, phase), M = 2^LOG2M points, first radix R0 = 2^(LOG2M mod 4):
//   1. fill fused with the first pass: a thread gathers the R0 consecutive positions of a first-pass
//      butterfly (code table read as one vector), does the R0-point DFT in registers, stores to smem;
//   2. the middle radix-16 passes in shared memory;
//   3. the last radix-16 pass fused with the output: butterfly i produces samples i + k M/16, which go
//      (scaled) straight to global memory -- coalesced over i -- including the cyclic prefix and, for
//      the odd-bin half of a 32K symbol, the in-place recombination with the even-bin half.
//
// C16 (chain mode): data cells arrive as 16-bit codes in cell-interleaved order.  Per symbol the CTA first
// copies the symbol's cells into a shared-memory staging area with bulk asynchronous copies (TMA), one per run of
// consecutive source cells (run_desc; for a time-interleaved PLP a run is a time-interleaver column); the carrier
// fill then gathers from shared memory and decodes through the constellation LUT (real part from the low byte's
// entry, imaginary from the high byte's -- in the same real-part table when the codes carry w~, see k_map).

// geometry of the carrier fill: a thread handles GPB first-pass butterflies (groups of R0 consecutive positions) per batch
template <int LOG2M, int T>
struct FillGeom {
  static constexpr int M = 1 << LOG2M;
  // 4K = 16 * 16 * 16: its first radix-16 pass (no twiddles) rides in the fill as well, like the 16K sub-transform's
  static constexpr int R0 = (LOG2M == 14 || LOG2M == 12) ? 16 : 1 << (LOG2M & 3);   // first radix (1 = no first pass)
  static constexpr int GROUPS = M / R0;             // first-pass butterflies
  static constexpr int INFL = LOG2M == 14 ? 16 : 8; // positions in flight per thread (16 where 128 registers are available)
  static constexpr int GPB0 = R0 >= INFL ? 1 : INFL / R0; // groups gathered per batch
  static constexpr int GPB = GPB0 * T > GROUPS ? GROUPS / T : GPB0;
  static constexpr int STEP = T * GPB;
  static_assert(GROUPS % STEP == 0, "fill batches must tile the transform");
};

// the carrier codes of one fill batch: the R0 codes of a group are contiguous and R0*4-byte aligned (one vector load)
template <int LOG2M, int T>
__device__ __forceinline__ void fill_load_codes(const int32_t *__restrict__ code, int g0,
                                                int (&c)[FillGeom<LOG2M, T>::GPB][FillGeom<LOG2M, T>::R0])
{
  typedef FillGeom<LOG2M, T> G;
  constexpr int R0 = G::R0;
#pragma unroll
  for (int b = 0; b < G::GPB; b++) {
    const int g = g0 + b * T;
    if (R0 == 4) {
      const int4 q4 = __ldg(reinterpret_cast<const int4 *>(code) + g);
      c[b][0] = q4.x; c[b][1 % R0] = q4.y; c[b][2 % R0] = q4.z; c[b][3 % R0] = q4.w;
    }
    else if (R0 == 8) {
      const int4 q4 = __ldg(reinterpret_cast<const int4 *>(code) + 2 * g), q5 = __ldg(reinterpret_cast<const int4 *>(code) + 2 * g + 1);
      c[b][0] = q4.x; c[b][1 % R0] = q4.y; c[b][2 % R0] = q4.z; c[b][3 % R0] = q4.w;
      c[b][4 % R0] = q5.x; c[b][5 % R0] = q5.y; c[b][6 % R0] = q5.z; c[b][7 % R0] = q5.w;
    }
    else if (R0 == 16) {
      // table laid out [quad q][group g][4] (ofdm_table_index): a warp's load of quad q is one contiguous 512 bytes
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int4 q4 = __ldg(reinterpret_cast<const int4 *>(code) + q * G::GROUPS + g);
        c[b][(4 * q) % R0] = q4.x; c[b][(4 * q + 1) % R0] = q4.y; c[b][(4 * q + 2) % R0] = q4.z; c[b][(4 * q + 3) % R0] = q4.w;
      }
    }
    else if (R0 == 2) {
      const int2 q2 = __ldg(reinterpret_cast<const int2 *>(code) + g);
      c[b][0] = q2.x; c[b][1 % R0] = q2.y;
    }
    else c[b][0] = __ldg(code + g);
  }
}

// shared-window addresses the chain-mode fill works with (see ofdm_fill)
struct FillSmem {
  uint32_t stage_s;        // staging area
  uint32_t lut_lane_s;     // real-part table + 4 * (lane mod copies)
  uint32_t im_ofs;         // distance of the imaginary-part table (0 with the single-table cell codes)
  uint32_t spool_m8_s;     // small pool - 8 bytes
  uint32_t esh;            // log2 of the bytes between table entries
};

// carrier fill of one (symbol, phase), fused with the first pass of radix R0.  POOL: the symbol has carriers taken
// from the big pool (L1 signalling / dummy cells); SINC: inverse-sinc equalisation factors are applied.
// `c` holds the codes of the thread's first batch (loaded by the caller ahead of the barrier that precedes the fill);
// the codes of batch n + 1 are fetched while batch n is processed.
// MT: the carrier codes carry the first entry of their constellation table (several tables, see OFDM_CODE_TAB_SHIFT).
// MISO: MISO group-2 carrier codes, bit 0 of a data code selects the component whose sign flips (OFDM_CODE_MISO_IM).
template <int LOG2M, int T, bool C16, bool POOL, bool SINC, bool MT = false, bool MISO = false>
__device__ __forceinline__ void ofdm_fill(float2 *x, const int32_t *__restrict__ code, const float *__restrict__ sinc,
                                          int (&c)[FillGeom<LOG2M, T>::GPB][FillGeom<LOG2M, T>::R0], const float2 *__restrict__ cells,
                                          const float2 *__restrict__ pool, const FillSmem fs, int stage_cap_dbg = 0, int lut_n_dbg = 0)
{
  typedef FillGeom<LOG2M, T> G;
  constexpr int R0 = G::R0, GPB = G::GPB;
#pragma unroll 1
  for (int g0 = threadIdx.x; g0 < G::GROUPS; g0 += G::STEP) {
    float2 v[GPB][R0];
#pragma unroll
    for (int b = 0; b < GPB; b++)
#pragma unroll
      for (int r = 0; r < R0; r++) {
        const int cc = c[b][r];
        if (C16) {
          // data cell: 16-bit code from the staging area through the LUT (a dummy read of offset 0 for the others);
          // small pool cell (null, pilots): (p + 1) << 17 -> spool[p]; big pool cell: sign bit set (POOL symbols only)
          const unsigned off = POOL && cc < 0 ? 0u : (unsigned)cc & (MISO ? 0x1FFFEu : 0x1FFFFu);
          // small pool cell: bits 17..20 only (with table bits a data code can exceed 0x20000 as well)
          BND(cc < 0 || (MT ? (unsigned)cc - 0x20000u < OFDM_CODE_SMALL_POOL : cc >= 0x20000) || off + 2 <= 2u * (unsigned)stage_cap_dbg);
          // explicit 32-bit shared-window addresses (one base register + the lane's table column): the generic-pointer
          // form made the compiler rebuild the window base and the lane offset for every carrier (≈ 10 instructions)
          unsigned sc;
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(sc) : "r"(fs.stage_s + off));
          // the tables are replicated 2^rep_shift times (entry e, copy c at (e << esh) + 4 c) and a lane reads copy
          // lane mod copies: with 32 copies no two lanes share a bank, with 16 only lanes l and l + 16 can collide
          float2 val;
          if constexpr (MT) {
            // the cell's own table starts at entry tb; pool and pilot carriers read the first (largest) table
            const unsigned tb = POOL && cc < 0 ? 0u : (unsigned)cc >> OFDM_CODE_TAB_SHIFT;
            BND(tb + (sc & 255u) < (unsigned)lut_n_dbg && tb + (sc >> 8) < (unsigned)lut_n_dbg);
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val.x) : "r"(fs.lut_lane_s + ((tb + (sc & 255u)) << fs.esh)));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val.y) : "r"(fs.lut_lane_s + fs.im_ofs + ((tb + (sc >> 8)) << fs.esh)));
          }
          else {
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val.x) : "r"(fs.lut_lane_s + ((sc & 255u) << fs.esh)));
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(val.y) : "r"(fs.lut_lane_s + fs.im_ofs + ((sc >> 8) << fs.esh)));
          }
          if constexpr (MISO) {
            // -conj(g) (bit 0 clear: negate Re) or conj(g) (bit 0 set: negate Im) of the paired cell; pool and pilot
            // carriers are overwritten below (their pool values are already transformed)
            const unsigned neg_im = (unsigned)cc << 31;
            val.x = __uint_as_float(__float_as_uint(val.x) ^ neg_im ^ 0x80000000u);
            val.y = __uint_as_float(__float_as_uint(val.y) ^ neg_im);
          }
          if (MT ? (unsigned)cc - 0x20000u < OFDM_CODE_SMALL_POOL : cc >= 0x20000) asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(val.x), "=f"(val.y) : "r"(fs.spool_m8_s + ((unsigned)cc >> 14)));
          if (POOL && cc < 0) val = __ldg(pool + (cc & 0x7FFFFFFF));
          v[b][r] = val;
        }
        else {
          const float2 *base = cc >= 0 ? cells : pool;
          v[b][r] = __ldg(base + (cc >= 0 ? cc : ~cc));
        }
      }
    if (g0 + G::STEP < G::GROUPS) fill_load_codes<LOG2M, T>(code, g0 + G::STEP, c);
#pragma unroll
    for (int b = 0; b < GPB; b++) {
      const int g = g0 + b * T;
      if (SINC) {
#pragma unroll
        for (int r = 0; r < R0; r++) {
          const float sf = __ldg(sinc + (R0 == 16 ? (((r >> 2) * G::GROUPS + g) * 4 + (r & 3)) : g * R0 + r));
          v[b][r] = __fmul2_rn(v[b][r], make_float2(sf, sf));
        }
      }
      if (R0 > 1) dft_reg<R0>(v[b]);
      float2 *xb = x + padx(g * R0);
#pragma unroll
      for (int k = 0; k < R0; k++) xb[k] = v[b][bitrev_c(k, R0)];
    }
  }
}

// ---- tensor memory (TMEM, sm_100): the 32K path keeps thread-private values there between its two phases.  Every
// tcgen05 instruction is warp-collective (.sync.aligned): all 32 lanes must execute it together.
constexpr int OFDM_PARK_COLS = 256;       // 512 threads x 64 words over the 128 lanes

// one warp: allocate NCOLS columns (power of two >= 32); the column base is written to the shared word at dst_s
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_s)
{
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(dst_s), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory"); }
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr)
{
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// four complex values to 8 consecutive columns of the thread's lane
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float2 (&v)[4])
{
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
               ::"r"(taddr), "f"(v[0].x), "f"(v[0].y), "f"(v[1].x), "f"(v[1].y), "f"(v[2].x), "f"(v[2].y), "f"(v[3].x), "f"(v[3].y));
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }
// the registers of tmem_ld4 hold the values only after tmem_wait_ld4 on them: the wait names them as operands, so
// the compiler cannot move a use of them above it
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float2 (&v)[4])
{
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x), "=f"(v[3].y)
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld4(float2 (&v)[4])
{
  asm volatile("tcgen05.wait::ld.sync.aligned;\n"
               : "+f"(v[0].x), "+f"(v[0].y), "+f"(v[1].x), "+f"(v[1].y), "+f"(v[2].x), "+f"(v[2].y), "+f"(v[3].x), "+f"(v[3].y));
}

// FMT: sink format (bit 0, SinkT) | OFDM_FMT_MT: chain mode with several constellation tables, the carrier codes carry
// their table's first entry (OFDM_CODE_TAB_SHIFT) | OFDM_FMT_MISO: MISO group-2 carrier codes (OFDM_CODE_MISO_IM)
constexpr int OFDM_FMT_MT = 2;
constexpr int OFDM_FMT_MISO = 4;
template <int LOG2M, int T, bool C16, int FMT, int SPLIT>
__global__ void __launch_bounds__(T, (LOG2M == 14 ? 1 : 1024 / T)) k_ofdm(const OfdmArgs a)
{
  constexpr bool MT = (FMT & OFDM_FMT_MT) != 0;
  constexpr bool MISO = (FMT & OFDM_FMT_MISO) != 0;
  static_assert(!MT || C16, "several constellation tables only in chain mode");
  static_assert(!MISO || C16, "MISO processing only in chain mode");
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float2 *x = reinterpret_cast<float2 *>(smem_raw);
  constexpr int M = 1 << LOG2M;
  uint8_t *stage = reinterpret_cast<uint8_t *>(x + padx(M));
  float *lut_re = reinterpret_cast<float *>(stage + 2 * a.stage_cap);
  const int lut_rep_shift = a.lut_rep_shift, lut_rep = 1 << lut_rep_shift;
  // one table when the cell codes carry w~ (Im = Re lut[w~]), else a second one for the imaginary parts
  const int lut_e = a.lut_n < 16 ? 16 : a.lut_n;      // table entries kept (a multiple of 16: the small pool behind stays 64-byte aligned)
  float *lut_im = a.lut_single ? lut_re : lut_re + lut_e * lut_rep;
  float2 *spool = reinterpret_cast<float2 *>(lut_re + (a.lut_single ? lut_e : 2 * lut_e) * lut_rep);      // first 8 pool cells: zero and the pilot values
  uint64_t *mbar = reinterpret_cast<uint64_t *>(spool + 8);                 // completion barriers: [0] staging copies, [1] descriptors
  const uint32_t mbar_s = (uint32_t)__cvta_generic_to_shared(mbar), dbar_s = mbar_s + 8;
  const int2 *descbuf = reinterpret_cast<const int2 *>(mbar + 2);           // the next symbol's copy descriptors
  const uint32_t desc_s = mbar_s + 16;
  if (C16) {
    // the constellation table goes through the (still unused) transform buffer: one L2 round trip, then replication
    if constexpr (MT) {
      for (int i = threadIdx.x; i < a.lut_n; i += T) x[i] = __ldg(a.lut + i);     // the tables together can exceed T entries
    }
    else if (threadIdx.x < a.lut_n) x[threadIdx.x] = __ldg(a.lut + threadIdx.x);
    if (threadIdx.x < 8) spool[threadIdx.x] = __ldg(a.pool + threadIdx.x);
    // carriers that are not data cells do a dummy read of staging slot 0 and look its code up: until a symbol with
    // data cells has been staged that slot must hold a valid code (the tables only have lut_n entries)
    if (threadIdx.x < 4) reinterpret_cast<uint32_t *>(stage)[threadIdx.x] = 0u;
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(mbar_s) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(dbar_s) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    for (int i = threadIdx.x; i < a.lut_n * lut_rep; i += T) {
      const float2 v = x[i >> lut_rep_shift];
      lut_re[i] = v.x;
      if (!a.lut_single) lut_im[i] = v.y;
    }
    __syncthreads();
  }
  static_assert(SPLIT == 1 || LOG2M == 14, "only 32K symbols are transformed as two halves");
  // 32K: the even-bin half E[n] of a symbol waits for the odd-bin phase in tensor memory (TMEM), 256 columns of this
  // CTA's allocation; see park_col below.  Warp 0 allocates, the column base goes through the first word of x (not
  // yet in use; the first fill is behind a barrier) to the other threads.
  uint32_t park_col = 0;
  if constexpr (SPLIT == 2) {
    uint32_t *tm_slot = reinterpret_cast<uint32_t *>(x);
    if (threadIdx.x < 32) {
      tmem_alloc<OFDM_PARK_COLS>((uint32_t)__cvta_generic_to_shared(tm_slot));
      tmem_relinquish();
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    // a warp reaches only the 32 TMEM lanes of its quadrant (warp mod 4); the four warps of a quadrant take 64
    // columns each: thread-private slots of 8 butterflies x 4 complex values (lane = thread, one column per word)
    const uint32_t warp = threadIdx.x >> 5;
    park_col = *tm_slot + ((32u * (warp & 3u)) << 16) + 64u * (warp >> 2);
  }
  constexpr int R0 = FillGeom<LOG2M, T>::R0;       // first radix, done inside the fill (1 = no first pass)
  constexpr int NLAST = M / 16;              // NPREV of the last radix-16 pass
  const int N = a.fft_n;
  const int units = a.frames * a.num_symbols;
  const int cp_from = N - a.gi;
  const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
  FillSmem fs;
  fs.stage_s = stage_s;
  fs.esh = 2u + (uint32_t)lut_rep_shift;
  fs.lut_lane_s = (uint32_t)__cvta_generic_to_shared(lut_re) + ((threadIdx.x & (uint32_t)(lut_rep - 1)) << 2);
  fs.im_ofs = a.lut_single ? 0u : 4u * (uint32_t)(lut_e * lut_rep);
  fs.spool_m8_s = (uint32_t)__cvta_generic_to_shared(spool) - 8u;
  // 16K sub-transform with 512 threads: every thread runs the same butterflies for every symbol, so their twiddle
  // bases stay in registers for the whole kernel (no L2 round trip at the start of each pass: L1 is ~2 KB here)
  // Pass schedule of the 16K sub-transform: radix 16 (in the fill, no twiddles), 16, 16, 4 (in the output).
  constexpr bool REGTW = LOG2M == 14;
  static_assert(!REGTW || T == 512, "the 16K schedule is written for 512 threads");
  float2 tw_p1 = make_float2(1.f, 0.f), tw_p2 = tw_p1, tw_last = tw_p1, tw_rec = tw_p1;
  if (REGTW) {
    tw_p1 = __ldg(a.tw + (threadIdx.x & 15) * (M / 256));       // pass with NPREV = 16:  W_M^{i M/256},  i = u mod 16
    tw_p2 = __ldg(a.tw + (threadIdx.x & 255) * (M / 4096));     // pass with NPREV = 256: W_M^{i M/4096}, i = u mod 256
    tw_last = __ldg(a.tw + threadIdx.x);                        // last pass: W_M^{tid}; butterfly tid + 512 j adds exp(j 2 pi j / 32)
    if (SPLIT == 2) tw_rec = __fmul2_rn(__ldg(a.tw_split + threadIdx.x), make_float2(a.norm, a.norm));   // W_N^{tid} * norm
  }
  // smaller transforms with at most one butterfly per thread and pass (M / 16 <= T): the thread's twiddle base of every
  // pass is the same for every symbol -- loaded once here instead of at the head of each pass, where the load's
  // latency was exposed (13 % of the 8K kernel's stall samples)
  static_assert(REGTW || M / 16 <= T, "one butterfly per thread and pass: the twiddle bases are loaded once");
  constexpr int NP1 = R0, NP2 = R0 * 16 < NLAST ? R0 * 16 : 1;       // NPREV of the middle passes (see below)
  if (!REGTW) {
    tw_p1 = __ldg(a.tw + (threadIdx.x & (NP1 - 1)) * (M / (NP1 * 16)));
    tw_p2 = __ldg(a.tw + (threadIdx.x & (NP2 - 1)) * (M / (NP2 * 16)));
    tw_last = (int)threadIdx.x < NLAST ? __ldg(a.tw + threadIdx.x) : make_float2(1.f, 0.f);
  }

  // C16: the cells of symbol `u` go to the staging area by bulk asynchronous copies (TMA, cp.async.bulk): one copy
  // per run of consecutive source cells -- the enclosing 16-byte aligned span of the frame's cell memory -- spread over
  // the threads, all completing on one mbarrier whose transaction count is the symbol's byte total.  Issued for symbol
  // u + gridDim.x as soon as symbol u's last fill has finished reading the staging area, so the copies run under the
  // FFT passes without occupying the load/store pipe.
  // The descriptors themselves (8 bytes per run, from L2) are fetched one symbol further ahead, by one more bulk copy
  // into shared memory, so issuing a symbol's copies never waits on global memory.
  uint32_t mphase = 0, dphase = 0;
  // (first run, run count) of a symbol's copy list; requested a symbol ahead of its use (cp1 below)
  auto run_range = [&](int u) {
    const int ul = u % a.num_symbols;
    return make_int2(__ldg(a.run_ptr + ul), __ldg(a.run_cnt + ul));
  };
  // one thread: fetch the descriptors of a symbol into descbuf (lists are 16-byte aligned and padded)
  auto desc_issue = [&](int2 rr) {
    if (rr.y <= 0) return;
    const uint32_t bytes = (uint32_t)((rr.y + 1) >> 1) * 16u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(dbar_s), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(desc_s), "l"(a.run_desc + rr.x), "r"(bytes), "r"(dbar_s) : "memory");
  };
  auto stage_issue = [&](int u, int2 rr) {
    if (rr.y <= 0) return;
    {
      uint32_t done;
      do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(done) : "r"(dbar_s), "r"(dphase) : "memory");
      } while (!done);
      dphase ^= 1u;
    }
    const int uf = u / a.num_symbols, ul = u - uf * a.num_symbols;
    const uint8_t *src = reinterpret_cast<const uint8_t *>(a.cells16 + (long long)uf * a.cells_stride);
    // the fill's reads of the staging area (generic proxy) are ordered before these writes (async proxy)
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    if (threadIdx.x == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar_s), "r"(__ldg(a.stage_bytes + ul)) : "memory");
#pragma unroll 2
    for (int i = threadIdx.x; i < rr.y; i += T) {
      const int2 d = descbuf[i];
      BND(i < a.desc_cap);
      BND(((unsigned)d.y >> 16) + ((unsigned)d.y & 0xFFFFu) <= (unsigned)a.stage_cap / 8u && d.x >= 0);
      BND(a.cells_len == 0 || (long long)uf * a.cells_stride * 2 + 16ll * (d.x + (d.y & 0xFFFF)) <= a.cells_len * 2 + 64);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                   ::"r"(stage_s + 16u * ((uint32_t)d.y >> 16)), "l"(src + 16ll * d.x), "r"(16u * ((uint32_t)d.y & 0xFFFFu)), "r"(mbar_s) : "memory");
    }
  };
  auto stage_wait = [&]() {
    uint32_t done;
    do {
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                   : "=r"(done) : "r"(mbar_s), "r"(mphase) : "memory");
    } while (!done);
    mphase ^= 1u;
  };

  int2 cp0 = make_int2(0, 0), cp1 = cp0;      // copy lists of this CTA's current and next symbol
  if (C16 && (int)blockIdx.x < units) {
    cp0 = run_range(blockIdx.x);
    if (threadIdx.x == 0) desc_issue(cp0);
  }
  for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
    const int f = unit / a.num_symbols, l = unit - f * a.num_symbols;
    if (C16 && unit + (int)gridDim.x < units) cp1 = run_range(unit + gridDim.x);
    const int variant = (a.frame_idx0 + (f % a.frames_per_channel)) % a.l1post_variants;
    const float2 *cells = a.cells + (long long)f * a.cells_stride;
    const float2 *pool = a.pool + (long long)variant * a.pool_stride;
    // output addressing in samples relative to a.out (element size depends on the sink format)
    typedef typename SinkT<FMT & 1>::type sample_t;
    sample_t *out = reinterpret_cast<sample_t *>(a.out) + (long long)f * a.out_stride;
    sample_t *sym = out + 2048 + (long long)l * (N + a.gi);
    BND(a.out_len == 0 || (long long)f * a.out_stride + 2048 + (long long)(l + 1) * (N + a.gi) <= a.out_len);

    if (l == 0)
      for (int i = threadIdx.x; i < 2048; i += T) {
        float2 p = __ldg(a.p1 + i);
        p.x *= a.sink_gain; p.y *= a.sink_gain;
        store_sample(out, i, p);
      }

    bool pool_sym = false;
    if (C16) pool_sym = __ldg(a.sym_flags + l) != 0;
    int c[FillGeom<LOG2M, T>::GPB][FillGeom<LOG2M, T>::R0];
    fill_load_codes<LOG2M, T>(a.code_pos + (long long)l * SPLIT * M, threadIdx.x, c);
    if (C16) {
      if (unit == (int)blockIdx.x) stage_issue(unit, cp0);      // first symbol of this CTA
      if (cp0.y > 0) stage_wait();
    }

    for (int phase = 0; phase < SPLIT; phase++) {
      const int32_t *code = a.code_pos + ((long long)l * SPLIT + phase) * M;
      const float *sinc = a.sinc_pos ? a.sinc_pos + (long long)phase * M : nullptr;
      if (phase) fill_load_codes<LOG2M, T>(code, threadIdx.x, c);
      __syncthreads();      // staging area landed (phase 0) / previous phase has finished reading x
      // every thread is past its reads of the descriptor buffer: the next symbol's list may come in
      if (C16 && phase == 0 && threadIdx.x == 0 && unit + (int)gridDim.x < units) desc_issue(cp1);
      // ---- 1. carrier fill (+ first pass)
      if (sinc) {
        if (pool_sym) ofdm_fill<LOG2M, T, C16, true, true, MT, MISO>(x, code, sinc, c, cells, pool, fs, a.stage_cap, a.lut_n);
        else ofdm_fill<LOG2M, T, C16, false, true, MT, MISO>(x, code, sinc, c, cells, pool, fs, a.stage_cap, a.lut_n);
      }
      else {
        if (pool_sym) ofdm_fill<LOG2M, T, C16, true, false, MT, MISO>(x, code, sinc, c, cells, pool, fs, a.stage_cap, a.lut_n);
        else ofdm_fill<LOG2M, T, C16, false, false, MT, MISO>(x, code, sinc, c, cells, pool, fs, a.stage_cap, a.lut_n);
      }
      __syncthreads();
      // every fill of the symbol has read its cells: the next symbol's cells may replace them (under the passes)
      if (C16 && phase == SPLIT - 1) {
        if (unit + (int)gridDim.x < units) stage_issue(unit + gridDim.x, cp1);
        cp0 = cp1;
      }
      // ---- 2. middle radix-16 passes
      if constexpr (REGTW) {
        fft_pass16x2<M, 16, T>(x, tw_p1); __syncthreads();
        fft_pass16x2<M, 256, T>(x, tw_p2); __syncthreads();
      }
      else {
        if (R0 * 16 < NLAST * 16 && R0 < NLAST) { fft_pass16<M, NP1, T>(x, tw_p1); __syncthreads(); }
        if (R0 * 16 < NLAST) { fft_pass16<M, NP2, T>(x, tw_p2); __syncthreads(); }
      }
      // ---- 3. last pass fused with scale + store (+ cyclic prefix, + 32K recombination)
      if constexpr (REGTW) {
        // radix 4 over the whole sub-transform: butterfly i = tid + 512 j (j < 8) reads x[i + q M/4] and produces the
        // samples i + k M/4.  W_M^i = W_M^tid * exp(j 2 pi j / 32); for the 32K recombination W_N^(i + k M/4) =
        // W_N^tid * exp(j 2 pi j / 64) * exp(j 2 pi k / 8).  32K: phase 0 parks its results E in TMEM (8 columns per
        // butterfly, no global stores); phase 1 requests butterfly j's E at the head of butterfly j and waits for it just
        // before the recombination.  The tcgen05 instructions stay outside the per-thread cyclic-prefix conditions.
        constexpr int NL = M / 4, NBT = NL / T;
        constexpr int XS = NL + NL / 16;                      // padx(q * NL) = q * XS
        sample_t *o = sym + a.gi + threadIdx.x;
        const bool odd_phase = SPLIT == 2 && phase == 1;
        if (odd_phase) tmem_wait_st();                        // phase 0's stores have landed
#pragma unroll
        for (int j = 0; j < NBT; j++) {
          const int i = threadIdx.x + j * T;
          const float2 *xb = x + padx(i);
          float2 e[4];
          if (odd_phase) tmem_ld4(park_col + 8u * j, e);
          float2 v[4];
#pragma unroll
          for (int q = 0; q < 4; q++) v[q] = xb[q * XS];
          const float2 w1 = j ? cmul(tw_last, w32(j)) : tw_last;
          const float2 w2 = cmul(w1, w1), w3 = cmul(w2, w1);
          v[1] = cmul(v[1], w1); v[2] = cmul(v[2], w2); v[3] = cmul(v[3], w3);
          dft_reg<4>(v);
          if (SPLIT == 1) {
            sample_t *ocp = sym + ((long long)threadIdx.x - cp_from);
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const float2 r = __fmul2_rn(v[bitrev_c(k, 4)], make_float2(a.norm, a.norm));
              store_sample(o, j * T + k * NL, r);
              if (i + k * NL >= cp_from) store_sample(ocp, j * T + k * NL, r);
            }
          }
          else if (phase == 0) {
            // even-bin half E[n], n = i + k M/4: read back only by this thread, in phase 1
            float2 r[4];
#pragma unroll
            for (int k = 0; k < 4; k++) r[k] = __fmul2_rn(v[bitrev_c(k, 4)], make_float2(a.norm, a.norm));
            tmem_st4(park_col + 8u * j, r);
          }
          else {
            sample_t *ocp = sym + ((long long)threadIdx.x + M - cp_from);
            const float2 wi = j ? cmul(tw_rec, w64(j)) : tw_rec;
            float2 r[4];
#pragma unroll
            for (int k = 0; k < 4; k++) r[k] = cmul(tw16(v[bitrev_c(k, 4)], 2 * k), wi);
            tmem_wait_ld4(e);
#pragma unroll
            for (int k = 0; k < 4; k++) {
              store_sample(o, j * T + k * NL, cadd(e[k], r[k]));
              const float2 hi = csub(e[k], r[k]);
              store_sample(o, j * T + k * NL + M, hi);
              if (i + k * NL + M >= cp_from) store_sample(ocp, j * T + k * NL, hi);
            }
          }
        }
      }
      else
#pragma unroll 1
      for (int i = threadIdx.x; i < NLAST; i += T) {
        const float2 *xb = x + padx(i);
        float2 v[16];
#pragma unroll
        for (int qd = 0; qd < 16; qd++) v[qd] = xb[padx(qd * NLAST)];
        apply_twiddles<16>(v, tw_last);
        dft_reg<16>(v);
        // sample t = i + k NLAST: one 64-bit base per destination, compile-time offsets k NLAST
        sample_t *o = sym + a.gi + i;
        sample_t *ocp = sym + ((long long)i - cp_from);       // cyclic prefix: sample t >= N - gi also goes to t - (N - gi)
#pragma unroll
        for (int k = 0; k < 16; k++) {
          float2 r = v[bitrev_c(k, 16)];
          r = __fmul2_rn(r, make_float2(a.norm, a.norm));
          store_sample(o, k * NLAST, r);
          if (i + k * NLAST >= cp_from) store_sample(ocp, k * NLAST, r);
        }
      }
    }
  }
  if constexpr (SPLIT == 2) {
    // every thread's TMEM accesses are complete (each load was waited for) before warp 0 frees the columns; the
    // kernel has no other way out
    tmem_fence_before_sync();
    __syncthreads();
    if (threadIdx.x < 32) {
      tmem_fence_after_sync();
      tmem_dealloc<OFDM_PARK_COLS>(park_col);
    }
  }
}

// bytes of one copy of the constellation table(s) in shared memory
static inline size_t lut_table_bytes(const OfdmArgs &a) { return (size_t)(a.lut_n < 16 ? 16 : a.lut_n) * 4 * (a.lut_single ? 1 : 2); }

template <int LOG2M, int T, bool C16, int FMT, int SPLIT>
static void launch_ofdm_t(const OfdmArgs &a, cudaStream_t s)
{
  constexpr int M = 1 << LOG2M;
  const size_t smem = (size_t)padx(M) * sizeof(float2) +
                      (C16 ? (size_t)a.stage_cap * 2 + ((size_t)lut_table_bytes(a) << a.lut_rep_shift) + 64 + 16 + (size_t)a.desc_cap * 8 : 0);
  const int units = a.frames * a.num_symbols;
  static bool attr[MAX_DEVICES];
  allow_smem(k_ofdm<LOG2M, T, C16, FMT, SPLIT>, 227 * 1024, attr);
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ofdm<LOG2M, T, C16, FMT, SPLIT>, T, smem);
  if (per_sm < 1) per_sm = 1;
  int blocks = sm_count() * per_sm;
  if (blocks > units) blocks = units;
  k_ofdm<LOG2M, T, C16, FMT, SPLIT><<<blocks, T, smem, s>>>(a);
  count_launch();
}

template <bool C16, int FMT>
static void launch_ofdm_c(const OfdmArgs &a, cudaStream_t s)
{
  switch (a.log2_m) {
    case 10: launch_ofdm_t<10, 256, C16, FMT, 1>(a, s); break;
    case 11: launch_ofdm_t<11, 256, C16, FMT, 1>(a, s); break;
    case 12: launch_ofdm_t<12, 256, C16, FMT, 1>(a, s); break;
    case 13: launch_ofdm_t<13, 512, C16, FMT, 1>(a, s); break;
    case 14:
      // 512 threads with up to 128 registers each: two butterflies per thread and pass, interleaved by the compiler;
      // 32K symbols (split = 2) as two 16K halves
      if (a.split == 2) launch_ofdm_t<14, 512, C16, FMT, 2>(a, s);
      else launch_ofdm_t<14, 512, C16, FMT, 1>(a, s);
      break;
    default: break;
  }
}

int launch_ofdm(const OfdmArgs &a0, cudaStream_t s)
{
  if (a0.frames * a0.num_symbols < 1) return 1;
  OfdmArgs a = a0;
  // up to 32 copies of the constellation table(s) (conflict-free: copy = lane), as many as shared memory allows (chain mode)
  // (without lowering the number of CTAs per SM that fit without replication; 2 resident CTAs at most are useful below 16K)
  a.lut_rep_shift = 0;
  if (a.cells16) {
    const size_t base = (size_t)padx(1 << a.log2_m) * sizeof(float2) + (size_t)a.stage_cap * 2 + 64 + 16 + (size_t)a.desc_cap * 8, sm_bytes = 227 * 1024;
    const size_t one = lut_table_bytes(a);
    size_t ctas = sm_bytes / (base + one + 1024);
    if (ctas < 1) ctas = 1;
    if (ctas > 2) ctas = 2;
    for (int sh = 5; sh > 0; sh--)
      if (base + (one << sh) + 1024 <= sm_bytes / ctas) { a.lut_rep_shift = sh; break; }
  }
  if (a.cells16) {
    switch ((a.out_fmt ? 1 : 0) | (a.lut_tables > 1 ? OFDM_FMT_MT : 0) | (a.miso ? OFDM_FMT_MISO : 0)) {
      case 0: launch_ofdm_c<true, 0>(a, s); break;
      case 1: launch_ofdm_c<true, 1>(a, s); break;
      case 2: launch_ofdm_c<true, 2>(a, s); break;
      case 3: launch_ofdm_c<true, 3>(a, s); break;
      case 4: launch_ofdm_c<true, 4>(a, s); break;
      case 5: launch_ofdm_c<true, 5>(a, s); break;
      case 6: launch_ofdm_c<true, 6>(a, s); break;
      case 7: launch_ofdm_c<true, 7>(a, s); break;
    }
  }
  else launch_ofdm_c<false, 0>(a, s);      // the drop-in block always emits complex64
  return 1 << a.lut_rep_shift;
}

// ================================================================================================
// K6  tone-reservation PAPR reduction (peak cancellation on the reserved carriers, see PaprArgs)
// ================================================================================================
// One cluster of CL CTAs per (frame, symbol); CTA r keeps samples [r N/CL, (r+1) N/CL) of c in shared memory for the
// whole iteration loop (32K: CL = 2, a 16K half each -- 256 KB do not fit one CTA).  Each iteration is one sweep over
// the samples that applies the previous update and tracks the new maximum as the 64-bit key
// float_bits(|c|^2) << 32 | (0xFFFFFFFF - n): the lowest index wins a tie, whatever the order of the reduction.  Warp
// maxima meet by shared-memory atomics in their CTA; with CL = 2 each CTA then stores its maximum into its partner's slot
// (DSMEM: a plain store -- there is no 64-bit max on the cluster's shared memory) and the key is the larger of the two.
// Keys rotate over three slots so that a slot is cleared one iteration before it is filled again.  Every CTA takes the same decisions from the same data: the
// reserved-carrier values R are kept (identically) in each.
constexpr int PAPR_MAX_THREADS = 1024;

// (not .aligned: the arrive follows a load whose address depends on the owner of c_m)
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release;\n" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;\n" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_rank()
{
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
// generic address of the same shared-memory variable in CTA `rank` of the cluster
template <class P>
__device__ __forceinline__ P *cluster_map(P *p, uint32_t rank)
{
  uint64_t r;
  asm volatile("mapa.u64 %0, %1, %2;\n" : "=l"(r) : "l"(reinterpret_cast<uint64_t>(p)), "r"(rank));
  return reinterpret_cast<P *>(r);
}

template <int CL>
__device__ __forceinline__ void papr_sync()
{
  if constexpr (CL == 1) __syncthreads();
  else { cluster_arrive(); cluster_wait(); }
}

// slot[0]: this CTA's maximum; slot[1] (CL = 2): the partner's, stored there by the partner.  Visible to every CTA of
// the cluster after the next papr_sync.
template <int CL>
__device__ __forceinline__ void papr_key_max(unsigned long long key, unsigned long long *slot, unsigned long long *rslot)
{
#pragma unroll
  for (int o = 16; o; o >>= 1) key = max(key, __shfl_xor_sync(0xFFFFFFFFu, key, o));
  if ((threadIdx.x & 31) == 0) atomicMax(slot, key);
  if constexpr (CL == 2) {
    __syncthreads();
    if (threadIdx.x == 0) rslot[1] = slot[0];
  }
}

__device__ __forceinline__ unsigned long long papr_key(float2 v, int n)
{
  const float p2 = v.x * v.x + v.y * v.y;
  return ((unsigned long long)__float_as_uint(p2) << 32) | (0xFFFFFFFFu - (uint32_t)n);
}

template <int CL, int FMT>
__global__ void __launch_bounds__(PAPR_MAX_THREADS) k_papr_tr(const PaprArgs a)
{
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int N = a.fft_n, H = N / CL, S = a.tones, T = blockDim.x, tid = threadIdx.x;
  float2 *c = reinterpret_cast<float2 *>(smem_raw);
  float2 *R = c + H;
  unsigned long long *keys = reinterpret_cast<unsigned long long *>(R + S);
  const uint32_t rank = CL == 2 ? cluster_rank() : 0u;
  unsigned long long *rkeys = CL == 2 ? cluster_map(keys, rank ^ 1u) : keys;      // [3][2], see papr_key_max
  const int unit = blockIdx.x / CL, f = unit / a.num_symbols, l = unit - f * a.num_symbols;
  const int set = __ldg(a.sym_set + l);
  BND(set >= 0 && set < a.sets);
  const float2 *kern = a.kernel + (long long)set * N;
  const int32_t *bins = a.bins + (long long)set * S;
  const long long sym0 = (long long)f * a.spf + 2048 + (long long)l * (N + a.gi);      // first CP sample
  BND(a.in_len == 0 || sym0 + a.gi + N <= a.in_len);
  const float2 *xin = a.in + sym0 + a.gi + (long long)rank * H;
  const float V = a.vclip, A2 = a.tone_max * a.tone_max;

  if (tid < 6) keys[tid] = 0ull;
  for (int t = tid; t < S; t += T) R[t] = make_float2(0.f, 0.f);
  papr_sync<CL>();      // the keys are cleared in every CTA before any of them adds to them

  // sweep 0: load the CTA's samples
  unsigned long long key = 0ull;
  for (int j = tid; j < H; j += T) {
    const float2 v = __ldg(xin + j);
    c[j] = v;
    key = max(key, papr_key(v, (int)rank * H + j));
  }
  papr_key_max<CL>(key, keys, rkeys);
  papr_sync<CL>();

  int applied = 0, reason = PAPR_STOP_LIMIT;
  for (int it = 0;; it++) {
    const unsigned long long K = CL == 2 ? max(keys[2 * (it % 3)], keys[2 * (it % 3) + 1]) : keys[2 * (it % 3)];
    if (tid == 0) keys[2 * ((it + 2) % 3)] = 0ull;      // slot of iteration it + 1's sweep: nobody reads or fills it now
    if (it == a.iterations) break;
    const int m = (int)(0xFFFFFFFFu - (uint32_t)K);
    BND(K != 0ull && m >= 0 && m < N);
    const float y = sqrtf(__uint_as_float((uint32_t)(K >> 32)));
    if (!(y > V)) { reason = PAPR_STOP_CLIP; break; }
    const int owner = m / H;
    const float2 cm = (CL == 1 || owner == (int)rank) ? c[m - owner * H] : cluster_map(c, (uint32_t)owner)[m - owner * H];
    if constexpr (CL == 2) cluster_arrive();      // c_m is read: the owner may update it once everyone has arrived
    const float s = (y - V) / y;
    const float bx = s * cm.x, by = s * cm.y;
    // the update's reserved-carrier values, dR_b = -beta exp(-j 2 pi b m / N) / (g |S|), checked against tone_max
    bool bad = false;
    for (int t = tid; t < S; t += T) {
      const int b = __ldg(bins + t);
      BND(b >= 0 && b < N);
      const float2 e = __ldg(a.tone_tw + (int)(((long long)b * m) & (N - 1)));
      const float2 r = make_float2(R[t].x - (bx * e.x - by * e.y) * a.tone_scale, R[t].y - (bx * e.y + by * e.x) * a.tone_scale);
      bad |= r.x * r.x + r.y * r.y > A2;
    }
    bad = __syncthreads_or(bad);
    if (bad) {
      if constexpr (CL == 2) cluster_wait();
      reason = PAPR_STOP_TONE;
      break;
    }
    for (int t = tid; t < S; t += T) {
      const int b = __ldg(bins + t);
      const float2 e = __ldg(a.tone_tw + (int)(((long long)b * m) & (N - 1)));
      R[t] = make_float2(R[t].x - (bx * e.x - by * e.y) * a.tone_scale, R[t].y - (bx * e.y + by * e.x) * a.tone_scale);
    }
    if constexpr (CL == 2) cluster_wait();
    // sweep: c_n -= beta p[(n - m) mod N] -- the kernel table streams from L2 in order, wrapping once
    key = 0ull;
    const int k0 = (int)rank * H - m;
    for (int j = tid; j < H; j += T) {
      const float2 q = __ldg(kern + ((k0 + j) & (N - 1)));
      float2 v = c[j];
      v.x -= bx * q.x - by * q.y;
      v.y -= bx * q.y + by * q.x;
      c[j] = v;
      key = max(key, papr_key(v, (int)rank * H + j));
    }
    papr_key_max<CL>(key, keys + 2 * ((it + 1) % 3), rkeys + 2 * ((it + 1) % 3));
    applied++;
    papr_sync<CL>();
  }
  if (rank == 0 && tid == 0) a.stats[unit] = (int16_t)(applied | reason << 8);

  typedef typename SinkT<FMT>::type sample_t;
  sample_t *sym = reinterpret_cast<sample_t *>(a.out) + sym0;
  const float gain = a.gain;
  if (!a.inplace || applied > 0) {
    BND(a.out_len == 0 || sym0 + a.gi + N <= a.out_len);
    const int cp_from = N - a.gi;
    for (int j = tid; j < H; j += T) {
      const int n = (int)rank * H + j;
      float2 v = c[j];
      if (!a.inplace) { v.x *= gain; v.y *= gain; }
      store_sample(sym, a.gi + n, v);
      if (n >= cp_from) store_sample(sym, n - cp_from, v);
    }
  }
  if (!a.inplace && l == 0 && rank == 0) {
    const float2 *p1 = a.in + (long long)f * a.spf;
    sample_t *o = reinterpret_cast<sample_t *>(a.out) + (long long)f * a.spf;
    for (int i = tid; i < 2048; i += T) {
      float2 v = __ldg(p1 + i);
      v.x *= gain; v.y *= gain;
      store_sample(o, i, v);
    }
  }
  if constexpr (CL == 2) papr_sync<CL>();      // no CTA leaves while its partner may still address its shared memory
}

template <int CL, int FMT>
static void launch_papr_t(const PaprArgs &a, cudaStream_t s)
{
  const int H = a.fft_n / CL;
  const int T = H >= 4096 ? PAPR_MAX_THREADS : (H / 4 < 256 ? 256 : H / 4);
  const size_t smem = (size_t)H * sizeof(float2) + (size_t)a.tones * sizeof(float2) + 6 * sizeof(unsigned long long);
  static bool attr[MAX_DEVICES];
  allow_smem(k_papr_tr<CL, FMT>, 227 * 1024, attr);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(a.frames * a.num_symbols * CL));
  cfg.blockDim = dim3((unsigned)T);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, k_papr_tr<CL, FMT>, a);
  count_launch();
}

void launch_papr_tr(const PaprArgs &a, cudaStream_t s)
{
  if (a.frames * a.num_symbols < 1) return;
  if (a.fft_n > 16384) {
    if (a.out_fmt) launch_papr_t<2, 1>(a, s);
    else launch_papr_t<2, 0>(a, s);
  }
  else {
    if (a.out_fmt) launch_papr_t<1, 1>(a, s);
    else launch_papr_t<1, 0>(a, s);
  }
}

} // namespace t2k
