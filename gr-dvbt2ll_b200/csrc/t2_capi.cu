// C ABI of libdvbt2ll_cuda.so (declared in include/dvbt2ll_cuda.h): handles own the host plan, the
// device copies of its tables, a CUDA stream and scratch buffers.  There is no CPU fallback: every
// *_work() call needs a CUDA device and fails with DVBT2LL_ERR_CUDA otherwise.
#include "../../include/dvbt2ll_cuda.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "t2_kernels.cuh"
#include "t2_plan.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) { g_err = msg; return code; }

#define CK(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) {                                                                      \
      cudaGetLastError(); /* not sticky: the next call must not inherit it */                     \
      return fail(DVBT2LL_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
    }                                                                                             \
  } while (0)

struct DevBuf {
  void *p; size_t cap;
  DevBuf() : p(0), cap(0) {}
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t ensure(size_t n)
  {
    if (n <= cap) return cudaSuccess;
    if (p) { cudaFree(p); p = 0; cap = 0; }
    cudaError_t e = cudaMalloc(&p, n);
    if (e == cudaSuccess) cap = n;
    return e;
  }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

template <class T>
cudaError_t upload(DevBuf &b, const std::vector<T> &v)
{
  cudaError_t e = b.ensure(v.size() * sizeof(T) + 16);
  if (e != cudaSuccess) return e;
  return cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
}

inline int align16(int n) { return (n + 15) & ~15; }

std::vector<t2::cfloat> make_twiddles(int n, int count)
{
  std::vector<t2::cfloat> w(count);
  const double k2pi = 6.283185307179586476925286766559;
  for (int i = 0; i < count; i++) {
    w[i].re = (float)std::cos(k2pi * i / n);
    w[i].im = (float)std::sin(k2pi * i / n);
  }
  return w;
}

// TS byte index, in a stream that starts on a packet boundary, at which FECFRAME j begins: j FECFRAMEs of `payload`
// bytes, 13 fewer for the first FECFRAME of every in-band signalling cycle of `cycle` FECFRAMEs (0: no in-band
// signalling).  In high efficiency mode the sync byte in front of every 187 payload bytes is not carried, and FECFRAME
// j starts right behind the last payload byte of FECFRAME j - 1.
long long ts_stream_pos(long long j, int payload, int cycle, int mode)
{
  const long long P = j * payload - (cycle > 0 ? 13 * ((j + cycle - 1) / cycle) : 0);     // payload bytes before it
  if (mode == t2::INPUTMODE_NORMAL || P == 0) return P;
  return P + (P - 1) / 187 + 1;
}

// Stream state of a TS-consuming handle (the drop-in BB block, the chain's generic work path), carried across calls
struct TsStream {
  long long fecframes;            // FECFRAMEs consumed so far
  uint8_t history[187];           // last 187 TS bytes consumed (CRC-8 of the packet in flight)
  int *h_err;                     // sync-error counter in mapped pinned host memory: no copy back per call
  TsStream() : fecframes(0), h_err(0) { std::memset(history, 0, sizeof(history)); }
  ~TsStream() { if (h_err) cudaFreeHost(h_err); }
  int init()
  {
    if (!h_err) {
      CK(cudaHostAlloc((void **)&h_err, 16, cudaHostAllocMapped | cudaHostAllocPortable));
      std::memset(h_err, 0, 16);
    }
    return 0;
  }
  // slide the 187-byte history window over `used` newly consumed bytes
  void note_consumed(const uint8_t *in, long long used)
  {
    if (used >= 187) std::memcpy(history, in + used - 187, 187);
    else if (used > 0) {
      std::memmove(history, history + used, 187 - (size_t)used);
      std::memcpy(history + 187 - used, in, (size_t)used);
    }
  }
};

} // namespace

// Device-resident hand-off between two adjacent drop-in blocks (dvbt2ll_link): the producer's last NSLOT outputs, each
// with the host range it stands for and the device buffer the same items still sit in.  A ring, not one record, because
// a scheduler with a thread per block lets the producer run ahead of its consumer by as many calls as the host buffer
// between them has room for.  The mutex is held only around the look-up / update of the records and the enqueueing of
// the consumer's kernels: the producer's reuse of a slot is ordered behind those kernels by an event on its own
// stream, so adjacent blocks driven by different threads still overlap.
// lazy (dvbt2ll_link_lazy_host): the producer leaves the host buffer unwritten; `pending` says a slot's items exist only
// in HBM, `taken_to` how far from the start the consumer has taken them.  Whatever was not taken is written to the host
// buffer before the slot is reused, and at once when the consumer asks for the range some other way (a miss), so the
// stream is never lost -- only late for readers other than the linked consumer.
struct LinkRec {
  enum { NSLOT = 4 };
  struct Slot {
    const uint8_t *host; size_t bytes; DevBuf buf; bool valid, pending; size_t taken_to;
    cudaEvent_t taken_ev; bool taken_valid;      // recorded behind the consumer's kernels that read `buf`
    Slot() : host(0), bytes(0), valid(false), pending(false), taken_to(0), taken_ev(0), taken_valid(false) {}
    ~Slot() { if (taken_ev) { cudaEventDestroy(taken_ev); cudaGetLastError(); } }
  } slot[NSLOT];
  std::mutex m;
  long long hits, misses, late_writes;
  bool lazy;
  int next;                                      // slot the producer's next call fills (the oldest)
  int item;                                      // bytes per item of the producer's output
  LinkRec() : hits(0), misses(0), late_writes(0), lazy(false), next(0), item(0) {}
};

// Automatic hand-off (dvbt2ll_set_auto_link / DVBT2LL_AUTO_LINK=1): every drop-in block keeps its outputs resident and
// registers its record here; a block that was not linked explicitly looks its input range up in the records of all the
// others, so a flowgraph built by unchanged Python gets the device-resident hand-off without calling dvbt2ll_link.
struct AutoLinks {
  std::mutex m;
  std::vector<std::weak_ptr<LinkRec> > recs;
  int on;
  AutoLinks() : on(-1) {}
  static AutoLinks &get() { static AutoLinks a; return a; }
  bool enabled()
  {
    std::lock_guard<std::mutex> g(m);
    if (on < 0) { const char *e = std::getenv("DVBT2LL_AUTO_LINK"); on = (e && e[0] == '1') ? 1 : 0; }
    return on == 1;
  }
  void add(const std::shared_ptr<LinkRec> &r) { std::lock_guard<std::mutex> g(m); recs.push_back(r); }
  void snapshot(std::vector<std::shared_ptr<LinkRec> > &out)
  {
    std::lock_guard<std::mutex> g(m);
    size_t w = 0;
    for (size_t i = 0; i < recs.size(); i++) {
      std::shared_ptr<LinkRec> p = recs[i].lock();
      if (p) { out.push_back(p); recs[w++] = recs[i]; }
    }
    recs.resize(w);
  }
};

// Process-wide registry of host page ranges registered by this library (cudaHostRegister), shared by all handles.
struct PinRegistry {
  struct Iv { uintptr_t a0, a1; std::vector<const void *> users; };
  std::mutex m;
  std::vector<Iv> ivs;            // disjoint page ranges registered by us
  static PinRegistry &get() { static PinRegistry r; return r; }
  static void add_user(Iv &iv, const void *u)
  {
    for (size_t i = 0; i < iv.users.size(); i++) if (iv.users[i] == u) return;
    iv.users.push_back(u);
  }
  void acquire(const void *user, uintptr_t p0, uintptr_t p1)
  {
    std::lock_guard<std::mutex> g(m);
    // gaps of [p0, p1) not covered by our ranges
    std::vector<Iv> sorted(ivs);
    std::sort(sorted.begin(), sorted.end(), [](const Iv &x, const Iv &y) { return x.a0 < y.a0; });
    std::vector<std::pair<uintptr_t, uintptr_t> > gaps;
    uintptr_t cur = p0;
    for (size_t i = 0; i < sorted.size() && cur < p1; i++) {
      if (sorted[i].a1 <= cur) continue;
      if (sorted[i].a0 >= p1) break;
      if (sorted[i].a0 > cur) gaps.push_back(std::make_pair(cur, sorted[i].a0));
      cur = sorted[i].a1;
    }
    if (cur < p1) gaps.push_back(std::make_pair(cur, p1));
    size_t done = 0;
    for (; done < gaps.size(); done++) {
      cudaPointerAttributes at;
      const bool foreign = cudaPointerGetAttributes(&at, (const void *)gaps[done].first) == cudaSuccess && at.type != cudaMemoryTypeUnregistered;
      cudaGetLastError();
      if (foreign || cudaHostRegister((void *)gaps[done].first, gaps[done].second - gaps[done].first, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        break;
      }
    }
    if (done < gaps.size()) {      // could not cover everything: undo this call's pieces, the range stays as it was
      for (size_t i = 0; i < done; i++) cudaHostUnregister((void *)gaps[i].first);
      cudaGetLastError();
      return;
    }
    for (size_t i = 0; i < gaps.size(); i++) {
      Iv iv; iv.a0 = gaps[i].first; iv.a1 = gaps[i].second;
      ivs.push_back(iv);
    }
    for (size_t i = 0; i < ivs.size(); i++)
      if (ivs[i].a0 < p1 && p0 < ivs[i].a1) add_user(ivs[i], user);
  }
  // boundaries of our registered ranges that fall strictly inside [p0, p1), ascending: a copy must not span two
  // separately registered ranges (or a registered and a pageable one), so it is issued piece by piece
  void cuts(uintptr_t p0, uintptr_t p1, std::vector<uintptr_t> &out)
  {
    std::lock_guard<std::mutex> g(m);
    for (size_t i = 0; i < ivs.size(); i++) {
      if (ivs[i].a0 > p0 && ivs[i].a0 < p1) out.push_back(ivs[i].a0);
      if (ivs[i].a1 > p0 && ivs[i].a1 < p1) out.push_back(ivs[i].a1);
    }
    std::sort(out.begin(), out.end());
    out.erase(std::unique(out.begin(), out.end()), out.end());
  }
  void release_all(const void *user)
  {
    std::lock_guard<std::mutex> g(m);
    for (size_t i = 0; i < ivs.size();) {
      std::vector<const void *> &u = ivs[i].users;
      u.erase(std::remove(u.begin(), u.end(), user), u.end());
      if (u.empty()) {
        cudaHostUnregister((void *)ivs[i].a0);
        cudaGetLastError();
        ivs.erase(ivs.begin() + i);
      }
      else i++;
    }
  }
};

// ------------------------------------------------------------------------------------------------
struct dvbt2ll_handle {
  enum Kind { BB, LDPC, MAP, FRAME, OFDM, CHAIN } kind;
  cudaStream_t stream;
  bool dev_ready;
  int warnings;
  DevBuf stage_in, stage_out;   // device staging for host-buffer work()
  // host buffers registered with cudaHostRegister on first sight (the scheduler's buffers are long-lived and reused)
  struct Pinned { uintptr_t a0, a1; };
  std::vector<Pinned> pinned;   // page ranges this handle has already asked the registry for (lock-free fast path)
  bool pin_enabled;
  std::shared_ptr<LinkRec> link_in, link_out;     // set by dvbt2ll_link (link_out also by the automatic hand-off)
  std::weak_ptr<LinkRec> auto_in;                 // automatic hand-off: where the input was found last time
  long long auto_hits;
  explicit dvbt2ll_handle(Kind k) : kind(k), stream(0), dev_ready(false), warnings(0), pin_enabled(false), auto_hits(0), bounce(0), bounce_cap(0), bounced_copies(0)
  {
    // opt-in (dvbt2ll_set_host_register or the environment): only safe when the caller's buffers outlive the handle,
    // as the GNU Radio scheduler's do -- a registration must never survive the munmap of its pages
    const char *e = std::getenv("DVBT2LL_HOST_REGISTER");
    if (e && e[0] == '1') pin_enabled = true;
  }
  virtual ~dvbt2ll_handle()
  {
    if (!pinned.empty()) PinRegistry::get().release_all(this);
    if (bounce) cudaFreeHost(bounce);
    if (stream) cudaStreamDestroy(stream);
  }
  // Make [p, p + n) page-locked (page granular).  Adjacent blocks share buffers (one's output is the next one's input)
  // and heap buffers share pages, so registrations are kept in one process-wide registry that only ever registers
  // the pages nobody registered yet: a copy never sees a partly registered range (CUDA rejects those).  Failure is
  // not an error: the copy then runs from pageable memory.
  // Only the pages that lie WHOLLY inside the buffer are registered: a page shared with some other heap object would
  // leave that object half registered, and CUDA rejects any copy from such a range (seen as "invalid argument" on a
  // plan-table upload whose std::vector happened to sit next to a registered buffer).  The up to two partial pages at
  // the ends travel as small pageable pieces (copy_host splits at the boundaries).
  void pin(const void *p, size_t n)
  {
    if (!pin_enabled || !p || n < (1u << 16)) return;
    const uintptr_t a0 = ((uintptr_t)p + 4095) & ~(uintptr_t)4095, a1 = ((uintptr_t)p + n) & ~(uintptr_t)4095;
    if (a1 <= a0) return;
    for (size_t i = 0; i < pinned.size(); i++)
      if (a0 >= pinned[i].a0 && a1 <= pinned[i].a1) return;
    if (pinned.size() >= 64) return;
    PinRegistry::get().acquire(this, a0, a1);
    Pinned e = { a0, a1 };
    pinned.push_back(e);
  }
  // host <-> device copy of a caller buffer on `s`, split at the boundaries of registered ranges when registration is on.
  // CUDA refuses a copy whose host range is only partly page-locked (e.g. pages some other component registered or
  // unregistered behind our back): such a piece goes through a page-locked bounce buffer of our own instead.
  void *bounce;
  size_t bounce_cap;
  long long bounced_copies;
  cudaError_t copy_piece(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s)
  {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, s);
    if (e == cudaSuccess || !pin_enabled) return e;
    cudaGetLastError();
    const size_t chunk = (size_t)4 << 20;
    if (!bounce) {
      if (cudaHostAlloc(&bounce, chunk, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return e; }
      bounce_cap = chunk;
    }
    bounced_copies++;
    for (size_t off = 0; off < bytes; off += bounce_cap) {
      const size_t n = bytes - off < bounce_cap ? bytes - off : bounce_cap;
      if (kind == cudaMemcpyHostToDevice) {
        std::memcpy(bounce, (const char *)src + off, n);
        if ((e = cudaMemcpyAsync((char *)dst + off, bounce, n, kind, s)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
      }
      else {
        if ((e = cudaMemcpyAsync(bounce, (const char *)src + off, n, kind, s)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
        std::memcpy((char *)dst + off, bounce, n);
      }
    }
    return cudaSuccess;
  }
  cudaError_t copy_host(void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s)
  {
    if (!pin_enabled || pinned.empty()) return cudaMemcpyAsync(dst, src, bytes, kind, s);
    const uintptr_t h0 = (uintptr_t)(kind == cudaMemcpyHostToDevice ? src : dst);
    std::vector<uintptr_t> cut;
    PinRegistry::get().cuts(h0, h0 + bytes, cut);
    cut.push_back(h0 + bytes);
    size_t off = 0;
    for (size_t i = 0; i < cut.size(); i++) {
      const size_t end = cut[i] - h0;
      cudaError_t e = copy_piece((char *)dst + off, (const char *)src + off, end - off, kind, s);
      if (e != cudaSuccess) return e;
      off = end;
    }
    return cudaSuccess;
  }
  virtual int output_multiple() const = 0;
  virtual int forecast(int noutput) const = 0;
  virtual int in_item() const = 0;
  virtual int out_item() const = 0;
  virtual int dev_init() = 0;
  // device-resident work on the given stream
  virtual int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s) = 0;
  // items work() must copy in for noutput outputs
  virtual long long input_items(int noutput) const { return forecast(noutput); }
  // TS-consuming handles (the BB block, the chain): their stream state, and work_device told whether the 187 bytes in
  // front of d_in hold the stream's history (work() puts it there; device-resident callers keep it there once anything
  // has been consumed)
  virtual TsStream *ts_stream() { return 0; }
  virtual int work_ts(const void *, int, void *, int, int *, cudaStream_t, int) { return fail(DVBT2LL_ERR_INVALID, "not a TS-consuming handle"); }
  virtual long long plan_get(const char *name, void *out, long long cap) const = 0;

  virtual int enter() { return ensure_device(); }
  int ensure_device()
  {
    if (dev_ready) return 0;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1) {
      cudaGetLastError();
      return fail(DVBT2LL_ERR_CUDA, "no CUDA device available (libdvbt2ll_cuda has no CPU fallback)");
    }
    if (!stream) CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    int r = dev_init();
    if (r) return r;
    dev_ready = true;
    return 0;
  }
};

namespace {

long long copy_out(const void *src, size_t bytes, void *out, long long cap)
{
  if (out && cap > 0) std::memcpy(out, src, (size_t)cap < bytes ? (size_t)cap : bytes);
  return (long long)bytes;
}
template <class T>
long long copy_vec(const std::vector<T> &v, void *out, long long cap) { return copy_out(v.data(), v.size() * sizeof(T), out, cap); }

long long dims_get(const t2::OfdmDims &d, void *out, long long cap)
{
  const int v[16] = { d.fft_n, d.fft_index, d.miso, d.n_p2, d.c_p2, d.c_data, d.n_fc, d.c_fc, d.c_ps, d.k_ext,
                      d.k_offset, d.dx, d.dy, d.gi, d.num_symbols, d.active_items };
  return copy_out(v, sizeof(v), out, cap);
}

// ================================================================================================
// BB framing + BCH (k_bb_bch): the plan, its device tables and the kernel's launch arguments, shared by the drop-in
// block and the chain's parameter sets
struct BbStage {
  t2::BbPlan plan;
  DevBuf d_scr, d_crc, d_tab, d_cols, d_ib;
  uint32_t crc_pos_mask[47][8];
  int init()
  {
    std::vector<uint8_t> scr(plan.scramble);
    scr.resize((scr.size() + 7) & ~(size_t)3, 0);      // kernel XORs the scrambler word-wise
    CK(upload(d_scr, scr));
    CK(upload(d_crc, std::vector<uint8_t>(plan.crc8_tab, plan.crc8_tab + 256)));   // byte table: the BB header's CRC-8
    // CRC-8 slicing-by-4 tables: S1 = byte table, S(k+1)[x] = S1[Sk[x]] (a byte followed by k zero bytes)
    std::vector<uint8_t> crc(1024);
    for (int x = 0; x < 256; x++) {
      uint8_t v = plan.crc8_tab[x];
      for (int k = 0; k < 4; k++) { crc[k * 256 + x] = v; v = plan.crc8_tab[v]; }
    }
    // the same four-byte step as parity masks (GF(2)-linear in the 32 bits): byte i of the word is followed by 3 - i more
    uint32_t crc_mask[8];
    for (int k = 0; k < 8; k++) {
      crc_mask[k] = 0;
      for (int i = 0; i < 4; i++)
        for (int j = 0; j < 8; j++)
          if ((crc[(3 - i) * 256 + (1 << j)] >> k) & 1) crc_mask[k] |= 1u << (8 * i + j);
    }
    // the whole packet at once: word j (of 47) contributes M4 followed by 46 - j further four-byte steps of its
    // 8-bit image; mask[j][k] collects the input bits that reach CRC bit k; the leading byte of word 0 is not data
    {
      auto step = [&](uint32_t t) { uint32_t c = 0; for (int k = 0; k < 8; k++) c |= (uint32_t)(__builtin_popcount(t & crc_mask[k]) & 1) << k; return c; };
      std::memset(crc_pos_mask, 0, sizeof(crc_pos_mask));
      for (int j = 0; j < 47; j++)
        for (int bit = 0; bit < 32; bit++) {
          uint32_t v = step(1u << bit);
          for (int r = 0; r < 46 - j; r++) v = step(v);
          for (int k = 0; k < 8; k++) if ((v >> k) & 1u) crc_pos_mask[j][k] |= 1u << bit;
        }
      for (int k = 0; k < 8; k++) crc_pos_mask[0][k] &= 0xFFFFFF00u;
    }
    CK(upload(d_tab, plan.bch_byte_tab));
    CK(upload(d_cols, plan.bch_shift_cols));
    CK(upload(d_ib, plan.inband_bytes));
    return 0;
  }
  // sync_errors: the caller's counter of payload sync bytes != 0x47 (device-visible)
  void fill_args(t2k::BbArgs &a, const uint8_t *d_ts_ptr, long long pitch, int channels, int frames, int count0,
                 int fb0, int hist_valid, uint8_t *d_out, int out_pitch, int *sync_errors) const
  {
    a.ts = d_ts_ptr; a.ts_pitch = pitch; a.hist_valid = hist_valid; a.n_channels = channels; a.frames = frames;
    a.count0 = count0; a.fec_block0 = fb0;
    a.kbch = plan.fec.kbch; a.nbch = plan.fec.nbch; a.bch_r = plan.fec.bch_r; a.payload_bytes = plan.payload_bytes;
    a.mode = plan.mode; a.inband = plan.inband ? 1 : 0; a.fecblocks = plan.fecblocks;
    a.chunk_bytes = plan.chunk_bytes; a.lead_zero_bytes = plan.lead_zero_bytes;
    a.scramble = d_scr.as<uint8_t>(); a.crc8_tab = d_crc.as<uint8_t>(); a.bch_tab = d_tab.as<uint32_t>();
    std::memcpy(a.crc8_pos_mask, crc_pos_mask, sizeof(crc_pos_mask));
    a.bch_cols = d_cols.as<uint32_t>(); a.inband_bytes = d_ib.as<uint8_t>();
    a.out = d_out; a.out_pitch = out_pitch; a.sync_errors = sync_errors;
    a.ts_len = 0; a.out_len = (long long)channels * frames * out_pitch;
    a.out_group = 0; a.out_group_stride = 0; a.out_group_off = 0;
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "bb.scramble") return copy_vec(plan.scramble, out, cap);
    if (n == "bb.crc8") return copy_out(plan.crc8_tab, 256, out, cap);
    if (n == "bb.bch_tab") return copy_vec(plan.bch_byte_tab, out, cap);
    if (n == "bb.bch_cols") return copy_vec(plan.bch_shift_cols, out, cap);
    if (n == "bb.inband") return copy_vec(plan.inband_bytes, out, cap);
    if (n == "bb.dims") {
      const int v[8] = { plan.fec.kbch, plan.fec.nbch, plan.fec.q, plan.fec.bch_r, plan.payload_bytes,
                         plan.chunk_bytes, plan.lead_zero_bytes, plan.fec.nldpc };
      return copy_out(v, sizeof(v), out, cap);
    }
    return -1;
  }
};

// the drop-in block: the stage, its stream state and the conversion of its packed codewords to one bit per byte
struct BbHandle : dvbt2ll_handle {
  BbStage st;
  TsStream ts;
  DevBuf d_packed;
  BbHandle() : dvbt2ll_handle(BB) {}
  TsStream *ts_stream() override { return &ts; }
  int output_multiple() const { return st.plan.fec.nbch; }
  int in_item() const { return 1; }
  int out_item() const { return 1; }
  int forecast(int noutput) const
  {
    // reference :207-216
    const t2::BbPlan &p = st.plan;
    const int base = (noutput - 80 - (p.fec.nbch - p.fec.kbch)) / 8;
    return p.mode == t2::INPUTMODE_NORMAL ? base : base + ((p.fec.kbch - 80) / 8) / 187 + 1;
  }
  int dev_init()
  {
    int r = st.init();
    return r ? r : ts.init();
  }
  // TS byte index at which FECFRAME j starts: one in-band signalling cycle per `fecblocks` FECFRAMEs
  long long stream_pos(long long j) const { return ts_stream_pos(j, st.plan.payload_bytes, st.plan.inband ? st.plan.fecblocks : 0, st.plan.mode); }
  long long input_items(int noutput) const override
  {
    return stream_pos(ts.fecframes + noutput / st.plan.fec.nbch) - stream_pos(ts.fecframes);
  }
  // the 187 bytes before d_in are read once anything has been consumed (see the header); at the very start of the
  // stream the history is all zero by definition
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    return work_ts(d_in, ninput, d_out, noutput, consumed, s, ts.fecframes > 0 ? 1 : 0);
  }
  int work_ts(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s, int hist_valid) override
  {
    const t2::BbPlan &p = st.plan;
    const int frames = noutput / p.fec.nbch;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    const long long need = input_items(noutput);
    if (ninput < need) return fail(DVBT2LL_ERR_SHORT, "bbheaderbch_bb: not enough input items");
    const int pitch = align16(p.fec.nbch / 8);
    CK(d_packed.ensure((size_t)frames * pitch));
    t2k::BbArgs a;
    st.fill_args(a, (const uint8_t *)d_in, 0, 1, frames, (int)(stream_pos(ts.fecframes) % 188),
                 p.inband ? (int)(ts.fecframes % p.fecblocks) : 0, hist_valid, d_packed.as<uint8_t>(), pitch, ts.h_err);
    a.ts_len = ninput;
    t2k::launch_bb_bch(a, s);
    t2k::launch_unpack_bits(d_packed.as<uint8_t>(), pitch, p.fec.nbch, (uint8_t *)d_out, frames, s);
    CK(cudaGetLastError());
    ts.fecframes += frames;
    if (consumed) *consumed = (int)need;
    return frames * p.fec.nbch;
  }
  long long plan_get(const char *name, void *out, long long cap) const { return st.plan_get(name, out, cap); }
};

// ================================================================================================
// LDPC encoding (k_ldpc), shared like BbStage
struct LdpcStage {
  t2::LdpcPlan plan;
  DevBuf d_rowptr, d_entries;
  int lane_per_row = 0;     // accumulation scheme of k_ldpc, chosen per code in init (DVBT2LL_LDPC_MODE=0|1 overrides)
  int init()
  {
    CK(upload(d_rowptr, plan.row_ptr));
    CK(upload(d_entries, plan.entries));
    // measured on B200 (tools/ldpc_mode_sweep.py, profiles/r2_ldpc_modes.txt)
    lane_per_row = ldpc_lane_per_row_default(plan.fec.nldpc, plan.fec.q);
    const char *e = std::getenv("DVBT2LL_LDPC_MODE");
    if (e && (e[0] == '0' || e[0] == '1')) lane_per_row = e[0] - '0';
    return 0;
  }
  static int ldpc_lane_per_row_default(int nldpc, int q)
  {
    // a lane per row wins for the low-rate codes (few table entries per row: the per-(row, word) bookkeeping dominates),
    // a lane per (row, word) for the others (consecutive lanes read consecutive words: fewer bank conflicts)
    return nldpc == 64800 ? (q >= 90 ? 1 : 0) : (q >= 18 ? 1 : 0);
  }
  void fill_args(t2k::LdpcArgs &a, const uint8_t *in, int in_pitch, uint8_t *out, int out_pitch, int frames) const
  {
    a.in = in; a.in_pitch = in_pitch; a.out = out; a.out_pitch = out_pitch; a.frames = frames;
    a.nbch = plan.fec.nbch; a.nldpc = plan.fec.nldpc; a.q = plan.fec.q; a.groups = plan.groups;
    a.row_ptr = d_rowptr.as<uint16_t>(); a.entries = d_entries.as<uint32_t>();
    a.lane_per_row = lane_per_row;
    a.in_len = (long long)frames * in_pitch + 64; a.out_len = (long long)frames * out_pitch;
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "ldpc.row_ptr") return copy_vec(plan.row_ptr, out, cap);
    if (n == "ldpc.entries") return copy_vec(plan.entries, out, cap);
    return -1;
  }
};

// the drop-in block: the stage and the conversion between one bit per byte and packed codewords
struct LdpcHandle : dvbt2ll_handle {
  LdpcStage st;
  DevBuf d_in_packed, d_out_packed;
  LdpcHandle() : dvbt2ll_handle(LDPC) {}
  int output_multiple() const { return st.plan.fec.nldpc; }
  int in_item() const { return 1; }
  int out_item() const { return 1; }
  int forecast(int noutput) const { return (noutput / st.plan.fec.nldpc) * st.plan.fec.nbch; }
  int dev_init() { return st.init(); }
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    const t2::FecSpec &f = st.plan.fec;
    const int frames = noutput / f.nldpc;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    if (ninput < frames * f.nbch) return fail(DVBT2LL_ERR_SHORT, "ldpc: not enough input items");
    const int ip = align16(f.nbch / 8), op = align16(f.nldpc / 8);
    CK(d_in_packed.ensure((size_t)frames * ip + 64));
    CK(d_out_packed.ensure((size_t)frames * op + 16));
    t2k::launch_pack_bits((const uint8_t *)d_in, f.nbch, d_in_packed.as<uint8_t>(), ip, frames, s);
    t2k::LdpcArgs a;
    st.fill_args(a, d_in_packed.as<uint8_t>(), ip, d_out_packed.as<uint8_t>(), op, frames);
    t2k::launch_ldpc(a, s);
    t2k::launch_unpack_ldpc(d_out_packed.as<uint8_t>(), op, f.nbch, f.nldpc, f.q, (uint8_t *)d_out, frames, s);
    CK(cudaGetLastError());
    if (consumed) *consumed = frames * f.nbch;
    return frames * f.nldpc;
  }
  long long plan_get(const char *name, void *out, long long cap) const { return st.plan_get(name, out, cap); }
};

// ================================================================================================
// bit interleaving + constellation mapping (k_map), shared like BbStage
struct MapStage {
  t2::MapPlan plan;
  DevBuf d_bitsrc, d_lut, d_qlut;
  int init()
  {
    CK(upload(d_bitsrc, plan.bit_src));
    CK(upload(d_lut, plan.lut));
    if (!plan.qpsk_lut.empty()) CK(upload(d_qlut, plan.qpsk_lut));
    return 0;
  }
  void fill_args(t2k::MapArgs &a, const uint8_t *in, int in_pitch, float2 *out, int frames) const
  {
    a.in = in; a.in_pitch = in_pitch; a.out = out; a.frames = frames;
    a.nldpc = plan.fec.nldpc; a.mod = plan.mod; a.cell_size = plan.cell_size; a.cyclic_delay = plan.cyclic_delay;
    a.bit_src = d_bitsrc.as<uint16_t>(); a.lut = d_lut.as<float2>();
    a.qpsk_lut = plan.qpsk_lut.empty() ? 0 : d_qlut.as<uint2>(); a.qpsk_lin_cells = a.qpsk_lut ? plan.qpsk_lin_cells : 0;
    a.qpsk_par_q = a.qpsk_lut ? plan.qpsk_par_q : 0; a.qpsk_nbch = plan.qpsk_nbch;
    a.ci_inv = 0; a.ci_inv4 = 0; a.ci_inv4_stride = 0; a.fec_shift = 0; a.fecblocks = 1; a.out16 = 0; a.out16_frame_stride = 0;
    a.in_len = (long long)frames * in_pitch; a.out_len = 0;
    a.ncol = plan.ncol;
    a.im_from_re = plan.im_from_re; a.im_mask_i = plan.im_mask_i; a.im_mask_q = plan.im_mask_q; a.im_flip = plan.im_flip;
    std::memcpy(a.col_of_bit, plan.col_of_bit, 16);
    std::memcpy(a.twist_of_col, plan.twist_of_col, 16);
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "map.bit_src") return copy_vec(plan.bit_src, out, cap);
    if (n == "map.lut") return copy_vec(plan.lut, out, cap);
    if (n == "map.qpsk") { const int v[3] = { plan.qpsk_lin_cells, plan.qpsk_par_q, plan.qpsk_nbch }; return copy_out(v, sizeof(v), out, cap); }
    if (n == "map.im_from_re") { const int v[4] = { plan.im_from_re, (int)plan.im_mask_i, (int)plan.im_mask_q, (int)plan.im_flip }; return copy_out(v, sizeof(v), out, cap); }
    return -1;
  }
};

// the drop-in block: the stage and the packing of the codeword items
struct MapHandle : dvbt2ll_handle {
  MapStage st;
  DevBuf d_packed;
  MapHandle() : dvbt2ll_handle(MAP) {}
  int output_multiple() const { return st.plan.cell_size; }
  int in_item() const { return 1; }
  int out_item() const { return 8; }
  int forecast(int noutput) const { return (noutput / st.plan.cell_size) * st.plan.fec.nldpc; }
  int dev_init() { return st.init(); }
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    const t2::MapPlan &p = st.plan;
    const int frames = noutput / p.cell_size;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    if (ninput < frames * p.fec.nldpc) return fail(DVBT2LL_ERR_SHORT, "interleavermod_bc: not enough input items");
    const int ip = align16(p.fec.nldpc / 8);
    CK(d_packed.ensure((size_t)frames * ip + 16));
    t2k::launch_pack_ldpc((const uint8_t *)d_in, p.fec.nbch, p.fec.nldpc, p.fec.q, d_packed.as<uint8_t>(), ip, frames, s);
    t2k::MapArgs a;
    st.fill_args(a, d_packed.as<uint8_t>(), ip, (float2 *)d_out, frames);
    t2k::launch_map(a, s);
    CK(cudaGetLastError());
    if (consumed) *consumed = frames * p.fec.nldpc;
    return frames * p.cell_size;
  }
  long long plan_get(const char *name, void *out, long long cap) const { return st.plan_get(name, out, cap); }
};

// ================================================================================================
struct FrameHandle : dvbt2ll_handle {
  t2::FramePlan plan;
  DevBuf d_code, d_pool;
  int t2_frame_num;
  FrameHandle() : dvbt2ll_handle(FRAME), t2_frame_num(0) {}
  int output_multiple() const { return plan.mapped_items; }
  int in_item() const { return 8; }
  int out_item() const { return 8; }
  int forecast(int noutput) const { return plan.stream_items * (noutput / plan.mapped_items); }
  int dev_init()
  {
    CK(upload(d_code, plan.code));
    CK(upload(d_pool, plan.pool.cells));
    return 0;
  }
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    const int frames = noutput / plan.mapped_items;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    if ((long long)ninput < (long long)frames * plan.stream_items)
      return fail(DVBT2LL_ERR_SHORT, "framemapperfint_cc: not enough input items");
    t2k::GatherArgs a;
    a.in = (const float2 *)d_in; a.in_stride = plan.stream_items;
    a.out = (float2 *)d_out; a.out_stride = plan.mapped_items;
    a.code = d_code.as<int32_t>(); a.n = plan.mapped_items; a.pool = d_pool.as<float2>();
    a.l1post_base = plan.pool.l1post_base; a.l1post_cells = plan.pool.l1post_cells; a.l1post_variants = plan.pool.l1post_variants;
    a.frames = frames; a.frame_idx0 = t2_frame_num;
    t2k::launch_gather(a, s);
    CK(cudaGetLastError());
    t2_frame_num = (t2_frame_num + frames) % plan.prm.t2frames;
    if (consumed) *consumed = frames * plan.stream_items;
    return frames * plan.mapped_items;
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "frame.code") return copy_vec(plan.code, out, cap);
    if (n == "frame.pool") return copy_vec(plan.pool.cells, out, cap);
    if (n == "frame.cell_perm") return copy_vec(plan.cell_perm, out, cap);
    if (n == "frame.fec_shift") return copy_vec(plan.fec_shift, out, cap);
    if (n == "frame.ci_dst") return copy_vec(plan.ci_dst, out, cap);
    if (n == "frame.ti_src") return copy_vec(plan.ti_src, out, cap);
    if (n == "frame.dims") return dims_get(plan.dims, out, cap);
    if (n == "frame.info") {
      const int v[12] = { plan.cell_size, plan.stream_items, plan.mapped_items, plan.eta_mod, plan.n_post, plan.n_punc,
                          plan.dummy_cells, plan.pool.l1post_base, plan.pool.l1post_cells, plan.pool.l1post_variants,
                          plan.pool_dummy, plan.pool_zero };
      return copy_out(v, sizeof(v), out, cap);
    }
    return -1;
  }
};

// ================================================================================================
struct OfdmDevice {
  DevBuf d_code, d_pool, d_p1, d_sinc, d_tw, d_tw_split, d_sym_flags;
  int log2_m, split;
  long long pool_stride;
  // c16: `code` holds staging slots (chain mode, 16-bit cells) and is re-encoded as the chain-mode carrier codes of
  // t2_kernels.cuh (2 * slot | (small pool cell + 1) << 17 | 0x80000000 + pool cell) for the kernel's branch-free fill;
  // with tab_base (several constellation tables) a data carrier's code also carries the first table entry of its cell's
  // PLP, tab_base[plp[carrier]] << OFDM_CODE_TAB_SHIFT; with miso (MISO group-2 codes, t2::compose_miso) a data carrier
  // whose cell sits at an odd place i of its symbol (op.code - op.sym_data_start) also carries OFDM_CODE_MISO_IM
  int init(const std::vector<int32_t> &code, const t2::CellPool &pool, const t2::OfdmPlan &op, bool c16 = false,
           const std::vector<uint8_t> *plp = 0, const int *tab_base = 0, bool miso = false)
  {
    // one copy of the pool per L1-post variant: in copy v the L1-post slot holds variant v, so the kernel
    // selects a pool base per frame instead of patching indices per cell
    {
      const int nv = pool.l1post_variants > 0 ? pool.l1post_variants : 1;
      pool_stride = (long long)pool.cells.size();
      std::vector<t2::cfloat> rep((size_t)nv * pool.cells.size());
      for (int v = 0; v < nv; v++) {
        std::copy(pool.cells.begin(), pool.cells.end(), rep.begin() + (size_t)v * pool.cells.size());
        for (int i = 0; i < pool.l1post_cells; i++)
          rep[(size_t)v * pool.cells.size() + pool.l1post_base + i] = pool.cells[pool.l1post_base + (size_t)v * pool.l1post_cells + i];
      }
      CK(upload(d_pool, rep));
    }
    CK(upload(d_p1, op.p1));
    const int N = op.dims.fft_n;
    split = N > 16384 ? 2 : 1;      // 32K: two 16K halves (even / odd bins), recombined in the kernel
    const int M = N / split;
    log2_m = 0;
    while ((1 << log2_m) < M) log2_m++;
    // carrier codes re-laid out per (symbol, phase) in the shared-memory position order of the FFT kernel:
    // sub-transform bin m of phase p is FFT bin b = split * m + p, i.e. centred spectrum index (b + N/2) mod N,
    // i.e. carrier k = that - left_nulls (null carriers outside [0, C_PS) take pool cell 0 = zero).
    const int L = op.dims.num_symbols, cps = op.dims.c_ps;
    std::vector<int> pos(M);
    for (int m = 0; m < M; m++) pos[m] = t2k::ofdm_table_index(t2k::ofdm_position_of_bin(m, log2_m), log2_m);
    std::vector<int32_t> code_pos((size_t)L * N, -1);
    std::vector<int32_t> sym_flags(L, 0);
    for (int l = 0; l < L; l++)
      for (int p = 0; p < split; p++)
        for (int m = 0; m < M; m++) {
          const int c = (split * m + p + N / 2) & (N - 1);
          const int k = c - op.left_nulls;
          int32_t v = (k >= 0 && k < cps) ? code[(size_t)l * cps + k] : -1;
          if (c16) {
            if (v >= 0) {
              if (v >= 65536) return fail(DVBT2LL_ERR_INVALID, "chain: staging slot out of range");
              v = 2 * v;
              if (tab_base) v |= tab_base[(*plp)[(size_t)l * cps + k]] << t2k::OFDM_CODE_TAB_SHIFT;
              if (miso && ((op.code[(size_t)l * cps + k] - op.sym_data_start[l]) & 1)) v |= t2k::OFDM_CODE_MISO_IM;
            }
            else if (~v < 8) v = (~v + 1) << 17;
            else { v = (int32_t)(0x80000000u | (uint32_t)(~v)); sym_flags[l] = 1; }
          }
          code_pos[((size_t)l * split + p) * M + pos[m]] = v;
        }
    CK(upload(d_code, code_pos));
    CK(upload(d_sym_flags, sym_flags));
    if (!op.inv_sinc.empty()) {
      std::vector<float> sinc_pos((size_t)N);
      for (int p = 0; p < split; p++)
        for (int m = 0; m < M; m++) sinc_pos[(size_t)p * M + pos[m]] = op.inv_sinc[(split * m + p + N / 2) & (N - 1)];
      CK(upload(d_sinc, sinc_pos));
    }
    CK(upload(d_tw, make_twiddles(M, M)));
    if (split == 2) CK(upload(d_tw_split, make_twiddles(N, M)));
    return 0;
  }
  void fill(t2k::OfdmArgs &a, const t2::OfdmPlan &op, const t2::CellPool &pool) const
  {
    a.code_pos = d_code.as<int32_t>(); a.pool = d_pool.as<float2>(); a.pool_stride = pool_stride;
    a.l1post_base = pool.l1post_base; a.l1post_cells = pool.l1post_cells; a.l1post_variants = pool.l1post_variants;
    a.p1 = d_p1.as<float2>(); a.sinc_pos = op.inv_sinc.empty() ? 0 : d_sinc.as<float>();
    a.tw = d_tw.as<float2>(); a.tw_split = split == 2 ? d_tw_split.as<float2>() : 0;
    a.fft_n = op.dims.fft_n; a.log2_m = log2_m; a.split = split;
    a.c_ps = op.dims.c_ps; a.left_nulls = op.left_nulls; a.gi = op.dims.gi; a.num_symbols = op.dims.num_symbols;
    a.norm = op.normalization;
    a.cells16 = 0; a.run_desc = 0; a.run_ptr = 0; a.run_cnt = 0; a.desc_cap = 0; a.stage_bytes = 0; a.stage_cap = 0; a.lut = 0; a.lut_n = 0; a.lut_single = 0;
    a.sym_flags = d_sym_flags.as<int32_t>();
    a.out_fmt = 0; a.sink_gain = 1.0f;
    a.cells_len = 0; a.out_len = 0; a.pool_len = pool_stride;
    a.lut_tables = 1;
    a.miso = 0;
  }
};

struct OfdmHandle : dvbt2ll_handle {
  t2::OfdmPlan plan;
  OfdmDevice dev;
  OfdmHandle() : dvbt2ll_handle(OFDM) {}
  int output_multiple() const { return plan.samples_per_frame; }
  int in_item() const { return 8; }
  int out_item() const { return 8; }
  int forecast(int noutput) const { return plan.dims.active_items * (noutput / plan.samples_per_frame); }
  int dev_init() { return dev.init(plan.code, plan.pool, plan); }
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    const int frames = noutput / plan.samples_per_frame;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    if ((long long)ninput < (long long)frames * plan.dims.active_items)
      return fail(DVBT2LL_ERR_SHORT, "pilotgenp1insert_cc: not enough input items");
    t2k::OfdmArgs a;
    dev.fill(a, plan, plan.pool);
    a.cells = (const float2 *)d_in; a.cells_stride = plan.dims.active_items;
    a.out = d_out; a.out_stride = plan.samples_per_frame;
    a.cells_len = (long long)frames * plan.dims.active_items; a.out_len = (long long)frames * plan.samples_per_frame;
    a.frames = frames; a.frame_idx0 = 0; a.frames_per_channel = frames;
    t2k::launch_ofdm(a, s);
    CK(cudaGetLastError());
    if (consumed) *consumed = frames * plan.dims.active_items;
    return frames * plan.samples_per_frame;
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "ofdm.code") return copy_vec(plan.code, out, cap);
    if (n == "ofdm.pool") return copy_vec(plan.pool.cells, out, cap);
    if (n == "ofdm.p1") return copy_vec(plan.p1, out, cap);
    if (n == "ofdm.carrier_type") return copy_vec(plan.carrier_type, out, cap);
    if (n == "ofdm.inv_sinc") return copy_vec(plan.inv_sinc, out, cap);
    if (n == "ofdm.sym_data_start") return copy_vec(plan.sym_data_start, out, cap);
    if (n == "ofdm.dims") return dims_get(plan.dims, out, cap);
    if (n == "ofdm.info") {
      int v[4] = { plan.left_nulls, plan.samples_per_frame, 0, 0 };
      std::memcpy(&v[2], &plan.normalization, 4);
      return copy_out(v, sizeof(v), out, cap);
    }
    return -1;
  }
};

// ================================================================================================
// the same table shifted by 0..3 entries: four consecutive entries at any phase become one aligned 8-byte load
std::vector<uint16_t> make_ci_inv4(const std::vector<uint16_t> &ci_inv, int *stride)
{
  const int nc = (int)ci_inv.size();
  *stride = (nc + 8 + 3) & ~3;
  std::vector<uint16_t> c4((size_t)4 * *stride, 0);
  for (int k = 0; k < 4; k++)
    for (int j = 0; j + k < nc; j++) {
      const int c = ci_inv[j + k];
      c4[(size_t)k * *stride + j] = (uint16_t)(c + 2 * (c >> 6));      // index in the kernel's padded code array
    }
  return c4;
}

struct ChainHandle : dvbt2ll_handle {
  // the stages of each PLP parameter set (fplan.plp_set: a distinct framesize, rate, constellation and rotation), built
  // from the set's first PLP, with that PLP's inverse cell permutation; the chain-wide BB fields (input mode, in-band
  // signalling) are fplan.prm's, and every set's BB launch counts sync errors in the chain's stream state
  struct Set {
    BbStage bb;
    LdpcStage ldpc;
    MapStage map;
    DevBuf d_ci_inv, d_ci_inv4;
    int ci4_stride;
    int bch_pitch() const { return align16(bb.plan.fec.nbch / 8); }
    int fec_pitch() const { return align16(bb.plan.fec.nldpc / 8); }
  };
  std::unique_ptr<Set[]> sets;     // [fplan.plp_sets]
  // FEC groups (see group_of): PLPs [p0, p1) with `blocks` FEC blocks per T2 frame, and their regions of the BCH / FEC
  // buffers, which hold the codewords [frame slot][block of the group] at the set's pitch
  struct Group { int p0, p1, blocks; size_t bch_off, fec_off; };
  std::vector<Group> grp;
  // constellation tables of the OFDM fill: one per distinct (constellation, rotation), the largest first; PLP p's
  // starts at entry lut_base[p]
  std::vector<t2::cfloat> luts;
  int lut_tables, lut_base[t2::MAX_PLP], lut_single;
  int lut_copies;      // copies of the table(s) k_ofdm kept in shared memory in the last run
  DevBuf d_luts;
  t2::FramePlan fplan;
  t2::OfdmPlan oplan;
  t2::Chain16Tables tables;
  OfdmDevice odev;
  DevBuf d_bch, d_fec, d_cells, d_ts_stage, d_out_stage, d_fec_shift, d_run_desc, d_run_ptr, d_run_cnt, d_stage_bytes;
  int stage_cap;
  int max_frames, device;
  int sink_fmt;          // 0 complex64 (what pilotgenp1insert_cc emits), 1 interleaved int16 I/Q
  float sink_gain;       // the flowgraph's multiply_const stage folded into the last kernel
  cudaStream_t stream2;
  // tone-reservation PAPR reduction (dvbt2ll_chain_set_papr_tr): k_papr_tr after k_ofdm when tr_iter > 0
  int tr_iter;
  float tr_vclip, tr_tone_max;
  bool tr_built, tr_uploaded;
  t2::PaprTrPlan tr;
  DevBuf d_tr_set, d_tr_bins, d_tr_kernel, d_tr_tw, d_tr_stats, d_tr_scratch;
  int tr_frames;         // frames whose counts the last run left in d_tr_stats (the "papr" tap)
  // MISO processing (dvbt2ll_chain_set_miso, dvbt2ll_chain_run_*_miso), built at first use: the pilot plan, carrier
  // tables and device tables of group g (0: TX1, 1: TX2 with MISO processing) over the chain's staging
  struct MisoGroup { t2::OfdmPlan op; t2::MisoTables tab; OfdmDevice dev; bool uploaded = false; };
  std::unique_ptr<MisoGroup> miso_g[2];
  bool miso_on;
  int last_frames;
  TsStream ts;           // stream state of the generic work() / work_device() path
  bool timing;
  enum { TIMING_SLOTS = 64 };
  cudaEvent_t ev[TIMING_SLOTS][5];     // per-run event sets so the timed loop never has to synchronise
  long long n_timed;
  ChainHandle() : dvbt2ll_handle(CHAIN), lut_tables(1), lut_single(0), lut_copies(0), max_frames(0), device(0), sink_fmt(0), sink_gain(1.0f), stream2(0), tr_iter(0), tr_vclip(0.f), tr_tone_max(0.f), tr_built(false), tr_uploaded(false), tr_frames(0), miso_on(false), last_frames(0), timing(false)
  {
    n_timed = 0;
    for (int s = 0; s < TIMING_SLOTS; s++) for (int i = 0; i < 5; i++) ev[s][i] = 0;
  }
  ~ChainHandle()
  {
    for (int s = 0; s < TIMING_SLOTS; s++) for (int i = 0; i < 5; i++) if (ev[s][i]) cudaEventDestroy(ev[s][i]);
    if (stream2) cudaStreamDestroy(stream2);
  }
  // every entry point: make the handle's device current for the calling thread (handles may be driven from any
  // thread, and one process may hold chains on several devices), then lazy device initialisation
  int enter() override
  {
    if (device >= 0) CK(cudaSetDevice(device));
    return ensure_device();
  }
  Set &set_of(int plp) const { return sets[fplan.plp_set[plp]]; }
  int first_plp(int set) const { int p = 0; while (fplan.plp_set[p] != set) p++; return p; }
  // The FEC group of a PLP: one LDPC and one mapper launch per group.  PLPs of a single parameter set form one group,
  // their codewords in the frame's block list, so a create_multiplp chain runs each stage once; with several sets
  // every PLP is a group of its own, whose cells FramePlan::plp_chain_off starts on a 16-byte boundary by the same rule.
  int group_of(int plp) const { return fplan.plp_sets > 1 ? plp : 0; }
  int F() const { return fplan.prm.fecblocks; }
  int P() const { return fplan.num_plp; }
  int Fp(int plp) const { return fplan.plp_first_block[plp + 1] - fplan.plp_first_block[plp]; }
  // cells per T2 frame in the 16-bit cell memory, padded so every frame starts on a 16-byte boundary (bulk copies)
  long long cells16_stride() const { return ((long long)fplan.plp_chain_off[P()] + 7) & ~7LL; }
  // TS byte index (per channel) at which T2 frame `frame` begins in PLP `plp`'s stream: the PLP's FEC blocks per T2
  // frame are its in-band signalling cycle
  long long stream_pos(long long frame, int plp = 0) const
  {
    return ts_stream_pos(frame * Fp(plp), set_of(plp).bb.plan.payload_bytes, fplan.prm.inband ? Fp(plp) : 0, fplan.prm.inputmode);
  }
  long long ts_bytes(long long first_frame, int n_frames, int plp = 0) const { return stream_pos(first_frame + n_frames, plp) - stream_pos(first_frame, plp); }
  long long ts_bytes_max(long long first_frame, int n_frames) const
  {
    long long m = 0;
    for (int pl = 0; pl < P(); pl++) m = std::max(m, ts_bytes(first_frame, n_frames, pl));
    return m;
  }
  long long ts_per_frame() const { return ts_bytes(0, 1); }
  // stream bytes that must precede the first TS byte of `first_frame` in every TS row: in normal input mode the CRC-8
  // that replaces the first sync byte covers the 187 bytes before the pointer
  long long history_bytes(long long first_frame) const { return (first_frame > 0 && fplan.prm.inputmode == t2::INPUTMODE_NORMAL) ? 187 : 0; }
  // the generic work path's stream position in T2 frames
  long long next_frame() const { return ts.fecframes / F(); }
  int output_multiple() const { return oplan.samples_per_frame; }
  int in_item() const { return 1; }
  int out_item() const { return sink_fmt ? 4 : 8; }
  int forecast(int noutput) const { return (int)(ts_per_frame() * (noutput / oplan.samples_per_frame)); }
  int dev_init()
  {
    int r;
    for (int s = 0; s < fplan.plp_sets; s++) {
      Set &x = sets[s];
      if ((r = x.bb.init()) || (r = x.ldpc.init()) || (r = x.map.init())) return r;
      const std::vector<uint16_t> &ci_inv = fplan.plp_cell_perm_inv[first_plp(s)];
      CK(upload(x.d_ci_inv, ci_inv));
      CK(upload(x.d_ci_inv4, make_ci_inv4(ci_inv, &x.ci4_stride)));
    }
    if ((r = ts.init())) return r;
    if ((r = odev.init(tables.code, tables.pool, oplan, true, &tables.plp, lut_tables > 1 ? lut_base : 0))) return r;
    CK(upload(d_luts, luts));
    CK(upload(d_fec_shift, fplan.fec_shift));
    CK(upload(d_run_desc, tables.run_desc));
    CK(upload(d_run_ptr, tables.run_ptr));
    CK(upload(d_run_cnt, tables.run_cnt));
    CK(upload(d_stage_bytes, tables.stage_bytes));
    stage_cap = (tables.max_slots + 7) & ~7;
    if ((size_t)(1 << odev.log2_m) * 8 * 17 / 16 + (size_t)stage_cap * 2 + 2048 + 96 + (size_t)(tables.max_runs + 2) * 8 > 227 * 1024)
      return fail(DVBT2LL_ERR_INVALID, "chain: the cells of one OFDM symbol do not fit the shared-memory staging area");
    grp.clear();
    size_t bch_end = 0, fec_end = 0;
    for (int pl = 0; pl < P(); pl++) {
      if (group_of(pl) == (int)grp.size()) grp.push_back(Group{ pl, pl, 0, bch_end, fec_end });
      Group &G = grp.back();
      G.p1 = pl + 1;
      G.blocks += Fp(pl);
      bch_end += (size_t)max_frames * Fp(pl) * set_of(pl).bch_pitch();
      fec_end += (size_t)max_frames * Fp(pl) * set_of(pl).fec_pitch();
    }
    CK(d_bch.ensure(bch_end + 64));
    CK(d_fec.ensure(fec_end + 64));
    CK(d_cells.ensure((size_t)max_frames * cells16_stride() * sizeof(uint16_t) + 64));   // 16-bit cell codes
    // the padding cells between frames and the slack behind the last one are never written by the mapper but travel
    // with the aligned bulk copies: give them a valid code once
    CK(cudaMemset(d_cells.p, 0, (size_t)max_frames * cells16_stride() * sizeof(uint16_t) + 64));
    for (int s = 0; s < TIMING_SLOTS; s++) for (int i = 0; i < 5; i++) CK(cudaEventCreate(&ev[s][i]));
    return 0;
  }
  // buf_frame: first T2-frame slot of the intermediate buffers to use; hist_valid < 0: history is present iff
  // first_frame > 0; tr_frame0: position of the batch's first frame in the tone-reservation counts (d_tr_stats)
  // d_out2 != NULL: MISO group 1 to d_out and group 2 with MISO processing to d_out2, from one pass of the front end
  int run(const void *d_ts, long long ts_pitch, int n_channels, int n_frames, long long first_frame, void *d_out, cudaStream_t s,
          int buf_frame = 0, int hist_valid = -1, int tr_frame0 = 0, void *d_out2 = 0)
  {
    const int frames = n_channels * n_frames;
    if (frames < 1) return 0;
    if (buf_frame + frames > max_frames) return fail(DVBT2LL_ERR_INVALID, "chain: batch larger than max_frames given at create");
    // the OFDM carrier tables of each output: the chain's own, or a MISO group's
    const MisoGroup *g1 = 0, *g2 = 0;
    if (d_out2 || miso_group2_out()) {
      int r = miso_upload(1);
      if (r) return r;
      g2 = miso_g[1].get();
      if (d_out2 && oplan.prm.misogroup != t2::MISO_TX1) {
        if ((r = miso_upload(0))) return r;
        g1 = miso_g[0].get();
      }
      if (!d_out2) { g1 = g2; g2 = 0; }
    }
    cudaEvent_t *tev = ev[n_timed % TIMING_SLOTS];
    if (timing) cudaEventRecord(tev[0], s);
    // a group's codewords of the batch: slot buf_frame onwards of its regions
    auto bch_buf = [&](const Group &G) { return d_bch.as<uint8_t>() + G.bch_off + (size_t)buf_frame * G.blocks * set_of(G.p0).bch_pitch(); };
    auto fec_buf = [&](const Group &G) { return d_fec.as<uint8_t>() + G.fec_off + (size_t)buf_frame * G.blocks * set_of(G.p0).fec_pitch(); };
    uint16_t *cell_buf = d_cells.as<uint16_t>() + (size_t)buf_frame * cells16_stride();
    // BB framing + BCH, PLP by PLP: row c * P + p of the TS holds PLP p of channel c; every PLP has its own stream
    // position (packet phase, in-band cycle = its FEC blocks per frame), and its codewords go to their place inside
    // its group's block list (streams begin on a packet boundary at frame 0)
    for (int pl = 0; pl < P(); pl++) {
      const Group &G = grp[group_of(pl)];
      Set &x = set_of(pl);
      const int fpl = Fp(pl), bp = x.bch_pitch();
      const int count0 = (int)(stream_pos(first_frame, pl) % 188);
      // every T2 frame begins an in-band signalling cycle (in-band phase 0)
      t2k::BbArgs ba;
      x.bb.fill_args(ba, (const uint8_t *)d_ts + (long long)pl * ts_pitch, ts_pitch * P(), n_channels, n_frames * fpl, count0, 0,
                     hist_valid >= 0 ? hist_valid : (first_frame > 0 ? 1 : 0), bch_buf(G), bp, ts.h_err);
      ba.fecblocks = fpl;
      ba.ts_len = ts_bytes(first_frame, n_frames, pl);
      ba.out_len = (long long)frames * G.blocks * bp;
      if (G.p1 - G.p0 > 1) {
        ba.out_group = fpl; ba.out_group_stride = G.blocks;
        ba.out_group_off = fplan.plp_first_block[pl] - fplan.plp_first_block[G.p0];
      }
      t2k::launch_bb_bch(ba, s);
    }
    if (timing) cudaEventRecord(tev[1], s);
    for (const Group &G : grp) {
      Set &x = set_of(G.p0);
      t2k::LdpcArgs la;
      x.ldpc.fill_args(la, bch_buf(G), x.bch_pitch(), fec_buf(G), x.fec_pitch(), frames * G.blocks);
      t2k::launch_ldpc(la, s);
    }
    if (timing) cudaEventRecord(tev[2], s);
    // the mapper writes the group's 16-bit cell codes, cell-interleaved, to its place in each frame's cell memory
    for (const Group &G : grp) {
      Set &x = set_of(G.p0);
      t2k::MapArgs ma;
      x.map.fill_args(ma, fec_buf(G), x.fec_pitch(), 0, frames * G.blocks);
      ma.out16 = cell_buf + fplan.plp_chain_off[G.p0]; ma.out16_frame_stride = cells16_stride();
      ma.ci_inv = x.d_ci_inv.as<uint16_t>(); ma.fec_shift = d_fec_shift.as<int32_t>() + fplan.plp_first_block[G.p0];
      ma.fecblocks = G.blocks;
      ma.ci_inv4 = x.d_ci_inv4.as<uint16_t>(); ma.ci_inv4_stride = x.ci4_stride;
      ma.im_from_re = lut_single;      // the w~ codes only when the OFDM fill keeps the single-table form for every PLP
      ma.out_len = (long long)frames * cells16_stride() - fplan.plp_chain_off[G.p0];
      t2k::launch_map(ma, s);
    }
    if (timing) cudaEventRecord(tev[3], s);
    // tone reservation: in place on d_out when the sink is complex64 at gain 1; otherwise k_ofdm writes complex64 at
    // gain 1 to a scratch (the buffer slots of buf_frame) and k_papr_tr applies the sink
    const bool tr_on = tr_iter > 0, tr_inplace = tr_on && sink_fmt == 0 && sink_gain == 1.0f;
    const long long spf = oplan.samples_per_frame;
    void *ofdm_out = d_out;
    if (tr_on) {
      int r = tr_upload();
      if (r) return r;
      CK(d_tr_stats.ensure((size_t)(tr_frame0 + frames) * oplan.dims.num_symbols * sizeof(int16_t)));
      if (!tr_inplace) {
        CK(d_tr_scratch.ensure((size_t)max_frames * spf * sizeof(float2)));
        ofdm_out = d_tr_scratch.as<float2>() + (size_t)buf_frame * spf;
      }
    }
    t2k::OfdmArgs oa;
    if (g1) { g1->dev.fill(oa, g1->op, g1->tab.pool); oa.miso = g1 == miso_g[1].get(); }
    else odev.fill(oa, oplan, tables.pool);
    oa.cells = 0; oa.cells_stride = cells16_stride();
    oa.cells16 = cell_buf; oa.run_desc = d_run_desc.as<int2>(); oa.run_ptr = d_run_ptr.as<int32_t>();
    oa.run_cnt = d_run_cnt.as<int32_t>(); oa.desc_cap = (tables.max_runs + 2) & ~1;
    oa.stage_bytes = d_stage_bytes.as<int32_t>(); oa.stage_cap = stage_cap;
    oa.lut = d_luts.as<float2>(); oa.lut_n = (int)luts.size(); oa.lut_tables = lut_tables; oa.lut_single = lut_single;
    oa.out = ofdm_out; oa.out_stride = oplan.samples_per_frame;
    oa.cells_len = (long long)frames * cells16_stride(); oa.out_len = (long long)frames * oplan.samples_per_frame;
    oa.out_fmt = sink_fmt; oa.sink_gain = sink_gain; oa.norm = oplan.normalization * sink_gain;
    if (ofdm_out != d_out) { oa.out_fmt = 0; oa.sink_gain = 1.0f; oa.norm = oplan.normalization; }
    oa.frames = frames; oa.frames_per_channel = n_frames;
    oa.frame_idx0 = (int)(first_frame % (tables.pool.l1post_variants > 0 ? tables.pool.l1post_variants : 1));
    lut_copies = t2k::launch_ofdm(oa, s);
    if (g2) {
      // group 2: the same cells, its own pilots and pool, the MISO form of the fill
      t2k::OfdmArgs o2 = oa;
      o2.code_pos = g2->dev.d_code.as<int32_t>(); o2.pool = g2->dev.d_pool.as<float2>(); o2.sym_flags = g2->dev.d_sym_flags.as<int32_t>();
      o2.out = d_out2;
      o2.miso = 1;
      t2k::launch_ofdm(o2, s);
    }
    if (tr_on) {
      t2k::PaprArgs pa;
      pa.in = (const float2 *)ofdm_out; pa.out = d_out;
      pa.out_fmt = sink_fmt; pa.gain = sink_gain; pa.inplace = tr_inplace ? 1 : 0;
      pa.spf = spf; pa.fft_n = oplan.dims.fft_n; pa.gi = oplan.dims.gi; pa.num_symbols = oplan.dims.num_symbols; pa.frames = frames;
      pa.iterations = tr_iter; pa.vclip = tr_vclip; pa.tone_max = tr_tone_max;
      pa.tone_scale = (float)(1.0 / ((double)oplan.normalization * tr.tones));
      pa.tones = tr.tones; pa.sets = tr.sets;
      pa.sym_set = d_tr_set.as<int32_t>(); pa.bins = d_tr_bins.as<int32_t>();
      pa.kernel = d_tr_kernel.as<float2>(); pa.tone_tw = d_tr_tw.as<float2>();
      pa.stats = d_tr_stats.as<int16_t>() + (size_t)tr_frame0 * oplan.dims.num_symbols;
      pa.in_len = pa.out_len = (long long)frames * spf;
      t2k::launch_papr_tr(pa, s);
      tr_frames = tr_frame0 + frames;
    }
    if (timing) { cudaEventRecord(tev[4], s); n_timed++; }
    CK(cudaGetLastError());
    if (buf_frame == 0) last_frames = frames;
    return frames;
  }
  bool miso_preamble() const { return oplan.prm.preamble == t2::PREAMBLE_T2_MISO || oplan.prm.preamble == t2::PREAMBLE_T2_LITE_MISO; }
  // set_miso(1) on a group-2 chain: run() emits group 2 with MISO processing
  bool miso_group2_out() const { return miso_on && oplan.prm.misogroup == t2::MISO_TX2; }
  // host tables of MISO group g (refused for a symbol with an odd cell count)
  int miso_build(int g)
  {
    if (miso_g[g]) return 0;
    std::unique_ptr<MisoGroup> m(new MisoGroup());
    t2::OfdmParams op = oplan.prm;
    op.misogroup = g ? t2::MISO_TX2 : t2::MISO_TX1;
    std::string err;
    if (!t2::build_ofdm_plan(op, &m->op, &err) || !t2::compose_miso(oplan, tables, m->op, g == 1, &m->tab, &err))
      return fail(DVBT2LL_ERR_INVALID, err);
    miso_g[g] = std::move(m);
    return 0;
  }
  int miso_upload(int g)
  {
    int r = miso_build(g);
    if (r) return r;
    MisoGroup &m = *miso_g[g];
    if (m.uploaded) return 0;
    if ((r = m.dev.init(m.tab.code, m.tab.pool, m.op, true, &m.tab.plp, lut_tables > 1 ? lut_base : 0, g == 1))) return r;
    m.uploaded = true;
    return 0;
  }
  int tr_upload()
  {
    if (tr_uploaded) return 0;
    CK(upload(d_tr_set, tr.sym_set));
    CK(upload(d_tr_bins, tr.bins));
    CK(upload(d_tr_kernel, tr.kernel));
    CK(upload(d_tr_tw, tr.tone_tw));
    tr_uploaded = true;
    return 0;
  }
  // the generic work path streams like the drop-in BB block: stream state carried across calls, 187 history bytes in
  // front of d_in once anything has been consumed (normal input mode)
  TsStream *ts_stream() override { return &ts; }
  long long input_items(int noutput) const override { return ts_bytes(next_frame(), noutput / oplan.samples_per_frame); }
  int work_device(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s)
  {
    return work_ts(d_in, ninput, d_out, noutput, consumed, s, ts.fecframes > 0 ? 1 : 0);
  }
  int work_ts(const void *d_in, int ninput, void *d_out, int noutput, int *consumed, cudaStream_t s, int hist_valid) override
  {
    const int frames = noutput / oplan.samples_per_frame;
    if (consumed) *consumed = 0;
    if (frames < 1) return 0;
    const long long need = input_items(noutput);
    if ((long long)ninput < need) return fail(DVBT2LL_ERR_SHORT, "chain: not enough input items");
    int r = run(d_in, 0, 1, frames, next_frame(), d_out, s, 0, hist_valid);
    if (r < 0) return r;
    ts.fecframes += (long long)frames * F();
    if (consumed) *consumed = (int)need;
    return frames * oplan.samples_per_frame;
  }
  long long plan_get(const char *name, void *out, long long cap) const
  {
    std::string n(name);
    if (n == "chain.code") return copy_vec(tables.code, out, cap);
    if (n == "chain.pool") return copy_vec(tables.pool.cells, out, cap);
    if (n == "chain.run_desc") return copy_vec(tables.run_desc, out, cap);
    if (n == "chain.run_ptr") return copy_vec(tables.run_ptr, out, cap);
    if (n == "chain.run_cnt") return copy_vec(tables.run_cnt, out, cap);
    if (n == "chain.stage_bytes") return copy_vec(tables.stage_bytes, out, cap);
    if (n == "ofdm.sym_data_start") return copy_vec(oplan.sym_data_start, out, cap);
    if (n == "frame.framed") return copy_vec(fplan.framed, out, cap);
    if (n == "frame.pool") return copy_vec(fplan.pool.cells, out, cap);
    if (n == "frame.info") {
      const int v[12] = { fplan.cell_size, fplan.stream_items, fplan.mapped_items, fplan.eta_mod, fplan.n_post, fplan.n_punc,
                          fplan.dummy_cells, fplan.pool.l1post_base, fplan.pool.l1post_cells, fplan.pool.l1post_variants,
                          fplan.pool_dummy, fplan.pool_zero };
      return copy_out(v, sizeof(v), out, cap);
    }
    if (n == "frame.plp") {
      int v[2 + t2::MAX_PLP + 1] = { fplan.num_plp, fplan.l1post_sig_bits };
      for (int i = 0; i <= fplan.num_plp; i++) v[2 + i] = fplan.plp_first_block[i];
      return copy_out(v, sizeof(int) * (3 + fplan.num_plp), out, cap);
    }
    if (n == "frame.fi_src") return copy_vec(fplan.fi_src, out, cap);
    if (miso_g[1] && n == "chain.miso_code") return copy_vec(miso_g[1]->tab.code, out, cap);
    if (miso_g[1] && n == "chain.miso_pool") return copy_vec(miso_g[1]->tab.pool.cells, out, cap);
    if (tr_built && n == "ofdm.tr_set") return copy_vec(tr.sym_set, out, cap);
    if (tr_built && n == "ofdm.tr_bins") return copy_vec(tr.bins, out, cap);
    if (tr_built && n == "ofdm.tr_kernel") return copy_vec(tr.kernel, out, cap);
    if (n == "frame.fec_shift") return copy_vec(fplan.fec_shift, out, cap);
    if (n == "frame.plp_cells") {
      // per PLP: cells per FECFRAME, first cell in the frame (PLP_START), first cell in the chain's cell memory
      int v[3 * t2::MAX_PLP];
      for (int i = 0; i < P(); i++) { v[3 * i] = fplan.plp_cell_size[i]; v[3 * i + 1] = fplan.plp_start[i]; v[3 * i + 2] = fplan.plp_chain_off[i]; }
      return copy_out(v, sizeof(int) * 3 * P(), out, cap);
    }
    if (n == "frame.plp_layout") {
      // per PLP: PLP_TYPE, PLP_GROUP_ID, cells per sub-slice; then SUB_SLICES_PER_FRAME, SUB_SLICE_INTERVAL, TYPE_2_START
      int v[3 * t2::MAX_PLP + 3];
      for (int i = 0; i < P(); i++) { v[3 * i] = fplan.plp_type[i]; v[3 * i + 1] = fplan.plp_group[i]; v[3 * i + 2] = fplan.plp_slice_cells[i]; }
      v[3 * P()] = fplan.num_subslices; v[3 * P() + 1] = fplan.subslice_interval; v[3 * P() + 2] = fplan.type2_start;
      return copy_out(v, sizeof(int) * (3 * P() + 3), out, cap);
    }
    if (n == "chain.luts") {
      // constellation tables of the OFDM fill: { tables, single-table form, copies in shared memory in the last run
      // (0 before any), first entry of each PLP's table }
      int v[3 + t2::MAX_PLP] = { lut_tables, lut_single, lut_copies };
      for (int i = 0; i < P(); i++) v[3 + i] = lut_base[i];
      return copy_out(v, sizeof(int) * (3 + P()), out, cap);
    }
    long long r;
    if ((r = sets[0].bb.plan_get(name, out, cap)) >= 0) return r;
    if ((r = sets[0].ldpc.plan_get(name, out, cap)) >= 0) return r;
    if ((r = sets[0].map.plan_get(name, out, cap)) >= 0) return r;
    if (n == "frame.code") return copy_vec(fplan.code, out, cap);
    if (n == "frame.ci_dst") return copy_vec(fplan.ci_dst, out, cap);
    if (n == "ofdm.code") return copy_vec(oplan.code, out, cap);
    if (n == "ofdm.dims") return dims_get(oplan.dims, out, cap);
    return -1;
  }
};

} // namespace

// ================================================================================================
extern "C" {

const char *dvbt2ll_last_error(void) { return g_err.c_str(); }
#ifdef DVBT2LL_DEBUG_BOUNDS
const char *dvbt2ll_version(void) { return "dvbt2ll-b200 0.2 (sm_100a, bounds-checking debug build)"; }
#else
const char *dvbt2ll_version(void) { return "dvbt2ll-b200 0.2 (sm_100a)"; }
#endif
long long dvbt2ll_kernel_launches(void) { return t2k::kernel_launch_count(); }

int dvbt2ll_device_available(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n > 0;
}

int dvbt2ll_output_multiple(const dvbt2ll_handle *h) { return h ? h->output_multiple() : DVBT2LL_ERR_INVALID; }
int dvbt2ll_forecast(const dvbt2ll_handle *h, int noutput) { return h ? h->forecast(noutput) : DVBT2LL_ERR_INVALID; }
int dvbt2ll_warnings(const dvbt2ll_handle *h) { return h ? h->warnings : 0; }
void dvbt2ll_destroy(dvbt2ll_handle *h) { delete h; }

long long dvbt2ll_plan_get(const dvbt2ll_handle *h, const char *name, void *out, long long cap)
{
  if (!h || !name) return -1;
  return h->plan_get(name, out, cap);
}

int dvbt2ll_work_device(dvbt2ll_handle *h, const void *d_in, int ninput, void *d_out, int noutput, int *consumed, void *stream)
{
  if (!h) return fail(DVBT2LL_ERR_INVALID, "null handle");
  int r = h->enter();
  if (r) return r;
  cudaStream_t s = stream ? (cudaStream_t)stream : h->stream;
  r = h->work_device(d_in, ninput, d_out, noutput, consumed, s);
  if (r >= 0 && !stream) CK(cudaStreamSynchronize(s));
  return r;
}

int dvbt2ll_work(dvbt2ll_handle *h, const void *in, int ninput, void *out, int noutput, int *consumed)
{
  if (!h) return fail(DVBT2LL_ERR_INVALID, "null handle");
  if (consumed) *consumed = 0;
  int r = h->enter();
  if (r) return r;
  const int om = h->output_multiple();
  const int frames = noutput / om;
  if (frames < 1) return 0;
  const int nout = frames * om;
  TsStream *ts = h->ts_stream();    // TS-consuming handles: history + stream position carried across calls
  ChainHandle *ch = h->kind == dvbt2ll_handle::CHAIN ? static_cast<ChainHandle *>(h) : 0;
  if (ch && ch->P() > 1) return fail(DVBT2LL_ERR_INVALID, "chain: a multi-PLP chain takes one TS per PLP: use dvbt2ll_chain_run_host / _run_device");
  const long long need = h->input_items(nout);
  if (ninput < need) return fail(DVBT2LL_ERR_SHORT, "not enough input items for the requested output");
  if (ch && frames > ch->max_frames) return fail(DVBT2LL_ERR_INVALID, "chain: more frames requested than max_frames given at create");
  DevBuf &d_in = h->stage_in;
  const size_t in_bytes = (size_t)need * h->in_item(), out_bytes = (size_t)nout * h->out_item();
  const size_t prefix = 192;
  // linked neighbours (dvbt2ll_link): upstream record first, then downstream -- one global lock order
  std::shared_ptr<LinkRec> found_in = h->link_in;  // the record the input is looked up in (outlives the lock on it)
  std::unique_lock<std::mutex> lk_in, lk_out;
  const bool auto_link = !ch && AutoLinks::get().enabled();
  if (auto_link && !h->link_out) {                 // every block is a producer under the automatic hand-off
    h->link_out = std::make_shared<LinkRec>();
    h->link_out->item = h->out_item();
    AutoLinks::get().add(h->link_out);
  }
  if (!found_in && auto_link && !ts) {
    // not linked explicitly: try the record that matched last time, then every other block's (one lock at a time)
    const uint8_t *ip = (const uint8_t *)in;
    std::vector<std::shared_ptr<LinkRec> > cand;
    if (std::shared_ptr<LinkRec> last = h->auto_in.lock()) cand.push_back(last);
    const size_t tried_first = cand.size();
    for (int pass = 0; pass < 2 && !found_in; pass++) {
      if (pass == 1) AutoLinks::get().snapshot(cand);
      for (size_t i = pass ? tried_first : 0; i < cand.size() && !found_in; i++) {
        LinkRec &L = *cand[i];
        if (cand[i] == h->link_out || L.item != h->in_item()) continue;
        std::unique_lock<std::mutex> g(L.m);
        for (int k = 0; k < LinkRec::NSLOT; k++) {
          const LinkRec::Slot &S = L.slot[k];
          if (S.valid && ip >= S.host && ip + (size_t)need * h->in_item() <= S.host + S.bytes) { found_in = cand[i]; break; }
        }
        if (found_in) lk_in = std::move(g);
      }
    }
    if (found_in) h->auto_in = found_in;
  }
  else if (found_in) lk_in = std::unique_lock<std::mutex>(found_in->m);
  if (h->link_out) lk_out = std::unique_lock<std::mutex>(h->link_out->m);
  // a lazily kept slot goes to the host buffer it stands for (late, but before anyone can miss it)
  auto write_back = [&](LinkRec &L, LinkRec::Slot &S) -> int {
    if (S.valid && S.pending && S.bytes) {
      CK(h->copy_host(const_cast<uint8_t *>(S.host), S.buf.p, S.bytes, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      L.late_writes++;
    }
    S.pending = false;
    return 0;
  };
  const uint8_t *resident = 0;           // the input items, if the upstream block left them in HBM
  LinkRec::Slot *taken = 0;
  if (found_in && !ts) {
    LinkRec &L = *found_in;
    const uint8_t *ip = (const uint8_t *)in;
    for (int k = 1; k <= LinkRec::NSLOT && !taken; k++) {         // newest first
      LinkRec::Slot &S = L.slot[(L.next - k + LinkRec::NSLOT) % LinkRec::NSLOT];
      if (S.valid && ip >= S.host && ip + in_bytes <= S.host + S.bytes) taken = &S;
    }
    if (taken) {
      resident = taken->buf.as<uint8_t>() + (ip - taken->host);
      L.hits++;
      if (!h->link_in) h->auto_hits++;
      const size_t o = (size_t)(ip - taken->host);
      if (o <= taken->taken_to && o + in_bytes > taken->taken_to) taken->taken_to = o + in_bytes;
      if (taken->taken_to >= taken->bytes) taken->pending = false;      // taken in full: the host copy is never needed
    }
    else {
      L.misses++;
      for (int k = 0; k < LinkRec::NSLOT; k++) {
        LinkRec::Slot &S = L.slot[k];
        if (S.valid && S.pending && ip < S.host + S.bytes && ip + in_bytes > S.host && (r = write_back(L, S)) < 0) return r;
      }
    }
  }
  LinkRec::Slot *mine = 0;               // where this call's output stays resident
  if (h->link_out) {
    LinkRec &L = *h->link_out;
    mine = &L.slot[L.next];
    if ((r = write_back(L, *mine)) < 0) return r;              // what the consumer did not take, before it is overwritten
    // an older slot standing for (part of) the host range this call writes is dead: the scheduler only hands that
    // range out again once its consumer is done with it
    for (int k = 0; k < LinkRec::NSLOT; k++) {
      LinkRec::Slot &S = L.slot[k];
      if (&S != mine && S.valid && (const uint8_t *)out < S.host + S.bytes && (const uint8_t *)out + out_bytes > S.host) {
        if ((r = write_back(L, S)) < 0) return r;
        S.valid = false;
      }
    }
    // the consumer's kernels may still be reading the slot: this block's stream goes behind them
    if (mine->taken_valid) CK(cudaStreamWaitEvent(h->stream, mine->taken_ev, 0));
    mine->valid = false;                                       // empty while this call works (and possibly reallocates)
    // all empty slots get their device buffer now (first call of the link, or a larger request): later calls must
    // not pay for an allocation each time they step to the next slot
    for (int k = 0; k < LinkRec::NSLOT; k++)
      if (!L.slot[k].valid) CK(L.slot[k].buf.ensure(out_bytes + 256));
    lk_out.unlock();
  }
  if (lk_in.owns_lock() && !resident) lk_in.unlock();
  DevBuf &d_out = mine ? mine->buf : h->stage_out;
  if (!resident) CK(d_in.ensure(prefix + in_bytes + 256));
  CK(d_out.ensure(out_bytes + 256));
  uint8_t *din = resident ? const_cast<uint8_t *>(resident) : d_in.as<uint8_t>() + prefix;
  cudaStream_t s = h->stream;
  // GNU Radio hands over pageable buffers; registering them (once per distinct buffer, they are reused call after
  // call) turns the two copies into DMA transfers at full PCIe rate instead of staged pageable copies
  if (!resident) h->pin(in, in_bytes);
  h->pin(out, out_bytes);
  if (ts) CK(cudaMemcpyAsync(din - 187, ts->history, 187, cudaMemcpyHostToDevice, s));
  if (!resident) CK(h->copy_host(din, in, in_bytes, cudaMemcpyHostToDevice, s));
  int used = 0;
  if (ts) r = h->work_ts(din, (int)need, d_out.p, nout, &used, s, 1);     // the history uploaded above
  else r = h->work_device(din, (int)need, d_out.p, nout, &used, s);
  if (r < 0) return r;
  if (resident) {
    // everything that reads the producer's device copy is enqueued: mark the point on this stream and let go of the record
    if (!taken->taken_ev) CK(cudaEventCreateWithFlags(&taken->taken_ev, cudaEventDisableTiming));
    CK(cudaEventRecord(taken->taken_ev, s));
    taken->taken_valid = true;
    lk_in.unlock();
  }
  const bool lazy_out = h->link_out && h->link_out->lazy;      // (only ever changed by this block's own thread)
  if (!lazy_out) CK(h->copy_host(out, d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (ts) {
    h->warnings = *ts->h_err;        // mapped host counter, complete after the synchronize
    ts->note_consumed((const uint8_t *)in, used);
  }
  if (mine) {
    lk_out.lock();
    LinkRec &L = *h->link_out;
    mine->host = (const uint8_t *)out; mine->bytes = out_bytes; mine->valid = true;
    mine->pending = lazy_out; mine->taken_to = 0;
    L.next = (L.next + 1) % LinkRec::NSLOT;
  }
  if (consumed) *consumed = used;
  return r;
}

// ---- transport-stream ingest helpers (host side; SURVEY 8(f) item 4) ---------------------------------------------
// first offset at which 0x47 repeats every 188 bytes over 5 packets (or to the end of a shorter buffer), -1 if none
long long dvbt2ll_ts_sync(const unsigned char *ts, size_t n)
{
  if (!ts) return -1;
  for (size_t off = 0; off < 188 && off < n; off++) {
    int ok = 0;
    size_t q = off;
    for (; q < n && ok < 5; q += 188, ok++)
      if (ts[q] != 0x47) break;
    if (ok == 5 || (ok > 0 && q >= n)) return (long long)off;
  }
  return -1;
}
// dst[0, dst_bytes) = bytes [pos, pos + dst_bytes) of the packet-aligned stream `src`, continued with null packets
// (PID 0x1FFF: 47 1F FF 10, payload FF) where pos runs past the last whole packet of src; pos < 0 reads as zeros
// (the history in front of the very first frame).  Returns the number of null-packet bytes written.
long long dvbt2ll_ts_fill(unsigned char *dst, size_t dst_bytes, const unsigned char *src, size_t src_bytes, long long pos)
{
  if (!dst) return -1;
  const long long whole = (long long)(src_bytes / 188) * 188;        // a trailing partial packet is dropped
  long long nulls = 0;
  for (size_t i = 0; i < dst_bytes; i++) {
    const long long q = pos + (long long)i;
    if (q < 0) dst[i] = 0;
    else if (q < whole && src) dst[i] = src[q];
    else {
      const int k = (int)(q % 188);
      dst[i] = k == 0 ? 0x47 : k == 1 ? 0x1F : k == 2 ? 0xFF : k == 3 ? 0x10 : 0xFF;
      nulls++;
    }
  }
  return nulls;
}

// plain synchronous copies between host and device memory, for hosts (tests, bench.py, language bindings) that hold raw
// device pointers handed out by this library (dvbt2ll_gather_wait) and have no CUDA runtime binding of their own
int dvbt2ll_copy_to_host(void *dst, const void *d_src, size_t bytes)
{
  CK(cudaMemcpy(dst, d_src, bytes, cudaMemcpyDeviceToHost));
  return 0;
}
int dvbt2ll_copy_to_device(void *d_dst, const void *src, size_t bytes)
{
  CK(cudaMemcpy(d_dst, src, bytes, cudaMemcpyHostToDevice));
  return 0;
}
void *dvbt2ll_device_alloc(size_t bytes)
{
  void *p = 0;
  if (cudaMalloc(&p, bytes) != cudaSuccess) { fail(DVBT2LL_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(cudaGetLastError())); return 0; }
  return p;
}
void dvbt2ll_device_free(void *p) { if (p) cudaFree(p); }
int dvbt2ll_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
int dvbt2ll_set_device(int device) { CK(cudaSetDevice(device)); return 0; }
void *dvbt2ll_stream_create(void)
{
  cudaStream_t s = 0;
  if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { fail(DVBT2LL_ERR_CUDA, "cudaStreamCreate failed"); cudaGetLastError(); return 0; }
  return (void *)s;
}
void dvbt2ll_stream_destroy(void *stream) { if (stream) cudaStreamDestroy((cudaStream_t)stream); }
int dvbt2ll_stream_synchronize(void *stream) { CK(cudaStreamSynchronize((cudaStream_t)stream)); return 0; }
int dvbt2ll_device_synchronize(void) { CK(cudaDeviceSynchronize()); return 0; }

void dvbt2ll_set_overfull_policy(int policy) { t2::set_overfull_policy(policy); }

void dvbt2ll_set_host_register(dvbt2ll_handle *h, int on) { if (h) h->pin_enabled = on != 0; }

int dvbt2ll_link(dvbt2ll_handle *producer, dvbt2ll_handle *consumer)
{
  if (!producer || !consumer || producer == consumer) return fail(DVBT2LL_ERR_INVALID, "link: two distinct handles needed");
  if (producer->out_item() != consumer->in_item()) return fail(DVBT2LL_ERR_INVALID, "link: item sizes differ");
  if (consumer->kind == dvbt2ll_handle::BB || consumer->kind == dvbt2ll_handle::CHAIN)
    return fail(DVBT2LL_ERR_INVALID, "link: a TS-consuming block keeps stream history in front of its input and cannot be a consumer");
  std::shared_ptr<LinkRec> L = std::make_shared<LinkRec>();
  L->item = producer->out_item();
  producer->link_out = L;
  consumer->link_in = L;
  return 0;
}

long long dvbt2ll_link_hits(const dvbt2ll_handle *consumer)
{
  if (!consumer) return 0;
  return consumer->link_in ? consumer->link_in->hits : consumer->auto_hits;
}

void dvbt2ll_set_auto_link(int on)
{
  AutoLinks &a = AutoLinks::get();
  std::lock_guard<std::mutex> g(a.m);
  a.on = on ? 1 : 0;
}

int dvbt2ll_link_lazy_host(dvbt2ll_handle *producer, int on)
{
  if (!producer || !producer->link_out) return fail(DVBT2LL_ERR_INVALID, "link_lazy_host: the handle is not the producer of a link");
  std::lock_guard<std::mutex> g(producer->link_out->m);
  producer->link_out->lazy = on != 0;
  return 0;
}

long long dvbt2ll_link_late_writes(const dvbt2ll_handle *producer) { return (producer && producer->link_out) ? producer->link_out->late_writes : 0; }

// ---- factories -----------------------------------------------------------------------------------
dvbt2ll_handle *dvbt2ll_bbheaderbch_create(int framesize, int rate, int mode, int inband, int fecblocks, int tsrate)
{
  BbHandle *h = new BbHandle();
  std::string err;
  if (mode != t2::INPUTMODE_NORMAL && mode != t2::INPUTMODE_HIEFF) { delete h; fail(DVBT2LL_ERR_INVALID, "bbheaderbch_bb: unknown input mode"); return 0; }
  if (!t2::build_bb_plan(framesize, rate, mode, inband, fecblocks, tsrate, &h->st.plan, &err)) { delete h; fail(DVBT2LL_ERR_INVALID, err); return 0; }
  return h;
}

dvbt2ll_handle *dvbt2ll_ldpc_create(int framesize, int rate)
{
  LdpcHandle *h = new LdpcHandle();
  std::string err;
  if (!t2::build_ldpc_plan(framesize, rate, &h->st.plan, &err)) { delete h; fail(DVBT2LL_ERR_INVALID, err); return 0; }
  return h;
}

dvbt2ll_handle *dvbt2ll_interleavermod_create(int framesize, int rate, int constellation, int rotation)
{
  MapHandle *h = new MapHandle();
  std::string err;
  if (!t2::build_map_plan(framesize, rate, constellation, rotation, &h->st.plan, &err)) { delete h; fail(DVBT2LL_ERR_INVALID, err); return 0; }
  return h;
}

dvbt2ll_handle *dvbt2ll_framemapperfint_create(int framesize, int rate, int constellation, int rotation, int fecblocks,
                                               int tiblocks, int carriermode, int fftsize, int guardinterval,
                                               int l1constellation, int pilotpattern, int t2frames, int numdatasyms,
                                               int paprmode, int version, int preamble, int inputmode,
                                               int reservedbiasbits, int l1scrambled, int inband)
{
  FrameHandle *h = new FrameHandle();
  std::string err;
  t2::FrameParams p = { framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize, guardinterval,
                        l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble, inputmode,
                        reservedbiasbits, l1scrambled, inband };
  if (!t2::build_frame_plan(p, &h->plan, &err)) { delete h; fail(DVBT2LL_ERR_INVALID, err); return 0; }
  if (h->plan.overfull) { h->warnings = 1; g_err = "Frame Mapper, too many FEC blocks in T2 frame."; }
  return h;
}

dvbt2ll_handle *dvbt2ll_pilotgenp1insert_create(int carriermode, int fftsize, int pilotpattern, int guardinterval,
                                                int numdatasyms, int paprmode, int version, int preamble,
                                                int misogroup, int equalization, int bandwidth, int vlength)
{
  OfdmHandle *h = new OfdmHandle();
  std::string err;
  t2::OfdmParams p = { carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble,
                       misogroup, equalization, bandwidth, vlength };
  if (!t2::build_ofdm_plan(p, &h->plan, &err)) { delete h; fail(DVBT2LL_ERR_INVALID, err); return 0; }
  return h;
}

// own_modcod: every PLP has its own framesize / rate / constellation / rotation (dvbt2ll_chain_create_plp_layout);
// otherwise they are the chain's, and an over-full frame follows the over-full policy like the reference's frame mapper.
// layout: PLP types, groups and sub-slices (NULL: type-1 PLPs of group 1, one sub-slice)
static dvbt2ll_handle *chain_create(const dvbt2ll_chain_params *c, int num_plp, const dvbt2ll_plp_params *plp, bool own_modcod,
                                    const dvbt2ll_plp_layout *layout, int max_frames, int device)
{
  std::unique_ptr<ChainHandle> h(new ChainHandle());
  std::string err;
  h->max_frames = max_frames; h->device = device;
  int fecblocks = 0;
  for (int p = 0; p < num_plp; p++) fecblocks += plp[p].fecblocks;
  // the frame's own FEC / modulation fields are PLP 0's
  t2::FrameParams fp = { plp[0].framesize, plp[0].rate, plp[0].constellation, plp[0].rotation, fecblocks, c->tiblocks,
                         c->carriermode, c->fftsize, c->guardinterval, c->l1constellation, c->pilotpattern, c->t2frames,
                         c->numdatasyms, c->paprmode, c->version, c->preamble, c->inputmode, c->reservedbiasbits,
                         c->l1scrambled, c->inband };
  fp.num_plp = num_plp;
  fp.plp_modcod = own_modcod ? 1 : 0;
  for (int p = 0; p < num_plp; p++) {
    fp.plp_fecblocks[p] = plp[p].fecblocks;
    fp.plp_framesize[p] = plp[p].framesize; fp.plp_rate[p] = plp[p].rate;
    fp.plp_constellation[p] = plp[p].constellation; fp.plp_rotation[p] = plp[p].rotation;
  }
  if (layout) {
    fp.plp_layout = 1;
    fp.num_subslices = layout->num_subslices;
    for (int p = 0; p < num_plp; p++) { fp.plp_type[p] = layout->type[p]; fp.plp_group[p] = layout->group[p]; }
  }
  t2::OfdmParams op = { c->carriermode, c->fftsize, c->pilotpattern, c->guardinterval, c->numdatasyms, c->paprmode,
                        c->version, c->preamble, c->misogroup, c->equalization, c->bandwidth, c->vlength };
  bool ok = t2::build_frame_plan(fp, &h->fplan, &err);
  // the stages of every parameter set, built from its first PLP: the same checks as a single-PLP chain's
  if (ok) h->sets.reset(new ChainHandle::Set[h->fplan.plp_sets]);
  for (int s = 0; ok && s < h->fplan.plp_sets; s++) {
    const dvbt2ll_plp_params &q = plp[h->first_plp(s)];
    ChainHandle::Set &x = h->sets[s];
    ok = ok && t2::build_bb_plan(q.framesize, q.rate, c->inputmode, c->inband, fecblocks, c->tsrate, &x.bb.plan, &err);
    ok = ok && t2::build_ldpc_plan(q.framesize, q.rate, &x.ldpc.plan, &err);
    ok = ok && t2::build_map_plan(q.framesize, q.rate, q.constellation, q.rotation, &x.map.plan, &err);
  }
  ok = ok && t2::build_ofdm_plan(op, &h->oplan, &err);
  ok = ok && t2::compose_chain16(h->fplan, h->oplan, &h->tables, &err);
  if (!ok) { fail(DVBT2LL_ERR_INVALID, err); return 0; }
  // one table per distinct (constellation, rotation), the largest first: the non-data carriers' look-ups (entry =
  // any cell code, see OFDM_CODE_TAB_SHIFT) stay inside it
  std::vector<int> order;
  for (int p = 0; p < num_plp; p++) order.push_back(p);
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return plp[x].constellation > plp[y].constellation; });
  h->lut_tables = 0;
  h->lut_single = 1;
  for (size_t i = 0; i < order.size(); i++) {
    const int p = order[i];
    const t2::MapPlan &mp = h->set_of(p).map.plan;
    h->lut_single &= mp.im_from_re;
    size_t j = 0;
    while (j < i && !(plp[order[j]].constellation == plp[p].constellation && plp[order[j]].rotation == plp[p].rotation)) j++;
    if (j < i) { h->lut_base[p] = h->lut_base[order[j]]; continue; }
    h->lut_base[p] = (int)h->luts.size();
    h->luts.insert(h->luts.end(), mp.lut.begin(), mp.lut.end());
    h->lut_tables++;
  }
  // several tables: a multiple of 16 entries, so the small pool behind them in shared memory stays 64-byte aligned
  // (k_ofdm rounds a lone 4-entry table up to 16 itself)
  if (h->lut_tables > 1) h->luts.resize((h->luts.size() + 15) & ~(size_t)15);
  if (h->luts.size() - 1 > t2k::OFDM_CODE_TAB_MAX) { fail(DVBT2LL_ERR_INVALID, "chain: constellation tables too large"); return 0; }
  if (h->fplan.overfull) { h->warnings = 1; g_err = "Frame Mapper, too many FEC blocks in T2 frame."; }
  return h.release();
}

dvbt2ll_handle *dvbt2ll_chain_create_plp_layout(const dvbt2ll_chain_params *c, int num_plp, const dvbt2ll_plp_params *plp,
                                                const dvbt2ll_plp_layout *layout, int max_frames, int device)
{
  if (!c || !plp || !layout || max_frames < 1) { fail(DVBT2LL_ERR_INVALID, "chain: bad arguments"); return 0; }
  if (num_plp < 1 || num_plp > t2::MAX_PLP) { fail(DVBT2LL_ERR_INVALID, "chain: number of PLPs out of range"); return 0; }
  for (int p = 0; p < num_plp; p++)
    if (plp[p].fecblocks < 1 || plp[p].fecblocks > 1023) { fail(DVBT2LL_ERR_INVALID, "chain: FEC blocks of a PLP out of range"); return 0; }
  return chain_create(c, num_plp, plp, true, layout, max_frames, device);
}

dvbt2ll_handle *dvbt2ll_chain_create_plps(const dvbt2ll_chain_params *c, int num_plp, const dvbt2ll_plp_params *plp, int max_frames,
                                          int device)
{
  dvbt2ll_plp_layout layout;
  layout.num_subslices = 1;
  for (int p = 0; p < t2::MAX_PLP; p++) { layout.type[p] = 1; layout.group[p] = 1; }
  return dvbt2ll_chain_create_plp_layout(c, num_plp, plp, &layout, max_frames, device);
}

dvbt2ll_handle *dvbt2ll_chain_create_multiplp(const dvbt2ll_chain_params *c, int num_plp, const int *plp_fecblocks, int max_frames, int device)
{
  if (!c || max_frames < 1) { fail(DVBT2LL_ERR_INVALID, "chain: bad arguments"); return 0; }
  if (num_plp < 1 || num_plp > t2::MAX_PLP || (num_plp > 1 && !plp_fecblocks)) { fail(DVBT2LL_ERR_INVALID, "chain: number of PLPs out of range"); return 0; }
  dvbt2ll_plp_params plp[t2::MAX_PLP];
  for (int p = 0; p < num_plp; p++) {
    const dvbt2ll_plp_params q = { num_plp > 1 ? plp_fecblocks[p] : c->fecblocks, c->framesize, c->rate, c->constellation, c->rotation };
    plp[p] = q;
  }
  return chain_create(c, num_plp, plp, false, 0, max_frames, device);
}

dvbt2ll_handle *dvbt2ll_chain_create(const dvbt2ll_chain_params *c, int max_frames, int device)
{
  return dvbt2ll_chain_create_multiplp(c, 1, 0, max_frames, device);
}

static ChainHandle *as_chain(const dvbt2ll_handle *h)
{
  return (h && h->kind == dvbt2ll_handle::CHAIN) ? static_cast<ChainHandle *>(const_cast<dvbt2ll_handle *>(h)) : 0;
}

long long dvbt2ll_chain_ts_bytes_per_frame(const dvbt2ll_handle *h) { ChainHandle *c = as_chain(h); return c ? c->ts_per_frame() : -1; }
long long dvbt2ll_chain_ts_bytes(const dvbt2ll_handle *h, long long first_frame, int n_frames)
{
  ChainHandle *c = as_chain(h);
  return c ? c->ts_bytes(first_frame, n_frames) : -1;
}
// stream bytes that must precede the first TS byte of `first_frame` in every row handed to dvbt2ll_chain_run_*
long long dvbt2ll_chain_history_bytes(const dvbt2ll_handle *h, long long first_frame)
{
  ChainHandle *c = as_chain(h);
  return c ? c->history_bytes(first_frame) : -1;
}
int dvbt2ll_chain_num_plp(const dvbt2ll_handle *h) { ChainHandle *c = as_chain(h); return c ? c->P() : -1; }
long long dvbt2ll_chain_plp_ts_bytes(const dvbt2ll_handle *h, int plp, long long first_frame, int n_frames)
{
  ChainHandle *c = as_chain(h);
  if (!c || plp < 0 || plp >= c->P()) return -1;
  return c->ts_bytes(first_frame, n_frames, plp);
}
long long dvbt2ll_chain_samples_per_frame(const dvbt2ll_handle *h) { ChainHandle *c = as_chain(h); return c ? c->oplan.samples_per_frame : -1; }
int dvbt2ll_chain_fecframes_per_frame(const dvbt2ll_handle *h) { ChainHandle *c = as_chain(h); return c ? c->F() : -1; }

// d_out2 != NULL: MISO group 1 to d_out and group 2 to d_out2 (dvbt2ll_chain_run_device_miso)
static int chain_run_device(ChainHandle *c, const void *d_ts, long long ts_pitch, int n_channels, int n_frames,
                            long long first_frame, void *d_out, void *d_out2, void *stream)
{
  int r = c->enter();
  if (r) return r;
  if (n_channels < 0 || n_frames < 0) return fail(DVBT2LL_ERR_INVALID, "chain: negative batch size");
  if (n_channels == 0 || n_frames == 0) return 0;
  if (c->P() > 1 && ts_pitch < c->ts_bytes_max(first_frame, n_frames))
    return fail(DVBT2LL_ERR_INVALID, "chain: with several PLPs the TS rows (channel * num_plp + plp) need a pitch of at least the longest PLP's bytes");
  return c->run(d_ts, ts_pitch, n_channels, n_frames, first_frame, d_out, stream ? (cudaStream_t)stream : c->stream, 0, -1, 0, d_out2);
}

int dvbt2ll_chain_run_device(dvbt2ll_handle *h, const void *d_ts, long long ts_pitch, int n_channels, int n_frames,
                             long long first_frame, void *d_out, void *stream)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  return chain_run_device(c, d_ts, ts_pitch, n_channels, n_frames, first_frame, d_out, 0, stream);
}

// out2 != NULL: MISO group 1 to out and group 2 to out2 (dvbt2ll_chain_run_host_miso)
static int chain_run_host(ChainHandle *c, const void *ts, long long ts_pitch, int n_channels, int n_frames,
                          long long first_frame, void *out, void *out2)
{
  int r;
  if (n_channels < 0 || n_frames < 0) return fail(DVBT2LL_ERR_INVALID, "chain: negative batch size");
  if (n_channels == 0 || n_frames == 0) return 0;
  const int P = c->P();                      // TS rows per channel (row = channel * P + plp)
  const long long per_ch = c->ts_bytes_max(first_frame, n_frames);
  const long long hist = c->history_bytes(first_frame);
  if (n_channels * P == 1 && ts_pitch < per_ch + hist) ts_pitch = per_ch + hist;      // a single row: the pitch is never used to step
  if (ts_pitch < per_ch + hist)
    return fail(DVBT2LL_ERR_INVALID, "chain: ts_pitch smaller than the TS bytes (+ 187 history bytes) of one channel");
  const long long dpitch = (per_ch + hist + 255) & ~255LL;
  const size_t ssz = c->sink_fmt ? 4 : 8;                                        // bytes per output sample
  const size_t out_bytes = (size_t)n_channels * n_frames * c->oplan.samples_per_frame * ssz;
  CK(c->d_ts_stage.ensure((size_t)n_channels * P * dpitch + 512));
  CK(c->d_out_stage.ensure(out2 ? 2 * out_bytes : out_bytes));
  uint8_t *base = c->d_ts_stage.as<uint8_t>() + 256;
  uint8_t *dout = c->d_out_stage.as<uint8_t>(), *dout2 = dout + out_bytes;
  const size_t ch_out = (size_t)n_frames * c->oplan.samples_per_frame;          // samples per channel
  // host layout: channel-major with pitch ts_pitch; when first_frame > 0 each channel pointer must be preceded
  // by 187 history bytes.  Channels are processed in groups on two streams so that the H2D copy and the
  // kernels of one group overlap the D2H copy of the previous one (the D2H copy dominates).
  if (!c->stream2) CK(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
  // every group writes its own part of the tone-reservation counts: size them for the whole call before the first
  if (c->tr_iter > 0) CK(c->d_tr_stats.ensure((size_t)n_channels * n_frames * c->oplan.dims.num_symbols * sizeof(int16_t)));
  int groups = n_channels >= 8 ? 8 : n_channels;
  while (groups > 1 && 2 * ((n_channels + groups - 1) / groups) * n_frames > c->max_frames) groups--;
  const int per = (n_channels + groups - 1) / groups;
  if (2 * per * n_frames > c->max_frames) groups = 1;
  int gi = 0;
  for (int c0 = 0; c0 < n_channels; c0 += (groups == 1 ? n_channels : per), gi++) {
    const int nc = groups == 1 ? n_channels : (c0 + per <= n_channels ? per : n_channels - c0);
    cudaStream_t s = (gi & 1) ? c->stream2 : c->stream;
    CK(cudaMemcpy2DAsync(base + (size_t)c0 * P * dpitch - hist, (size_t)dpitch, (const uint8_t *)ts + (size_t)c0 * P * ts_pitch - hist,
                         (size_t)ts_pitch, (size_t)(per_ch + hist), (size_t)nc * P, cudaMemcpyHostToDevice, s));
    r = c->run(base + (size_t)c0 * P * dpitch, dpitch, nc, n_frames, first_frame, dout + (size_t)c0 * ch_out * ssz, s,
               groups == 1 ? 0 : (gi & 1) * per * n_frames, -1, c0 * n_frames, out2 ? dout2 + (size_t)c0 * ch_out * ssz : 0);
    if (r < 0) return r;
    CK(cudaMemcpyAsync((uint8_t *)out + (size_t)c0 * ch_out * ssz, dout + (size_t)c0 * ch_out * ssz, (size_t)nc * ch_out * ssz,
                       cudaMemcpyDeviceToHost, s));
    if (out2)
      CK(cudaMemcpyAsync((uint8_t *)out2 + (size_t)c0 * ch_out * ssz, dout2 + (size_t)c0 * ch_out * ssz, (size_t)nc * ch_out * ssz,
                         cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaStreamSynchronize(c->stream2));
  return n_channels * n_frames;
}

int dvbt2ll_chain_run_host(dvbt2ll_handle *h, const void *ts, long long ts_pitch, int n_channels, int n_frames,
                           long long first_frame, void *out)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  int r = c->enter();
  if (r) return r;
  return chain_run_host(c, ts, ts_pitch, n_channels, n_frames, first_frame, out, 0);
}

// the dual MISO calls: a MISO preamble, tone reservation off, both outputs given
static int miso_dual_check(ChainHandle *c, const void *out1, const void *out2)
{
  if (!c->miso_preamble()) return fail(DVBT2LL_ERR_INVALID, "chain: MISO outputs need preamble T2_MISO or T2_LITE_MISO");
  if (c->tr_iter > 0) return fail(DVBT2LL_ERR_INVALID, "chain: the MISO dual call does not apply tone reservation; switch it off");
  if (!out1 || !out2) return fail(DVBT2LL_ERR_INVALID, "chain: the MISO dual call needs both outputs");
  return c->miso_build(1);
}

int dvbt2ll_chain_run_device_miso(dvbt2ll_handle *h, const void *d_ts, long long ts_pitch, int n_channels, int n_frames,
                                  long long first_frame, void *d_out1, void *d_out2, void *stream)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  const int r = miso_dual_check(c, d_out1, d_out2);
  return r ? r : chain_run_device(c, d_ts, ts_pitch, n_channels, n_frames, first_frame, d_out1, d_out2, stream);
}

int dvbt2ll_chain_run_host_miso(dvbt2ll_handle *h, const void *ts, long long ts_pitch, int n_channels, int n_frames,
                                long long first_frame, void *out1, void *out2)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  int r = miso_dual_check(c, out1, out2);
  if (r) return r;
  if ((r = c->enter())) return r;
  return chain_run_host(c, ts, ts_pitch, n_channels, n_frames, first_frame, out1, out2);
}

long long dvbt2ll_chain_tap(dvbt2ll_handle *h, const char *stage, void *out, long long cap)
{
  ChainHandle *c = as_chain(h);
  if (!c || !stage) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  if (!c->dev_ready || c->last_frames < 1) return fail(DVBT2LL_ERR_INVALID, "chain: nothing has run yet");
  const size_t nfec = (size_t)c->last_frames * c->F();
  const void *src; size_t bytes;
  std::string n(stage);
  if ((n.compare(0, 4, "bch.") == 0 || n.compare(0, 4, "fec.") == 0) && n.size() > 4) {
    // PLP p's codewords [channel][frame][block] at its own pitch, out of its group's region
    char *end = 0;
    const long p = std::strtol(n.c_str() + 4, &end, 10);
    if (*end || p < 0 || p >= c->P()) return fail(DVBT2LL_ERR_INVALID, "chain: unknown tap");
    const bool fec = n[0] == 'f';
    const ChainHandle::Group &G = c->grp[c->group_of((int)p)];
    const size_t pitch = fec ? c->set_of((int)p).fec_pitch() : c->set_of((int)p).bch_pitch(), row = c->Fp((int)p) * pitch;
    bytes = (size_t)c->last_frames * row;
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaDeviceSynchronize());
    if (!out || cap <= 0) return (long long)bytes;
    std::vector<uint8_t> h(bytes);
    const uint8_t *region = fec ? c->d_fec.as<uint8_t>() + G.fec_off : c->d_bch.as<uint8_t>() + G.bch_off;
    CK(cudaMemcpy2D(h.data(), row, region + (size_t)(c->fplan.plp_first_block[p] - c->fplan.plp_first_block[G.p0]) * pitch,
                    G.blocks * pitch, row, c->last_frames, cudaMemcpyDeviceToHost));
    std::memcpy(out, h.data(), (size_t)cap < bytes ? (size_t)cap : bytes);
    return (long long)bytes;
  }
  if ((n == "bch" || n == "fec") && c->grp.size() != 1)
    return fail(DVBT2LL_ERR_INVALID, "chain: the PLPs have their own FEC parameters: use the taps bch.<plp> / fec.<plp>");
  if (n == "bch") { src = c->d_bch.p; bytes = nfec * c->sets[0].bch_pitch(); }
  else if (n == "fec") { src = c->d_fec.p; bytes = nfec * c->sets[0].fec_pitch(); }
  else if (n == "cells") { src = c->d_cells.p; bytes = (size_t)c->last_frames * c->cells16_stride() * sizeof(uint16_t); }
  else if (n == "papr") {
    if (c->tr_iter < 1 || c->tr_frames < 1) return fail(DVBT2LL_ERR_INVALID, "chain: the tone-reservation stage is off");
    src = c->d_tr_stats.p; bytes = (size_t)c->tr_frames * c->oplan.dims.num_symbols * sizeof(int16_t);
  }
  else return fail(DVBT2LL_ERR_INVALID, "chain: unknown tap");
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaDeviceSynchronize());
  if (out && cap > 0) CK(cudaMemcpy(out, src, (size_t)cap < bytes ? (size_t)cap : bytes, cudaMemcpyDeviceToHost));
  return (long long)bytes;
}

int dvbt2ll_chain_set_sink(dvbt2ll_handle *h, int format, float gain)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  if (format != 0 && format != 1) return fail(DVBT2LL_ERR_INVALID, "chain: sink format must be 0 (complex64) or 1 (int16 I/Q)");
  c->sink_fmt = format;
  c->sink_gain = gain;
  return 0;
}

int dvbt2ll_chain_set_papr_tr(dvbt2ll_handle *h, int iterations, float vclip, float tone_max)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  const int pm = c->oplan.prm.paprmode;
  if (pm != t2::PAPR_TR && pm != t2::PAPR_BOTH) return fail(DVBT2LL_ERR_INVALID, "chain: tone reservation needs paprmode TR or BOTH");
  if (iterations < 0 || iterations > 64) return fail(DVBT2LL_ERR_INVALID, "chain: tone-reservation iterations must be 0 (off) .. 64");
  if (!(std::isfinite(vclip) && vclip > 0.f) || !(std::isfinite(tone_max) && tone_max > 0.f))
    return fail(DVBT2LL_ERR_INVALID, "chain: tone-reservation vclip and tone_max must be finite and > 0");
  if (!c->tr_built) {
    std::string err;
    if (!t2::build_papr_tr_plan(c->oplan, &c->tr, &err)) return fail(DVBT2LL_ERR_INVALID, err);
    c->tr_built = true;
  }
  c->tr_iter = iterations; c->tr_vclip = vclip; c->tr_tone_max = tone_max;
  return 0;
}

int dvbt2ll_chain_set_miso(dvbt2ll_handle *h, int on)
{
  ChainHandle *c = as_chain(h);
  if (!c) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  if (!c->miso_preamble()) return fail(DVBT2LL_ERR_INVALID, "chain: MISO processing needs preamble T2_MISO or T2_LITE_MISO");
  if (on) {
    const int r = c->miso_build(1);
    if (r) return r;
  }
  c->miso_on = on != 0;
  return 0;
}

void dvbt2ll_chain_enable_timing(dvbt2ll_handle *h, int on)
{
  ChainHandle *c = as_chain(h);
  if (c) { c->timing = on != 0; c->n_timed = 0; }
}

int dvbt2ll_chain_stage_ms(dvbt2ll_handle *h, float *ms5)
{
  ChainHandle *c = as_chain(h);
  if (!c || !ms5) return fail(DVBT2LL_ERR_INVALID, "not a chain handle");
  if (!c->timing || !c->dev_ready || c->n_timed < 1) return fail(DVBT2LL_ERR_INVALID, "chain: timing not enabled or nothing run");
  // average over the runs recorded since timing was enabled (at most the last TIMING_SLOTS)
  const long long n = c->n_timed < ChainHandle::TIMING_SLOTS ? c->n_timed : ChainHandle::TIMING_SLOTS;
  for (int i = 0; i < 5; i++) ms5[i] = 0.f;
  for (long long k = 0; k < n; k++) {
    cudaEvent_t *e = c->ev[(c->n_timed - 1 - k) % ChainHandle::TIMING_SLOTS];
    CK(cudaEventSynchronize(e[4]));
    float t;
    for (int i = 0; i < 4; i++) { CK(cudaEventElapsedTime(&t, e[i], e[i + 1])); ms5[i] += t; }
    CK(cudaEventElapsedTime(&t, e[0], e[4]));
    ms5[4] += t;
  }
  for (int i = 0; i < 5; i++) ms5[i] /= (float)n;
  return 0;
}

} // extern "C"
