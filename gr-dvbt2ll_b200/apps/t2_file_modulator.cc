// t2_file_modulator -- the step before and after the hot path for a file-based mux (SURVEY.md 8(f) items 1 and 4):
// transport-stream FILE(S) in (one per PLP), complex baseband FILE out, through the C ABI of libdvbt2ll_cuda.so.
// It stands where the shipped flowgraph has ule_source and uhd_usrp_sink (apps/vv009-4kshort.grc:1663-1697).
//
// TS ingest: the reader acquires packet sync (0x47 every 188 bytes over 5 packets, dvbt2ll_ts_sync), starts the stream
// on a packet boundary and, when a file ends inside a T2 frame, completes the frame with null packets (PID 0x1FFF,
// dvbt2ll_ts_fill) -- what a rate-adapting source does when the multiplex runs dry.  Frames are modulated in batches
// of `batch` T2 frames per call (stream position carried by first_frame + the 187 history bytes in front of a batch).
//
// usage: t2_file_modulator [--config c1|c2|c3|c4] [--plp-blocks a,b,..] [--plp BLOCKS[:FRAMESIZE:RATE:CONSTELLATION:ROTATION]]...
//                          [--frames N] [--batch B] [--sc16 GAIN] [--papr-tr ITER:VCLIP:TONEMAX] [--miso 1|2|both [--out2 FILE2]]
//                          --out FILE  TS_FILE [TS_FILE ...]
// --plp, once per PLP: its FEC blocks per T2 frame and, optionally, its own FEC type, code rate, constellation and
// rotation (enum values of dvbt2ll_config.h; the config's where omitted).
// --papr-tr: paprmode = PAPR_TR and tone-reservation PAPR reduction on the reserved carriers (dvbt2ll_chain_set_papr_tr).
// The reserved carriers take cells away: a config whose FEC blocks no longer fit is refused as over-full; lower its
// block count with --plp BLOCKS (c1: 7, c3: 200, c4: 119; c2 fits as it is).
// --miso: preamble = T2_MISO; 1 or 2 emits that transmitter group (2 with MISO processing, dvbt2ll_chain_set_miso);
// both writes group 1 to --out and group 2 to --out2 from one FEC pass (dvbt2ll_chain_run_host_miso).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dvbt2ll_cuda.h"

namespace {

// the five BASELINE.json per-channel configurations (enum values of dvbt2ll_config.h), as in python/dvbt2ll_b200/configs.py
bool named_config(const std::string &n, dvbt2ll_chain_params *p)
{
  dvbt2ll_chain_params c;
  std::memset(&c, 0, sizeof(c));
  c.l1constellation = 3; c.t2frames = 2; c.bandwidth = 4; c.tsrate = 4000000; c.tiblocks = 3;
  if (n == "c1") { c.framesize = 0; c.rate = 4; c.constellation = 3; c.rotation = 1; c.fecblocks = 8; c.fftsize = 2; c.guardinterval = 0; c.pilotpattern = 6; c.numdatasyms = 3; c.vlength = 4096; }
  else if (n == "c2") { c.framesize = 1; c.rate = 0; c.constellation = 0; c.rotation = 0; c.fecblocks = 19; c.fftsize = 1; c.guardinterval = 3; c.pilotpattern = 0; c.numdatasyms = 100; c.vlength = 8192; }
  else if (n == "c3") { c.framesize = 1; c.rate = 2; c.constellation = 3; c.rotation = 1; c.fecblocks = 202; c.carriermode = 1; c.fftsize = 5; c.guardinterval = 4; c.pilotpattern = 6; c.numdatasyms = 59; c.vlength = 32768; }
  else if (n == "c4") { c.framesize = 1; c.rate = 1; c.constellation = 2; c.rotation = 1; c.fecblocks = 120; c.fftsize = 4; c.guardinterval = 1; c.pilotpattern = 3; c.numdatasyms = 100; c.vlength = 16384; }
  else return false;
  *p = c;
  return true;
}

std::vector<unsigned char> read_file(const char *path)
{
  std::vector<unsigned char> v;
  FILE *f = std::fopen(path, "rb");
  if (!f) return v;
  unsigned char buf[1 << 16];
  size_t n;
  while ((n = std::fread(buf, 1, sizeof(buf), f)) > 0) v.insert(v.end(), buf, buf + n);
  std::fclose(f);
  return v;
}

} // namespace

int main(int argc, char **argv)
{
  std::string cfg = "c1", out_path, out2_path, miso;
  std::vector<int> plp_blocks;
  std::vector<dvbt2ll_plp_params> plps;
  std::vector<int> plp_own;          // --plp entries that name their own parameters
  std::vector<const char *> inputs;
  int frames = -1, batch = 4, sc16 = 0;
  float gain = 1.0f;
  int tr_iter = 0;
  float tr_vclip = 0.f, tr_tone_max = 0.f;
  for (int i = 1; i < argc; i++) {
    std::string a = argv[i];
    if (a == "--config" && i + 1 < argc) cfg = argv[++i];
    else if (a == "--out" && i + 1 < argc) out_path = argv[++i];
    else if (a == "--out2" && i + 1 < argc) out2_path = argv[++i];
    else if (a == "--miso" && i + 1 < argc) miso = argv[++i];
    else if (a == "--frames" && i + 1 < argc) frames = std::atoi(argv[++i]);
    else if (a == "--batch" && i + 1 < argc) batch = std::atoi(argv[++i]);
    else if (a == "--sc16" && i + 1 < argc) { sc16 = 1; gain = (float)std::atof(argv[++i]); }
    else if (a == "--papr-tr" && i + 1 < argc) {
      if (std::sscanf(argv[++i], "%d:%f:%f", &tr_iter, &tr_vclip, &tr_tone_max) != 3) {
        std::fprintf(stderr, "--papr-tr ITER:VCLIP:TONEMAX\n");
        return 2;
      }
    }
    else if (a == "--plp-blocks" && i + 1 < argc) {
      for (char *t = std::strtok(argv[++i], ","); t; t = std::strtok(0, ",")) plp_blocks.push_back(std::atoi(t));
    }
    else if (a == "--plp" && i + 1 < argc) {
      int v[5] = { 0, -1, -1, -1, -1 };
      const int n = std::sscanf(argv[++i], "%d:%d:%d:%d:%d", &v[0], &v[1], &v[2], &v[3], &v[4]);
      if (n != 1 && n != 5) { std::fprintf(stderr, "--plp BLOCKS[:FRAMESIZE:RATE:CONSTELLATION:ROTATION]\n"); return 2; }
      dvbt2ll_plp_params q = { v[0], v[1], v[2], v[3], v[4] };
      plps.push_back(q);
      plp_own.push_back(n == 5);
    }
    else inputs.push_back(argv[i]);
  }
  dvbt2ll_chain_params prm;
  const bool miso_ok = miso.empty() ? out2_path.empty() : (miso == "both") == !out2_path.empty() && (miso == "1" || miso == "2" || miso == "both");
  if (!named_config(cfg, &prm) || out_path.empty() || inputs.empty() || batch < 1 || (!plps.empty() && !plp_blocks.empty()) || !miso_ok) {
    std::fprintf(stderr, "usage: %s [--config c1..c4] [--plp-blocks a,b,.. | --plp BLOCKS[:FRAMESIZE:RATE:CONSTELLATION:ROTATION]...] [--frames N] [--batch B] [--sc16 GAIN] [--papr-tr ITER:VCLIP:TONEMAX] [--miso 1|2|both [--out2 FILE2]] --out FILE TS_FILE...\n", argv[0]);
    return 2;
  }
  bool own = false;
  for (size_t p = 0; p < plps.size(); p++) {
    if (plp_own[p]) { own = true; continue; }
    plps[p].framesize = prm.framesize; plps[p].rate = prm.rate; plps[p].constellation = prm.constellation; plps[p].rotation = prm.rotation;
  }
  if (!own)
    for (size_t p = 0; p < plps.size(); p++) plp_blocks.push_back(plps[p].fecblocks);
  const int P = own ? (int)plps.size() : plp_blocks.empty() ? 1 : (int)plp_blocks.size();
  if ((int)inputs.size() != P) { std::fprintf(stderr, "one TS file per PLP expected (%d)\n", P); return 2; }
  if (P == 1 && !own && !plps.empty()) prm.fecblocks = plps[0].fecblocks;
  if (tr_iter) prm.paprmode = 2;      // PAPR_TR
  if (!miso.empty()) { prm.preamble = 1; prm.misogroup = miso == "2" ? 1 : 0; }      // PREAMBLE_T2_MISO, MISO_TX1 / TX2
  dvbt2ll_handle *h = own ? dvbt2ll_chain_create_plps(&prm, P, plps.data(), batch, -1)
                    : P == 1 ? dvbt2ll_chain_create(&prm, batch, -1) : dvbt2ll_chain_create_multiplp(&prm, P, plp_blocks.data(), batch, -1);
  if (!h) { std::fprintf(stderr, "chain: %s\n", dvbt2ll_last_error()); return 1; }
  if (sc16 && dvbt2ll_chain_set_sink(h, 1, gain) < 0) { std::fprintf(stderr, "%s\n", dvbt2ll_last_error()); return 1; }
  if (tr_iter && dvbt2ll_chain_set_papr_tr(h, tr_iter, tr_vclip, tr_tone_max) < 0) { std::fprintf(stderr, "%s\n", dvbt2ll_last_error()); return 1; }
  if (!miso.empty() && dvbt2ll_chain_set_miso(h, 1) < 0) { std::fprintf(stderr, "%s\n", dvbt2ll_last_error()); return 1; }

  // ---- ingest: sync acquisition per file; whole T2 frames available = limited by the shortest PLP (then null filled)
  std::vector<std::vector<unsigned char> > ts(P);
  std::vector<size_t> start(P, 0);
  long long avail = -1;
  for (int p = 0; p < P; p++) {
    ts[p] = read_file(inputs[p]);
    long long off = dvbt2ll_ts_sync(ts[p].data(), ts[p].size());
    if (off < 0) { std::fprintf(stderr, "%s: no transport-stream sync found\n", inputs[p]); return 1; }
    start[p] = (size_t)off;
    // frames this file fills at least partly
    long long n = 0;
    while (dvbt2ll_chain_plp_ts_bytes(h, p, 0, (int)n) < (long long)(ts[p].size() - start[p])) n++;
    if (avail < 0 || n > avail) avail = n;
  }
  if (frames < 0 || frames > avail) frames = (int)avail;
  const long long S = dvbt2ll_chain_samples_per_frame(h);
  const size_t ssz = sc16 ? 4 : 8;
  FILE *fo = std::fopen(out_path.c_str(), "wb");
  if (!fo) { std::fprintf(stderr, "cannot write %s\n", out_path.c_str()); return 1; }
  FILE *fo2 = 0;
  if (!out2_path.empty() && !(fo2 = std::fopen(out2_path.c_str(), "wb"))) { std::fprintf(stderr, "cannot write %s\n", out2_path.c_str()); return 1; }
  std::vector<unsigned char> out((size_t)batch * S * ssz), out2(fo2 ? out.size() : 0), rows;
  long long nulls = 0;
  for (int f0 = 0; f0 < frames; f0 += batch) {
    const int n = frames - f0 < batch ? frames - f0 : batch;
    const long long hist = dvbt2ll_chain_history_bytes(h, f0);
    long long width = 0;
    for (int p = 0; p < P; p++) { const long long b = dvbt2ll_chain_plp_ts_bytes(h, p, f0, n); if (b > width) width = b; }
    const size_t pitch = (size_t)(hist + width);
    rows.assign(pitch * P, 0);
    for (int p = 0; p < P; p++) {
      const long long pos = dvbt2ll_chain_plp_ts_bytes(h, p, 0, f0), len = dvbt2ll_chain_plp_ts_bytes(h, p, f0, n);
      // [pos - hist, pos + len) of the aligned stream, null packets where the file has ended
      nulls += dvbt2ll_ts_fill(rows.data() + pitch * p, (size_t)(hist + len), ts[p].data() + start[p], ts[p].size() - start[p], pos - hist);
    }
    const int r = fo2 ? dvbt2ll_chain_run_host_miso(h, rows.data() + hist, (long long)pitch, 1, n, f0, out.data(), out2.data())
                      : dvbt2ll_chain_run_host(h, rows.data() + hist, (long long)pitch, 1, n, f0, out.data());
    if (r < 0) { std::fprintf(stderr, "chain: %s\n", dvbt2ll_last_error()); return 1; }
    std::fwrite(out.data(), ssz, (size_t)n * S, fo);
    if (fo2) std::fwrite(out2.data(), ssz, (size_t)n * S, fo2);
  }
  std::fclose(fo);
  if (fo2) std::fclose(fo2);
  std::printf("%d T2 frame(s), %lld samples, %lld null-packet bytes inserted, %lld kernel launches\n", frames, (long long)frames * S, nulls,
              dvbt2ll_kernel_launches());
  dvbt2ll_destroy(h);
  return 0;
}
