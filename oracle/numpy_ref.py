"""TEST INFRASTRUCTURE ONLY -- the block API of oracle/ref.py over the numpy restatement (oracle/t2oracle.py).

The parity tests compare the CUDA path with the unmodified reference through oracle/ref.py.  That needs
oracle/_ref/libdvbt2ll_ref.so, which can only be built where the reference sources are present; they are not part
of this repository.  Elsewhere the tests compare with this module instead.  It is NOT the reference: it is the
restatement, which matches the reference's own output where that output is stored (tests/golden/chain_*.json,
written by tools/make_golden.py from oracle/_ref) and which the parity tests found equal to the reference on all
their inputs while oracle/_ref was built.

So that a later change to the restatement cannot move with a change to the CUDA path, every output this module
hands out is checked against a digest recorded from it (LEDGER, keyed by the block, its parameters, the call number
on the instance and the input bytes): SHA-256 (96 bits) for bits and cells, RMS plus a seeded sample for baseband.  An input
with no recorded output is an error.  To re-record after a deliberate change, run the suite with
DVBT2LL_RECORD_REFERENCE=<file> and replace LEDGER with that file.
Reference-only behaviour (its broken short-code encoder, its over-full-frame forecast) is not modelled.
"""
import atexit
import hashlib
import json
import os

import numpy as np

from oracle import t2oracle as O

# the restatement encodes every code, including the three the reference's own encoder cannot (ref.REF_LDPC_BROKEN)
REF_LDPC_BROKEN = frozenset()

LEDGER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "numpy_ref_ledger.json")
_RECORD = os.environ.get("DVBT2LL_RECORD_REFERENCE")
_ledger = None


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:32]


def _digest(out, baseband):
    if baseband:
        rms = float(np.sqrt(np.mean(np.abs(out.astype(np.complex128)) ** 2)))
        pick = np.random.default_rng(out.size).choice(out.size, min(4, out.size), replace=False)
        return {"n": int(out.size), "rms": rms, "iq": [round(float(v) / rms, 7) for v in out[pick].view(np.float32)]}
    return _sha(out)[:24]


def _pinned(key, out, baseband=False):
    """Check `out` against the digest recorded for `key` (or record it).  Returns out."""
    global _ledger
    if _ledger is None:
        if _RECORD:
            _ledger = {}
            atexit.register(lambda: json.dump(_ledger, open(_RECORD, "w"), sort_keys=True, separators=(",", ":")))
        else:
            with open(LEDGER) as f:
                _ledger = json.load(f)
    out = np.asarray(out)
    got = _digest(out, baseband)
    k = hashlib.sha256(key.encode()).hexdigest()[:24]
    if _RECORD:
        _ledger[k] = got
        return out
    want = _ledger.get(k)
    assert want is not None, "numpy_ref: no recorded output for this input (%s)" % key[:120]
    if isinstance(got, dict):
        rms = want["rms"]
        assert got["n"] == want["n"] and abs(got["rms"] - rms) <= 1e-6 * rms and \
            np.abs(np.array(got["iq"]) - np.array(want["iq"])).max() <= 1e-6, "numpy_ref: baseband differs from the record"
    else:
        assert got == want, "numpy_ref: output differs from the record (%s)" % key[:120]
    return out


class Block(object):
    """One block: `step(data, nframes)` runs nframes frames from data and returns (items out, items consumed)."""
    warnings = 0

    def __init__(self, output_multiple, input_per_frame, step, name, baseband=False):
        self.output_multiple = output_multiple
        self._in = input_per_frame
        self._step = step
        self._name, self._baseband, self._calls = name, baseband, 0

    def forecast(self, noutput):
        return (noutput // self.output_multiple) * self._in

    def work(self, data, nframes):
        out, used = self._step(data, nframes)
        self._calls += 1
        key = "%s|%d|%d|%d|%s" % (self._name, self._calls, nframes, used, _sha(np.asarray(data)[:used]))
        return _pinned(key, out, self._baseband), used


class BbHeaderBch(Block):
    def __init__(self, framesize, rate, mode, inband, fecblocks, tsrate):
        self.bb = O.BbHeaderBch(framesize, rate, mode, inband, fecblocks, tsrate)
        self.fs, self.rate = framesize, rate
        p = self.bb.p
        Block.__init__(self, p["nbch"], (p["kbch"] - 80) // 8, self.bb.work,
                       "bbheaderbch%r" % ((framesize, rate, mode, inband, fecblocks, tsrate),))

    @property
    def warnings(self):
        return self.bb.warnings

    def ldpc(self, bch_bits, frame_size):
        info = np.asarray(bch_bits[:self.bb.p["nbch"]], np.uint8)
        cw = O.ldpc_encode(info[None], self.fs, self.rate)[0][:frame_size]
        return _pinned("ldpc|%d|%d|%s" % (self.fs, self.rate, _sha(info)), cw)


def _per_frame(frame_work, n):
    """step() of a block whose restatement takes one frame of n complex items per call"""
    def step(x, nframes):
        x = np.asarray(x[:nframes * n], np.complex64)
        return np.concatenate([frame_work(x[f * n:(f + 1) * n]) for f in range(nframes)]), nframes * n
    return step


def bbheaderbch(framesize, rate, mode, inband, fecblocks, tsrate):
    return BbHeaderBch(framesize, rate, mode, inband, fecblocks, tsrate)


def interleavermod(framesize, rate, constellation, rotation):
    N = O.fec_params(framesize, rate)["nldpc"]
    cell_size = N // (2 * (constellation + 1))

    def step(fec, nframes):
        cw = np.asarray(fec[:nframes * N], np.uint8).reshape(nframes, N)
        return O.interleavermod(cw, framesize, rate, constellation, rotation).reshape(-1), nframes * N
    return Block(cell_size, N, step, "interleavermod%r" % ((framesize, rate, constellation, rotation),))


def framemapper(framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize, guardinterval,
                l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble, inputmode,
                reservedbiasbits, l1scrambled, inband):
    args = (framesize, rate, constellation, rotation, fecblocks, tiblocks, carriermode, fftsize, guardinterval,
            l1constellation, pilotpattern, t2frames, numdatasyms, paprmode, version, preamble, inputmode,
            reservedbiasbits, l1scrambled, inband)
    fm = O.FrameMapper(dict(framesize=framesize, rate=rate, constellation=constellation, rotation=rotation,
                            fecblocks=fecblocks, tiblocks=tiblocks, carriermode=carriermode, fftsize=fftsize,
                            guardinterval=guardinterval, l1constellation=l1constellation, pilotpattern=pilotpattern,
                            t2frames=t2frames, numdatasyms=numdatasyms, paprmode=paprmode, version=version,
                            preamble=preamble, inputmode=inputmode, reservedbiasbits=reservedbiasbits,
                            l1scrambled=l1scrambled, inband=inband))
    b = Block(fm.mapped_items, fm.stream_items, _per_frame(fm.work, fm.stream_items), "framemapper%r" % (args,))
    b.warnings = int(fm.dummy < 0)      # the reference warns when the FEC blocks do not fit the T2 frame
    return b


def pilotgen(carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble, misogroup,
             equalization, bandwidth, vlength):
    args = (carriermode, fftsize, pilotpattern, guardinterval, numdatasyms, paprmode, version, preamble, misogroup,
            equalization, bandwidth, vlength)
    pg = O.PilotGen(dict(carriermode=carriermode, fftsize=fftsize, pilotpattern=pilotpattern,
                         guardinterval=guardinterval, numdatasyms=numdatasyms, paprmode=paprmode, version=version,
                         preamble=preamble, misogroup=misogroup, equalization=equalization, bandwidth=bandwidth,
                         vlength=vlength))
    d = pg.d
    b = Block(pg.p1.size + d["L"] * (d["N"] + d["gi"]), d["active"], _per_frame(pg.work, d["active"]),
              "pilotgen%r" % (args,), baseband=True)

    def get_int_array(name):
        """the reference's carrier maps: p2_carrier_map, fc_carrier_map, data_carrier_map:<symbol>"""
        l = {"p2_carrier_map": 0, "fc_carrier_map": d["L"] - 1}.get(name)
        l = int(name.split(":")[1]) if l is None else l
        return _pinned("carrier_map%r|%s" % (args, name), pg.carrier_map(l))
    b.get_int_array = get_int_array
    return b


class Chain(object):
    """The reference flowgraph order, one T2 frame per run_frame() with state carried across frames (as ref.Chain)."""

    def __init__(self, cfg):
        self.cfg = cfg = dict(cfg)
        self.bb = bbheaderbch(cfg["framesize"], cfg["rate"], cfg["inputmode"], cfg["inband"], cfg["fecblocks"],
                              cfg["tsrate"])
        self.im = interleavermod(cfg["framesize"], cfg["rate"], cfg["constellation"], cfg["rotation"])
        self.fm = framemapper(*[cfg[k] for k in (
            "framesize", "rate", "constellation", "rotation", "fecblocks", "tiblocks", "carriermode", "fftsize",
            "guardinterval", "l1constellation", "pilotpattern", "t2frames", "numdatasyms", "paprmode", "version",
            "preamble", "inputmode", "reservedbiasbits", "l1scrambled", "inband")])
        self.pg = pilotgen(*[cfg[k] for k in (
            "carriermode", "fftsize", "pilotpattern", "guardinterval", "numdatasyms", "paprmode", "version",
            "preamble", "misogroup", "equalization", "bandwidth", "vlength")])
        p = O.fec_params(cfg["framesize"], cfg["rate"])
        self.frame_size, self.nbch, self.kbch = p["nldpc"], p["nbch"], p["kbch"]
        self.ts_pos = 0

    def ts_bytes_per_t2_frame(self):
        return self.cfg["fecblocks"] * ((self.kbch - 80) // 8)

    def run_frame(self, ts):
        F = self.cfg["fecblocks"]
        bch, used = self.bb.work(ts[self.ts_pos:], F)
        self.ts_pos += used
        fec = O.ldpc_encode(bch.reshape(F, self.nbch), self.cfg["framesize"], self.cfg["rate"]).reshape(-1)
        fec = _pinned("ldpc_frame|%d|%d|%s" % (self.cfg["framesize"], self.cfg["rate"], _sha(bch)), fec)
        cells, _ = self.im.work(fec, F)
        mapped, _ = self.fm.work(cells, 1)
        samples, _ = self.pg.work(mapped, 1)
        return {"bch": bch, "fec": fec, "cells": cells, "mapped": mapped, "samples": samples, "ts_used": used}
