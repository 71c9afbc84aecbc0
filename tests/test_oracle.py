"""Pins the numpy oracle restatement (oracle/t2oracle.py) to the UNMODIFIED reference (oracle/_ref) and to
the committed golden fixtures, and checks reference-independent known answers (SURVEY.md section 4)."""
import numpy as np
import pytest

from dvbt2ll_b200 import configs as K
from oracle import t2oracle as O
from common import bits_equal, cells_equal, max_err_over_rms, load_golden, sha, fm_args, pg_args


@pytest.mark.parametrize("name", ["c1", "c2", "c4"])
def test_oracle_chain_equals_reference(reflib, name):
    cfg = K.resolve(name)
    ch = reflib.Chain(cfg)
    ts = K.make_ts(2 * ch.ts_bytes_per_t2_frame() + 1000)
    o = O.chain(cfg, ts, 2)
    r = [ch.run_frame(ts) for _ in range(2)]
    cat = lambda k: np.concatenate([x[k] for x in r])   # noqa: E731
    assert o["ts_used"] == sum(x["ts_used"] for x in r)
    assert bits_equal(o["bch"], cat("bch"))
    assert bits_equal(o["fec"], cat("fec"))
    assert cells_equal(o["cells"], cat("cells"))
    assert cells_equal(o["mapped"], cat("mapped"))
    assert max_err_over_rms(o["samples"], cat("samples")) < 1e-6


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_oracle_matches_golden(name):
    """Golden fixtures were produced by the reference itself (tools/make_golden.py): both stored T2 frames (the second
    one checks the state carried across frames)."""
    g = load_golden("chain_%s.json" % name)
    cfg = K.resolve(name)
    nfr = 2
    n = g["frames"][0]["ts_used"]
    ts = K.make_ts(2 * n + 1000)
    assert sha(ts[:4096]) == g["ts_head_sha256"]
    o = O.chain(cfg, ts, nfr)
    F = cfg["fecblocks"]
    for fr in range(nfr):
        gf = g["frames"][fr]
        nb, nf = o["bch"].size // nfr, o["fec"].size // nfr
        assert sha(np.packbits(o["bch"][fr * nb:(fr + 1) * nb])) == gf["bch_sha256"]
        assert sha(np.packbits(o["fec"][fr * nf:(fr + 1) * nf])) == gf["fec_sha256"]
        nc, nm, ns = o["cells"].size // nfr, o["mapped"].size // nfr, gf["n_samples"]
        assert sha(o["cells"][fr * nc:(fr + 1) * nc]) == gf["cells_sha256"]
        assert sha(o["mapped"][fr * nm:(fr + 1) * nm]) == gf["mapped_sha256"]
        head = np.array(gf["samples_head"], dtype=np.float32).view(np.complex64)
        s = o["samples"][fr * ns:(fr + 1) * ns]
        assert np.abs(s[:head.size] - head).max() <= 1e-6 * gf["samples_rms"]
    assert F * ((O.fec_params(cfg["framesize"], cfg["rate"])["kbch"] - 80) // 8) == g["frames"][0]["ts_used"]


@pytest.mark.parametrize("mode,inband", [(1, 0), (0, 1), (1, 1)])
def test_oracle_bbheader_modes(reflib, mode, inband):
    fs, rate = 0, O.C3_5
    a = O.BbHeaderBch(fs, rate, mode, inband, 3, 4000000)
    b = reflib.bbheaderbch(fs, rate, mode, inband, 3, 4000000)
    ts = K.make_ts(20000)
    pa = pb = 0
    for n in (1, 3, 2):
        xa, ua = a.work(ts[pa:], n)
        xb, ub = b.work(ts[pb:], n)
        assert ua == ub and bits_equal(xa, xb)
        pa += ua
        pb += ub


@pytest.mark.parametrize("fs,rate,con,rot", [(1, O.C3_5, 1, 1), (1, O.C1_2, 0, 1), (0, O.C1_3, 0, 0), (0, O.C2_5, 2, 1),
                                             (0, O.C1_3, 3, 0), (1, O.C5_6, 2, 0), (0, O.C3_4, 1, 0), (1, O.C3_4, 3, 1)])
def test_oracle_ldpc_and_mapper_modes(reflib, fs, rate, con, rot):
    rng = np.random.default_rng(11)
    p = O.fec_params(fs, rate)
    info = rng.integers(0, 2, (2, p["nbch"]), dtype=np.uint8)
    fec = O.ldpc_encode(info, fs, rate)
    if (fs, rate) not in reflib.REF_LDPC_BROKEN:
        rbb = reflib.bbheaderbch(fs, rate, 0, 0, 1, 0)
        want = np.stack([rbb.ldpc(info[f], p["nldpc"]) for f in range(2)])
        assert bits_equal(fec, want)
    cells = O.interleavermod(fec, fs, rate, con, rot)
    rim = reflib.interleavermod(fs, rate, con, rot)
    assert cells_equal(cells.reshape(-1), rim.work(fec.reshape(-1), 2)[0])


def test_oracle_frame_and_pilot_variants(reflib):
    rng = np.random.default_rng(12)
    base = K.resolve("c1")
    variants = [dict(base, l1constellation=0, fecblocks=6), dict(base, l1constellation=1, fecblocks=7),
                dict(base, l1constellation=2, fecblocks=7, tiblocks=0),
                dict(base, version=2, l1scrambled=1, reservedbiasbits=1, inband=1, inputmode=1),
                dict(base, fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
                     fecblocks=18, paprmode=2, vlength=2048),
                dict(K.resolve("c2"), preamble=K.PREAMBLE_T2_MISO, misogroup=1, fecblocks=18, tiblocks=5, equalization=1)]
    for cfg in variants:
        fm, rf = O.FrameMapper(cfg), reflib.framemapper(*fm_args(cfg))
        assert fm.mapped_items == rf.output_multiple
        for _ in range(3):
            x = (rng.standard_normal(fm.stream_items) + 1j * rng.standard_normal(fm.stream_items)).astype(np.complex64)
            y = fm.work(x)
            assert cells_equal(y, rf.work(x, 1)[0])
        pg, rp = O.PilotGen(cfg), reflib.pilotgen(*pg_args(cfg))
        for l in range(pg.d["L"]):
            if l < pg.d["n_p2"]:
                m = rp.get_int_array("p2_carrier_map")
            elif pg.d["n_fc"] and l == pg.d["L"] - 1:
                m = rp.get_int_array("fc_carrier_map")
            else:
                m = rp.get_int_array("data_carrier_map:%d" % l)
            assert np.array_equal(pg.carrier_map(l), m)
        assert max_err_over_rms(pg.work(y), rp.work(y, 1)[0]) < 1e-6


def _wide_configs():
    import json
    import os
    with open(os.path.join(os.path.dirname(__file__), "golden", "fuzz_configs_r2w.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("idx", [0, 2, 3, 5, 9, 13, 19, 22])
def test_oracle_wide_parameter_sets(reflib, idx):
    """MISO / T2-Lite preambles, MISO group 2, all PAPR signalling modes, reserved-bias bits, every bandwidth
    (tools/make_fuzz_configs.py ... wide): frame mapper bit-exact and pilot generator within 1e-6 of RMS of the
    reference for eight of the committed random sets (the GPU sweep runs all 24 through the chain)."""
    rng = np.random.default_rng(40 + idx)
    cfg = K.resolve(_wide_configs()[idx])
    fm, rf = O.FrameMapper(cfg), reflib.framemapper(*fm_args(cfg))
    assert fm.mapped_items == rf.output_multiple
    y = None
    for _ in range(cfg["t2frames"] + 1):
        x = (rng.standard_normal(fm.stream_items) + 1j * rng.standard_normal(fm.stream_items)).astype(np.complex64)
        y = fm.work(x)
        assert cells_equal(y, rf.work(x, 1)[0])
    pg, rp = O.PilotGen(cfg), reflib.pilotgen(*pg_args(cfg))
    assert max_err_over_rms(pg.work(y), rp.work(y, 1)[0]) < 1e-6


# ---- known answers that do not depend on the reference code ------------------------------------------
def test_bch_codewords_divisible_by_generator():
    rng = np.random.default_rng(5)
    for r, k in ((160, 43040), (192, 32208), (168, 12432)):
        msg = rng.integers(0, 2, (1, k), dtype=np.uint8)
        cw = np.concatenate([msg, O.bch_parity(msg, r)], axis=1)[0]
        g = O.bch_generator(r)
        assert g.size == r + 1
        # polynomial long division over GF(2), highest order first
        rem = cw.copy()
        gh = g[::-1]
        for i in range(k):
            if rem[i]:
                rem[i:i + r + 1] ^= gh
        assert not rem.any()


def test_ldpc_parity_checks():
    rng = np.random.default_rng(6)
    for fs, rate in ((1, O.C2_3), (0, O.C4_5), (1, O.C3_5)):
        p = O.fec_params(fs, rate)
        info = rng.integers(0, 2, (1, p["nbch"]), dtype=np.uint8)
        cw = O.ldpc_encode(info, fs, rate)[0]
        ii, pi = O.ldpc_edges(O._LDPC_TAB[(fs, rate)], p["q"], p["nbch"], p["nldpc"])
        P = p["nldpc"] - p["nbch"]
        s = np.bincount(pi, weights=cw[ii], minlength=P).astype(np.int64) & 1
        par = cw[p["nbch"]:]
        prev = np.concatenate([[0], par[:-1]])
        assert not np.any(s ^ par ^ prev)


def test_crc8_check_value_and_constellation_power():
    t = O.crc8_table()
    crc = 0
    for v in b"123456789":
        crc = int(t[crc ^ v])
    assert crc == 0xBC           # CRC-8/DVB-S2 check value
    for con in range(4):
        for rot in (0, 1):
            lut = O.constellation(con, rot)
            assert abs(np.mean(np.abs(lut) ** 2) - 1.0) < 1e-6


def test_frequency_interleaver_is_permutation():
    for fi, lim in ((0, 764), (2, 3328), (3, 6208), (5, 27404), (5, 22432)):
        for odd in (False, True):
            H = O.freq_interleaver_H(fi, lim, odd)
            assert np.array_equal(np.sort(H), np.arange(lim))
