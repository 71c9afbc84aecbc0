"""GPU parity tests added in round 2: full-size channels against the reference itself, the three short LDPC codes the
reference's own encoder cannot run, the streaming / device-resident / linked variants of the drop-in path, the
reference's over-full frame behaviour, several devices in one process and the ordered multi-GPU reassembly."""
import ctypes as C

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from dvbt2ll_b200 import shard
from common import bits_equal, cells_equal, mer_db, max_err_over_rms, fm_args

pytestmark = pytest.mark.gpu

MER_MIN_DB = 90.0
MAX_ERR_OVER_RMS = 1e-5


def test_full_size_channels_against_reference(reflib):
    """BASELINE config 5 at full size: channels 17 and 63 of the 64-channel launch (seeds + 17, + 63) against the
    unmodified reference flowgraph run on the same TS -- not against the repo's own kernels."""
    cfg = K.resolve("c3")
    nch = 64
    ch = T.Chain(cfg, max_frames=nch)
    n_ts = ch.ts_bytes_per_frame
    ts = np.stack([K.make_ts(n_ts, seed=K.TS_SEED + c) for c in range(nch)])
    out = ch.run_host(ts, nch, 1)
    for c in (17, 63):
        want = reflib.Chain(cfg).run_frame(np.concatenate([ts[c], np.zeros(1024, np.uint8)]))["samples"]
        assert mer_db(out[c], want) >= MER_MIN_DB, c
        assert max_err_over_rms(out[c], want) <= MAX_ERR_OVER_RMS, c


@pytest.mark.parametrize("rate", [K.C1_2, K.C3_4, K.C5_6])
def test_chain_short_codes_stage_taps_match_oracle(rate):
    """Short FECFRAME 1/2, 3/4, 5/6 end to end, with the chain's bch and fec taps: the reference's dead-code LDPC overruns
    its table for these (oracle/ref.py REF_LDPC_BROKEN), so the checker is the numpy restatement (address-table scatter
    form, H.c = 0)."""
    from oracle import t2oracle as O
    cfg = K.resolve(dict(K.CONFIGS["c1"], rate=rate))
    nframes = 2
    ch = T.Chain(cfg, max_frames=nframes)
    ts = K.make_ts(ch.ts_bytes(0, nframes) + 16, seed=K.TS_SEED + rate)
    out = ch.run_host(ts[:ch.ts_bytes(0, nframes)], 1, nframes)[0]
    want = O.chain(cfg, ts, nframes)
    F = cfg["fecblocks"]
    p = O.fec_params(cfg["framesize"], rate)
    bch = np.unpackbits(ch.tap("bch").reshape(nframes * F, -1)[:, :p["nbch"] // 8], axis=1).reshape(-1)
    assert bits_equal(bch, np.asarray(want["bch"]).reshape(-1))
    # FECFRAMEs: the chain keeps the parity in interleaved-row ("u") order; put the oracle's codewords in that order
    fec = np.unpackbits(ch.tap("fec").reshape(nframes * F, -1)[:, :p["nldpc"] // 8], axis=1)
    w = np.asarray(want["fec"]).reshape(nframes * F, p["nldpc"])
    q = p["q"]
    par = w[:, p["nbch"]:].reshape(nframes * F, 360, q).transpose(0, 2, 1).reshape(nframes * F, -1)
    assert bits_equal(fec, np.concatenate([w[:, :p["nbch"]], par], axis=1))
    s = np.asarray(want["samples"]).reshape(-1)
    assert mer_db(out, s) >= MER_MIN_DB
    assert max_err_over_rms(out, s) <= MAX_ERR_OVER_RMS


def test_chain_32k_int16_multichannel():
    """32K + int16 sink with several channels: run_host alternates channel groups on two streams whose 32K transforms
    run at the same time, and every channel's int16 output must still match its complex64 output."""
    cfg = K.resolve("c3")
    nch = 6
    ch = T.Chain(cfg, max_frames=nch)
    n_ts = ch.ts_bytes_per_frame
    ts = np.stack([K.make_ts(n_ts, seed=K.TS_SEED + 100 + c) for c in range(nch)])
    f32 = ch.run_host(ts, nch, 1)
    ch.set_sink(1, 0.2)
    for _ in range(3):                      # the race needs both streams busy at once: repeat
        q = ch.run_host(ts, nch, 1)
        want = np.clip(np.rint(f32.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(nch, -1, 2)
        assert q.shape == want.shape and q.dtype == np.int16
        assert np.abs(q.astype(np.int64) - want.astype(np.int64)).max() <= 1


def test_bb_work_device_streams_with_history():
    """dvbt2ll_work_device on the BB block, two calls on one device-resident stream: the second call starts inside a
    packet, so its first CRC-8 covers bytes consumed by the first call (read from in front of d_in)."""
    from oracle import t2oracle as O
    fs, rate = K.FECFRAME_SHORT, K.C3_5
    bb = T.bbheaderbch_bb(fs, rate, 0, 0, 1, 0)
    ob = O.BbHeaderBch(fs, rate, 0, 0, 1, 0)
    nbch = bb.output_multiple
    per = bb.forecast(nbch)
    assert per % 188 != 0                    # frames do not end on packet boundaries
    nfr = (2, 3)
    ts = K.make_ts(sum(nfr) * per + 400, seed=77)
    dev_ts = T.DeviceBuffer(256 + ts.size, data=np.concatenate([np.zeros(256, np.uint8), ts]))
    L = T.lib()
    pos = 0
    got = []
    for n in nfr:
        d_out = T.DeviceBuffer(n * nbch)
        used = C.c_int(0)
        r = L.dvbt2ll_work_device(bb._h, dev_ts.ptr + 256 + pos, ts.size - pos, d_out.ptr, n * nbch, C.byref(used), None)
        assert r == n * nbch, T.last_error()
        got.append(d_out.to_host(np.uint8))
        pos += used.value
        d_out.free()
    want, used2 = ob.work(ts, sum(nfr))
    assert pos == used2
    assert bits_equal(np.concatenate(got), want)


def test_chain_wrapper_first_frame_history(reflib):
    """Chain.run_host(first_frame > 0): rows start with the 187 history bytes; two channels, frames 1..2 of three."""
    cfg = K.resolve("c1")
    nch, nframes = 2, 3
    ch = T.Chain(cfg, max_frames=nch * nframes)
    n_all = ch.ts_bytes(0, nframes)
    S = ch.samples_per_frame
    ts = np.stack([K.make_ts(n_all, seed=K.TS_SEED + 5 + c) for c in range(nch)])
    full = ch.run_host(ts, nch, nframes)
    lo, hi = shard.ts_slice_for_frames(ch, 1, 2)
    assert lo == ch.ts_bytes(0, 1) - 187 and hi == n_all
    part = ch.run_host(np.ascontiguousarray(ts[:, lo:hi]), nch, 2, first_frame=1)
    assert np.array_equal(part.view(np.uint32), full[:, S:].view(np.uint32))
    with pytest.raises(ValueError):
        ch.run_host(np.ascontiguousarray(ts[:, lo + 187:hi]), nch, 2, first_frame=1)      # history missing
    # and the reference agrees on the frames of channel 1
    rc = reflib.Chain(cfg)
    for fr in range(nframes):
        want = rc.run_frame(np.concatenate([ts[1], np.zeros(512, np.uint8)]))["samples"]
        assert mer_db(full[1, fr * S:(fr + 1) * S], want) >= MER_MIN_DB


def test_chain_generic_work_streams():
    """dvbt2ll_work on a chain handle streams: packet phase, CRC history, in-band phase and L1 FRAME_IDX carry over."""
    cfg = K.resolve(dict(K.CONFIGS["c1"], inband=1, version=2, fecblocks=7))
    ch = T.Chain(cfg, max_frames=4)
    S = ch.samples_per_frame
    n_all = ch.ts_bytes(0, 4)
    ts = K.make_ts(n_all + 64, seed=9)
    want = ch.run_host(ts[:n_all], 1, 4)[0]
    pos = 0
    got = []
    for n in (1, 2, 1):
        out, used = ch.work(ts[pos:], n)
        assert out.size == n * S
        got.append(out)
        pos += used
    assert pos == n_all
    assert np.array_equal(np.concatenate(got).view(np.uint32), want.view(np.uint32))


def test_overfull_frame_warn_policy(compiled_ref):
    """An over-full T2 frame: refused by default, reproduced like the reference (warn, truncate) with the opt-in policy."""
    cfg = K.resolve(dict(K.CONFIGS["c1"], fecblocks=9))
    T.set_overfull_policy(False)
    with pytest.raises(ValueError):
        T.framemapperfint_cc(*fm_args(cfg))
    T.set_overfull_policy(True)
    try:
        fm = T.framemapperfint_cc(*fm_args(cfg))
        assert fm.warnings == 1
        rf = compiled_ref.framemapper(*fm_args(cfg))
        assert rf.warnings == 1
        assert fm.output_multiple == rf.output_multiple
        # (the reference's forecast() asks for 0 items here: its divisor is the grown private frame length; the
        # drop-in keeps asking for what general_work really reads, stream_items)
        n_in = fm.forecast(fm.output_multiple)
        assert n_in == cfg["fecblocks"] * 2025 and rf.forecast(rf.output_multiple) == 0
        rng = np.random.default_rng(5)
        x = (rng.standard_normal(2 * n_in) + 1j * rng.standard_normal(2 * n_in)).astype(np.complex64)
        for fr in range(2):           # both L1-post variants
            a, ua = fm.work(x[fr * n_in:(fr + 1) * n_in], 1)
            b, ub = rf.work(x[fr * n_in:(fr + 1) * n_in], 1)
            assert ua == ub
            assert cells_equal(a, b)
        # the fused chain follows the same rule
        ch = T.Chain(cfg, max_frames=2)
        assert ch.warnings == 1
        ts = K.make_ts(ch.ts_bytes(0, 2) + 512, seed=3)
        out = ch.run_host(ts[:ch.ts_bytes(0, 2)], 1, 2)[0]
        rc = compiled_ref.Chain(cfg)
        S = ch.samples_per_frame
        for fr in range(2):
            want = rc.run_frame(ts)["samples"]
            assert mer_db(out[fr * S:(fr + 1) * S], want) >= MER_MIN_DB
    finally:
        T.set_overfull_policy(False)


def test_dropin_host_register_and_link(reflib):
    """The per-block path with long-lived buffers: registered on first sight, and with the device-resident hand-off
    between adjacent handles -- same items as the reference either way."""
    cfg = K.resolve("c1")
    F = cfg["fecblocks"]
    ts = K.make_ts(3 * F * 2000, seed=21)
    rc = reflib.Chain(cfg)
    refs = [rc.run_frame(ts) for _ in range(2)]
    for link in (False, True):
        B = T.blocks_for(cfg)
        order = [B["bb"], B["ldpc"], B["im"], B["fm"], B["pg"]]
        for blk in order:
            blk.set_host_register(True)
        if link:
            for i in range(4):
                order[i].link_to(order[i + 1])
        nfr = [F, F, F, 1, 1]
        bufs = [np.empty(n * blk.output_multiple, dtype=blk.out_dtype) for blk, n in zip(order, nfr)]
        need = B["bb"].forecast(F * B["bb"].output_multiple) + 400
        ts_buf = np.empty(need, np.uint8)
        pos = 0
        for fr in range(2):
            ts_buf[:] = ts[pos:pos + need]
            _, used = order[0].work_into(ts_buf, bufs[0], nfr[0])
            pos += used
            for i in range(1, 5):
                order[i].work_into(bufs[i - 1], bufs[i], nfr[i])
            r = refs[fr]
            assert used == r["ts_used"]
            assert bits_equal(bufs[0], r["bch"]) and bits_equal(bufs[1], r["fec"])
            assert cells_equal(bufs[2], r["cells"]) and cells_equal(bufs[3], r["mapped"])
            assert mer_db(bufs[4], r["samples"]) >= MER_MIN_DB
        hits = sum(blk.link_hits for blk in order[1:])
        assert hits == (8 if link else 0)
        del order, B          # handles (and their registrations) go before the buffers
        del bufs, ts_buf


def test_dropin_link_lazy_host(reflib):
    """dvbt2ll_link_lazy_host: intermediate host buffers are not written while the linked consumer takes every item
    from HBM (the last block's output is still exact); what the consumer does not take is written late -- when the
    producer reuses the slot, or at once when the consumer asks for an overlapping range that is not resident."""
    cfg = K.resolve("c1")
    F = cfg["fecblocks"]
    ts = K.make_ts(9 * F * 2000, seed=22)
    rc = reflib.Chain(cfg)
    refs = [rc.run_frame(ts) for _ in range(7)]
    B = T.blocks_for(cfg)
    order = [B["bb"], B["ldpc"], B["im"], B["fm"], B["pg"]]
    bb, ldpc = order[0], order[1]
    for i in range(4):
        order[i].link_to(order[i + 1], lazy_host=True)
    nfr = [F, F, F, 1, 1]
    bufs = [np.empty(n * blk.output_multiple, dtype=blk.out_dtype) for blk, n in zip(order, nfr)]
    need = bb.forecast(F * bb.output_multiple) + 400
    nbch, nldpc = bb.output_multiple, ldpc.output_multiple
    pos = 0
    # A. every hand-off hits: the intermediate host buffers keep their sentinel, the baseband is exact
    for b in bufs[:4]:
        b.view(np.uint8)[:] = 0xA5
    _, used = bb.work_into(ts[pos:pos + need].copy(), bufs[0], F)
    pos += used
    for i in range(1, 5):
        order[i].work_into(bufs[i - 1], bufs[i], nfr[i])
    assert mer_db(bufs[4], refs[0]["samples"]) >= MER_MIN_DB
    assert all((b.view(np.uint8) == 0xA5).all() for b in bufs[:4])
    assert sum(blk.link_hits for blk in order[1:]) == 4 and sum(blk.link_late_writes for blk in order[:4]) == 0
    # B. (a fresh BB -> LDPC pair with only that edge lazy, so the LDPC block's own output goes to the host)
    #    The producer keeps its last four outputs resident (a thread-per-block scheduler lets it run ahead); items the
    #    consumer did not take are written to their host buffer when their slot is reused, four calls later.
    del order, bb, ldpc
    B2 = T.blocks_for(cfg)
    bb, ldpc = B2["bb"], B2["ldpc"]
    bb.link_to(ldpc, lazy_host=True)
    outs = [np.full(F * nbch, 0xA5, np.uint8) for _ in range(6)]       # stay alive: lazy slots are written to them later
    pos = 0
    for k in range(2):
        _, used = bb.work_into(ts[pos:pos + need].copy(), outs[k], F)
        pos += used
    assert all((o == 0xA5).all() for o in outs) and bb.link_late_writes == 0
    # the consumer takes frame 0 in full (one frame behind the producer: found in the ring) and half of frame 1
    fec0 = np.empty(F * nldpc, np.uint8)
    ldpc.work_into(outs[0], fec0, F)
    half = np.empty((F // 2) * nldpc, np.uint8)
    ldpc.work_into(outs[1][:(F // 2) * nbch], half, F // 2)
    assert ldpc.link_hits == 2 and bits_equal(fec0, refs[0]["fec"]) and bits_equal(half, refs[1]["fec"][:half.size])
    assert all((o == 0xA5).all() for o in outs) and bb.link_late_writes == 0
    for k in range(2, 6):          # calls 5 and 6 reuse the slots of frames 0 (taken in full: nothing to write) and 1
        _, used = bb.work_into(ts[pos:pos + need].copy(), outs[k], F)
        pos += used
    assert bb.link_late_writes == 1 and (outs[0] == 0xA5).all() and bits_equal(outs[1], refs[1]["bch"])
    assert all((o == 0xA5).all() for o in outs[2:])
    # C. the consumer asks for a range that overlaps a resident output without lying inside it (one FECFRAME further
    #    on): not resident, so that output is written back at once and the items come from the host as usual
    big = np.full((F + 1) * nbch + 4096, 0xA5, np.uint8)
    rec = big[128:128 + F * nbch]
    _, used = bb.work_into(ts[pos:pos + need].copy(), rec, F)          # frame 6
    assert (big == 0xA5).all()
    big[128 + F * nbch:128 + (F + 1) * nbch] = refs[6]["bch"][:nbch]
    out = np.empty(F * nldpc, np.uint8)
    late = bb.link_late_writes
    ldpc.work_into(big[128 + nbch:128 + (F + 1) * nbch], out, F)
    assert bb.link_late_writes == late + 1 and bits_equal(rec, refs[6]["bch"])
    assert bits_equal(out[:(F - 1) * nldpc], refs[6]["fec"][nldpc:]) and bits_equal(out[(F - 1) * nldpc:], refs[6]["fec"][:nldpc])
    del B, B2, bb, ldpc


def test_dropin_auto_link(reflib):
    """dvbt2ll_set_auto_link: no link() calls; every block finds its input among the other blocks' resident outputs by
    host address (the producer may be a frame ahead), the items are the reference's."""
    cfg = K.resolve("c1")
    F = cfg["fecblocks"]
    ts = K.make_ts(4 * F * 2000, seed=23)
    rc = reflib.Chain(cfg)
    refs = [rc.run_frame(ts) for _ in range(3)]
    T.set_auto_link(True)
    try:
        B = T.blocks_for(cfg)
        order = [B["bb"], B["ldpc"], B["im"], B["fm"], B["pg"]]
        nfr = [F, F, F, 1, 1]
        # two host slots per edge: the BB block runs one frame ahead of the rest
        bufs = [[np.empty(n * blk.output_multiple, dtype=blk.out_dtype) for _ in range(2)] for blk, n in zip(order, nfr)]
        need = B["bb"].forecast(F * B["bb"].output_multiple) + 400
        pos = 0
        _, used = order[0].work_into(ts[pos:pos + need].copy(), bufs[0][0], F)
        pos += used
        for fr in range(3):
            if fr + 1 < 3:
                _, used = order[0].work_into(ts[pos:pos + need].copy(), bufs[0][(fr + 1) % 2], F)
                pos += used
            for i in range(1, 5):
                order[i].work_into(bufs[i - 1][fr % 2], bufs[i][fr % 2], nfr[i])
            r = refs[fr]
            assert bits_equal(bufs[0][fr % 2], r["bch"]) and bits_equal(bufs[1][fr % 2], r["fec"])
            assert cells_equal(bufs[2][fr % 2], r["cells"]) and cells_equal(bufs[3][fr % 2], r["mapped"])
            assert mer_db(bufs[4][fr % 2], r["samples"]) >= MER_MIN_DB
        assert [blk.link_hits for blk in order] == [0, 3, 3, 3, 3]
        del order, B
    finally:
        T.set_auto_link(False)


def _run_gather(devices, cfg_name="c1", nch_total=5, nfr=2, steps=5, sink=0):
    """`len(devices)` ranks in ONE process (rank r on devices[r]): every step each rank runs its channels and the
    parts are reassembled in order on rank 0's device. Returns (list of per-step slots as host arrays, expected)."""
    cfg = K.resolve(cfg_name)
    world = len(devices)
    counts = [len(shard.channels_for_rank(nch_total, world, r)) for r in range(world)]
    chains, ts_dev, gs, streams = [], [], [], []
    ssz = 4 if sink else 8
    one = T.Chain(cfg, max_frames=1)
    S, n_ts = one.samples_per_frame, one.ts_bytes_per_frame
    offs, sizes, slot_bytes = shard.slot_layout(counts, nfr * S * ssz)
    ts_all = np.stack([K.make_ts(nfr * n_ts, seed=K.TS_SEED + c) for c in range(nch_total)])
    for r in range(world):
        T.set_device(devices[r])
        ch = T.Chain(cfg, max_frames=max(1, counts[r] * nfr), device=devices[r])
        if sink:
            ch.set_sink(1, 0.2)
        chains.append(ch)
        mine = shard.channels_for_rank(nch_total, world, r)
        ts_dev.append(T.DeviceBuffer(max(16, len(mine) * nfr * n_ts), data=ts_all[mine] if mine else None))
        gs.append(T.Gather(r, world, 0, devices[r], slot_bytes, max(16, sizes[r]), n_slots=2))
        streams.append(T.stream_create())
    blobs = [g.export() for g in gs]
    for g in gs:
        g.connect(blobs)
    T.set_device(devices[0])
    consumer = T.stream_create()
    slots = []
    for k in range(steps):
        for r in range(world):
            T.set_device(devices[r])
            p = gs[r].acquire(k, offs[r], streams[r])
            if counts[r]:
                chains[r].run_device(ts_dev[r].ptr, nfr * n_ts, counts[r], nfr, 0, p, streams[r])
            gs[r].push(k, offs[r], sizes[r], streams[r])
        T.set_device(devices[0])
        slot = gs[0].wait(k, consumer)
        assert T.lib().dvbt2ll_stream_synchronize(consumer) == 0, T.last_error()
        host = np.empty(slot_bytes // ssz, dtype=np.complex64 if not sink else np.int32)
        T.copy_to_host(host, slot)
        slots.append(host)
        gs[0].release(k, consumer)
    for r in range(world):
        T.set_device(devices[r])
        T.device_synchronize()
    for g in gs[1:] + gs[:1]:
        g.close()
    for r in range(world):
        T.set_device(devices[r])
        T.stream_destroy(streams[r])
    T.set_device(devices[0])
    T.stream_destroy(consumer)
    T.set_device(devices[0])
    ref_chain = T.Chain(cfg, max_frames=nch_total * nfr, device=devices[0])
    if sink:
        ref_chain.set_sink(1, 0.2)
    want = ref_chain.run_host(ts_all, nch_total, nfr)
    want = want.reshape(-1) if not sink else np.ascontiguousarray(want).view(np.int32).reshape(-1)
    return slots, want


@pytest.mark.parametrize("sink", [0, 1])
def test_gather_two_ranks_one_device(sink):
    """The ordered reassembly (dvbt2ll_gather_*) with two ranks on ONE device: ring reuse over five steps with two
    slots exercises arrival counters, slot release and back-pressure; the slot equals the single-launch output."""
    slots, want = _run_gather([0, 0], sink=sink)
    for k, s in enumerate(slots):
        assert np.array_equal(s.view(np.uint32), want.view(np.uint32)), "step %d" % k


def test_gather_three_ranks_ragged_one_device():
    slots, want = _run_gather([0, 0, 0], nch_total=4, nfr=1, steps=4)      # parts of 2, 1, 1 channels
    for s in slots:
        assert np.array_equal(s.view(np.uint32), want.view(np.uint32))


@pytest.mark.skipif(T.device_count() < 2, reason="needs two GPUs")
def test_two_devices_in_one_process(reflib):
    """Chains on device 0 AND device 1 of one process (function attributes and the SM count are per device), then the
    reassembly across the two devices over NVLink peer access."""
    cfg = K.resolve("c3")
    outs = []
    ts = K.make_ts(T.Chain(cfg, max_frames=1).ts_bytes_per_frame, seed=K.TS_SEED + 2)
    for d in (0, 1):
        ch = T.Chain(cfg, max_frames=1, device=d)
        outs.append(ch.run_host(ts, 1, 1)[0])
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
    want = reflib.Chain(cfg).run_frame(np.concatenate([ts, np.zeros(1024, np.uint8)]))["samples"]
    assert mer_db(outs[1], want) >= MER_MIN_DB
    slots, want = _run_gather([0, 1], cfg_name="c4", nch_total=4, nfr=1, steps=5)
    for s in slots:
        assert np.array_equal(s.view(np.uint32), want.view(np.uint32))


def test_ldpc_both_accumulation_schemes(monkeypatch):
    """k_ldpc picks a lane per (row, word) or a lane per row by code; both must give the oracle's codewords."""
    from oracle import t2oracle as O
    rng = np.random.default_rng(12)
    for fs, rate in ((1, K.C1_2), (1, K.C2_3), (0, K.C1_3), (0, K.C4_5)):
        p = O.fec_params(fs, rate)
        info = rng.integers(0, 2, 3 * p["nbch"], dtype=np.uint8)
        want = O.ldpc_encode(info.reshape(3, p["nbch"]), fs, rate).reshape(-1)
        for mode in ("0", "1"):
            monkeypatch.setenv("DVBT2LL_LDPC_MODE", mode)
            fec, _ = T.ldpc_bb(fs, rate).work(info, 3)
            assert bits_equal(fec, want), (fs, rate, mode)


@pytest.mark.parametrize("name", ["c1", "c3"])
def test_dropin_blocks_device_resident_any_alignment(name):
    """dvbt2ll_work_device on the four blocks behind the BB stage, items resident in HBM: the vectorised kernels (8-byte
    bit-format conversions, 16-byte cell stores, paired frame-mapper gathers) taken with aligned buffers and the scalar
    ones taken with byte- / cell-misaligned buffers both reproduce the host-buffer path (which the other tests tie to the
    reference) bit for bit."""
    cfg = K.resolve(name)
    b = T.blocks_for(cfg)
    F = cfg["fecblocks"]
    nfr = 2
    rng = np.random.default_rng(5)
    nbch = b["bb"].output_multiple
    bits = rng.integers(0, 2, size=nfr * F * nbch, dtype=np.uint8)
    # host path = the checker here (itself bit-exact against the reference in test_blocks_match_reference)
    fec, _ = b["ldpc"].work(bits, nfr * F)
    cells, _ = b["im"].work(fec, nfr * F)
    mapped, _ = b["fm"].work(cells.view(np.complex64), nfr)
    stages = (("ldpc", bits, fec, 1, 1, nfr * F), ("im", fec, cells.view(np.complex64), 1, 8, nfr * F),
              ("fm", cells.view(np.complex64), mapped.view(np.complex64), 8, 8, nfr))
    for k, x, want, isz, osz, n in stages:
        blk = T.blocks_for(cfg)[k]          # fresh block: the frame mapper carries its T2 frame counter
        for in_ofs, out_ofs in ((0, 0), (isz, osz), (0, osz), (isz, 0)):
            if in_ofs or out_ofs:
                blk = T.blocks_for(cfg)[k]
            raw = np.ascontiguousarray(x).view(np.uint8)
            d_in = T.DeviceBuffer(raw.size + 64, data=np.concatenate([np.zeros(in_ofs, np.uint8), raw]))
            nout = n * blk.output_multiple
            d_out = T.DeviceBuffer(nout * osz + 64)
            r, used = blk.work_device(d_in.ptr + in_ofs, raw.size // isz, d_out.ptr + out_ofs, nout, None)
            assert r == nout and used == raw.size // isz
            got = np.empty(nout * osz + 64, np.uint8)
            T.copy_to_host(got, d_out.ptr)
            got = got[out_ofs:out_ofs + nout * osz]
            assert np.array_equal(got, np.ascontiguousarray(want).view(np.uint8)[:nout * osz]), (k, in_ofs, out_ofs)
            d_in.free(); d_out.free()
