"""CPU: G.711 mu-law / A-law input (CVAD_PCM_ULAW / CVAD_PCM_ALAW) in everything that runs without a GPU -- the decode rule
against the standard and audioop, the native feeder's framing, payloads and row snapshots on 1-byte samples, and the
Python plumbing.  The GPU decode stage is covered by tests/test_gpu_g711.py."""
import re
import struct
import warnings

import numpy as np
import pytest

from conftest import ROOT, synth_streams


def _feeder(**kw):
    from real_time_vad.engine.feeder import StreamFeeder
    return StreamFeeder(None, **kw)


def _g711_standard(law):
    """G.711's expansion tables restated from the segment / step description of the standard, scaled to 16 bits.
    mu-law: the code is sent inverted; segment e (bits 4-6), step m (bits 0-3), sign bit 7 set = negative; magnitude in
    14-bit units (2m + 33) 2^e - 33.  A-law: the even bits are sent inverted (XOR 0x55); sign bit 7 set = positive;
    magnitude in 13-bit units 2m + 1 in segment 0, (2m + 33) 2^(e - 1) in segment e >= 1."""
    out = np.zeros(256, np.int64)
    for code in range(256):
        if law == "ulaw":
            c = code ^ 0xFF
            e, m, neg = (c >> 4) & 7, c & 15, bool(c & 0x80)
            mag = 4 * ((2 * m + 33) * 2 ** e - 33)
        else:
            c = code ^ 0x55
            e, m, neg = (c >> 4) & 7, c & 15, not (c & 0x80)
            mag = 8 * ((2 * m + 1) if e == 0 else (2 * m + 33) * 2 ** (e - 1))
        out[code] = -mag if neg else mag
    return out


@pytest.mark.parametrize("law", ["ulaw", "alaw"])
def test_decode_tables_follow_the_standard_and_audioop(law):
    from real_time_vad.utils.audio import G711_LINEAR, AudioUtils
    want = _g711_standard(law)
    assert np.array_equal(G711_LINEAR[law].astype(np.int64), want)
    span = {"ulaw": 32124, "alaw": 32256}[law]
    assert want.min() == -span and want.max() == span
    if law == "ulaw":
        assert want[0x7F] == 0 and want[0xFF] == 0
    codes = np.arange(256, dtype=np.uint8)
    x = AudioUtils.g711_to_float32(codes, law)
    assert x.dtype == np.float32
    assert np.array_equal(x, AudioUtils.pcm_to_float32(want.astype(np.int16).tobytes()))
    assert np.array_equal(x, AudioUtils.g711_to_float32(codes.tobytes(), law))
    with pytest.raises(Exception, match="uint8"):
        AudioUtils.g711_to_float32(codes.astype(np.int16), law)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        try:
            import audioop
        except ImportError:
            return
    lin = audioop.ulaw2lin(bytes(range(256)), 2) if law == "ulaw" else audioop.alaw2lin(bytes(range(256)), 2)
    assert np.array_equal(np.frombuffer(lin, "<i2").astype(np.int64), want)


def test_header_constants_equal_capi():
    from real_time_vad.engine import capi
    h = (ROOT / "include" / "cutter_vad_b200.h").read_text()
    consts = dict(re.findall(r"#define (CVAD_PCM_\w+) (\d+)", h))
    assert int(consts["CVAD_PCM_ULAW"]) == capi.PCM_ULAW == 3
    assert int(consts["CVAD_PCM_ALAW"]) == capi.PCM_ALAW == 4
    assert capi.pcm_dtype(capi.PCM_ULAW) == capi.pcm_dtype(capi.PCM_ALAW) == np.uint8
    assert capi.pcm_dtype(capi.PCM_F32) == np.float32 and capi.pcm_dtype(capi.PCM_S16_32768) == np.int16


def _codes(n, L, seed):
    return np.random.default_rng(seed).integers(0, 256, (n, L), dtype=np.uint8)


@pytest.mark.parametrize("pcm_format", [3, 4])
@pytest.mark.parametrize("src_rate,frame_len,hop,push", [(8000, 256, 256, "160"), (16000, 480, 480, "random"),
                                                         (16000, 512, 256, "random"), (0, 0, 0, "random")])
def test_gather_frames_equal_split_into_frames_of_the_byte_stream(pcm_format, src_rate, frame_len, hop, push):
    """Whatever the push sizes (160-byte telephony packets or random), the frames stepped for a stream are
    split_into_frames of its byte stream, and the gathered rows stay 16-byte aligned."""
    from vad_oracle import split_into_frames
    rates = [8000, 16000, 24000, 48000, 8000, 16000, 8000]
    n, L = len(rates), 12000
    wire = _codes(n, L, seed=pcm_format)
    f = _feeder(max_streams=16, pcm_format=pcm_format, frame_len=frame_len or 512, hop=hop or 512,
                src_rate=src_rate, capacity_frames=4)
    slots = [1, 2, 4, 7, 9, 12, 15]
    for k, s in enumerate(slots):
        f.open(s, src_rate=rates[k] if src_rate == 0 else 0)
    flen = {s: (rates[k] * 512 // 16000 if src_rate == 0 else frame_len) for k, s in enumerate(slots)}
    fhop = {s: (flen[s] if src_rate == 0 else hop) for s in slots}
    rng = np.random.default_rng(2)
    pos = np.zeros(n, int)
    got = {s: [] for s in slots}
    for _ in range(2000):
        for k, s in enumerate(slots):
            if pos[k] < L:
                m = 160 if push == "160" else int(rng.integers(1, 1400))
                chunk = np.ascontiguousarray(wire[k, pos[k]:pos[k] + m])
                if k % 2:
                    f.push_bytes(s, chunk.tobytes())
                else:
                    f.push(s, chunk)
                pos[k] += m
        r = f.gather_only()
        assert r.raw_stride % 16 == 0
        if r.raw is not None:
            assert r.raw.dtype == np.uint8
        for row, (s, c) in enumerate(zip(r.slots, r.counts)):
            s = int(s)
            for j in range(c):
                got[s].append(r.raw[row, j * fhop[s]:j * fhop[s] + flen[s]].copy())
        if (pos >= L).all() and r.slots.size == 0:
            break
    for k, s in enumerate(slots):
        want = split_into_frames(wire[k], flen[s], fhop[s])
        assert len(got[s]) == len(want) and np.array_equal(np.stack(got[s]), want), s
    f.close()


def _deliver_pair(pcm_format, payload, denoise, frame_len, hop, seed, n=6, T=100):
    """The same scripted probabilities / flags through a G.711 feeder and a PCM_F32 feeder fed the decoded audio."""
    from real_time_vad.engine import capi
    from real_time_vad.utils.audio import G711_LINEAR, AudioUtils
    from vad_oracle import StateMachine
    law = "ulaw" if pcm_format == capi.PCM_ULAW else "alaw"
    rng = np.random.default_rng(seed)
    L = (T - 1) * hop + frame_len
    audio = synth_streams(n, L, seed=seed)
    # codes of real audio (so that the gate sees samples on both sides of 0.01), plus random codes in one stream
    lin = np.clip(np.round(audio * 32767.0), -32768, 32767).astype(np.int16)
    order = np.argsort(G711_LINEAR[law])
    sorted_lin = G711_LINEAR[law][order]
    idx = np.clip(np.searchsorted(sorted_lin, lin), 0, 255)
    wire = order[idx].astype(np.uint8)
    wire[1] = _codes(1, L, seed)[0]
    decoded = AudioUtils.g711_to_float32(wire, law).reshape(n, L)
    probs = np.clip(0.5 + 0.5 * np.sin(np.arange(T)[None, :] / rng.uniform(3, 9, (n, 1)) + rng.uniform(0, 6, (n, 1)))
                    + 0.15 * rng.standard_normal((n, T)), 0, 1).astype(np.float32)
    fg = _feeder(max_streams=8, pcm_format=pcm_format, frame_len=frame_len, hop=hop, capacity_frames=5)
    ff = _feeder(max_streams=8, pcm_format=capi.PCM_F32, frame_len=frame_len, hop=hop, capacity_frames=5)
    sms = [StateMachine(0.5, 0.35, 0.8, 0.95, 2 + s % 2, 3 + s % 3) for s in range(n)]
    for f in (fg, ff):
        for s in range(n):
            f.open(s, payload=payload, vad_start_probability=0.5, enable_denoising=denoise)
    done = np.zeros(n, int)
    pos = np.zeros(n, int)
    n_seg = n_cont = 0
    while (done < T).any():
        for s in range(n):
            m = int(rng.integers(150, 2600))
            if pos[s] < L:
                fg.push(s, np.ascontiguousarray(wire[s, pos[s]:pos[s] + m]))
                ff.push(s, np.ascontiguousarray(decoded[s, pos[s]:pos[s] + m]))
            pos[s] += m
        gg, gf = fg.gather_only(), ff.gather_only()
        assert np.array_equal(gg.slots, gf.slots) and np.array_equal(gg.counts, gf.counts)
        if gg.slots.size == 0:
            continue
        Tm = int(gg.counts.max())
        p = np.zeros((gg.slots.size, Tm), np.float32)
        fl = np.zeros((gg.slots.size, Tm), np.uint8)
        for row, (s, c) in enumerate(zip(gg.slots, gg.counts)):
            for j in range(c):
                p[row, j] = probs[s, done[s] + j]
                fl[row, j] = sms[s].step(float(p[row, j]))
            done[s] += c
        rg, rf = fg.deliver_only(p, fl), ff.deliver_only(p, fl)
        assert len(rg.deliveries) == len(rf.deliveries)
        for a, b in zip(rg.deliveries, rf.deliveries):
            assert (a.slot, a.stream, a.step_frame, a.flags, a.prob) == (b.slot, b.stream, b.step_frame, b.flags, b.prob)
            for x, y in ((a.frame, b.frame), (a.segment, b.segment)):
                assert (x is None) == (y is None)
                if x is not None:
                    assert x.dtype == np.float32 and x.tobytes() == y.tobytes()
            n_seg += a.segment is not None and a.segment.size > 0
            n_cont += a.frame is not None
        for s in range(n):
            assert fg.is_active(s) == ff.is_active(s)
    fg.close()
    ff.close()
    return n_seg, n_cont


@pytest.mark.parametrize("pcm_format", [3, 4])
@pytest.mark.parametrize("payload,denoise,frame_len,hop", [(3, True, 480, 480), (3, False, 512, 512), (2, True, 512, 256),
                                                           (1, True, 512, 512)])
def test_deliver_equals_a_float32_feeder_fed_the_decoded_audio(pcm_format, payload, denoise, frame_len, hop):
    n_seg, n_cont = _deliver_pair(pcm_format, payload, denoise, frame_len, hop, seed=31 + payload)
    assert (n_seg >= 4) == (payload >= 2)
    assert (n_cont > 50) == (payload == 3)


def test_rows_move_between_g711_feeders_and_other_formats_are_refused():
    from real_time_vad.engine import capi
    from real_time_vad.engine.feeder import FeederError, set_row_payloads
    wire = _codes(3, 5000, seed=4)
    a = _feeder(max_streams=8, pcm_format=capi.PCM_ULAW, frame_len=480, hop=480)
    for s in (1, 3, 5):
        a.open(s, payload=capi.PAYLOAD_FRAMES, vad_start_probability=0.5)
    for k, s in enumerate((1, 3, 5)):
        a.push(s, np.ascontiguousarray(wire[k, :1000 + 333 * k]))
    g = a.gather_only()
    p = np.full((g.slots.size, int(g.counts.max())), 0.9, np.float32)
    fl = np.zeros_like(p, dtype=np.uint8)
    a.deliver_only(p, fl)                                  # above-threshold frames: every stream holds a pre-roll
    blob = a.export_rows([1, 3, 5])
    hd = struct.unpack_from("<IIiiiiii", blob, 0)
    assert hd[2] == capi.PCM_ULAW
    pend = [a.pending(s) for s in (1, 3, 5)]
    assert pend == [(1000 + 333 * k) % 480 for k in range(3)]
    n_pre = [struct.unpack_from("<qqq", blob, pos + 40)[1] for pos in _row_offsets(blob, 1)]
    assert all(x > 0 for x in n_pre)
    # set_row_payloads walks the 1-byte rows: lowering the payload mode of the last row only rewrites that field
    low = set_row_payloads(blob, [capi.PAYLOAD_FRAMES, capi.PAYLOAD_FRAMES, capi.PAYLOAD_NONE])
    assert len(low) == len(blob)
    offs = _row_offsets(blob, 1)
    assert struct.unpack_from("<i", low, offs[2] + 8)[0] == capi.PAYLOAD_NONE
    assert struct.unpack_from("<i", low, offs[1] + 8)[0] == capi.PAYLOAD_FRAMES
    b = _feeder(max_streams=8, pcm_format=capi.PCM_ULAW, frame_len=480, hop=480)
    b.import_rows([0, 2, 6], blob)
    assert [b.pending(s) for s in (0, 2, 6)] == pend
    assert b.export_rows([0, 2, 6]) == blob
    for k, (s, t) in enumerate(zip((1, 3, 5), (0, 2, 6))):
        tail = np.ascontiguousarray(wire[k, 1000 + 333 * k:1000 + 333 * k + 480])
        a.push(s, tail)
        b.push(t, tail)
    ra, rb = a.gather_only(), b.gather_only()
    assert np.array_equal(ra.counts, rb.counts) and np.array_equal(ra.raw, rb.raw)
    for other in (capi.PCM_S16_32768, capi.PCM_ALAW, capi.PCM_F32):
        c = _feeder(max_streams=8, pcm_format=other, frame_len=480, hop=480)
        with pytest.raises(FeederError, match="PCM format"):
            c.import_rows([0, 2, 6], blob)
        assert c.pending(0) == 0
        c.close()
    with pytest.raises(FeederError):
        _feeder(max_streams=4, pcm_format=5)
    with pytest.raises(FeederError):
        _feeder(max_streams=4, pcm_format=-1)
    a.close()
    b.close()


def _row_offsets(blob, es):
    n = struct.unpack_from("<i", blob, 24)[0]
    pos, out = 32, []
    for _ in range(n):
        out.append(pos)
        n_pending, n_pre, n_seg = struct.unpack_from("<qqq", blob, pos + 40)
        pos += 64 + n_pending * es + (n_pre + n_seg) * 4
    assert pos == len(blob)
    return out


def test_sharded_manager_forwards_pcm_format():
    from real_time_vad.core.sharded_manager import ShardedVADManager
    from real_time_vad.engine import capi
    seen = {}

    def factory(**kw):
        seen.update(kw)
        return object()

    ShardedVADManager(16, rank=0, world_size=2, manager_factory=factory, pcm_format=capi.PCM_ALAW, source_rate=8000)
    assert seen["pcm_format"] == capi.PCM_ALAW and seen["source_rate"] == 8000
