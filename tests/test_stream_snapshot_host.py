"""CPU: the host side of stream snapshots -- the cvad_stream_state record layout, feeder row export / import between
feeders built without an engine (carried samples, skipped samples, pre-roll and segment, mixed rates, refused blobs) and
the StreamSnapshot container."""
import subprocess

import numpy as np
import pytest

from conftest import ROOT, synth_streams

HEADER = ROOT / "include" / "cutter_vad_b200.h"


def _feeder(**kw):
    from real_time_vad.engine.feeder import StreamFeeder
    return StreamFeeder(None, **kw)


def test_stream_state_record_matches_state_dtype(tmp_path):
    from real_time_vad.engine import capi
    fields = ["h", "c", "frames_done", "vad_start_probability", "vad_end_probability", "is_voice_active",
              "voice_start_frame_count", "voice_end_frame_count", "n_start", "n_end", "enable_denoising"]
    src = tmp_path / "state_layout.c"
    src.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "{HEADER}"\n'
                   'int main(){printf("%zu", sizeof(cvad_stream_state));' +
                   "".join(f'printf(" %zu", offsetof(cvad_stream_state, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / "state_layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    dt = capi.STATE_DTYPE
    assert got == [1072] + [dt.fields[f][1] for f in fields]
    assert dt.itemsize == 1072 and list(dt.names) == fields


def _gather_rows(f, want_slots):
    """One gather_only: {slot: [frames as arrays]} for the slots of interest."""
    r = f.gather_only()
    out = {}
    for row, (s, c) in enumerate(zip(r.slots, r.counts)):
        out[int(s)] = (int(c), r.raw[row].copy())
    return {s: out.get(s) for s in want_slots}, r


def _continue_equal(a, b, slot_map, audio, pos, frame_len, hop, rounds=12, seed=5):
    """Push identical pieces into both feeders and compare every gathered row (A's slot -> B's slot)."""
    rng = np.random.default_rng(seed)
    for _ in range(rounds):
        for k, (sa, sb) in enumerate(slot_map.items()):
            m = int(rng.integers(50, 1500))
            piece = np.ascontiguousarray(audio[k, pos[k]:pos[k] + m])
            pos[k] += m
            if piece.size:
                a.push(sa, piece)
                b.push(sb, piece)
        ga, _ = _gather_rows(a, list(slot_map))
        gb, _ = _gather_rows(b, list(slot_map.values()))
        for sa, sb in slot_map.items():
            if ga[sa] is None or gb[sb] is None:
                assert ga[sa] is None and gb[sb] is None, (sa, sb)
                continue
            ca, ra = ga[sa]
            cb, rb = gb[sb]
            assert ca == cb
            need = (ca - 1) * hop + frame_len
            assert np.array_equal(ra[:need], rb[:need])
        for sa, sb in slot_map.items():
            assert a.pending(sa) == b.pending(sb)


@pytest.mark.parametrize("frame_len,hop,pcm", [(512, 512, 0), (512, 256, 1), (400, 640, 2), (480, 480, 1)])
def test_rows_carry_pending_and_skipped_samples(frame_len, hop, pcm):
    """Carried samples (fewer than a frame), and with hop > frame_len the samples between frames that had not arrived
    yet (skp): after export -> import into other slots of another feeder, both frame the same audio identically."""
    n, L = 6, 40000
    audio = synth_streams(n, L, seed=11)
    if pcm:
        audio = np.clip(np.round(audio * 32767.0), -32768, 32767).astype(np.int16)
    kw = dict(pcm_format=pcm, frame_len=frame_len, hop=hop, capacity_frames=4)
    a, b = _feeder(max_streams=16, **kw), _feeder(max_streams=32, **kw)
    src = [1, 2, 4, 7, 9, 15]
    dst = [30, 3, 17, 0, 22, 8]
    for s in src:
        a.open(s)
    rng = np.random.default_rng(2)
    pos = np.zeros(n, int)
    for _ in range(5):
        for k, s in enumerate(src):
            m = int(rng.integers(100, 1700))
            a.push(s, np.ascontiguousarray(audio[k, pos[k]:pos[k] + m]))
            pos[k] += m
        a.gather_only()
    if hop > frame_len:                                  # a row that ran ahead of its samples (skp > 0)
        a.push(src[0], np.ascontiguousarray(audio[0, pos[0]:pos[0] + frame_len]))
        pos[0] += frame_len
        a.gather_only()
    pend = [a.pending(s) for s in src]
    assert any(pend)
    blob = a.export_rows(src)
    b.import_rows(dst, blob)
    assert [b.pending(s) for s in dst] == pend
    _continue_equal(a, b, dict(zip(src, dst)), audio, pos, frame_len, hop)
    a.close()
    b.close()


def test_rows_carry_pre_roll_and_segment():
    """Pre-roll and half-built segment assembled by deliver_only move with the row: scripted probabilities and flags
    delivered to both feeders afterwards produce identical delivery records and payloads."""
    from real_time_vad.engine import capi
    n, T, F = 4, 40, 480
    audio = synth_streams(n, F * T, seed=4)
    a, b = _feeder(max_streams=8, frame_len=F, hop=F), _feeder(max_streams=8, frame_len=F, hop=F)
    for s in range(n):
        a.open(s, payload=capi.PAYLOAD_FRAMES, vad_start_probability=0.5, enable_denoising=s % 2 == 0)
    # per stream, frame t: probability and flags (a start at 6, an end at 30; stream 1 starts late, in pre-roll at the cut)
    probs = np.full((n, T), 0.2, np.float32)
    flags = np.zeros((n, T), np.uint8)
    for s in range(n):
        st = 6 + 8 * (s == 1)
        probs[s, st - 2:30] = 0.9
        flags[s, st] = capi.FLAG_STARTED
        flags[s, st + 1:30] = capi.FLAG_CONTINUING
        flags[s, 30] = capi.FLAG_ENDED
    cut = 13                                             # stream 1: frames 12..13 above threshold, start at 14

    def run(f, ids, t0, t1):
        out = []
        for t in range(t0, t1):
            for s, sid in zip(range(n), ids):
                f.push(sid, np.ascontiguousarray(audio[s, t * F:(t + 1) * F]))
            g = f.gather_only()
            k = {int(x): i for i, x in enumerate(g.slots)}
            p = np.zeros((len(k), 1), np.float32)
            fl = np.zeros((len(k), 1), np.uint8)
            for s, sid in zip(range(n), ids):
                p[k[sid], 0], fl[k[sid], 0] = probs[s, t], flags[s, t]
            r = f.deliver_only(p, fl)
            inv = dict(zip(ids, range(n)))
            out += [(t, inv[d.slot], d.flags, None if d.frame is None else d.frame.tobytes(),
                     None if d.segment is None else d.segment.tobytes()) for d in r.deliveries]
        return sorted(out, key=lambda d: (d[0], d[1]))       # (rows are in slot order, and the slots differ)

    run(a, list(range(n)), 0, cut + 1)
    dst = [5, 2, 7, 0]
    b.import_rows(dst, a.export_rows(list(range(n))))
    assert [b.is_active(s) for s in dst] == [a.is_active(s) for s in range(n)] == [True, False, True, True]
    wa = run(a, list(range(n)), cut + 1, T)
    wb = run(b, dst, cut + 1, T)
    assert wa == wb
    ends = [d for d in wa if d[2] & capi.FLAG_ENDED]
    assert len(ends) == n and all(len(d[4]) == 4 * F * (30 - (6 + 8 * (d[1] == 1)) + 3) for d in ends)
    a.close()
    b.close()


def test_mixed_rate_rows():
    from real_time_vad.engine import capi
    plan = {0: 8000, 3: 16000, 4: 24000, 6: 48000}
    a, b = _feeder(max_streams=8, src_rate=0), _feeder(max_streams=8, src_rate=0)
    x = {}
    for s, r in plan.items():
        a.open(s, src_rate=r, payload=capi.PAYLOAD_SEGMENTS)
        n_in = r * 512 // 16000
        x[s] = (np.arange(n_in * 6 + 33, dtype=np.float32) * 1e-4 + s)
        a.push(s, x[s][:n_in * 2 + 33])
    a.gather_only()
    dst = {0: 7, 3: 1, 4: 2, 6: 5}
    b.import_rows(list(dst.values()), a.export_rows(list(dst)))
    for s, t in dst.items():
        assert b.pending(t) == a.pending(s) == 33
        n_in = plan[s] * 512 // 16000
        a.push(s, x[s][n_in * 2 + 33:])
        b.push(t, x[s][n_in * 2 + 33:])
    ra, rb = a.gather_only(), b.gather_only()
    rows_a = {int(s): (int(c), ra.raw[k]) for k, (s, c) in enumerate(zip(ra.slots, ra.counts))}
    rows_b = {int(s): (int(c), rb.raw[k]) for k, (s, c) in enumerate(zip(rb.slots, rb.counts))}
    for s, t in dst.items():
        n_in = plan[s] * 512 // 16000
        assert rows_a[s][0] == rows_b[t][0] == 4
        assert np.array_equal(rows_a[s][1][:4 * n_in], rows_b[t][1][:4 * n_in])
        assert np.array_equal(rows_a[s][1][:4 * n_in], x[s][n_in * 2:n_in * 6])
    # a fixed-rate feeder does not take mixed rows
    c = _feeder(max_streams=8, src_rate=48000)
    from real_time_vad.engine.feeder import FeederError
    with pytest.raises(FeederError, match="framing"):
        c.import_rows([0, 1, 2, 3], a.export_rows(list(dst)))
    for f in (a, b, c):
        f.close()


def test_refused_blobs_change_no_row():
    from real_time_vad.engine import capi
    from real_time_vad.engine.feeder import FeederError
    a = _feeder(max_streams=8, frame_len=512, hop=256)
    for s in (0, 1):
        a.open(s, payload=capi.PAYLOAD_SEGMENTS)
        a.push(s, np.full(700 + s, 0.1, np.float32))
    blob = a.export_rows([0, 1])
    with pytest.raises(FeederError, match="not open"):
        a.export_rows([0, 2])
    with pytest.raises(FeederError, match="twice"):
        a.export_rows([0, 0])
    t = _feeder(max_streams=8, frame_len=512, hop=256)
    for s in (3, 4):
        t.open(s)
        t.push(s, np.full(100 * s, 0.2, np.float32))

    def refused(target, ids, data, match):
        before = [target.pending(s) for s in ids]
        with pytest.raises(FeederError, match=match) as ei:
            target.import_rows(ids, data)
        assert ei.value.code in (capi.E_INVALID, capi.E_CAPACITY)
        assert [target.pending(s) for s in ids] == before

    bad = bytearray(blob)
    bad[0] ^= 0xFF
    refused(t, [3, 4], bytes(bad), "magic")
    bad = bytearray(blob)
    bad[4] = 2
    refused(t, [3, 4], bytes(bad), "version")
    for cut in (10, 40, 32 + 64 + 10, len(blob) - 1):
        refused(t, [3, 4], blob[:cut], None)
    refused(t, [3, 4], blob + b"\0", "after the last row")
    bad = bytearray(blob)
    bad[32 + 8] = 7                                       # payload mode of row 0
    refused(t, [3, 4], bytes(bad), "payload")
    refused(t, [3], blob, "rows")
    with pytest.raises(FeederError, match="out of range") as ei:
        t.import_rows([3, 9], blob)
    assert ei.value.code == capi.E_CAPACITY and t.pending(3) == 300
    for other in (_feeder(max_streams=8, frame_len=512, hop=512), _feeder(max_streams=8, frame_len=512, hop=256, pcm_format=1)):
        for s in (3, 4):
            other.open(s)
            other.push(s, np.full(10, 1, other.dtype))
        refused(other, [3, 4], blob, "framing|PCM")
        other.close()
    t.import_rows([3, 4], blob)
    assert [t.pending(3), t.pending(4)] == [700, 701]
    a.close()
    t.close()


def _snapshot(n=3):
    from real_time_vad import VADConfig
    from real_time_vad.core.stream_snapshot import SnapshotStream, StreamSnapshot
    from real_time_vad.engine import capi
    rng = np.random.default_rng(0)
    f = _feeder(max_streams=8, frame_len=512, hop=512)
    for s in range(n):
        f.open(s)
        f.push(s, rng.standard_normal(100 + s).astype(np.float32) * 0.1)
    states = np.zeros(n, capi.STATE_DTYPE)
    states["h"] = rng.standard_normal((n, 128))
    states["c"] = rng.standard_normal((n, 128))
    states["frames_done"] = [5, 0, 77]
    states["n_start"], states["n_end"] = 3, 4
    streams = [SnapshotStream(s + 10, VADConfig(vad_start_probability=0.4)._to_serializable_dict(), 2, s == 1,
                              [rng.standard_normal(512).astype(np.float32)] * s, [rng.standard_normal(512).astype(np.float32)])
               for s in range(n)]
    snap = StreamSnapshot("v5", 0x0123456789abcdef, 0, 512, 512, 16000, streams, states, f.export_rows(list(range(n))))
    f.close()
    return snap


def test_stream_snapshot_round_trips_through_bytes():
    from real_time_vad import StreamSnapshot, VADConfig
    snap = _snapshot()
    data = snap.to_bytes()
    back = StreamSnapshot.from_bytes(data)
    assert back.to_bytes() == data
    assert back.fingerprint == snap.fingerprint and back.source_rate == 16000 and back.feeder_rows == snap.feeder_rows
    assert back.states.tobytes() == snap.states.tobytes()
    for x, y in zip(snap.streams, back.streams):
        assert (x.stream_id, x.payload, x.active) == (y.stream_id, y.payload, y.active)
        assert VADConfig.from_dict(dict(y.config)) == VADConfig.from_dict(dict(x.config))
        assert [f.tobytes() for f in x.pre_roll] == [f.tobytes() for f in y.pre_roll]
        assert [f.tobytes() for f in x.segment] == [f.tobytes() for f in y.segment]
    assert b"pickle" not in data and data[:8] == b"CVADSNAP"


def test_corrupt_or_truncated_snapshots_are_rejected():
    from real_time_vad import StreamSnapshot, VADError
    data = _snapshot().to_bytes()
    for cut in [0, 7, 12, 19, 25, len(data) // 2, len(data) - 1]:
        with pytest.raises(VADError, match="invalid stream snapshot"):
            StreamSnapshot.from_bytes(data[:cut])
    with pytest.raises(VADError, match="invalid stream snapshot"):
        StreamSnapshot.from_bytes(data + b"x")
    bad = bytearray(data)
    bad[3] ^= 1
    with pytest.raises(VADError, match="magic"):
        StreamSnapshot.from_bytes(bytes(bad))
    bad = bytearray(data)
    bad[8] = 9
    with pytest.raises(VADError, match="version"):
        StreamSnapshot.from_bytes(bytes(bad))
    bad = bytearray(data)
    bad[21] ^= 0x55                                       # inside the JSON header
    with pytest.raises(VADError, match="invalid stream snapshot"):
        StreamSnapshot.from_bytes(bytes(bad))


def test_header_stream_list_must_be_a_list_of_distinct_streams():
    import json
    import struct
    from real_time_vad import StreamSnapshot, VADError
    data = _snapshot().to_bytes()
    hlen = struct.unpack_from("<Q", data, 12)[0]
    header = json.loads(data[20:20 + hlen])

    def rebuilt(h):
        hb = json.dumps(h).encode()
        return data[:12] + struct.pack("<Q", len(hb)) + hb + data[20 + hlen:]

    assert StreamSnapshot.from_bytes(rebuilt(header)).stream_ids == [10, 11, 12]
    for bad in (5, "x", [1, 2, 3], None):
        with pytest.raises(VADError, match="invalid stream snapshot"):
            StreamSnapshot.from_bytes(rebuilt(dict(header, streams=bad)))
    dup = json.loads(json.dumps(header))
    dup["streams"][2]["id"] = 10
    with pytest.raises(VADError, match="twice"):
        StreamSnapshot.from_bytes(rebuilt(dup))


def test_rows_imported_without_audio_keep_no_pre_roll_or_segment():
    """A row's payload mode may be lowered before import (a restored stream that no longer wants audio): the carried
    pre-roll and segment are then dropped, so the end record hands over an empty segment."""
    from real_time_vad.engine import capi
    from real_time_vad.engine.feeder import set_row_payloads
    a = _feeder(max_streams=4, frame_len=512, hop=512)
    a.open(0, payload=capi.PAYLOAD_SEGMENTS, vad_start_probability=0.5)
    a.push(0, np.full(1024, 0.3, np.float32))
    a.gather_only()
    a.deliver_only(np.array([[0.9, 0.9]], np.float32), np.array([[capi.FLAG_STARTED, capi.FLAG_CONTINUING]], np.uint8))
    blob = a.export_rows([0])

    def end_segment(payload):
        b = _feeder(max_streams=4, frame_len=512, hop=512)
        b.import_rows([1], set_row_payloads(blob, [payload]))
        b.push(1, np.full(512, 0.3, np.float32))
        b.gather_only()
        r = b.deliver_only(np.array([[0.1]], np.float32), np.array([[capi.FLAG_ENDED]], np.uint8))
        b.close()
        return r.deliveries[0].segment

    assert end_segment(capi.PAYLOAD_SEGMENTS).size == 3 * 512
    assert end_segment(capi.PAYLOAD_EVENTS).size == 0
    a.close()


def test_export_rows_while_other_threads_push():
    """Rows may grow between sizing the blob and filling it: the export is repeated, never refused."""
    import threading
    from real_time_vad.engine.feeder import StreamFeeder
    f = _feeder(max_streams=4, frame_len=512, hop=512, capacity_frames=2)
    f.open(0)
    stop = threading.Event()
    x = np.full(4096, 0.1, np.float32)

    def producer():
        while not stop.is_set():
            f.push(0, x)

    t = threading.Thread(target=producer)
    t.start()
    try:
        sizes = [len(f.export_rows([0])) for _ in range(200)]
    finally:
        stop.set()
        t.join()
    assert sizes == sorted(sizes) and sizes[-1] > sizes[0]
    g = StreamFeeder(None, max_streams=4, frame_len=512, hop=512)
    g.import_rows([2], f.export_rows([0]))
    assert g.pending(2) == f.pending(0)
    f.close()
    g.close()
