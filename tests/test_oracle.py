"""Pins of the CPU oracle (test infrastructure) -- CPU only.

The reference is C# and ships no golden vectors for this path; no .NET runtime exists here.  The
oracle is therefore pinned by (1) an INDEPENDENT native decoder (FFmpeg's vorbis decoder, fixture
tests/golden/ffmpeg_pin_<name>.npz made by make_ffmpeg_pin.py) under the reference's own test convention
(NVorbis.Tests/AssetTest.cs:131-194: 16-bit PCM, |diff| <= 2 LSB, here even <= 1), (2) closed forms
and invariants that do not depend on any decoder, (3) the workload counts SURVEY.md measured with a
separate symbol-level walker, (4) regression digests of its own output (oracle_golden.json)."""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_binding as ob
from conftest import FILES, GOLDEN, load_file

GOLD = json.load(open(os.path.join(GOLDEN, "oracle_golden.json")))


def q16(x):
    return np.clip((x * np.float32(32768.0)).astype(np.int64), -32768, 32767)


def ffmpeg_pin(name):
    """FFmpeg's 16-bit PCM of `name`, [frames, channels] (stored by make_ffmpeg_pin.encode)."""
    z = np.load(os.path.join(GOLDEN, "ffmpeg_pin_%s.npz" % name))
    d = (z["lo"].astype(np.uint16) | (z["hi"].astype(np.uint16) << 8)).view(np.int16)
    for _ in range(2):
        d = np.cumsum(d, axis=1, dtype=np.int16)
    return d.T


@pytest.mark.parametrize("name", FILES)
def test_oracle_vs_independent_decoder(name):
    pin = ffmpeg_pin(name).astype(np.int64)
    s = ob.OracleStream(load_file(name))
    s.set_clip(False)
    pcm, _, _ = s.decode_all()
    n = pcm.shape[0]
    assert n <= pin.shape[0] and pin.shape[1] == s.channels  # FFmpeg does not apply the end-of-stream granule trim
    diff = np.abs(q16(pcm) - pin[:n])
    assert diff.max() <= 1, "oracle differs from FFmpeg by %d LSB" % diff.max()


@pytest.mark.parametrize("name", FILES)
def test_container_and_codebooks(name):
    s = ob.OracleStream(load_file(name))
    assert s.crc_failures() == 0 and s.waste_bits() == 0
    for b in range(s.book_count()):
        info = s.book_info(b)
        used = int((s.book_lengths(b) > 0).sum())
        if used > 1:
            assert abs(s.book_kraft(b) - 1.0) < 1e-12, "book %d is not a complete prefix code" % b
        assert info["max_bits"] <= 32


@pytest.mark.parametrize("name", FILES)
def test_golden_digests(name):
    g = GOLD[name]
    data = load_file(name)
    s = ob.OracleStream(data)
    assert (s.channels, s.sample_rate, list(s.block_sizes)) == (g["channels"], g["sample_rate"], g["block_sizes"])
    assert s.total_samples == g["total_samples"]
    pk = s.audio_packets()
    assert len(pk) == g["audio_packets"] and sum(len(p["data"]) for p in pk) == g["packet_bytes"]
    h = hashlib.sha256()
    nsc = 0
    for p in pk:
        d = s.dump_packet(p["data"], want_floats=False)
        assert d["bits_read"] <= 8 * len(p["data"])  # no packet over-reads
        h.update(np.int32([d["status"], d["mode"], d["block_size"], d["bits_read"]] + d["info"] + d["post_count"]).tobytes())
        h.update(d["scalars"].tobytes())
        h.update(d["classes"].tobytes())
        h.update(d["raw_posts"].tobytes())
        for c, k in enumerate(d["post_count"]):
            h.update(d["final_y"][c][:k].tobytes())
            h.update(d["step_flags"][c][:k].tobytes())
        nsc += d["scalars_n"]
    assert nsc == g["decode_scalar_calls"]
    assert h.hexdigest() == g["stage_sha256"]
    for clip in (True, False):
        key = "clip" if clip else "noclip"
        t = ob.OracleStream(data)
        t.set_clip(clip)
        pcm, counts, fault = t.decode_all()
        assert pcm.shape[0] == g["samples_" + key] and fault == g["fault_" + key]
        assert len(counts) == g["read_calls_" + key] and t.has_clipped == g["has_clipped_" + key]
        assert hashlib.sha256(pcm.tobytes()).hexdigest() == g["pcm_sha256_" + key]


def test_survey_workload_counts():
    """SURVEY.md 8(d): counts measured with a separate throw-away walker in the survey session."""
    want = {"1test": (25, 270, 17318), "2test": (310, 21174, 315790), "3test": (366, 209944, 288094),
            "issue6test": (606, 112540, 548160)}
    for name, (pk, calls, samples) in want.items():
        g = GOLD[name]
        assert (g["audio_packets"], g["decode_scalar_calls"], g["samples_clip"]) == (pk, calls, samples)


def test_1test_pcm_fixture():
    ref = np.load(os.path.join(GOLDEN, "1test_pcm.npy"))
    s = ob.OracleStream(load_file("1test"))
    pcm, _, _ = s.decode_all()
    assert np.array_equal(pcm.view(np.uint32), ref.view(np.uint32))
    # SURVEY Appendix C anchors (independent float64 NumPy decoder): rms 0.00660, peak +0.19060 @ 739
    assert abs(float(np.sqrt((pcm.astype(np.float64) ** 2).mean())) - 0.00660) < 5e-5
    assert int(np.argmax(pcm[:, 0])) == 739 and abs(float(pcm[739, 0]) - 0.19060) < 1e-4


@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192])
def test_imdct_vs_float64_direct_form(n):
    """Mdct.Reverse == y[i] = sum_k X[k] cos(pi/(2n) (2i+1+n/2)(2k+1)) (SURVEY A6), no scaling."""
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n // 2).astype(np.float32)
    y = ob.imdct(x)
    i = np.arange(n)[:, None]
    k = np.arange(n // 2)[None, :]
    ref = (np.cos(np.pi / (2 * n) * (2 * i + 1 + n // 2) * (2 * k + 1)) * x.astype(np.float64)[None, :]).sum(axis=1)
    assert np.abs(y - ref).max() <= 3e-6 * np.abs(ref).max() + 1e-6


@pytest.mark.parametrize("n", [64, 128])
def test_imdct_below_256_is_not_a_transform_in_the_reference(n):
    """Quirk Q10 (DESIGN.md): Mdct.CalcReverse always runs step-3 iterations 0, 1 and the fused
    ld-6/-5/-4 pass (Mdct.cs:200-249), which is two/one pass too many for n = 64/128, so the reference
    (and this restatement of it) does not compute an IMDCT there.  The GPU path refuses such streams."""
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n // 2).astype(np.float32)
    y = ob.imdct(x)
    i = np.arange(n)[:, None]
    k = np.arange(n // 2)[None, :]
    ref = (np.cos(np.pi / (2 * n) * (2 * i + 1 + n // 2) * (2 * k + 1)) * x.astype(np.float64)[None, :]).sum(axis=1)
    assert np.abs(y - ref).max() > 0.1


def test_window_and_db_table_closed_forms():
    for n in (128, 1024):
        w = ob.window_slope(n)
        i = np.arange(n)
        ref = np.sin(np.pi / 2 * np.sin(np.pi / 2 * (i + 0.5) / n) ** 2)
        assert np.abs(w - ref).max() < 3e-7
    t = ob.inverse_db_table()
    ref = np.exp(0.11512925 * (np.arange(256) * 0.546875 - 139.453125))
    assert np.abs(t / ref - 1).max() < 2e-6
    assert t[255] == np.float32(1.0)


def test_packet_geometry_table():
    """SURVEY A7 table for 256/2048."""
    assert ob.packet_info(256, 2048, 0, 1, 1) == [128, 0, 0, 128, 128, 256]
    assert ob.packet_info(256, 2048, 1, 1, 1) == [1024, 1, 0, 1024, 1024, 2048]
    assert ob.packet_info(256, 2048, 1, 0, 0) == [128, 0, 448, 576, 1472, 1600]


def test_crc_known_answer():
    # Ogg CRC-32 (poly 0x04c11db7, init 0, no reflection): the first page of 1test.ogg carries its own CRC
    d = load_file("1test")
    nseg = d[26]
    plen = 27 + nseg + sum(d[27:27 + nseg])
    page = bytearray(d[:plen])
    want = int.from_bytes(page[22:26], "little")
    page[22:26] = b"\0\0\0\0"
    assert ob.crc_ogg(bytes(page)) == want


# ---- (5) an independent second reading of the integer stages ------------------------------------------
def _pin_digest(seq):
    return hashlib.sha256(",".join(str(int(x)) for x in seq).encode()).hexdigest()[:16]


@pytest.mark.parametrize("name", FILES)
def test_integer_stages_vs_independent_walker(name):
    """tests/golden/stage_pin.json was produced by tests/golden/make_stage_pin.py: a pure-Python symbol walker
    written from the algorithm notes (SURVEY.md Appendix A) and sharing no code with oracle/ -- its own Ogg
    splitter, codeword assignment and bit reader.  Every audio packet: DecodeScalar sequence, raw posts,
    final Y, step flags and partition classes of the C oracle must equal that second reading."""
    pin = json.load(open(os.path.join(GOLDEN, "stage_pin.json")))[name]
    s = ob.OracleStream(load_file(name))
    pk = s.audio_packets()
    assert len(pk) == len(pin)
    for i, (p, w) in enumerate(zip(pk, pin)):
        o = s.dump_packet(p["data"])
        if w is None:
            assert o["status"] != 0
            continue
        what = "%s packet %d" % (name, i)
        assert o["status"] == 0, what
        assert o["scalars_n"] == w["n_scalars"] and _pin_digest(o["scalars"][:o["scalars_n"]]) == w["scalars"], what
        assert o["classes_n"] == w["n_classes"] and _pin_digest(o["classes"][:o["classes_n"]]) == w["classes"], what
        counts = [max(int(o["post_count"][c]), 0) for c in range(s.channels)]
        assert counts == w["post_counts"], what
        assert _pin_digest([v for c in range(s.channels) for v in o["raw_posts"][c][:counts[c]]]) == w["raw_posts"], what
        assert _pin_digest([v for c in range(s.channels) for v in o["final_y"][c][:counts[c]]]) == w["final_y"], what
        assert _pin_digest([v for c in range(s.channels) for v in o["step_flags"][c][:counts[c]]]) == w["step_flags"], what
        assert o["bits_read"] == w["bits"], what


def test_bench_imdct_ola_matches_the_reference_restatement():
    """bench.py's config-3 CPU baseline (oracle/vo_bench.c: Mdct.Reverse + OverlapBuffers + interleaved clipped
    store per synthetic stream) produces the samples tests/cases.py's block-by-block restatement produces."""
    import cases
    rng = np.random.default_rng(5)
    ch, n_streams, n_blocks = 2, 3, 17
    flags = rng.integers(0, 2, (n_streams, n_blocks)).astype(np.uint8)
    sizes = np.where(flags.reshape(-1) & 1, 1024, 128)
    spectra = (rng.standard_normal(int(sizes.sum()) * ch) * 0.05).astype(np.float32)
    n, _, chk = ob.bench_imdct_ola(spectra, flags, ch, 256, 2048, 2)
    total, ref_sum, off = 0, 0.0, 0
    for s in range(n_streams):
        nfl = int(sum((2048 if f & 1 else 256) // 2 * ch for f in flags[s]))
        ref = cases.reference_imdct_ola(flags[s], spectra[off:off + nfl], ch, 256, 2048)
        off += nfl
        total += ref.size
        ref_sum += float(np.clip(ref, -0.99999994, 0.99999994).astype(np.float64).sum())
    assert n == total
    assert abs(chk - ref_sum) <= 1e-3 * max(1.0, abs(ref_sum)) + 1e-2
