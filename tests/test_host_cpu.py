"""Host-side logic of the Python mirror that needs no GPU (the C-ABI library only has to load)."""
from soundsym_b200 import api


def test_audacity_labels_known_answers(tmp_path):
    """src/sound.rs:561-571 checks tests/vowel.txt for these values; the same three lines in the same format here."""
    p = tmp_path / "labels.txt"
    p.write_text("0.7065779155923718\t0.7619218551399829\to\n0.7619218551399829\t1.0201935730288352\ts\n"
                 "5.4\t5.59353222977394\tning\n3.0\n\nx\ty\n")
    t = api.audacity_labels_to_timestamps(str(p))
    assert len(t) == 6
    assert abs(t[0][0] - 0.7065779155923718) < 1e-10 and abs(t[2][1] - 5.59353222977394) < 1e-10
    assert t[1] == (0.7619218551399829, 1.0201935730288352, "s") and t[2][2] == "ning"
    assert t[3] == (3.0, 0.0, None)    # missing fields: 0.0 / None
    assert t[4] == (0.0, 0.0, None)    # blank line: trim().split('\t') yields one empty field
    assert t[5] == (0.0, 0.0, None)    # unparsable numbers: 0.0


def test_write_wav_rounding(tmp_path):
    import numpy as np
    api._write_wav_i32(str(tmp_path / "a.wav"), np.array([0.0, 0.5, -0.5, 1.0, -1.0, 2.0, -2.0, float("nan")]), 44100)
    pcm, sr, bits = api._read_wav_pcm(str(tmp_path / "a.wav"))
    assert bits == 32 and sr == 44100.0
    assert pcm.tolist() == [0, 1073741823, -1073741823, 2147483647, -2147483647, 2147483647, -2147483648, 0]


def test_bench_sharding_and_algorithmic_bytes():
    """bench.py's host logic: shards are contiguous, cover every segment once and are balanced by frames (SURVEY.md 8e);
    the pairwise-streaming byte count (SURVEY.md 8d) is additive over shards."""
    import importlib.util
    import os
    import numpy as np
    from soundsym_b200 import synth
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    d, doff = synth.segments(5000, 13, seed=7)
    q, qoff = synth.segments(300, 13, seed=8)
    whole = bench.algorithmic_bytes(doff, qoff, 0, len(doff) - 1)
    lens_d, lens_q = np.diff(doff).astype(np.int64), np.diff(qoff).astype(np.int64)
    assert whole == int((lens_d[:, None] + lens_q[None, :]).sum()) * 13 * 4  # sum over pairs of (Lq + Ld) * C * 4 B
    for n in (1, 2, 4, 8):
        cuts = bench.shard_bounds(doff, n)
        assert cuts[0] == 0 and cuts[-1] == len(doff) - 1 and all(a <= b for a, b in zip(cuts, cuts[1:]))
        frames = [int(doff[b] - doff[a]) for a, b in zip(cuts, cuts[1:])]
        assert sum(frames) == int(doff[-1]) and max(frames) - min(frames) <= 2 * 32  # within a segment or two of even
        assert sum(bench.algorithmic_bytes(doff, qoff, a, b) for a, b in zip(cuts, cuts[1:])) == whole


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 .npy files that round-trip the u32 indices exactly; past the size cap, the same
    seeded sample of queries on every run; --steps 0 and unsupported configurations are refused."""
    import importlib.util
    import os
    import sys
    import numpy as np
    import pytest
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(5)
    idx = rng.integers(0, 100000, size=(1000, 4)).astype(np.uint32)
    idx[3, 2:] = 0xFFFFFFFF
    dist = rng.uniform(0.0, 50.0, size=(1000, 4))
    bench.dump_outputs(str(tmp_path / "all"), idx, dist)
    out = {n: np.load(str(tmp_path / "all" / (n + ".npy"))) for n in ("query_ids", "indices", "distances")}
    assert all(a.dtype == np.float64 for a in out.values())
    assert np.array_equal(out["query_ids"], np.arange(1000)) and np.array_equal(out["distances"], dist)
    assert np.array_equal(out["indices"].astype(np.uint32), idx) and out["indices"][3, 3] == 0xFFFFFFFF
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 4096 + 72 * 100)  # room for 100 rows of k = 4
    samples = []
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), idx, dist)
        ids = np.load(str(tmp_path / run / "query_ids.npy")).astype(np.int64)
        assert len(ids) == 100 and np.all(np.diff(ids) > 0)
        assert np.array_equal(np.load(str(tmp_path / run / "indices.npy")).astype(np.uint32), idx[ids])
        assert np.array_equal(np.load(str(tmp_path / run / "distances.npy")), dist[ids])
        samples.append(ids)
    assert np.array_equal(samples[0], samples[1])
    for argv in (["--steps", "0"], ["--config", "5", "--dump-outputs", str(tmp_path)],
                 ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()


def test_synth_is_seeded():
    import numpy as np
    from soundsym_b200 import synth
    a, ao = synth.segments(50, 13, seed=3)
    b, bo = synth.segments(50, 13, seed=3)
    assert np.array_equal(a, b) and np.array_equal(ao, bo) and int(ao[-1]) == a.shape[0]
    assert np.diff(ao).min() >= 4 and np.diff(ao).max() <= 32
    x = synth.audio(0.5, seed=1)
    assert np.array_equal(x, synth.audio(0.5, seed=1)) and x.shape == (22050,) and np.abs(x).max() <= 1.0


def test_cpp_mirror_file_helpers_match_python_mirror(tmp_path):
    """The C++ mirror's Audacity-label parser, 32-bit WAV writer and PCM reader (include/soundsym.hpp) against the Python
    mirror's, on the same bytes. Host code only: the binary never creates a context."""
    import json
    import os
    import subprocess
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "host_helpers")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "host_helpers.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "soundsym_b200"), "-lsoundsym_b200",
                           "-Wl,-rpath," + os.path.join(root, "soundsym_b200")])
    labels = tmp_path / "labels.txt"
    labels.write_text("0.7065779155923718\t0.7619218551399829\to\n1.5\t2.25\n\n3\t4\tning ning\nx\t1\tz\n")
    wav = str(tmp_path / "w.wav")
    out = json.loads(subprocess.run([exe, str(labels), wav], capture_output=True, text=True, check=True).stdout)
    py = api.audacity_labels_to_timestamps(str(labels))
    assert out["n"] == len(py) == 5
    assert [tuple(s) for s in out["stamps"]] == [tuple(t) for t in py]
    pcm, sr, bits = api._read_wav_pcm(wav)
    assert bits == 32 and sr == out["sr"] == 22050.0
    ref = np.array([0.0, 0.5, -0.5, 1.0, -1.0, 2.0, -2.0, float("nan"), 0.123456789])
    api._write_wav_i32(str(tmp_path / "p.wav"), ref, 22050)
    pcm2, _, _ = api._read_wav_pcm(str(tmp_path / "p.wav"))
    assert np.array_equal(pcm, pcm2)                                   # both writers produce the same samples
    assert np.array_equal(np.array(out["back"]), pcm.astype(np.float64) / 2147483647.0)  # reader: s / (i32::MAX >> 0)


def test_wav_reader_rejects_what_hound_rejects(tmp_path):
    """_read_wav_pcm accepts integer PCM only (hound::WavReader at src/sound.rs:117 yields i32 samples; float WAVs, a data
    chunk before fmt, truncated fmt chunks and odd bit depths are errors), and 8-bit samples are unsigned offset-128."""
    import struct
    import numpy as np
    import pytest

    def wav(chunks):
        body = b"WAVE" + b"".join(cid + struct.pack("<I", len(b)) + b + (b"\0" if len(b) & 1 else b"") for cid, b in chunks)
        return b"RIFF" + struct.pack("<I", len(body)) + body

    def fmt(tag, bits, sr=8000, extra=b""):
        return struct.pack("<HHIIHH", tag, 1, sr, sr * bits // 8, max(bits // 8, 1), bits) + extra

    def load(name, data):
        p = tmp_path / name
        p.write_bytes(data)
        return api._read_wav_pcm(str(p))

    pcm, sr, bits = load("u8.wav", wav([(b"fmt ", fmt(1, 8)), (b"data", bytes([0, 128, 255]))]))
    assert bits == 8 and sr == 8000.0 and pcm.tolist() == [-128, 0, 127]
    pcm, _, bits = load("s24.wav", wav([(b"LIST", b"abc"), (b"fmt ", fmt(1, 24)), (b"data", bytes([0xFF, 0xFF, 0xFF, 0x01, 0x00, 0x80]))]))
    assert bits == 24 and pcm.tolist() == [-1, -8388607]
    ext = fmt(0xFFFE, 16, extra=struct.pack("<HHI", 22, 16, 4) + struct.pack("<H", 1) + b"\0" * 14)
    pcm, _, bits = load("ext.wav", wav([(b"fmt ", ext), (b"data", struct.pack("<hh", -2, 7))]))
    assert bits == 16 and pcm.tolist() == [-2, 7]
    for name, data in [
        ("float.wav", wav([(b"fmt ", fmt(3, 32)), (b"data", b"\0" * 8)])),           # IEEE float
        ("order.wav", wav([(b"data", b"\0" * 8), (b"fmt ", fmt(1, 16))])),           # data before fmt
        ("short.wav", wav([(b"fmt ", fmt(1, 16)[:10]), (b"data", b"\0" * 8)])),      # truncated fmt
        ("bits.wav", wav([(b"fmt ", fmt(1, 4)), (b"data", b"\0" * 8)])),             # bits < 8 (was a division by zero)
        ("nodata.wav", wav([(b"fmt ", fmt(1, 16))])),
        ("junk.wav", b"RIFFxxxxWAVX"),
    ]:
        with pytest.raises(ValueError):
            load(name, data)
