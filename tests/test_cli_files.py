"""SURVEY §8(f) N2: the file front-end of the reference's `nnnoiseless` binary (src/nnnoiseless.rs; tests/cli.rs).

CPU: decoders against an independent restatement (also on excerpts of the reference's own WAV fixtures), the WAV writer
against Python's `wave`, the CLI's error behaviour, the oracle resampler's properties.
GPU: resampler and whole-file results against the oracle."""
import os
import struct
import subprocess
import wave

import numpy as np
import pytest

import oracle
from nnnoiseless_b200 import files
from nnnoiseless_b200.synth import synth_streams

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _wav_bytes(x, rate, bits=16, fmt=1, extensible=False, extra_chunk=False):
    """x: [n][ch] float in the i16 range -> RIFF/WAVE bytes with the requested sample encoding."""
    n, ch = x.shape
    if fmt == 3:
        payload = (x / 32767.0).astype("<f4").tobytes()
        nbytes = 4
    else:
        nbytes = (bits + 7) // 8
        v = np.round(x).astype(np.int64)
        v = v >> (16 - bits) if bits < 16 else v << (bits - 16)
        if nbytes == 1:
            payload = (v + 128).astype(np.uint8).tobytes()
        else:
            u = (v & ((1 << (8 * nbytes)) - 1)).astype(np.uint64)
            payload = np.stack([(u >> (8 * i)) & 0xFF for i in range(nbytes)], -1).astype(np.uint8).tobytes()
    body = struct.pack("<HHIIHH", 0xFFFE if extensible else fmt, ch, rate, rate * ch * nbytes, ch * nbytes, bits)
    if extensible:
        guid = struct.pack("<H", fmt) + bytes.fromhex("000000001000800000aa00389b71")
        body += struct.pack("<HHI", 22, bits, (1 << ch) - 1) + guid
    chunks = b"fmt " + struct.pack("<I", len(body)) + body
    if extra_chunk:
        chunks += b"LIST" + struct.pack("<I", 5) + b"abcde" + b"\0"      # odd-sized chunk + pad byte
    chunks += b"data" + struct.pack("<I", len(payload)) + payload
    return b"RIFF" + struct.pack("<I", 4 + len(chunks)) + b"WAVE" + chunks


def _signal(n, ch, seed):
    x = synth_streams(ch, (n + 479) // 480, seed=seed)[:, :n]
    return np.ascontiguousarray(x.T)                                      # [n][ch]


@pytest.mark.parametrize("kw", [dict(bits=16), dict(bits=8), dict(bits=24), dict(bits=32), dict(bits=12), dict(fmt=3, bits=32),
                                dict(bits=24, extensible=True), dict(bits=16, extra_chunk=True)])
def test_wav_decoder_matches_restatement(tmp_path, kw):
    x = _signal(3000, 2, seed=4)
    data = _wav_bytes(x, 44100, **kw)
    p = tmp_path / "in.wav"
    p.write_bytes(data)
    got, rate = files.read_audio(str(p))
    want, wrate = oracle.decode_wav(data)
    assert rate == wrate == 44100.0 and got.shape == want.shape == (3000, 2)
    assert np.array_equal(got, want)
    if kw.get("bits") in (16, 24, 32) and kw.get("fmt", 1) == 1:
        assert np.array_equal(got, np.round(x))                           # >= 16 bits: lossless round trip


@pytest.mark.parametrize("name,ch", [("mono.wav", 1), ("stereo.wav", 2), ("mono-float.wav", 1)])
def test_reference_fixtures_decode(name, ch):
    """The reference's test_data/<name> (written by hound) cut to frames 60000..64095: every chunk before `data` kept
    byte for byte (mono-float.wav's `fact` and `PEAK` included), the RIFF and data sizes set to the excerpt's."""
    path = os.path.join(GOLDEN, name.replace(".wav", "_excerpt.wav"))
    got, rate = files.read_audio(path)
    want, wrate = oracle.decode_wav(open(path, "rb").read())
    assert rate == wrate == 44100.0 and got.shape == (4096, ch)
    assert np.array_equal(got, want)


def test_raw_decoder_and_errors(tmp_path):
    pcm = np.arange(-6, 6, dtype="<i2")
    p = tmp_path / "a.raw"
    p.write_bytes(pcm.tobytes())
    got, rate = files.read_audio(str(p), channels=3, sample_rate=16000)
    assert rate == 16000.0 and np.array_equal(got, pcm.astype(np.float32).reshape(4, 3))
    p.write_bytes(pcm.tobytes()[:-1])
    with pytest.raises(files.NnnoiselessError, match="even number of bytes"):      # src/nnnoiseless.rs:68-70
        files.read_audio(str(p))
    p.write_bytes(pcm.tobytes()[:-2])
    with pytest.raises(files.NnnoiselessError, match="multiple of 3 samples"):     # :88-91
        files.read_audio(str(p), channels=3)
    with pytest.raises(files.NnnoiselessError, match="Failed to open input file"):
        files.read_audio(str(tmp_path / "missing.raw"))


@pytest.mark.parametrize("ch", [1, 2, 5])
def test_wav_writer_readable(tmp_path, ch):
    pcm = np.round(_signal(1000, ch, seed=9)).astype(np.int16)
    p = tmp_path / "o.wav"
    files.write_audio(str(p), pcm)
    data = p.read_bytes()
    back, rate = oracle.decode_wav(data)
    assert rate == 48000.0 and np.array_equal(back, pcm.astype(np.float32))          # spec at src/nnnoiseless.rs:278-283
    assert struct.unpack("<I", data[4:8])[0] == len(data) - 8
    if ch <= 2:                                                                      # Python's wave refuses WAVE_FORMAT_EXTENSIBLE
        with wave.open(str(p)) as w:
            assert (w.getnchannels(), w.getframerate(), w.getsampwidth(), w.getnframes()) == (ch, 48000, 2, 1000)
    q = tmp_path / "o.raw"
    files.write_audio(str(q), pcm)
    assert q.read_bytes() == pcm.astype("<i2").tobytes()


def test_cli_invalid_wav(tmp_path):
    """tests/cli.rs::invalid_wav: a non-RIFF input, by extension and with --wav-in."""
    (tmp_path / "input.wav").write_bytes(bytes(4800))
    r = subprocess.run([files.CLI_PATH, str(tmp_path / "input.wav"), str(tmp_path / "output.wav")], capture_output=True, text=True)
    assert r.returncode != 0 and "no RIFF tag found" in r.stderr
    (tmp_path / "input.raw").write_bytes(bytes(4800))
    r = subprocess.run([files.CLI_PATH, "--wav-in", str(tmp_path / "input.raw"), str(tmp_path / "output.wav")], capture_output=True,
                       text=True)
    assert r.returncode != 0 and "no RIFF tag found" in r.stderr


def test_cli_argument_errors(tmp_path):
    r = subprocess.run([files.CLI_PATH], capture_output=True, text=True)
    assert r.returncode != 0 and "<INPUT>" in r.stderr
    r = subprocess.run([files.CLI_PATH, "--sample-rate", "abc", "a", "b"], capture_output=True, text=True)
    assert r.returncode != 0 and "--sample-rate" in r.stderr
    r = subprocess.run([files.CLI_PATH, "--model", str(tmp_path / "nope.rnn"), "a", "b"], capture_output=True, text=True)
    assert r.returncode != 0 and "Failed to open model file" in r.stderr
    (tmp_path / "bad.rnn").write_bytes(b"\x01\x02\x03")
    r = subprocess.run([files.CLI_PATH, "--model", str(tmp_path / "bad.rnn"), "a", "b"], capture_output=True, text=True)
    assert r.returncode != 0 and "Failed to parse model file" in r.stderr
    assert subprocess.run([files.CLI_PATH, "--help"], capture_output=True).returncode == 0


def test_cli_inputs_shorter_than_two_frames(tmp_path):
    """The first frame's output is discarded (src/nnnoiseless.rs:319-327): < 960 samples in -> an empty but valid output."""
    (tmp_path / "short.raw").write_bytes(bytes(2 * 700))
    r = subprocess.run([files.CLI_PATH, str(tmp_path / "short.raw"), str(tmp_path / "o.wav")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    back, rate = oracle.decode_wav((tmp_path / "o.wav").read_bytes())
    assert rate == 48000.0 and back.shape == (0, 1)
    r = subprocess.run([files.CLI_PATH, str(tmp_path / "short.raw"), str(tmp_path / "o.raw")], capture_output=True, text=True)
    assert r.returncode == 0 and (tmp_path / "o.raw").read_bytes() == b""


def test_oracle_resampler_properties():
    n = np.arange(44100)
    x = (10000 * np.sin(2 * np.pi * 1000 * n / 44100)).astype(np.float32)
    y = oracle.resample(x, 44100 / 48000)[:, 0]
    assert abs(len(y) - 48000) <= 1
    # a depth-8 windowed sinc centred between ring frames 8 and 9: output k sits at source time (k + 1) r - 8
    t = (np.arange(len(y)) + 1) * (44100 / 48000) - 8
    ref = 10000 * np.sin(2 * np.pi * 1000 * t / 44100)
    assert np.sqrt(np.mean((y[200:-200] - ref[200:-200]) ** 2)) < 1e-3 * 10000
    # channels are independent and interleaved
    x2 = np.stack([x, -0.5 * x], -1)
    y2 = oracle.resample(x2, 44100 / 48000)
    assert np.array_equal(y2[:, 0], y) and np.allclose(y2[:, 1], -0.5 * y, atol=2e-3)
    # the start-up (ring still filling) is causal: nothing comes out before the first source sample went in
    imp = np.zeros(64, np.float32)
    imp[0] = 1000.0
    assert oracle.resample(imp, 0.5)[0, 0] == 0.0


def _oracle_file(model, x, rate):
    x48 = x if rate == 48000 else oracle.resample(x, rate / 48000.0)
    return oracle.cli_frames(model, x48)


@pytest.mark.gpu
@pytest.mark.parametrize("rate,ch", [(44100, 1), (16000, 2), (96000, 3), (8000, 1), (47999, 1)])
def test_resampler_matches_oracle(rate, ch):
    x = _signal(rate // 4, ch, seed=rate)
    want = oracle.resample(x, rate / 48000.0)
    got = files.resample(x, rate / 48000.0)
    assert got.shape == want.shape
    # same f64 formula per tap; CUDA's sin/cos differ from glibc's in the last ulp, which only rarely survives the
    # rounding of each tap to f32: bit-equal almost everywhere, 1e-6 relative otherwise
    assert (got != want).mean() < 0.02
    assert np.max(np.abs(got - want)) <= 4e-3


@pytest.mark.gpu
def test_cli_basic_usage(tmp_path):
    """tests/cli.rs::basic_usage: 4800 zero bytes of raw input."""
    (tmp_path / "input.raw").write_bytes(bytes(4800))
    r = subprocess.run([files.CLI_PATH, str(tmp_path / "input.raw"), str(tmp_path / "output.raw")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "output.raw").read_bytes() == bytes(4 * 960)       # 5 frames in, the first one's output discarded


@pytest.mark.gpu
def test_cli_golden_vector(tmp_path, reference_output):
    """The reference's golden pair is exactly a CLI run: testing.raw -> reference_output.raw (src/lib.rs:196-213)."""
    src = os.path.join(os.path.dirname(__file__), "golden", "testing.raw")
    r = subprocess.run([files.CLI_PATH, src, str(tmp_path / "out.raw")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = np.frombuffer((tmp_path / "out.raw").read_bytes(), "<i2").astype(np.float64)
    ref = reference_output.astype(np.float64)
    assert got.shape == ref.shape
    assert np.sum((ref - got) ** 2) / np.sum(got ** 2) < 1e-4              # the metric of src/lib.rs:184-194
    assert np.max(np.abs(ref - got)) <= 1


@pytest.mark.gpu
def test_files_match_oracle_batch_and_single(tmp_path, builtin_bytes):
    model = oracle.Model(builtin_bytes)
    specs = [("a.wav", 44100, 1, dict(bits=16)), ("b.wav", 48000, 2, dict(bits=16)), ("c.wav", 44100, 1, dict(fmt=3, bits=32)),
             ("d.wav", 32000, 3, dict(bits=24, extensible=True)), ("e.raw", 48000, 1, None), ("f.wav", 22050, 2, dict(bits=8))]
    pairs, wants = [], []
    for i, (name, rate, ch, kw) in enumerate(specs):
        n = int(rate * (0.35 + 0.1 * i)) + 17 * i                        # different lengths: shorter files are padded in the batch
        x = _signal(n, ch, seed=20 + i)
        p = tmp_path / name
        if kw is None:
            p.write_bytes(np.round(x).astype("<i2").tobytes())
            dec = np.round(x).astype(np.float32)
        else:
            data = _wav_bytes(x, rate, **kw)
            p.write_bytes(data)
            dec, _ = oracle.decode_wav(data)
        pairs.append((str(p), str(tmp_path / ("out_" + name))))
        wants.append(_oracle_file(model, dec, rate))
    files.denoise_files(pairs)
    for (name, rate, ch, kw), (_, outp), want in zip(specs, pairs, wants):
        raw = open(outp, "rb").read()
        if name.endswith(".wav"):
            got, orate = oracle.decode_wav(raw)
            assert orate == 48000.0
            got = got.astype(np.int16)
        else:
            got = np.frombuffer(raw, "<i2").reshape(-1, ch)
        assert got.shape == want.shape and got.shape[0] % 480 == 0 and got.shape[0] > 0
        d = np.abs(got.astype(np.int32) - want.astype(np.int32))
        assert d.max() <= 1 and (d != 0).mean() < 1e-2, (name, d.max(), (d != 0).mean())
    # one file alone == the same file inside the batch, bit for bit (streams are independent)
    single = tmp_path / "single.wav"
    files.denoise_file(pairs[3][0], str(single))
    assert single.read_bytes() == open(pairs[3][1], "rb").read()
    # raw multi-channel input with --sample-rate / --channels through the binary
    x = _signal(12000, 2, seed=77)
    (tmp_path / "g.raw").write_bytes(np.round(x).astype("<i2").tobytes())
    r = subprocess.run([files.CLI_PATH, "--sample-rate", "24000", "--channels=2", "--wav-out", str(tmp_path / "g.raw"),
                        str(tmp_path / "g.out")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got, _ = oracle.decode_wav((tmp_path / "g.out").read_bytes())
    want = _oracle_file(model, np.round(x).astype(np.float32), 24000)
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    assert got.shape == want.shape and d.max() <= 1 and (d != 0).mean() < 1e-2


def test_wav_decoder_fuzz_never_misreads(tmp_path):
    """Mutated / truncated WAV images: the decoder either fails with a message or agrees with the restatement."""
    from hypothesis import given, settings, strategies as st

    x = _signal(200, 2, seed=1)
    good = _wav_bytes(x, 44100, bits=16, extra_chunk=True)
    p = tmp_path / "f.wav"

    @settings(max_examples=200, deadline=None)
    @given(st.lists(st.tuples(st.integers(0, 79), st.integers(0, 255)), max_size=4), st.integers(-60, 0))
    def check(edits, cut):
        b = bytearray(good)
        for pos, val in edits:
            b[pos] = val                                   # the first 80 bytes hold every header field
        b = bytes(b[:len(b) + cut])
        p.write_bytes(b)
        try:
            got, rate = files.read_audio(str(p), wav=True)
        except files.NnnoiselessError as e:
            assert str(e)
            return
        try:
            want, wrate = oracle.decode_wav(b)
        except Exception:
            return                                         # the restatement is stricter about some malformed headers
        if want.shape == got.shape and wrate == rate:
            assert np.array_equal(got, want)

    check()
