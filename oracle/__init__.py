"""ctypes binding of the CPU oracle (TEST INFRASTRUCTURE -- see oracle/nno_oracle.h).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
The product package nnnoiseless_b200 never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libnno_oracle.so")
FRAME_SIZE = 480
NB_BANDS = 22
NB_FEATURES = 42


def _cpu_stamp():
    """The Makefile uses -march=native: rebuild when the host CPU differs from the one that built the .so."""
    try:
        with open("/proc/cpuinfo") as f:
            txt = f.read()
        model = [l for l in txt.splitlines() if l.startswith("model name")][:1]
        flags = [l for l in txt.splitlines() if l.startswith("flags")][:1]
        return "|".join(model + flags)
    except OSError:
        return "unknown"


def build(force=False):
    """Compile oracle/nno_oracle.c with gcc (see oracle/Makefile)."""
    src = [os.path.join(_HERE, f) for f in ("nno_oracle.c", "nno_oracle.h", "Makefile")]
    stamp_path = os.path.join(_HERE, "_build", "cpu.stamp")
    stamp = _cpu_stamp()
    try:
        with open(stamp_path) as f:
            same_cpu = f.read() == stamp
    except OSError:
        same_cpu = False
    if (not force and same_cpu and os.path.exists(_LIB_PATH)
            and all(os.path.getmtime(_LIB_PATH) >= os.path.getmtime(s) for s in src)):
        return _LIB_PATH
    subprocess.run(["make", "-C", _HERE, "-B"], check=True, capture_output=True)
    with open(stamp_path, "w") as f:
        f.write(stamp)
    return _LIB_PATH


class Taps(C.Structure):
    _fields_ = [
        ("pitch", C.c_int32),
        ("silence", C.c_int32),
        ("vad", C.c_float),
        ("pitch_gain", C.c_float),
        ("features", C.c_float * NB_FEATURES),
        ("gains", C.c_float * NB_BANDS),
        ("ex", C.c_float * NB_BANDS),
        ("ep", C.c_float * NB_BANDS),
        ("exp", C.c_float * NB_BANDS),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.nno_model_from_bytes.restype = C.c_void_p
        L.nno_model_from_bytes.argtypes = [C.c_char_p, C.c_size_t]
        L.nno_model_free.argtypes = [C.c_void_p]
        L.nno_model_describe.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        L.nno_state_new.restype = C.c_void_p
        L.nno_state_new.argtypes = [C.c_void_p]
        L.nno_state_free.argtypes = [C.c_void_p]
        L.nno_process_frame.restype = C.c_float
        L.nno_process_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.nno_get_taps.argtypes = [C.c_void_p, C.POINTER(Taps)]
        L.nno_rfft960.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.nno_irfft960.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.nno_pitch_only.restype = C.c_int32
        L.nno_pitch_only.argtypes = [C.c_void_p, C.c_void_p]
        L.nno_set_fft_mode.argtypes = [C.c_int]
        L.nno_tansig.restype = C.c_float
        L.nno_tansig.argtypes = [C.c_float]
        L.nno_sigmoid.restype = C.c_float
        L.nno_sigmoid.argtypes = [C.c_float]
        L.nno_tansig_table.restype = C.POINTER(C.c_float)
        L.nno_run_batch.restype = C.c_double
        L.nno_run_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.nno_resample.restype = C.c_long
        L.nno_resample.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_double, C.c_void_p, C.c_long]
        L.nno_cli_frames.restype = C.c_long
        L.nno_cli_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_long]
        L.nno_train_new.restype = C.c_void_p
        L.nno_train_free.argtypes = [C.c_void_p]
        L.nno_train_set_params.argtypes = [C.c_void_p, C.c_void_p]
        L.nno_train_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.nno_train_band_lp.restype = C.c_int32
        L.nno_train_band_lp.argtypes = [C.c_int32]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Model:
    def __init__(self, data: bytes):
        self._h = lib().nno_model_from_bytes(data, len(data))
        if not self._h:
            raise ValueError("oracle: model bytes rejected")

    def describe(self):
        out = (C.c_int32 * 18)()
        lib().nno_model_describe(self._h, out)
        return [tuple(out[3 * i:3 * i + 3]) for i in range(6)]

    def __del__(self):
        if getattr(self, "_h", None):
            lib().nno_model_free(self._h)
            self._h = None


def model_accepts(data: bytes) -> bool:
    h = lib().nno_model_from_bytes(data, len(data))
    if h:
        lib().nno_model_free(h)
    return bool(h)


class State:
    def __init__(self, model: Model):
        self.model = model
        self._h = lib().nno_state_new(model._h)

    def process_frame(self, frame: np.ndarray):
        frame = np.ascontiguousarray(frame, dtype=np.float32)
        assert frame.shape == (FRAME_SIZE,)
        out = np.empty(FRAME_SIZE, np.float32)
        vad = lib().nno_process_frame(self._h, _ptr(out), _ptr(frame))
        return out, float(vad)

    def taps(self) -> Taps:
        t = Taps()
        lib().nno_get_taps(self._h, C.byref(t))
        return t

    def pitch_only(self, buf1728):
        buf = np.ascontiguousarray(buf1728, dtype=np.float32)
        assert buf.shape == (1728,)
        return int(lib().nno_pitch_only(self._h, _ptr(buf)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().nno_state_free(self._h)
            self._h = None


def tansig_table() -> np.ndarray:
    """The 201-entry table of the reference's table tanh (src/util.rs:3-27), float32 values, entry i at x = i / 25."""
    return np.ctypeslib.as_array(lib().nno_tansig_table(), shape=(201,)).copy()


def set_fft_mode(mode: int):
    """0 = the pinned f32 Stockham FFT (default), 1 = f64 DFT sums rounded once, 2 = f32 Stockham with another radix order."""
    lib().nno_set_fft_mode(int(mode))


def rfft960(x):
    x = np.ascontiguousarray(x, dtype=np.float32)
    re = np.empty(481, np.float32)
    im = np.empty(481, np.float32)
    lib().nno_rfft960(_ptr(x), _ptr(re), _ptr(im))
    return re + 1j * im


def irfft960(X):
    re = np.ascontiguousarray(X.real, dtype=np.float32)
    im = np.ascontiguousarray(X.imag, dtype=np.float32)
    out = np.empty(960, np.float32)
    lib().nno_irfft960(_ptr(re), _ptr(im), _ptr(out))
    return out


def run_batch(model: Model, x: np.ndarray, n_threads=0, want_out=True, want_taps=True):
    """x: [B][T][480] float32.  Returns dict(out, vad, pitch, seconds, threads)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    B, T, F = x.shape
    assert F == FRAME_SIZE
    out = np.empty_like(x) if want_out else None
    vad = np.empty((B, T), np.float32) if want_taps else None
    pitch = np.empty((B, T), np.int32) if want_taps else None
    used = C.c_int(0)
    secs = lib().nno_run_batch(model._h, _ptr(x), _ptr(out), _ptr(vad), _ptr(pitch), B, T, n_threads, C.byref(used))
    return dict(out=out, vad=vad, pitch=pitch, seconds=float(secs), threads=int(used.value))


class Trainer:
    """One lane of the training-data generator (src/training.rs main loop + NoiseSimulator::next_frame)."""

    def __init__(self):
        self._h = lib().nno_train_new()

    def set_params(self, params44: np.ndarray):
        """params44: one record laid out like nno_sim_params (44 bytes)."""
        buf = np.ascontiguousarray(params44)
        assert buf.nbytes == 44
        lib().nno_train_set_params(self._h, _ptr(buf))

    def frame(self, signal, noise):
        signal = np.ascontiguousarray(signal, dtype=np.float32)
        noise = np.ascontiguousarray(noise, dtype=np.float32)
        assert signal.shape == (FRAME_SIZE,) and noise.shape == (FRAME_SIZE,)
        row = np.empty(87, np.float32)
        lib().nno_train_frame(self._h, _ptr(signal), _ptr(noise), _ptr(row))
        return row

    def __del__(self):
        if getattr(self, "_h", None):
            lib().nno_train_free(self._h)
            self._h = None


def train_band_lp(lowpass: int) -> int:
    return int(lib().nno_train_band_lp(int(lowpass)))


def resample(x: np.ndarray, ratio: float) -> np.ndarray:
    """Resample::next_sample (src/nnnoiseless.rs:104-131) until dry.  x: [n][channels] -> [k][channels]."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    if x.ndim == 1:
        x = x[:, None]
    n, ch = x.shape
    cap = int(n / ratio) + 16
    out = np.empty((cap, ch), np.float32)
    k = lib().nno_resample(_ptr(x), n, ch, float(ratio), _ptr(out), cap)
    return out[:k]


def cli_frames(model: Model, x48: np.ndarray) -> np.ndarray:
    """main's frame loop (src/nnnoiseless.rs:301-330).  x48: [n][channels] float32 at 48 kHz -> int16 [m][channels]."""
    x48 = np.ascontiguousarray(x48, dtype=np.float32)
    if x48.ndim == 1:
        x48 = x48[:, None]
    n, ch = x48.shape
    out = np.empty((max(n, 1), ch), np.int16)
    m = lib().nno_cli_frames(model._h, _ptr(x48), n, ch, _ptr(out), out.shape[0])
    return out[:m]


def decode_wav(data: bytes):
    """Independent (struct-based) restatement of what hound + wav_samples (src/nnnoiseless.rs:190-228) yield:
    -> (samples [n][channels] float32, sample_rate).  Integer PCM 8/16/24/32-bit and 32-bit float."""
    import struct
    if data[:4] != b"RIFF":
        raise ValueError("no RIFF tag found")
    if data[8:12] != b"WAVE":
        raise ValueError("no WAVE tag found")
    p, fmt = 12, None
    while p + 8 <= len(data):
        cid, ln = data[p:p + 4], struct.unpack("<I", data[p + 4:p + 8])[0]
        p += 8
        if cid == b"fmt ":
            tag, ch, rate, _, align, bits = struct.unpack("<HHIIHH", data[p:p + 16])
            if tag == 0xFFFE:
                tag = struct.unpack("<H", data[p + 24:p + 26])[0]
            fmt = (tag, ch, rate, align // ch, bits)
        elif cid == b"data":
            tag, ch, rate, nbytes, bits = fmt
            raw = np.frombuffer(data[p:p + ln], np.uint8)
            n = ln // nbytes
            if tag == 3:
                v = raw[:n * 4].view("<f4").astype(np.float32) * np.float32(32767.0)
            else:
                b = raw[:n * nbytes].reshape(n, nbytes).astype(np.int64)
                if nbytes == 1:
                    s = b[:, 0] - 128
                else:
                    s = sum(b[:, i] << (8 * i) for i in range(nbytes))
                    s = np.where(s >= 1 << (8 * nbytes - 1), s - (1 << (8 * nbytes)), s)
                v = (s << (16 - bits) if bits < 16 else s >> (bits - 16)).astype(np.float32)
            return v.reshape(-1, ch), float(rate)
        p += ln + (ln & 1)
    raise ValueError("no data chunk found")
