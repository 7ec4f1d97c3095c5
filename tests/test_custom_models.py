"""The three GRU kernels on model shapes other than the built-in one.

The loader accepts any layer widths from 0 to 127 whose sizes chain and whose GRU input widths 42 + nd + nv and
42 + nv + nn fit a signed header byte (nd, nv, nn, ndn: widths of input_dense, vad_gru, noise_gru, denoise_gru).  The
shape decides which GRU kernel runs: rnn_tc.cu (tcgen05 + TMEM) when build_model_tc can pack the model into its TMEM and
shared-memory budget, rnn_mma.cu (mma.sync) when it cannot or with NNB_RNN_MMA=1, rnn.cu (FP32) with NNB_RNN_FP32=1.

* CPU: nnb_tc_pack_selftest (the host replay of the tcgen05 kernel's phases from its packed model image) over a grid of
  widths, mixed activations and both weight styles.
* GPU: a fixed list of shapes through each kernel, checked against a float64 restatement of the network
  (src/rnn.rs:251-379) fed with the GPU's own features and silence flags; a check that shapes the tcgen05 kernel
  rejects really run the mma.sync kernel; and a few shapes end to end against the C oracle.
"""
import ctypes as C
import functools
import hashlib
import itertools
import os
import time

import numpy as np
import pytest

import oracle
import nnnoiseless_b200 as nb
from conftest import synth_streams

TANH, SIGMOID, RELU = 0, 1, 2
BUILTIN_ACTS = (TANH, RELU, RELU, RELU, SIGMOID, SIGMOID)   # layer order of src/rnn.rs:189-194
TANH_ACTS = (TANH, TANH, TANH, TANH, SIGMOID, SIGMOID)
ACT_MS = 0.4   # mean square assumed for a hidden activation when sizing the scaled weights


# ---- model images ---------------------------------------------------------------------------------------------------
def layer_dims(nd, nv, nn, ndn):
    """(kind, inputs, neurons) of the six layers in file order (src/rnn.rs:189-194)."""
    return [("dense", 42, nd), ("gru", nd, nv), ("gru", 42 + nd + nv, nn), ("gru", 42 + nv + nn, ndn),
            ("dense", ndn, 22), ("dense", nv, 1)]


def legal(nd, nv, nn, ndn):
    return 42 + nd + nv <= 127 and 42 + nv + nn <= 127


@functools.lru_cache(maxsize=None)
def feature_mean_square():
    """Sum over the 42 features of their mean square on synth_streams (oracle taps; dominated by the band energies)."""
    with open(nb.BUILTIN_WEIGHTS_PATH, "rb") as f:
        m = oracle.Model(f.read())
    x = synth_streams(4, 16, seed=3).reshape(4, 16, 480)
    acc, n = 0.0, 0
    for s in range(4):
        st = oracle.State(m)
        for t in range(16):
            st.process_frame(x[s, t])
            acc += float((np.array(st.taps().features, np.float64) ** 2).sum())
            n += 1
    return acc / n


def make_model(nd, nv, nn, ndn, acts=TANH_ACTS, seed=0, scale="scaled"):
    """A model image that RnnModel::from_bytes accepts: per layer the header [ni, nn, act], the int8 weights
    ([ni][nn] dense, [ni][3 nn] and [nn][3 nn] for a GRU, gate order z | r | h) and the biases.

    scale="scaled": weights and biases ~ N(0, sigma) rounded and clipped to +-127, sigma per layer such that a
    pre-activation (bias + sum of weight * input) / 256 has unit variance on synth_streams features and hidden
    activations of mean square ACT_MS -- gates stay away from saturation, where a packing error would hide.
    scale="full": uniform integers in [-127, 127], like the built-in model (whose weights have p99 = 127)."""
    assert legal(nd, nv, nn, ndn)
    rng = np.random.default_rng(seed)
    fms = feature_mean_square() if scale == "scaled" else 0.0
    # mean square of the inputs of each layer: features, then hidden activations
    in_ms = [fms, nd * ACT_MS, (nd + nv) * ACT_MS + fms, (nv + nn) * ACT_MS + fms, ndn * ACT_MS, nv * ACT_MS]
    out = bytearray()
    for (kind, ni, n), act, ms in zip(layer_dims(nd, nv, nn, ndn), acts, in_ms):
        out += bytes([ni, n, act])
        cnt = ni * n + n if kind == "dense" else 3 * n * ni + 3 * n * n + 3 * n
        if scale == "full":
            v = rng.integers(-127, 128, cnt)
        else:
            rec = n * ACT_MS if kind == "gru" else 0.0
            sigma = 256.0 / np.sqrt(ms + rec + 1.0)
            v = np.clip(np.rint(rng.normal(0.0, sigma, cnt)), -127, 127)
        out += v.astype(np.int8).tobytes()
    data = bytes(out)
    assert oracle.model_accepts(data), (nd, nv, nn, ndn)
    assert nb.RnnModel.from_bytes(data) is not None, (nd, nv, nn, ndn)
    return data


def parse_model(data):
    """Model image -> list of (kind, act, W or (W, R), bias) as float64, W [ni][n] / [ni][3n], R [n][3n]."""
    b = np.frombuffer(data, np.int8)
    p, layers = 0, []
    for kind in ("dense", "gru", "gru", "gru", "dense", "dense"):
        ni, n, act = int(b[p]), int(b[p + 1]), int(b[p + 2])
        p += 3
        g = 1 if kind == "dense" else 3
        w = b[p:p + g * n * ni].astype(np.float64).reshape(ni, g * n); p += g * n * ni
        r = None
        if kind == "gru":
            r = b[p:p + 3 * n * n].astype(np.float64).reshape(n, 3 * n); p += 3 * n * n
        bias = b[p:p + g * n].astype(np.float64); p += g * n
        layers.append((kind, act, w, r, bias))
    assert p == len(b)
    return layers


# ---- float64 restatement of the network (src/rnn.rs:251-379, src/util.rs:3-53) -------------------------------------
@functools.lru_cache(maxsize=None)
def _table():
    return oracle.tansig_table().astype(np.float64)


def tansig(x):
    """The reference's table tanh (src/util.rs:29-45), evaluated in float64."""
    tab = _table()
    ax = np.minimum(np.abs(x), 8.0)
    i = np.floor(0.5 + 25.0 * ax)
    d = ax - 0.04 * i
    y = tab[i.astype(np.int64)]
    y = np.where(x < 0, -1.0, 1.0) * (y + d * (1.0 - y * y) * (1.0 - y * d))
    return np.where(~(x < 8.0), 1.0, np.where(~(x > -8.0), -1.0, y))


def activate(act, x):
    if act == TANH:
        return tansig(x)
    if act == SIGMOID:
        return 0.5 + 0.5 * tansig(0.5 * x)
    return np.maximum(x, 0.0)


class Reference:
    """The network on a batch of streams in float64, with its own float64 GRU state."""

    def __init__(self, data, n_streams):
        self.L = parse_model(data)
        self.h = [np.zeros((n_streams, self.L[k][4].size // 3)) for k in (1, 2, 3)]
        self.lastg = np.zeros((n_streams, 22))

    def _dense(self, k, x):
        _, act, w, _, b = self.L[k]
        return activate(act, (b + x @ w) / 256.0)

    def _gru(self, k, x, h):
        _, act, w, r, b = self.L[k]
        n = h.shape[1]
        zr = (b[:2 * n] + x @ w[:, :2 * n] + h @ r[:, :2 * n]) / 256.0
        z, rg = activate(SIGMOID, zr[:, :n]), activate(SIGMOID, zr[:, n:])
        c = activate(act, (b[2 * n:] + x @ w[:, 2 * n:] + (rg * h) @ r[:, 2 * n:]) / 256.0)  # reset before the product
        return z * h + (1.0 - z) * c

    def step(self, feat, silent):
        """feat [B][42], silent [B] bool -> gains [B][22], vad [B]; silent streams keep their state and get vad 0.
        The gains are those the taps report: the network's, floored at 0.6 x the previous frame's (src/denoise.rs:107),
        a 1-Lipschitz map that passes any error of the network's through."""
        f = feat.astype(np.float64)
        hv, hn, hd = self.h
        d = self._dense(0, f)
        nv = self._gru(1, d, hv)
        vad = self._dense(5, nv)[:, 0]
        nn_ = self._gru(2, np.concatenate([d, nv, f], 1), hn)
        nd_ = self._gru(3, np.concatenate([nv, nn_, f], 1), hd)
        gains = np.maximum(self._dense(4, nd_), 0.6 * self.lastg)
        keep = silent[:, None]
        self.h = [np.where(keep, o, n) for o, n in zip(self.h, (nv, nn_, nd_))]
        self.lastg = np.where(keep, self.lastg, gains)
        return gains, np.where(silent, 0.0, vad)


def pack_selftest(data, seed=0):
    L = nb.lib()
    L.nnb_tc_pack_selftest.restype = C.c_double
    L.nnb_tc_pack_selftest.argtypes = [C.c_char_p, C.c_size_t, C.c_int]
    return L.nnb_tc_pack_selftest(data, len(data), seed)


# ---- CPU: the tcgen05 packing over a grid of shapes -----------------------------------------------------------------
SWEEP_WIDTHS = (0, 1, 3, 7, 8, 9, 15, 16, 17, 24, 31, 32, 48, 56, 57, 63, 64, 65, 72, 85, 96, 97, 127)


def sweep_shapes():
    """Every legal (nd, nv, nn) over SWEEP_WIDTHS, each with two denoise widths taken in turn from the same list (the
    full product is ~100,000 shapes); plus the shapes the GPU tests use."""
    out = set(s for s, _ in GPU_SHAPES)
    k = 0
    for nd, nv, nn in itertools.product(SWEEP_WIDTHS, repeat=3):
        if legal(nd, nv, nn, 0):
            for j in (0, 11):
                out.add((nd, nv, nn, SWEEP_WIDTHS[(k + j) % len(SWEEP_WIDTHS)]))
            k += 1
    return sorted(out)


def test_tcgen05_packing_sweep():
    """For every shape: the tcgen05 packing either refuses the model (-2: the mma.sync kernel runs it) or its host replay
    equals the direct evaluation within 2e-5.  Activations are mixed (relu included) and a third of the models use
    full-range weights."""
    t0 = time.time()
    shapes = sweep_shapes()
    bad, n_tc = [], 0
    for i, shp in enumerate(shapes):
        rng = np.random.default_rng(i)
        acts = tuple(int(a) for a in rng.integers(0, 3, 6))
        data = make_model(*shp, acts=acts, seed=i, scale="full" if i % 3 == 0 else "scaled")
        e = pack_selftest(data, seed=i)
        if e == -2.0:
            continue
        n_tc += 1
        if not 0.0 <= e < 2e-5:
            bad.append((shp, acts, e))
    print("packing sweep: %d shapes, %d on tcgen05, %d failing, %.1f s" % (len(shapes), n_tc, len(bad), time.time() - t0))
    assert len(shapes) > 8000 and n_tc > 0.5 * len(shapes)
    no_chunk = [b for b in bad if b[2] == -3.0]
    wrong = [b for b in bad if b[2] != -3.0]
    assert not bad, ("%d shapes with a phase whose MMA is missing or has N = 0 (-3), first: %s; %d shapes with a replay "
                     "error, noise widths %s, first: %s" % (len(no_chunk), [b[0] for b in no_chunk[:8]], len(wrong),
                                                            sorted(set(b[0][2] for b in wrong)), wrong[:4]))


def test_make_model_matches_loader():
    """The generator writes what the loader reads: the same image back, the same layer headers as the oracle sees."""
    data = make_model(13, 31, 19, 22, acts=BUILTIN_ACTS, seed=5)
    assert nb.RnnModel.from_bytes(data).to_bytes() == data
    dims = [(ni, n) for _, ni, n in layer_dims(13, 31, 19, 22)]
    assert oracle.Model(data).describe() == [d + (a,) for d, a in zip(dims, BUILTIN_ACTS)]
    assert [w.shape for _, _, w, _, _ in parse_model(data)] == [(42, 13), (13, 93), (86, 57), (92, 66), (22, 22), (31, 1)]


# ---- GPU ------------------------------------------------------------------------------------------------------------
GPU_SHAPES = [
    ((24, 24, 48, 96), "the built-in shape (and activations) with random weights"),
    ((1, 1, 1, 1), "one neuron per layer: every phase is one padded tile"),
    ((0, 0, 0, 0), "every layer empty: the gains come from the output bias alone"),
    ((0, 0, 48, 96), "no dense or vad layer: nothing feeds vad_output"),
    ((24, 24, 48, 0), "no denoise GRU: nothing feeds denoise_output"),
    ((13, 31, 19, 22), "widths that are not multiples of 4: unaligned state rows"),
    ((8, 8, 64, 8), "noise width 64: its candidate met vad_output's accumulators"),
    ((16, 16, 60, 16), "noise width 60, the same overlap"),
    ((24, 24, 61, 24), "noise width 61, the same overlap"),
    ((8, 8, 72, 8), "noise width 72"),
    ((24, 24, 48, 127), "denoise width 127: beyond the tcgen05 budget"),
    ((43, 42, 43, 127), "the widest legal GRU inputs: beyond the tcgen05 budget"),
    ((85, 0, 85, 64), "widest dense and noise layers, no vad GRU: beyond the tcgen05 budget"),
    ((0, 1, 73, 89), "fits the TMEM columns, not the 227 KB of shared memory: beyond the tcgen05 budget"),
    ((32, 32, 32, 32), "every width a multiple of 16"),
    ((31, 17, 40, 56), "relu dense layer and relu GRU candidates"),
]
FALLBACK_SHAPES = [(24, 24, 48, 127), (43, 42, 43, 127), (85, 0, 85, 64), (0, 1, 73, 89)]   # the mma.sync kernel's
GPU_ACTS = {(24, 24, 48, 96): BUILTIN_ACTS, (31, 17, 40, 56): (RELU, RELU, RELU, RELU, SIGMOID, SIGMOID)}
KERNELS = {"default": {}, "mma": {"NNB_RNN_MMA": "1"}, "fp32": {"NNB_RNN_FP32": "1"}}
B_GPU, T_GPU = 161, 24   # one full 128-stream tcgen05 tile + a partial one of 33; not a multiple of 32
ISOLATED_ATOL = 1e-4


def gpu_model(shape):
    return make_model(*shape, acts=GPU_ACTS.get(shape, TANH_ACTS), seed=sum(shape) + 7 * shape[2])


@functools.lru_cache(maxsize=None)
def gpu_input():
    """[T][B][480]: synth_streams; every fourth stream is quiet (1/512) for frames 0-7 and digital zeros for frames
    8-15, so it goes silent mid-run (the GRU state must then stay untouched) and comes back at frame 16."""
    x = synth_streams(B_GPU, T_GPU, seed=606).reshape(B_GPU, T_GPU, 480)
    x[3::4, :8] *= 1.0 / 512.0
    x[3::4, 8:16] = 0.0
    return np.ascontiguousarray(x.transpose(1, 0, 2))


def _batch(data, n_streams, env):
    os.environ.update(env)
    try:
        return nb.DenoiseBatch(n_streams, nb.RnnModel.from_bytes(data))
    finally:
        for k in env:
            del os.environ[k]


@functools.lru_cache(maxsize=None)
def gpu_run(shape, kernel):
    """Frame by frame through one kernel: features, silence, gains and vad of every frame, and a digest of the output."""
    data = gpu_model(shape)
    b = _batch(data, B_GPU, KERNELS[kernel])
    x = gpu_input()
    feats, sil, gains, vads, h = [], [], [], [], hashlib.sha256()
    for t in range(T_GPU):
        o, v = b.process_host(x[t:t + 1])
        tp = b.taps()
        feats.append(tp["features"].copy()); sil.append(tp["silence"].astype(bool)); gains.append(tp["gains"].copy())
        vads.append(v[0].copy())
        h.update(o.tobytes())
    return dict(features=np.stack(feats), silence=np.stack(sil), gains=np.stack(gains), vad=np.stack(vads), out=h.hexdigest())


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("shape", [s for s, _ in GPU_SHAPES], ids=lambda s: "x".join(map(str, s)))
def test_gru_kernel_against_float64(shape, kernel):
    """Gains and VAD of every non-silent frame within ISOLATED_ATOL of the float64 network run on the GPU's own
    features and silence flags (so the FFT's rounding cancels out); silent frames return VAD 0."""
    r = gpu_run(shape, kernel)
    sil = r["silence"]
    assert sil[:, 3::4].any() and not sil[:, 0::4].any()   # the quiet streams went silent, the loud ones never
    ref = Reference(gpu_model(shape), B_GPU)
    worst_g = worst_v = 0.0
    for t in range(T_GPU):
        g, v = ref.step(r["features"][t], sil[t])
        live = ~sil[t]
        dg, dv = np.abs(r["gains"][t][live] - g[live]), np.abs(r["vad"][t][live] - v[live])
        assert np.isfinite(dg).all() and np.isfinite(dv).all(), t   # a NaN must fail, not vanish in max()
        worst_g = max([worst_g, *dg.ravel()])
        worst_v = max([worst_v, *dv.ravel()])
        assert np.all(r["vad"][t][sil[t]] == 0.0), t
    print("isolated %-14s %-7s worst |gain| %.3g  worst |vad| %.3g  (tcgen05 self-test %g)"
          % ("x".join(map(str, shape)), kernel, worst_g, worst_v, pack_selftest(gpu_model(shape))))
    assert worst_g <= ISOLATED_ATOL and worst_v <= ISOLATED_ATOL


def test_gpu_shapes_kernel_choice():
    """Which GPU shapes the tcgen05 packing refuses is exactly FALLBACK_SHAPES; its replay passes on all the others."""
    e = {s: pack_selftest(gpu_model(s)) for s, _ in GPU_SHAPES}
    assert sorted(s for s in e if e[s] == -2.0) == sorted(FALLBACK_SHAPES)
    assert all(0.0 <= e[s] < 2e-5 for s in e if s not in FALLBACK_SHAPES), e


@pytest.mark.gpu
@pytest.mark.parametrize("shape", FALLBACK_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_default_kernel_is_mma_when_tcgen05_refuses(shape):
    """A model the tcgen05 packing refuses runs on the mma.sync kernel: the default handle gives the NNB_RNN_MMA=1
    handle's output and VAD bit for bit."""
    assert pack_selftest(gpu_model(shape)) == -2.0
    a, b = gpu_run(shape, "default"), gpu_run(shape, "mma")
    assert a["out"] == b["out"] and np.array_equal(a["vad"], b["vad"])


E2E_SHAPES = [(13, 31, 19, 22), (8, 8, 64, 8), (32, 32, 32, 32), (43, 42, 43, 127)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", E2E_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_custom_model_end_to_end_against_oracle(shape):
    """The whole frame path with a custom model against the C oracle: pitch bit-exact, output rel-RMS <= 1e-5, VAD
    within 1e-4.  Every fourth stream starts with 8 frames of digital silence."""
    from test_gpu_parity import check_against_oracle
    data = gpu_model(shape)
    x = synth_streams(B_GPU, T_GPU, seed=707).reshape(B_GPU, T_GPU, 480)
    x[3::4, :8] = 0.0
    ref = oracle.run_batch(oracle.Model(data), x, n_threads=0)
    b = nb.DenoiseBatch(B_GPU, nb.RnnModel.from_bytes(data))
    outs, vads, pitches = [], [], []
    for t in range(T_GPU):
        o, v = b.process_host(np.ascontiguousarray(x[:, t][None]))
        outs.append(o[0]); vads.append(v[0]); pitches.append(b.taps()["pitch"].copy())
    assert np.array_equal(np.stack(pitches, 1), ref["pitch"])
    check_against_oracle(np.stack(outs), np.stack(vads), None, ref, x)
