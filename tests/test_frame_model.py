"""CPU: the exact float32 model of K3 (oracle/frame_model.py).  Its tables are the device's own (the probe's host image
equals ewk_host_table and the oracle's tables); with the stand-in log it sits far inside the device tests' old
tolerances against the float64 oracle; its loader classifier equals a brute-force restatement of the kernel's tests;
each FMA contraction site it restates is pinned (inputs exist where the other readings give other bits); and the faults
that pass the old tolerances change its bits."""
import numpy as np
import pytest
import scipy.fft

from helpers import K3Probe, mfcc_rel_l2
from oracle import ewk_oracle as O
from oracle import frame_model as M
from oracle import librosa_restated as L
from oracle.resample_restated import fmaf32


@pytest.fixture(scope="module")
def tables(tmp_path_factory):
    img, sizes = K3Probe(tmp_path_factory.mktemp("k3_probe")).tables()
    assert sizes == (M.DEVICE_TABLES.itemsize, M.FRAME_IMAGE_OFFSET, M.FRAME_TABLES.itemsize)
    return M.Tables.from_image(img)


@pytest.fixture(scope="module")
def inputs(golden_matcher):
    g = golden_matcher
    return {n: g[f"in_{n}"].astype(np.float32) for n in ("word", "speech_like", "noise42", "stream_3s_i16")}


def test_tables_match_library_and_oracle(tables):
    from easywakeword_b200 import _lib
    t = tables.flat
    assert np.array_equal(t["hann"], _lib.host_table(0))
    assert np.array_equal(tables.mel_dense(), _lib.host_table(1).reshape(128, 257))
    assert np.array_equal(t["dct_t"].reshape(128, 20).T, _lib.host_table(2).reshape(20, 128))
    assert np.array_equal(t["hann"], L.hann_window().astype(np.float32))
    assert np.array_equal(tables.mel_dense(), L.mel_filterbank())
    dct = scipy.fft.dct(np.eye(128), type=2, norm="ortho", axis=0)[:20]
    assert np.abs(t["dct_t"].reshape(128, 20).T - dct).max() < 1e-7
    m = np.arange(256)
    assert np.abs(t["w256"][:, 0] + 1j * t["w256"][:, 1] - np.exp(-2j * np.pi * m / 256)).max() < 1e-7
    assert np.array_equal(tables.hw.reshape(-1), t["hann"])                          # lane layout of the window
    assert tables.ft["n_mfcc"] == 20 and tables.ft["preemph"] == 0


def segment_with(y, T, fault=None, log_fn=M.log_mel_standin):
    """The model's pipeline with an optional fault applied to the loaded frames."""
    x = M.frame_samples(y)
    if fault is not None:
        x = fault(x.copy())
    lm = M.log_mel(M.power_spectrum(x, T), T, log_fn)
    floor = np.float32(lm.max()) - np.float32(80.0)
    mf = M.dct20(np.maximum(lm, floor), T)
    mean, std = M.pool(mf)
    return mf, mean, std


def test_model_against_float64_oracle(tables, inputs):
    """The stand-in-log model against the float64 oracle: worst per-frame relative L2 and worst score error."""
    tm, ts = M.segment(inputs["word"], tables)["mean"], M.segment(inputs["word"], tables)["std"]
    om, os_ = O.extract_mfcc(inputs["word"])
    worst_l2, worst_score = 0.0, 0.0
    for name, y in inputs.items():
        r = M.segment(y, tables)
        worst_l2 = max(worst_l2, float(mfcc_rel_l2(r["frames"].T, O.mfcc_frames(y)).max()))
        cm, cs = O.extract_mfcc(y)
        with np.errstate(all="ignore"):
            ref = float(O.similarity_from_features(om, os_, cm, cs))
        worst_score = max(worst_score, abs(float(M.score(tm, ts, r["mean"], r["std"])) - ref))
    print(f"model vs float64 oracle: worst per-frame rel. L2 {worst_l2:.2e}, worst score error {worst_score:.2e}")
    assert worst_l2 < 2e-6 and worst_score < 1e-3


def test_preemphasis_and_n_mfcc_against_oracle(tables, inputs):
    y = inputs["speech_like"]
    for pre, n in ((0.97, 13), (0.5, 1)):
        r = M.segment(y, tables, preemphasis=pre, n_mfcc=n)
        ref = O.mfcc_frames(y, pre, 20)
        assert mfcc_rel_l2(r["frames"].T, ref).max() < 2e-6
        m, s = O.extract_mfcc(y, pre, 20)
        assert np.allclose(r["mean"][:n], m[:n], rtol=1e-5, atol=1e-4) and not r["mean"][n:].any() and not r["std"][n:].any()


def brute_branch(start, length, ring, fmt, aligned, t):
    """PcmReader.fast_base / odd_base and load_frame_pairs_raw's even test, statement by statement."""
    f0 = 160 * t - 256
    q = fmt == "i16"

    def base(odd):
        if f0 < 0 or f0 + 512 > length:
            return -1
        p = start + f0
        if ring:
            if p >= ring:
                p -= ring
            if p + 512 > ring:
                return -1
        if (p & 1) != odd:
            return -1
        if not odd:
            return p if aligned else -1
        if q:
            if not aligned:
                return -1
            if not ring and f0 + 513 > length:
                return -1
        return p
    if base(0) >= 0:
        return M.FAST
    if base(1) >= 0:
        return M.ODD
    p00 = start + f0
    even = (p00 & 1) == 0 and (ring == 0 or (ring & 1) == 0) and aligned
    if even and ring:
        return M.MASKED_RING
    if even:
        return M.MASKED_LINEAR
    return M.SCALAR


def test_loader_classifier():
    rng = np.random.default_rng(1)
    seen = set()
    for _ in range(400):
        ring = int(rng.choice([0, 0, 2048, 4096, 176000]))
        length = int(rng.integers(1, 4000 if ring == 0 else min(ring, 4000)))
        start = int(rng.integers(0, ring if ring else 5000))
        fmt, aligned = str(rng.choice(["f32", "i16"])), bool(rng.integers(0, 4) > 0)
        t = np.arange(1 + length // 160)
        got = M.loader_branch(start, length, ring, fmt, aligned, t)
        want = [brute_branch(start, length, ring, fmt, aligned, int(i)) for i in t]
        assert list(got) == want, (start, length, ring, fmt, aligned)
        seen |= set(want)
    assert seen == {M.FAST, M.ODD, M.MASKED_RING, M.MASKED_LINEAR, M.SCALAR}


def differs(*vals):
    """True when every pair of the given arrays differs somewhere."""
    return all(not np.array_equal(a, b) for i, a in enumerate(vals) for b in vals[i + 1:])


def test_contraction_sites_are_pinned():
    """For every site the model fuses, the SASS reading, the unfused form and the other fusion give different bits on
    ordinary inputs, so that a wrong reading fails the device tests."""
    rng = np.random.default_rng(2)
    a, b, c, d = (rng.standard_normal(20000).astype(np.float32) for _ in range(4))
    # Hann into the first butterfly: fma(x, h, fl(x4 h4)) vs fl(x h) + fl(x4 h4) vs fma(x4, h4, fl(x h))
    assert differs(fmaf32(a, b, c * d), a * b + c * d, fmaf32(c, d, a * b))
    # cmul re = fma(ax, bx, -fl(ay by)), im = fma(ay, bx, fl(ax by)); the untangle and the power have the same shapes
    assert differs(fmaf32(a, b, -(c * d)), a * b - c * d, fmaf32(-c, d, a * b))
    assert differs(fmaf32(c, b, a * d), c * b + a * d, fmaf32(a, d, c * b))
    assert differs(fmaf32(a, a, c * c), a * a + c * c, fmaf32(c, c, a * a))
    # Chan merge: fl(M2 + fma(fl(d d), q, part)) vs fl(M2 + fl(fl(d d) q) + part)
    q, part, M2 = np.abs(b), np.abs(c), np.abs(d)
    assert differs(M2 + fmaf32(a * a, q, part), M2 + ((a * a) * q + part))


def test_model_sites_reach_the_output(tables, inputs):
    """The model's fused multiply-adds reach its output: computed unfused, its frames change."""
    y = inputs["speech_like"]
    base = M.segment(y, tables)["frames"]
    orig = M.fmaf32
    try:
        M.fmaf32 = lambda x, y_, z: (np.asarray(x, np.float32) * np.asarray(y_, np.float32)) + np.asarray(z, np.float32)
        unfused = M.segment(y, tables)["frames"]
    finally:
        M.fmaf32 = orig
    assert not np.array_equal(base, unfused)


def test_faults_change_bits_within_old_tolerances(tables, inputs):
    """Faults of the size the old tolerances cannot see change the model's bits.  Frame samples 1 and 511 read as 0,
    and TEN_LOG10_2 one float32 ulp low stay within 1e-4 per-frame relative L2 of the float64 oracle; these two, frame
    sample 2 read as 0 and the Hann taps shifted by one sample all move no score by 0.01."""
    def z(*idx):
        def f(x):
            x[:, list(idx)] = 0.0
            return x
        return f

    def coarse_log(S):
        x = np.maximum(np.asarray(S, np.float32), np.float32(1e-10))
        return (np.nextafter(M.TEN_LOG10_2, np.float32(0)) * np.log2(x.astype(np.float64)).astype(np.float32)).astype(np.float32)
    assert np.float32(3.0103) == M.TEN_LOG10_2, "3.0103f is the same float32 as 10 log10(2): no fault at all"
    ft = tables.ft.copy()
    ft["hw"] = np.roll(tables.flat["hann"], 1).reshape(256, 2)
    shifted = M.Tables(tables.flat, ft)
    faults = {"samples 1, 511 zero": dict(fault=z(1, 511)), "sample 2 zero": dict(fault=z(2)),
              "TEN_LOG10_2 one ulp low": dict(log_fn=coarse_log), "Hann shifted by one": dict(T=shifted)}
    tm, ts = M.segment(inputs["word"], tables)["mean"], M.segment(inputs["word"], tables)["std"]
    for name, kw in faults.items():
        worst_l2, worst_score, changed = 0.0, 0.0, False
        for y in (inputs["word"], inputs["speech_like"], inputs["noise42"]):
            mf0, m0, s0 = segment_with(y, tables)
            mf, m, s = segment_with(y, kw.get("T", tables), kw.get("fault"), kw.get("log_fn", M.log_mel_standin))
            changed |= not np.array_equal(mf, mf0) or not np.array_equal(m, m0)
            worst_l2 = max(worst_l2, float(mfcc_rel_l2(mf.T, O.mfcc_frames(y)).max()))
            with np.errstate(all="ignore"):
                worst_score = max(worst_score, abs(float(M.score(tm, ts, m, s)) - float(M.score(tm, ts, m0, s0))))
        print(f"{name}: worst per-frame rel. L2 vs oracle {worst_l2:.1e}, worst score change {worst_score:.1e}")
        assert changed, name
        assert worst_score < 0.01, name
        if name in ("samples 1, 511 zero", "TEN_LOG10_2 one ulp low"):
            assert worst_l2 < 1e-4, name
