"""CPU: template analysis (WakeWord._analyze_reference_audio_duration) pinned bit for bit.  Four statements of the frame
RMS agree on every frame: the exact 32-chain model (oracle/vad_model.py), the restated librosa.feature.rms
(oracle/librosa_restated.py), librosa's own lines over a strided view, and the package's host rule
(easywakeword_b200.wakeword).  The durations agree too, and the near-threshold templates the GPU tests use are shown
to separate librosa's arithmetic from a double-accumulated one."""
import numpy as np
import pytest

from easywakeword_b200.wakeword import analyze_reference_audio_duration as host_rule, template_frame_rms
from oracle import ewk_oracle as O, librosa_restated as L, vad_model as V

LENGTHS = [0, 1, 159, 160, 161, 199, 200, 201, 399, 400, 401] + [160 * k + d for k in (3, 7, 64, 257) for d in (-1, 1)]
LONG = 480_017                                              # about 30 s: 3001 frames


def librosa_lines(y):
    """librosa 0.11 feature.rms(frame_length=400, hop_length=160, center=True, pad_mode='constant') as its source reads:
    np.pad, util.frame (as_strided windows, moveaxis, slice every hop), util.abs2 -> np.square(dtype=float32),
    np.mean(axis=-2, keepdims=True), np.sqrt."""
    y = np.pad(np.asarray(y, dtype=np.float32), [(200, 200)], mode="constant")
    xw = np.lib.stride_tricks.as_strided(y, shape=(len(y) - 400 + 1, 400), strides=y.strides + y.strides)
    x = np.moveaxis(xw, -1, -2)[..., ::160]
    power = np.mean(np.square(x, dtype=np.float32), axis=-2, keepdims=True)
    return np.sqrt(power)[0]


def amplitude_classes(n, rng):
    """(name, float32 signal of length n) covering subnormal squares to above full scale, silence, impulse, DC."""
    g = rng.standard_normal(n).astype(np.float32)
    out = [(f"noise*{a:g}", (g * np.float32(a)).astype(np.float32)) for a in (1e-22, 3e-20, 1e-19, 1e-6, 0.003, 0.5, 10.0)]
    mix = g * np.float32(0.01)
    mix[rng.random(n) < 0.1] *= np.float32(1e-18)                 # tiny values among ordinary ones
    out.append(("mixed", mix.astype(np.float32)))
    out.append(("zeros", np.zeros(n, np.float32)))
    imp = np.zeros(n, np.float32)
    if n:
        imp[n // 2] = np.float32(0.7)
    out.append(("impulse", imp))
    out.append(("dc", np.full(n, np.float32(0.25))))
    out.append(("dc_odd", np.full(n, np.float32(-0.123456789))))
    return out


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def _cases():
    rng = np.random.default_rng(20261021)
    for n in LENGTHS + [LONG]:
        for name, y in amplitude_classes(n, rng):
            yield n, name, y


def test_four_statements_of_frame_rms_agree_bit_for_bit():
    frames = 0
    with np.errstate(under="ignore"):
        for n, name, y in _cases():
            m = V.frame_rms(y)
            assert len(m) == 1 + n // 160, (n, name)
            for other, what in ((L.rms(y, frame_length=400, hop_length=160)[0], "librosa_restated.rms"),
                                (librosa_lines(y), "librosa lines"), (template_frame_rms(y), "host rule")):
                assert other.dtype == np.float32, what
                assert np.array_equal(_bits(other), _bits(m)), (n, name, what, int(np.sum(_bits(other) != _bits(m))))
            frames += len(m)
    assert frames > 40_000


def test_durations_agree_with_the_model():
    with np.errstate(under="ignore"):
        for n, name, y in _cases():
            r = V.analyze(y)
            d = V.duration(y)
            assert host_rule(y) == d and O.analyze_reference_audio_duration(y) == d, (n, name)
            assert r["n_frames"] == 1 + n // 160
            if name == "zeros":
                assert not r["voiced"] and r["first_frame"] == r["last_frame"] == -1 and r["duration_s"] == 0.0
                assert r["max_rms"] == 0 and r["threshold"] == 0
            if name == "impulse" and n:
                # one sample lights up the frames whose window holds it: [p - 199, p + 200] -> 2 or 3 frames
                assert r["voiced"] and r["duration_s"] == 0.2


def test_empty_template_is_one_zero_frame_not_voiced():
    r = V.analyze(np.zeros(0, np.float32))
    assert r["n_frames"] == 1 and not r["voiced"] and r["duration_s"] == 0.0
    assert V.frame_rms(np.zeros(0, np.float32)).tolist() == [0.0]
    assert host_rule(np.zeros(0, np.float32)) is None and O.analyze_reference_audio_duration(np.zeros(0, np.float32)) is None


def test_threshold_is_float32_times_float32_tenth():
    rng = np.random.default_rng(5)
    for _ in range(200):
        y = (rng.standard_normal(int(rng.integers(400, 4000))) * rng.uniform(1e-3, 2)).astype(np.float32)
        r = V.analyze(y)
        thr = np.float32(np.float32(r["max_rms"]) * np.float32(0.1))
        assert _bits(r["threshold"]) == _bits(thr)
        rms = L.rms(y, frame_length=400, hop_length=160)[0]
        ref_thr = np.max(rms) * 0.1                              # the reference's line under NEP 50
        assert ref_thr.dtype == np.float32 and _bits(ref_thr) == _bits(thr)


def test_host_rule_takes_float64_input_as_float32():
    rng = np.random.default_rng(11)
    for k in range(40):
        y64 = rng.standard_normal(int(rng.integers(1, 30000))) * rng.uniform(1e-4, 1.0)
        y64[: int(rng.integers(0, len(y64)))] *= 1e-3
        assert host_rule(y64) == host_rule(y64.astype(np.float32)) == V.duration(y64.astype(np.float32)), k
        assert np.array_equal(_bits(template_frame_rms(y64)), _bits(V.frame_rms(y64.astype(np.float32)))), k
    for y in V.near_threshold_templates(7, 6):
        assert host_rule(y.astype(np.float64)) == host_rule(y) == V.duration(y)


def test_row_by_row_restatement_and_double_accumulation_differ_from_librosa():
    """Two arithmetics the repository used before, kept as facts: the fancy-indexed [400, F] copy that
    librosa_restated.rms once reduced row by row (it produced tests/golden/vad.npz's rms_* arrays), and K6's earlier
    double accumulation across lanes.  Each differs from librosa's pairwise float32 sum in a large share of frames."""
    from oracle.librosa_restated import frame_signal
    rng = np.random.default_rng(3)
    n_frames = n_rows = n_double = 0
    for _ in range(40):
        y = (rng.standard_normal(int(rng.integers(8000, 32000))) * rng.uniform(1e-3, 1.0)).astype(np.float32)
        m = _bits(V.frame_rms(y))
        rows = np.sqrt(np.mean(np.abs(frame_signal(np.pad(y, 200), 400, 160)) ** 2, axis=0))
        n_rows += int(np.sum(_bits(rows) != m))
        n_double += int(np.sum(_bits(V.frame_rms_double(y)) != m))
        n_frames += len(m)
    assert n_rows > 0.3 * n_frames, (n_rows, n_frames)
    assert n_double > 0.1 * n_frames, (n_double, n_frames)


def test_near_threshold_templates_change_duration_under_double_accumulation():
    """The GPU tests' near-threshold set: the model, the restated rms and the host rule agree on every template, and
    K6's earlier double accumulation gives another duration on a good share of them.  If a change to the construction
    let that share drop, the set would stop showing anything, so it is asserted here."""
    ys = V.near_threshold_templates(2026, 40)
    differ = 0
    for i, y in enumerate(ys):
        d = V.duration(y)
        assert d is not None and host_rule(y) == d and O.analyze_reference_audio_duration(y) == d, i
        r_double = V.analyze(y, rms=V.frame_rms_double(y))
        differ += r_double["duration_s"] != d
    # each pair straddles the threshold: the voiced member has the longer duration
    for lo, hi in zip(ys[0::2], ys[1::2]):
        assert V.duration(hi) > V.duration(lo)
    assert differ >= 8, (differ, len(ys))                    # 10 of these 80


@pytest.mark.parametrize("seed", [0, 1])
def test_model_chains_against_numpy_pairwise_sum_on_random_frames(seed):
    """The model's 32 chains against np.add.reduce on contiguous float32 rows of 400 (numpy's own pairwise sum)."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((4000, 400)) * np.exp(rng.uniform(-12, 3, (4000, 1)))).astype(np.float32)
    sq = x * x
    assert np.array_equal(_bits(V._chain_sums(sq)), _bits(np.add.reduce(sq, axis=1)))
