"""CPU: pin oracle/ (the checker) against the reference-generated goldens and the reference's
own known-answer tests for this path (SURVEY §8(c))."""
import os

import numpy as np
import pytest

from oracle import ewk_oracle as O
from oracle import librosa_restated as L
from easywakeword_b200 import synth
from helpers import detect_stream_for, sha

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- Appendix A anchors of the restated front-end ---------------------------------------
def test_mel_filterbank_anchors():
    M = L.mel_filterbank()
    assert M.shape == (128, 257) and M.dtype == np.float32
    assert int((M > 0).sum()) == 504
    assert np.unravel_index(M.argmax(), M.shape) == (3, 3)
    assert abs(float(M.max()) - 0.042366076) < 1e-9
    assert abs(float(L.hz_to_mel(8000.0)) - 45.245640471924965) < 1e-12
    nnz = (M > 0).sum(axis=1)
    assert nnz.min() == 1 and nnz.max() == 12


def test_mel_and_dct_against_torchaudio():
    ta = pytest.importorskip("torchaudio")
    import scipy.fft
    fb = ta.functional.melscale_fbanks(257, 0.0, 8000.0, 128, 16000, norm="slaney", mel_scale="slaney").T.numpy()
    assert np.abs(fb - L.mel_filterbank()).max() < 1e-6
    d = ta.functional.create_dct(20, 128, "ortho").T.numpy()
    D = scipy.fft.dct(np.eye(128), axis=0, type=2, norm="ortho")[:20]
    assert np.abs(D - d).max() < 1e-5


def test_hann_window():
    w = L.hann_window(512)
    assert w[0] == 0 and abs(w[256] - 1) < 1e-15 and abs(w.sum() - 256) < 1e-9 and abs((w ** 2).sum() - 192) < 1e-9


def test_bundled_word_anchor(word):
    assert len(word) == 15503
    m = L.mfcc(word)
    assert m.shape == (20, 97) and m.dtype == np.float32
    np.testing.assert_allclose(m.mean(1)[:4], [-530.33685, 98.579170, -19.178118, 25.856405], rtol=2e-6)


# ---- reference known-answer tests (tests/test_wakeword_simulated.py:104-205, 330-360) ----
@pytest.mark.parametrize("sig", ["sine440", "speech_like"])
def test_self_similarity_is_exactly_100(sig, golden_matcher):
    a = golden_matcher[f"in_{sig}"]
    m = O.WordMatcherOracle()
    m.set_reference(a)
    ok, sim = m.matches(a)
    assert ok and sim == 100.0


def test_reference_inequalities(golden_matcher):
    m = O.WordMatcherOracle()
    m.set_reference(golden_matcher["in_sine440"])
    assert m.matches(golden_matcher["in_sine880"])[1] < 100.0
    assert m.matches(golden_matcher["in_noise42"])[1] < 100.0
    assert m.matches(golden_matcher["in_sine440_half"])[1] > 50.0
    # LEARNINGS.md:92-93 doc pins ("89 %+", "77 %+")
    assert 89.0 < m.matches(golden_matcher["in_sine880"])[1] < 90.5
    assert 77.0 < m.matches(golden_matcher["in_noise42"])[1] < 79.0


def test_no_reference_raises():
    with pytest.raises(ValueError, match="No reference word set"):
        O.WordMatcherOracle().calculate_similarity(np.zeros(16000, np.float32))


# ---- oracle == reference (goldens written by the reference's classes) ---------------------
def test_matcher_equals_reference_goldens(golden_matcher, word):
    g = golden_matcher
    tpl = {"word": word, "sine440": g["in_sine440"], "speech_like": g["in_speech_like"]}
    ms = {}
    for k, a in tpl.items():
        ms[k] = O.WordMatcherOracle()
        ms[k].set_reference(a)
        assert np.array_equal(ms[k].reference_mfcc_mean, g[f"tpl_{k}_mean"])
        assert np.array_equal(ms[k].reference_mfcc_std, g[f"tpl_{k}_std"])
    for name in g["names"]:
        a = g[f"in_{name}"]
        mean, std = O.extract_mfcc(a)
        assert np.array_equal(mean, g[f"mean_{name}"], equal_nan=True), name
        assert np.array_equal(std, g[f"std_{name}"], equal_nan=True), name
        assert np.array_equal(O.mfcc_frames(a), g[f"mfcc_{name}"]), name
        assert g[f"mfcc_{name}"].shape == (20, 1 + len(a) // 160)
        for k in tpl:
            ok, sim = ms[k].matches(a)
            assert np.array_equal(np.float64(sim), g[f"score_{k}_{name}"], equal_nan=True), (k, name)
            assert bool(ok) == bool(g[f"match_{k}_{name}"])


def test_detect_equals_reference_goldens(golden_detect, word):
    g, cases = golden_detect
    n_events = n_nomatch = 0
    for c in cases:
        n = c["name"]
        s = detect_stream_for(c, word)
        assert sha(s) == str(g[f"{n}_stream_sha"]), f"synthetic stream for {n} drifted"
        o = O.detect_stream(s, word, block=c["block"], fast=True, **c["params"])
        assert o["full_tick"] == int(g[f"{n}_full_tick"])
        assert o["ticks_run"] == int(g[f"{n}_ticks_run"])
        assert np.array_equal(o["trace_tick"], g[f"{n}_trace_tick"])
        assert np.array_equal(o["trace_silent"], g[f"{n}_trace_silent"])
        assert np.array_equal(o["trace_thr"], g[f"{n}_trace_thr"])
        assert [e["tick"] for e in o["events"]] == list(g[f"{n}_ev_tick"])
        assert [e["seg_len"] for e in o["events"]] == list(g[f"{n}_ev_len"])
        assert np.array_equal(np.array([e["score"] for e in o["events"]]), g[f"{n}_ev_score"])
        assert [e["matched"] for e in o["events"]] == list(g[f"{n}_ev_match"])
        assert o["timeouts"] == list(g[f"{n}_timeouts"])
        n_events += len(o["events"])
        n_nomatch += sum(not e["matched"] for e in o["events"])
    assert n_events >= 50 and n_nomatch >= 8


def test_config1_expected_events(golden_detect):
    """SURVEY §8(d) config 1: ring full at tick 101, one level-2 call at tick 156, 17 600 samples, 99.5034."""
    g, _ = golden_detect
    assert int(g["config1_full_tick"]) == 101
    assert list(g["config1_ev_tick"]) == [156] and list(g["config1_ev_len"]) == [17600]
    assert abs(float(g["config1_ev_score"][0]) - 99.5034) < 1e-3 and bool(g["config1_ev_match"][0])


def test_slow_and_fast_threshold_paths_identical(word):
    c = dict(seed=2004, seconds=30, noise=0.012, gain=(2.0, 5.0))
    s = detect_stream_for(c, word)
    a = O.detect_stream(s, word, block=512, fast=False, max_ticks=200)
    b = O.detect_stream(s, word, block=512, fast=True, max_ticks=200)
    assert np.array_equal(a["trace_thr"], b["trace_thr"]) and np.array_equal(a["trace_silent"], b["trace_silent"])


def test_dense_equals_reference_goldens(golden_dense, word):
    g = golden_dense
    tpls = [word, g["tpl2"]]
    for si in range(2):
        x, _ = synth.stream(int(g[f"s{si}_seed"]), 12.0, word, gain=(1.0, 4.0), zero_gaps=int(g[f"s{si}_zero_gaps"]))
        x = synth.from_int16(synth.to_int16(x))
        assert sha(x) == str(g[f"s{si}_sha"])
        hops = g[f"s{si}_hops"][::6]
        sc = O.dense_scores(x, tpls, hops)
        np.testing.assert_array_equal(sc.astype(np.float64), g[f"s{si}_scores"][::6])


def test_level3_preprocessing_and_vad(word):
    y = O.prepare_for_level3(word.astype(np.float64) + 0.01)
    assert abs(np.max(np.abs(y)) - 1.0) < 1e-12 and abs(np.mean(np.clip(y, -1, 1))) < 0.05
    assert O.analyze_reference_audio_duration(word) == pytest.approx(0.69)
    assert O.auto_speech_durations(word) == (pytest.approx(0.69), pytest.approx(1.38))
    assert O.auto_speech_durations(word, user_min=0.5) == (0.5, 1.0)
    assert O.auto_speech_durations(np.zeros(100, np.float32)) [1] >= O.auto_speech_durations(np.zeros(100, np.float32))[0] > 0


def test_full_mfcc_front_end_against_torchaudio(word):
    """Independent implementation of the whole librosa.feature.mfcc chain: torchaudio.transforms.MFCC configured with
    librosa's defaults (periodic Hann, center + zero padding, power 2, Slaney mel/norm, power_to_db with the global
    top_db=80 floor, ortho DCT-II).  Agreement to ~1e-6 per-frame relative L2 pins the restated librosa layer to a
    second code base, including the floor path (digital-silence padding)."""
    torch = pytest.importorskip("torch")
    ta = pytest.importorskip("torchaudio")
    tr = ta.transforms.MFCC(sample_rate=16000, n_mfcc=20, dct_type=2, norm="ortho", log_mels=False,
                            melkwargs=dict(n_fft=512, hop_length=160, n_mels=128, center=True, pad_mode="constant",
                                           power=2.0, norm="slaney", mel_scale="slaney", f_min=0.0, f_max=8000.0,
                                           window_fn=torch.hann_window))
    cases = {
        "word": word,
        "noise": (np.random.default_rng(0).standard_normal(16000) * 0.01).astype(np.float32),
        "zeros_word_zeros": np.concatenate([np.zeros(3000, np.float32), word, np.zeros(2000, np.float32)]),
        "sine440": synth.sine(440),
    }
    for name, x in cases.items():
        got = tr(torch.from_numpy(x)).numpy()
        ref = L.mfcc(x)
        assert got.shape == ref.shape, name
        err = np.linalg.norm(got - ref, axis=0) / np.linalg.norm(ref, axis=0)
        assert err.max() < 2e-5, (name, float(err.max()))


_TRANSFORMERS_CHECK = r"""
import json, sys
import numpy as np, scipy.fft
sys.path.insert(0, sys.argv[1])
import transformers.audio_utils as au
from oracle import librosa_restated as L
from easywakeword_b200 import synth
word = np.load(sys.argv[1] + "/tests/golden/reference_word.npz")["pcm_i16"].astype(np.float32) / np.float32(32768)
fb = au.mel_filter_bank(257, 128, 0.0, 8000.0, 16000, norm="slaney", mel_scale="slaney")
win = au.window_function(512, "hann", periodic=True)
cases = {
    "word": word,
    "noise": (np.random.default_rng(3).standard_normal(16000) * 0.05).astype(np.float32),
    "word_gap_word": np.concatenate([word[:6000], np.zeros(4000, np.float32), word[6000:]]),
    "sine440": synth.sine(440),
}
out = {}
for name, x in cases.items():
    db = au.spectrogram(x.astype(np.float64), win, 512, 160, fft_length=512, power=2.0, center=True, pad_mode="constant",
                        mel_filters=fb, mel_floor=1e-10, log_mel="dB", reference=1.0, min_value=1e-10, db_range=80.0,
                        dtype=np.float64)
    got = scipy.fft.dct(db, axis=0, type=2, norm="ortho")[:20]
    ref = L.mfcc(x)
    out[name] = [list(got.shape) == list(ref.shape), float((np.linalg.norm(got - ref, axis=0) / np.linalg.norm(ref, axis=0)).max())]
print("RESULT " + json.dumps(out))
"""


def test_full_mfcc_front_end_against_transformers_spectrogram():
    """A third code base for the same chain: transformers.audio_utils (the Whisper / CLAP feature-extractor numerics) —
    `spectrogram(power=2, center, constant padding, periodic Hann, Slaney filter bank, log_mel="dB", db_range=80)` in
    float64, then scipy's ortho DCT-II.  The restated librosa layer agrees with it to ~1e-7 per-frame relative L2,
    floor path included (a digital-silence gap inside the word): three independent implementations, one answer.
    Runs in a fresh interpreter: with oracle/shim's stand-in `librosa` on sys.path (oracle/ref_harness.py puts it
    there) transformers would take its librosa/soxr branch at import."""
    import json
    import subprocess
    import sys
    pytest.importorskip("transformers")
    r = subprocess.run([sys.executable, "-c", _TRANSFORMERS_CHECK, REPO], capture_output=True, text=True, timeout=600)
    if r.returncode != 0 and "No module named" in r.stderr:
        pytest.skip(r.stderr.strip().splitlines()[-1])
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads(next(l for l in r.stdout.splitlines() if l.startswith("RESULT "))[7:])
    assert len(res) == 4
    for name, (same_shape, err) in res.items():
        assert same_shape, name
        assert err < 2e-6, (name, err)


def test_vad_goldens_durations_exact_rms_within_sum_bound(golden_vad):
    """oracle.analyze_reference_audio_duration / librosa_restated.rms and the package's host rule against the
    values WakeWord._analyze_reference_audio_duration (wakeword.py:854-898) returned for the same WAVs.

    The golden rms_* arrays came through the first restatement of librosa.feature.rms, which reduced a fancy-indexed
    [400, F] copy row by row in float32 instead of librosa's pairwise sum over each contiguous frame
    (oracle/vad_model.py).  They still equal that row-by-row statement bit for bit, and differ from librosa's
    arithmetic in the last bits of about half the frames, at most 53 ulps: within the error bound of a 400-term
    sequential float32 sum, 399 * 2^-24 of the sum of squares, half that on the RMS.  The durations are exact under the
    corrected arithmetic; the RMS is pinned bit for bit against the model in tests/test_vad_model.py."""
    from oracle import ewk_oracle as O, librosa_restated as L
    from easywakeword_b200.wakeword import analyze_reference_audio_duration as host_rule
    g = golden_vad
    for name in [str(n) for n in g["names"]]:
        audio = g[f"pcm_{name}"].astype(np.float32) / np.float32(32768.0)
        ref = float(g[f"duration_{name}"])
        for fn in (O.analyze_reference_audio_duration, host_rule):
            d = fn(audio)
            if np.isnan(ref):
                assert d is None, name
            else:
                assert d is not None and d == ref, (name, d, ref)
        gr32 = g[f"rms_{name}"]
        rows = np.sqrt(np.mean(np.abs(L.frame_signal(np.pad(audio, 200), 400, 160)) ** 2, axis=0))
        assert rows.dtype == np.float32 and np.array_equal(rows, gr32), name     # how the goldens were made
        rms = L.rms(y=audio, frame_length=400, hop_length=160)[0].astype(np.float64)
        gr = gr32.astype(np.float64)
        assert rms.shape == gr.shape and np.all(np.abs(rms - gr) <= 399 * 2.0**-25 * gr), name
        assert np.abs(rms - gr).max() <= 1e-6 * max(float(gr.max()), 1e-30), name
        smin, smax = O.auto_speech_durations(audio)
        assert (smin, smax) == ((0.3, 2.0) if np.isnan(ref) else (ref, 2.0 * ref)), name


# ---- N3: the resampling oracle (parity unpinned vs soxr; arithmetic pinned here)
@pytest.mark.parametrize("sr", [8000, 22050, 44100, 48000])
def test_resample_oracle_matches_scipy_polyphase_with_same_filter(sr):
    """oracle.resample_restated evaluates out[n] = sum_k x[k] g(n M / L - k); scipy.signal.upfirdn(h, x, L, M) with
    h[i] = g((i - c) / L) is an independent implementation of the same sum."""
    from scipy import signal
    from oracle import resample_restated as R
    rng = np.random.default_rng(sr)
    x = rng.standard_normal(3000)
    d = R.design(sr)
    L, M, W = d["L"], d["M"], d["W"]
    c = W * L                                               # prototype centre
    h = R.kernel((np.arange(2 * c + 1) - c) / L, d)
    full = signal.upfirdn(h, x, up=L, down=1)               # full[i] = sum_k x[k] h[i - k L] = sum_k x[k] g((i - c)/L - k)
    n_out = R.out_len(len(x), sr)
    ref = full[c + np.arange(n_out) * M]                    # time n M / L
    got = R.resample(x, sr, table_dtype=np.float64).astype(np.float64)
    assert np.abs(got - ref).max() <= 2e-6 * np.abs(ref).max()   # float32 rounding of the oracle's output


@pytest.mark.parametrize("sr", [11025, 44100, 48000, 96000])
def test_resample_oracle_tones(sr):
    """Pass-band tones come out at unit gain and the right phase (ideal band-limited interpolation), content above
    8 kHz is rejected by > 120 dB, and the output length is librosa's ceil(n * 16000 / sr)."""
    from oracle import resample_restated as R
    n = sr // 2
    t = np.arange(n) / sr
    lower = min(sr, 16000)
    for f in (300.0, 0.45 * lower * 0.9):
        y = R.resample(np.sin(2 * np.pi * f * t), sr)
        assert len(y) == int(np.ceil(n * 16000 / sr))
        to = np.arange(len(y)) / 16000
        mid = slice(700, len(y) - 700)
        assert np.abs(y[mid] - np.sin(2 * np.pi * f * to)[mid]).max() < 5e-6
    if sr > 2 * 9000:
        y = R.resample(np.sin(2 * np.pi * 9000.0 * t), sr)
        assert np.abs(y[700:-700]).max() < 1e-6             # < -120 dB


def test_preemphasis_restatement_is_lfilter_with_librosa_state():
    """oracle.librosa_restated.preemphasis == the closed form of scipy.signal.lfilter([1, -a], [1], y, zi=2 y0 - y1)
    in float32; coefficient 0 is the identity (the reference's call, wakeword.py:561-563, applies none)."""
    from oracle import librosa_restated as L
    rng = np.random.default_rng(3)
    y = (rng.standard_normal(5000) * 0.1).astype(np.float32)
    for a in (0.97, 0.5):
        out = L.preemphasis(y, a)
        assert out.dtype == np.float32
        na = np.float32(-a)
        ref = np.empty_like(y)
        ref[0] = (np.float32(2) * y[0] - y[1]) + y[0]
        ref[1:] = (na * y[:-1]) + y[1:]                       # fl(fl(-a y[n-1]) + y[n]) in float32
        assert np.abs(out - ref).max() <= 1e-7
    assert np.array_equal(O.mfcc_frames(y, preemphasis=0.0), O.mfcc_frames(y))
    m13 = O.mfcc_frames(y, n_mfcc=13)
    assert m13.shape[0] == 13 and np.array_equal(m13, O.mfcc_frames(y)[:13])


@pytest.mark.parametrize("sr", [44100, 48000, 22050, 8000])
def test_resample_oracle_against_an_independent_kaiser_sinc_resampler(sr):
    """N3 stays PARITY UNPINNED against the reference's soxr (no soxr / librosa binary offline, no resampled golden in the
    reference).  What can be stated: on band-limited content (twelve tones below 0.8 of the lower Nyquist) the restated
    converter agrees with an independent implementation of band-limited resampling — torchaudio's Kaiser-windowed sinc
    interpolator in its 'kaiser_best' setting — to 2e-5 of a 1.3 full-scale signal, i.e. to the two filters' pass-band
    ripple.  Differences between any two such filters (soxr HQ included) live in the 0.913 .. 1.0 transition band."""
    torch = pytest.importorskip("torch")
    torchaudio = pytest.importorskip("torchaudio")
    from oracle import resample_restated as R
    t = np.arange(int(sr * 0.5)) / sr
    fmax = 0.8 * min(sr, 16000) / 2
    rng = np.random.default_rng(0)
    x = sum(rng.uniform(0.05, 0.2) * np.sin(2 * np.pi * f * t + rng.uniform(0, 6)) for f in rng.uniform(100, fmax, 12)).astype(np.float32)
    y = R.resample(x, sr)
    z = torchaudio.functional.resample(torch.from_numpy(x), sr, 16000, lowpass_filter_width=64, rolloff=0.9475,
                                       resampling_method="sinc_interp_kaiser", beta=14.769656459379492).numpy()
    n = min(len(y), len(z))
    assert abs(len(y) - len(z)) <= 1
    dev = float(np.abs(y[:n][400:n - 400] - z[:n][400:n - 400]).max())
    assert dev <= 5e-5, dev
