"""GPU parity: K6 template_vad (ewk_analyze_templates, SURVEY §8(f) N2) vs the durations the reference's own
WakeWord._analyze_reference_audio_duration returned (tests/golden/vad.npz) and vs the oracle on random templates.
Durations and voiced spans are integers times 0.01 s: they must be identical.  Frame RMS equals the exact model of
librosa's arithmetic (oracle/vad_model.py) bit for bit.  The goldens' rms_* arrays came through an earlier restatement
of librosa.feature.rms with another summation order; tests/test_oracle.py bounds the model's distance from them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from easywakeword_b200 import _lib
    c = _lib.Context(device=0, n_streams=0, max_templates=1)
    yield c
    c.close()


def test_durations_match_reference_goldens(ctx, golden_vad):
    from oracle import vad_model as V
    g = golden_vad
    names = [str(n) for n in g["names"]]
    audios = [g[f"pcm_{n}"].astype(np.float32) / np.float32(32768.0) for n in names]
    res, rms = ctx.analyze_templates(audios, want_rms=True)
    for i, n in enumerate(names):
        ref = float(g[f"duration_{n}"])
        assert res["n_frames"][i] == 1 + len(audios[i]) // 160 == len(rms[i]), n
        if np.isnan(ref):
            assert not res["voiced"][i] and res["first_frame"][i] == -1, n
        else:
            assert res["voiced"][i] and res["duration_s"][i] == ref, (n, res["duration_s"][i], ref)
        m = V.frame_rms(audios[i])
        assert np.array_equal(rms[i].view(np.uint32), m.view(np.uint32)), n
        assert res["max_rms"][i].view(np.uint32) == m.max().view(np.uint32), n


def test_random_templates_match_oracle(ctx):
    from oracle import ewk_oracle as O, vad_model as V
    rng = np.random.default_rng(2024)
    audios = []
    for k in range(64):
        n = int(rng.integers(1, 40000))
        x = rng.standard_normal(n).astype(np.float32) * np.float32(0.003)
        a, b = sorted(rng.integers(0, n, 2))
        x[a:b] += rng.standard_normal(b - a).astype(np.float32) * np.float32(rng.uniform(0.02, 0.5))
        if k % 9 == 0:
            x[:] = 0
        audios.append(x)
    audios.append(np.zeros(0, np.float32))                    # empty template: one all-zero frame, not voiced
    res, rms = ctx.analyze_templates(audios, want_rms=True)
    for i, x in enumerate(audios):
        assert np.array_equal(rms[i].view(np.uint32), V.frame_rms(x).view(np.uint32)), i
        d = O.analyze_reference_audio_duration(x) if len(x) else None
        if d is None:
            assert not res["voiced"][i], i
        else:
            assert res["voiced"][i] and res["duration_s"][i] == d, (i, res["duration_s"][i], d)


def test_bank_default_durations_come_from_device_vad(word):
    """WakeWordBank without explicit durations: min = VAD duration of the first template, max = 2 * min
    (the _auto_calculate_speech_durations contract, reference tests/test_wakeword_simulated.py:687-775)."""
    from easywakeword_b200.bank import WakeWordBank
    from oracle import ewk_oracle as O
    bank = WakeWordBank(2, [word, word[:8000]], device=0)
    try:
        smin, smax = O.auto_speech_durations(word)
        assert bank.params["speech_duration_min"] == smin and bank.params["speech_duration_max"] == smax
        assert bank.template_vad["duration_s"][1] == O.analyze_reference_audio_duration(word[:8000])
    finally:
        bank.close()
