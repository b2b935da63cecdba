"""K6 (template_vad_kernel, ewk_analyze_templates) pinned bit for bit against oracle/vad_model.py: every field of
ewk_vad_result and every frame RMS, at the length and amplitude classes of tests/test_vad_model.py, templates of more
than 256 frames, many templates at unaligned offsets of one packed buffer, host and device input.  Near-threshold
templates, where one ulp of frame RMS moves the first voiced frame, give the model's and the host rule's durations, and
WakeWordBank's automatic durations equal the WakeWord facade's for them."""
import ctypes as C
import struct

import numpy as np
import pytest

from oracle import vad_model as V
from test_vad_model import LENGTHS, LONG, amplitude_classes

pytestmark = pytest.mark.gpu

FIELDS = ("max_rms", "threshold", "first_frame", "last_frame", "n_frames", "voiced")


@pytest.fixture(scope="module")
def ctx():
    from easywakeword_b200 import _lib
    c = _lib.Context(device=0, n_streams=0, max_templates=1)
    yield c
    c.close()


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def analyze_packed(ctx, pcm, offs, lens, where):
    """ewk_analyze_templates on one packed float32 buffer (host or device) -> (results, list of frame RMS)."""
    from easywakeword_b200 import _lib
    n = len(offs)
    offs = np.ascontiguousarray(offs, np.int64)
    lens = np.ascontiguousarray(lens, np.int64)
    frames = 1 + lens // 160
    out = np.zeros(n, _lib.VAD_DTYPE)
    rms = np.full(int(frames.sum()), np.nan, np.float32)
    if where == "host":
        ptr = pcm.ctypes.data
    else:
        import torch
        t = torch.from_numpy(pcm).cuda()
        torch.cuda.synchronize()
        ptr = t.data_ptr()
    rc = ctx.lib.ewk_analyze_templates(ctx.h, C.cast(ptr, C.POINTER(C.c_float)), _lib.HOST if where == "host" else _lib.DEVICE,
                                       _lib.i64ptr(offs), _lib.i64ptr(lens), n, out.ctypes.data, _lib.f32ptr(rms), len(rms))
    assert rc == 0, ctx.lib.ewk_last_error(ctx.h)
    return out, np.split(rms, np.cumsum(frames)[:-1])


def assert_matches_model(res, rms, ys, what):
    for i, y in enumerate(ys):
        m_rms = V.frame_rms(y)
        if not np.array_equal(bits(rms[i]), bits(m_rms)):
            bad = np.flatnonzero(bits(rms[i]) != bits(m_rms))
            raise AssertionError(f"{what} template {i} (len {len(y)}): {len(bad)} of {len(m_rms)} frame RMS differ, "
                                 f"e.g. {[(int(b), float(rms[i][b]), float(m_rms[b])) for b in bad[:4]]}")
        m = V.analyze(y, rms=m_rms)
        r = res[i]
        for f in FIELDS:
            assert bits(r[f]) == bits(m[f]) if f in ("max_rms", "threshold") else int(r[f]) == m[f], (what, i, f, r[f], m[f])
        assert float(r["duration_s"]) == m["duration_s"], (what, i, float(r["duration_s"]), m["duration_s"])


def test_length_and_amplitude_classes_bit_for_bit(ctx):
    """Every class of tests/test_vad_model.py, including a 30 s template (3001 frames: each warp runs the frame loop
    375 times), through the Python API (host input, one packed buffer)."""
    rng = np.random.default_rng(20261021)
    ys = [y for n in LENGTHS + [LONG] for _, y in amplitude_classes(n, rng)]
    res, rms = ctx.analyze_templates(ys, want_rms=True)
    assert_matches_model(res, rms, ys, "classes")
    assert sum(len(r) for r in rms) > 40_000


@pytest.mark.parametrize("where", ["host", "device"])
def test_many_templates_at_unaligned_offsets(ctx, where):
    """One buffer, templates at odd offsets with stray samples between them (not read: a template is zero outside its
    own samples), some overlapping, some longer than 256 frames."""
    rng = np.random.default_rng(77 if where == "host" else 78)
    pcm = (rng.standard_normal(700_001) * 0.05).astype(np.float32)
    pcm[rng.random(len(pcm)) < 0.01] *= np.float32(40.0)          # loud stray samples next to the templates
    offs, lens = [], []
    for k in range(90):
        n = int(rng.choice([0, 1, 160, 401, 4001, 41_000, 60_321])) + int(rng.integers(0, 3))
        o = int(rng.integers(0, len(pcm) - n))
        offs.append(o), lens.append(n)
    for k in range(0, 90, 3):                                      # shape some of them: silence, a burst, a quiet tail
        o, n = offs[k], lens[k]
        if n > 4000:
            pcm[o:o + n // 3] *= np.float32(1e-4)
    res, rms = analyze_packed(ctx, pcm, offs, lens, where)
    ys = [pcm[o:o + n] for o, n in zip(offs, lens)]
    assert_matches_model(res, rms, ys, where)
    assert max(len(r) for r in rms) > 256


@pytest.mark.parametrize("where", ["host", "device"])
def test_near_threshold_durations(ctx, where):
    """Templates built on the threshold (oracle.vad_model.near_threshold_templates, the set tests/test_vad_model.py
    shows to separate librosa's arithmetic from a double-accumulated one): device duration == model == host rule."""
    from easywakeword_b200.wakeword import analyze_reference_audio_duration as host_rule
    ys = V.near_threshold_templates(2026, 40)
    lens = [len(y) for y in ys]
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]) + 3
    pcm = np.zeros(int(offs[-1] + lens[-1] + 5), np.float32)
    for o, y in zip(offs, ys):
        pcm[o:o + len(y)] = y
    res, rms = analyze_packed(ctx, pcm, offs, lens, where)
    bad = [i for i, y in enumerate(ys) if float(res["duration_s"][i]) != V.duration(y)]
    assert not bad, f"{len(bad)} of {len(ys)} near-threshold templates changed duration on the device: {bad}"
    assert_matches_model(res, rms, ys, "near-threshold")
    for i, y in enumerate(ys):
        assert float(res["duration_s"][i]) == host_rule(y), i


def _write_f32_wav(path, y):
    """IEEE-float WAV (format tag 3): the template's float32 samples reach librosa.load's stand-in unchanged."""
    data = np.asarray(y, "<f4").tobytes()
    fmt = struct.pack("<HHIIHH", 3, 1, 16000, 16000 * 4, 4, 32)
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 4 + 8 + len(fmt) + 8 + len(data)) + b"WAVE")
        f.write(b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data)


def test_bank_auto_durations_equal_the_facade(tmp_path):
    """WakeWordBank (K6) and WakeWord (host rule) set the same speech_duration_min / max from the same near-threshold
    template: the pairs where the double-accumulated arithmetic disagrees, and a few more."""
    from easywakeword_b200.bank import WakeWordBank
    from easywakeword_b200.wakeword import WakeWord, load_wav_16k

    class Stt:
        def transcribe(self, audio):
            return ""

    ys = V.near_threshold_templates(2026, 40)
    pick = [i for i, y in enumerate(ys) if V.analyze(y, rms=V.frame_rms_double(y))["duration_s"] != V.duration(y)]
    pick = sorted(set(pick) | {0, 1, 2, 3})
    assert len(pick) >= 10
    for i in pick:
        p = str(tmp_path / f"t{i}.wav")
        _write_f32_wav(p, ys[i])
        assert np.array_equal(load_wav_16k(p), ys[i])
        ww = WakeWord("hello", p, transcriber=Stt())
        bank = WakeWordBank(1, [p], device=0)
        try:
            assert (bank.params["speech_duration_min"], bank.params["speech_duration_max"]) == \
                (ww.speech_duration_min, ww.speech_duration_max), i
            assert ww.speech_duration_min == V.duration(ys[i]), i
        finally:
            bank.close()
