"""GPU: the drop-in classes (WordMatcher / SoundBuffer / WakeWord / WakeWordBank) with the reference's
own test scenarios (tests/test_wakeword_simulated.py:104-205, 298-360; tests/test_cross_platform.py:
69-109) and against the oracle restatement of SoundBuffer."""
import wave

import numpy as np
import pytest

from easywakeword_b200 import synth

pytestmark = pytest.mark.gpu


class _NullSource:
    def start(self): pass
    def stop(self): pass


@pytest.fixture()
def wav(tmp_path, word_i16):
    p = tmp_path / "word.wav"
    with wave.open(str(p), "wb") as w:
        w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(word_i16.tobytes())
    return str(p)


def _wav_roundtrip(x):
    return (np.rint(x.astype(np.float64) * 32767.0) / 32768.0).astype(np.float32)


# ---- WordMatcher: the reference's TestWordMatcher / TestCrossPlatformMFCC scenarios
def test_wordmatcher_reference_scenarios(golden_matcher):
    from easywakeword_b200.wakeword import WordMatcher
    a440 = _wav_roundtrip(synth.sine(440))
    m = WordMatcher(sample_rate=16000)
    with pytest.raises(ValueError, match="No reference word set"):
        m.calculate_similarity(np.zeros(16000, np.float32))
    m.set_reference(a440, "test")
    ok, sim = m.matches(a440)
    assert ok and sim == 100.0                                   # test_self_match
    assert m.calculate_similarity(a440) == m.calculate_similarity(a440) == 100.0   # deterministic
    ok2, sim2 = m.matches(_wav_roundtrip(synth.sine(880)))
    assert sim2 < 100.0 and abs(float(sim2) - float(golden_matcher["score_sine440_sine880"])) <= 0.01
    np.random.seed(42)
    noise = np.random.randn(16000).astype(np.float32) * 0.1
    assert m.matches(noise)[1] < 100.0
    assert m.matches(a440 * 0.5, threshold=75.0)[1] > 50.0       # test_audio_normalization
    mean, std = m.extract_mfcc(a440)
    assert len(mean) == 20 and len(std) == 20 and np.isfinite(mean).all() and np.isfinite(std).all()
    assert m.mfcc(a440).shape == (20, 101)
    sp = _wav_roundtrip(synth.speech_like(1.0))
    m2 = WordMatcher()
    m2.set_reference(sp, "speech")
    assert m2.matches(sp) == (True, 100.0)                        # test_speech_like_audio_matching
    assert m.reference_word == "test" and m2.reference_word == "speech"
    assert m.matches(a440)[1] == 100.0                            # two matchers keep separate templates


def test_wordmatcher_load_reference_from_file(wav, word, golden_matcher):
    from easywakeword_b200.wakeword import WordMatcher
    m = WordMatcher()
    m.load_reference_from_file(wav, "test_word")
    assert m.reference_word == "test_word"
    ref_mean = golden_matcher["tpl_word_mean"]
    assert np.linalg.norm(m.reference_mfcc_mean - ref_mean) <= 1e-4 * np.linalg.norm(ref_mean)
    ok, sim = m.matches(word, threshold=75.0)
    assert ok and sim >= 75.0


# ---- SoundBuffer vs the oracle restatement of the reference's SoundBuffer
@pytest.mark.parametrize("block", [512, 1600])
def test_soundbuffer_follows_reference(block, word):
    from easywakeword_b200.wakeword import SoundBuffer
    from oracle.ewk_oracle import SoundBufferOracle
    x, _ = synth.stream(77, 4.5, word, noise_sigma=0.008, gain=(2.0, 3.0), inserts_per_10s=(2, 2))
    sb = SoundBuffer(seconds=2, source=_NullSource())
    ob = SoundBufferOracle(seconds=2, fast=True)
    assert sb.is_silent() and sb.frame_size == 0 and not sb.is_buffer_full()
    n_silent = 0
    for i, p in enumerate(range(0, len(x) - block, block)):
        blk = x[p:p + block]
        sb._add_sound_to_buffer(blk.reshape(-1, 1), block, None, None)
        ob.add_block(blk)
        if i % 3 == 2:
            assert sb.is_silent() == ob.is_silent(), (i, sb.silence_threshold, ob.silence_threshold)
            n_silent += ob.is_silent()
            np.testing.assert_allclose(sb.silence_threshold, ob.silence_threshold, rtol=1e-12)
            assert sb.is_buffer_full() == ob.is_buffer_full()
            assert sb.pointer == ob.pointer and sb.samples_collected == ob.samples_collected
    assert sb.frame_size == block and 0 < n_silent
    assert ob.silence_threshold > 0.006                          # the adaptive branch was exercised
    for n in (0.1, 0.5, 2.0, 5.0):
        a, b = sb.return_last_n_seconds(n), ob.return_last_n_seconds(n)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    assert np.array_equal(sb.data, ob.data)
    assert len(sb.return_last_n_seconds(0)) == 0
    sb.stop()


# ---- WakeWord end to end: scripted audio source, fake clock, stub transcriber
def test_wakeword_waitforit_detects_inserted_word(wav, word, monkeypatch):
    import easywakeword_b200.wakeword as W
    x = (np.random.default_rng(7).standard_normal(16000 * 8) * 0.002).astype(np.float32)
    x[16000 * 4:16000 * 4 + len(word)] += 3.0 * word

    class Clock:
        """time() = k*0.1; sleep() feeds the next 0.1 s of audio through the PortAudio callback."""
        def __init__(self): self.k, self.buf, self.fed = 0, None, 0
        def time(self): return self.k * 0.1
        def sleep(self, dt):
            self.k += 1
            while self.fed + 512 <= min(len(x), self.k * 1600):
                self.buf._add_sound_to_buffer(x[self.fed:self.fed + 512].reshape(-1, 1), 512, None, None)
                self.fed += 512
    clk = Clock()
    monkeypatch.setattr(W, "time", clk)

    class Stt:
        calls = 0
        def transcribe(self, audio):
            Stt.calls += 1
            assert np.max(np.abs(audio)) <= 1.0
            return "Computer!"

    ww = W.WakeWord("computer", wav, numberofwords=1, timeout=30, buffer_seconds=2, transcriber=Stt())
    ww._sound_buffer = W.SoundBuffer(seconds=2, source=_NullSource())
    clk.buf = ww._sound_buffer
    assert ww.waitforit() == "Computer!"
    assert Stt.calls == 1 and 50 < clk.k < 70 and not ww.is_listening()
    # the same stream through the oracle makes the same single level-2 call at the same tick
    from oracle import ewk_oracle as O
    o = O.detect_stream(x, word, block=512, buffer_seconds=2, fast=True, speech_duration_min=ww.speech_duration_min,
                        speech_duration_max=ww.speech_duration_max)
    assert [e["tick"] for e in o["events"]] == [clk.k]
    ww.stop()


# ---- WakeWordBank: callback surface over many streams
def test_bank_run_reports_matches(word):
    from easywakeword_b200.bank import WakeWordBank
    from oracle import ewk_oracle as O
    n = 6
    xs = [synth.stream(5000 + i, 25.0, word, gain=(2.0, 4.0))[0] for i in range(n)]
    q = np.stack([synth.to_int16(x) for x in xs])
    bank = WakeWordBank(n, [word], frame_size=1600)
    assert bank.params["speech_duration_min"] == pytest.approx(0.69)
    hits = []
    log = bank.run((np.ascontiguousarray(q[:, p:p + 8000]) for p in range(0, q.shape[1], 8000)),
                   on_match=lambda s, t, sc, txt: hits.append((s, t, sc)))
    bank.close()
    want = []
    for i in range(n):
        o = O.detect_stream(synth.from_int16(q[i]), word, block=1600, fast=True, speech_duration_min=0.69,
                            speech_duration_max=1.38)
        want += [(i, e["tick"]) for e in o["events"] if e["matched"]]
    assert sorted((s, t) for s, t, _ in hits) == sorted(want) and len(want) >= 4
    assert all(sc >= 75.0 for _, _, sc in hits)


# ---- N1: batched level-3 pre-processing on the device; N4: several reference templates, best one wins
def test_bank_level3_handoff_and_multi_template(word):
    from easywakeword_b200.bank import WakeWordBank
    from oracle import ewk_oracle as O
    other = synth.synthetic_word(seed=3, duration=0.8)
    n = 4
    xs = []
    for i in range(n):
        x, _ = synth.stream(6000 + i, 40.0, word if i % 2 == 0 else other, gain=(2.0, 4.0), inserts_per_10s=(2, 3))
        xs.append(x)
    q = np.stack([synth.to_int16(x) for x in xs])
    bank = WakeWordBank(n, [word, other], frame_size=1600, similarity_threshold=75.0,
                        speech_duration_min=0.5, speech_duration_max=1.6)
    heard = []

    class Stt:
        def transcribe(self, audio):
            assert audio.dtype == np.float32 and np.max(np.abs(audio)) <= 1.0
            heard.append(audio)
            return "computer"

    log = bank.run((np.ascontiguousarray(q[:, p:p + 16000]) for p in range(0, q.shape[1], 16000)),
                   on_match=lambda s, t, sc, txt: None, transcriber=Stt())
    ev = [e for e in log if e["kind"] == 2]
    assert len(ev) >= 4 and len(heard) == sum(bool(e["matched"]) for e in ev)
    # N4: the event's template is the best-scoring slot, equal to the oracle's argmax over both templates
    mats = [O.WordMatcherOracle(), O.WordMatcherOracle()]
    mats[0].set_reference(word); mats[1].set_reference(other)
    # ring content is gone for old events; recompute from the source streams
    for e in ev:
        seg = synth.from_int16(q[e["stream"], e["seg_start"]:e["seg_start"] + e["seg_len"]])
        sc = [float(m.calculate_similarity(seg)) for m in mats]
        assert abs(float(e["score"]) - max(sc)) <= 0.01
        if abs(sc[0] - sc[1]) > 0.02:
            assert int(e["template_slot"]) == int(np.argmax(sc))
    # N1: device pre-processing == the reference formula (float64) rounded to float32, bit for bit on an int16 ring
    last = [e for e in ev if e["matched"]][-2:]
    got = bank.prepare_for_transcription(last)
    for e, g in zip(last, got):
        seg = synth.from_int16(q[e["stream"], e["seg_start"]:e["seg_start"] + e["seg_len"]]).astype(np.float64)
        assert np.array_equal(g.view(np.uint32), O.prepare_for_level3(seg).astype(np.float32).view(np.uint32))
    bank.close()
