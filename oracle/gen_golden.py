"""ORACLE — TEST INFRASTRUCTURE ONLY.  Writes tests/golden/*.npz from the REFERENCE'S OWN CODE.

Run in the build container (needs /root/reference):   python -m oracle.gen_golden

Every value in the fixtures is produced by /root/reference/easywakeword/wakeword.py run
unmodified on oracle/shim (see oracle/ref_harness.py): WordMatcher.extract_mfcc /
calculate_similarity / matches, SoundBuffer and WakeWord._detect_word under the fake clock.
The inputs are either stored (small) or regenerated in the tests from the recorded seeds via
easywakeword_b200/synth.py (a sha256 of each regenerated stream is stored to catch drift).
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, _REPO)

from easywakeword_b200 import synth  # noqa: E402
from oracle import ref_harness as H  # noqa: E402

GOLDEN = os.path.join(_REPO, "tests", "golden")
REF_WAV = os.path.join(H.REFERENCE_ROOT, "reference_word.wav")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def matcher_cases(word):
    """name -> float32 audio; mirrors the signals of the reference's hot-path tests
    (tests/test_wakeword_simulated.py:107-205, 330-360; tests/test_cross_platform.py:72-109)."""
    cases = {}
    cases["word"] = word
    # reference tests write PCM16 WAVs and read them back: lrint(x*32767)/32768
    def via_wav(x):
        return (np.rint(x.astype(np.float64) * 32767.0) / 32768.0).astype(np.float32)
    cases["sine440"] = via_wav(synth.sine(440))
    cases["sine880"] = via_wav(synth.sine(880))
    cases["sine440_raw"] = synth.sine(440)
    cases["speech_like"] = via_wav(synth.speech_like(1.0))
    np.random.seed(42)
    cases["noise42"] = np.random.randn(16000).astype(np.float32) * 0.1
    cases["sine440_half"] = via_wav(synth.sine(440)) * 0.5
    cases["word_half"] = word * np.float32(0.5)
    cases["zeros_word_zeros"] = np.concatenate([np.zeros(3000, np.float32), word, np.zeros(2000, np.float32)])
    rng = np.random.default_rng(0)
    cases["noise_sigma01_1s"] = (rng.standard_normal(16000) * 0.01).astype(np.float32)
    x, _ = synth.stream(77, 3.0, word, gain=(2.0, 3.0), inserts_per_10s=(1, 1))
    cases["stream_3s_i16"] = synth.from_int16(synth.to_int16(x))        # 48000 samples: the 3.0 s cap
    for n in (1, 100, 159, 160, 161, 511, 512, 513, 1000, 4000):
        cases[f"noise_n{n}"] = (np.random.default_rng(n).standard_normal(n) * 0.05).astype(np.float32)
    cases["word_loud_in_noise"] = (np.random.default_rng(5).standard_normal(20000) * 0.002).astype(np.float32)
    cases["word_loud_in_noise"][2000:2000 + len(word)] += 3.0 * word
    return cases


def gen_matcher(mod, word):
    cases = matcher_cases(word)
    out = {"names": np.array(list(cases))}
    templates = {"word": word, "sine440": cases["sine440"], "speech_like": cases["speech_like"]}
    ms = {}
    for tn, ta in templates.items():
        m = mod.WordMatcher(sample_rate=16000)
        m.set_reference(ta, tn)
        ms[tn] = m
        out[f"tpl_{tn}_mean"] = m.reference_mfcc_mean
        out[f"tpl_{tn}_std"] = m.reference_mfcc_std
    import librosa  # the shim: same function WordMatcher calls (wakeword.py:561)
    for name, a in cases.items():
        out[f"in_{name}"] = a
        mean, std = ms["word"].extract_mfcc(a)
        out[f"mean_{name}"] = mean
        out[f"std_{name}"] = std
        out[f"mfcc_{name}"] = librosa.feature.mfcc(y=a, sr=16000, n_mfcc=20, n_fft=512, hop_length=160)
        with np.errstate(all="ignore"):
            for tn, m in ms.items():
                ok, sim = m.matches(a, threshold=75.0)
                out[f"score_{tn}_{name}"] = np.float64(sim)
                out[f"match_{tn}_{name}"] = np.bool_(ok)
    np.savez_compressed(os.path.join(GOLDEN, "matcher.npz"), **out)
    return {n: float(out[f"score_word_{n}"]) for n in cases}


DETECT_CASES = [
    # name, seed, seconds, block, noise_sigma, gain, extra params
    dict(name="config1", special="config1", block=512, params=dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=30)),
    dict(name="b1600_quiet", seed=2001, seconds=60, block=1600, noise=0.002, gain=(1.0, 4.0),
         params=dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=30)),
    dict(name="b512_quiet", seed=2002, seconds=60, block=512, noise=0.002, gain=(1.0, 4.0),
         params=dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=30)),
    dict(name="b1600_loudnoise", seed=2003, seconds=60, block=1600, noise=0.01, gain=(2.0, 5.0),
         params=dict(speech_duration_min=0.5, speech_duration_max=1.6, timeout=30)),
    dict(name="b512_loudnoise", seed=2004, seconds=60, block=512, noise=0.012, gain=(2.0, 5.0),
         params=dict(speech_duration_min=0.5, speech_duration_max=1.6, timeout=12)),
    dict(name="b800_short_timeout", seed=2005, seconds=50, block=800, noise=0.003, gain=(1.5, 3.0),
         params=dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=5, pre_speech_silence=0.5,
                     post_speech_silence=0.3)),
    dict(name="b1024_defaults", seed=2006, seconds=50, block=1024, noise=0.002, gain=(2.0, 4.0),
         params=dict(similarity_threshold=90.0)),
    dict(name="b1600_distractors_thr97", seed=2008, seconds=80, block=1600, noise=0.002, gain=(1.5, 4.0),
         distractor_prob=0.5, inserts=(2, 3),
         params=dict(speech_duration_min=0.5, speech_duration_max=1.6, timeout=30, similarity_threshold=97.0)),
    dict(name="b512_distractors_thr98", seed=2009, seconds=80, block=512, noise=0.006, gain=(2.0, 5.0),
         distractor_prob=0.6, inserts=(2, 3),
         params=dict(speech_duration_min=0.5, speech_duration_max=1.6, timeout=20, similarity_threshold=98.0)),
    dict(name="b320_zero_gaps", seed=2007, seconds=40, block=320, noise=0.004, gain=(2.0, 4.0), zero_gaps=6,
         params=dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=30)),
    # a short timeout with restarts at block 512 and 0.6-1.5 s durations, which no case above covers
    dict(name="b512_timeout8", seed=4242, seconds=25, block=512, noise=0.003, gain=(2.0, 4.0),
         params=dict(speech_duration_min=0.6, speech_duration_max=1.5, timeout=8)),
]


def detect_stream_for(case, word):
    if case.get("special") == "config1":     # SURVEY §8(d) config 1
        rng = np.random.default_rng(7)
        s = (rng.standard_normal(400000) * 0.002).astype(np.float32)
        s[224000:224000 + len(word)] += (3.0 * word).astype(np.float32)
        return s
    x, _ = synth.stream(case["seed"], case["seconds"], word, noise_sigma=case["noise"], gain=case["gain"],
                        zero_gaps=case.get("zero_gaps", 0), distractor_prob=case.get("distractor_prob", 0.0),
                        inserts_per_10s=case.get("inserts", (1, 3)))
    return synth.from_int16(synth.to_int16(x))   # device-representable: q/32768


def gen_detect(word):
    out = {"names": np.array([c["name"] for c in DETECT_CASES]), "cases_json": np.array(json.dumps(DETECT_CASES))}
    summary = {}
    for c in DETECT_CASES:
        s = detect_stream_for(c, word)
        r = H.run_reference_stream(s, word, block=c["block"], **c["params"])
        n = c["name"]
        out[f"{n}_stream_sha"] = np.array(sha(s))
        out[f"{n}_full_tick"] = np.int64(r["full_tick"])
        out[f"{n}_ticks_run"] = np.int64(r["ticks_run"])
        out[f"{n}_trace_tick"] = r["trace_tick"]
        out[f"{n}_trace_silent"] = r["trace_silent"]
        out[f"{n}_trace_thr"] = r["trace_thr"]
        out[f"{n}_ev_tick"] = np.array([e["tick"] for e in r["events"]], dtype=np.int64)
        out[f"{n}_ev_len"] = np.array([e["seg_len"] for e in r["events"]], dtype=np.int64)
        out[f"{n}_ev_score"] = np.array([e["score"] for e in r["events"]], dtype=np.float64)
        out[f"{n}_ev_match"] = np.array([e["matched"] for e in r["events"]], dtype=np.bool_)
        out[f"{n}_timeouts"] = np.array(r["timeouts"], dtype=np.int64)
        summary[n] = dict(ticks=int(r["ticks_run"]), events=[(e["tick"], e["seg_len"], round(e["score"], 4), e["matched"])
                                                               for e in r["events"]], timeouts=r["timeouts"],
                          thr_range=(float(r["trace_thr"].min()), float(r["trace_thr"].max())),
                          silent_frac=float(r["trace_silent"].mean()))
    np.savez_compressed(os.path.join(GOLDEN, "detect.npz"), **out)
    return summary


def gen_dense(mod, word):
    """Reference WordMatcher.calculate_similarity on the dense windows of A9 (strided hops)."""
    from oracle.ewk_oracle import dense_window
    tpl2 = synth.synthetic_word(seed=3, duration=0.61)
    templates = [word, tpl2]
    out = {"tpl2": tpl2}
    for si, (seed, zero_gaps) in enumerate([(3001, 0), (3002, 4)]):
        x, _ = synth.stream(seed, 12.0, word, gain=(1.0, 4.0), zero_gaps=zero_gaps)
        x = synth.from_int16(synth.to_int16(x))
        hops = np.arange(200, 1200, 7)
        sc = np.full((len(hops), len(templates)), np.nan)
        for ki, tpl in enumerate(templates):
            m = mod.WordMatcher(sample_rate=16000)
            m.set_reference(tpl, "t")
            nb, ln = dense_window(len(tpl))
            for hi, h in enumerate(hops):
                s0 = 160 * (int(h) - nb)
                with np.errstate(all="ignore"):
                    sc[hi, ki] = m.calculate_similarity(x[s0:s0 + ln])
        out[f"s{si}_seed"] = np.int64(seed)
        out[f"s{si}_zero_gaps"] = np.int64(zero_gaps)
        out[f"s{si}_sha"] = np.array(sha(x))
        out[f"s{si}_hops"] = hops
        out[f"s{si}_scores"] = sc
    np.savez_compressed(os.path.join(GOLDEN, "dense.npz"), **out)
    return {k: (float(np.nanmin(v)), float(np.nanmax(v))) for k, v in out.items() if k.endswith("_scores")}


def gen_vad(mod, word):
    """WakeWord._analyze_reference_audio_duration (wakeword.py:854-898), the reference's own method run on PCM16
    WAV files (the only template format its loader is given), plus librosa.feature.rms frame values through
    the shim.  Stored: the int16 samples of every case, the returned duration (NaN for None) and the frame RMS."""
    import tempfile
    import types
    import wave

    import librosa  # shim

    def i16(x):
        return np.clip(np.rint(np.asarray(x, np.float64) * 32767.0), -32768, 32767).astype(np.int16)

    rng = np.random.default_rng(11)
    cases = {
        "word": np.rint(word.astype(np.float64) * 32768.0).astype(np.int16),
        "zeros_word_zeros": i16(np.concatenate([np.zeros(3000), word, np.zeros(2000)])),
        "speech_like": i16(synth.speech_like(1.0)),
        "sine440": i16(synth.sine(440)),
        "noise": i16(rng.standard_normal(16000) * 0.05),
        "quiet_then_burst": i16(np.concatenate([rng.standard_normal(8000) * 0.001, rng.standard_normal(4000) * 0.2,
                                                rng.standard_normal(6000) * 0.001])),
        "all_zeros": np.zeros(8000, np.int16),
        "tiny_100": i16(rng.standard_normal(100) * 0.1),
        "short_click": i16(np.concatenate([np.zeros(4000), [0.9, -0.9, 0.9], np.zeros(4000)])),
        "synth_word_1": i16(synth.synthetic_word(seed=1, duration=0.45)),
        "synth_word_2": i16(synth.synthetic_word(seed=2, duration=1.3)),
        "word_in_noise": i16(np.concatenate([rng.standard_normal(5000) * 0.004, 0.8 * word + rng.standard_normal(len(word)) * 0.004,
                                             rng.standard_normal(7000) * 0.004])),
        "two_bursts": i16(np.concatenate([np.zeros(1600), rng.standard_normal(3200) * 0.3, np.zeros(6400),
                                          rng.standard_normal(1600) * 0.3, np.zeros(3200)])),
    }
    out, summary = {"names": np.array(list(cases))}, {}
    with tempfile.TemporaryDirectory() as td:
        for name, pcm in cases.items():
            path = os.path.join(td, name + ".wav")
            with wave.open(path, "wb") as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(16000); w.writeframes(pcm.tobytes())
            stub = types.SimpleNamespace(wavword=path, _log=lambda *a, **k: None)
            dur = mod.WakeWord._analyze_reference_audio_duration(stub)
            audio, sr = librosa.load(path, sr=None)
            assert sr == 16000 and np.array_equal(audio, pcm.astype(np.float32) / np.float32(32768.0))
            rms = librosa.feature.rms(y=audio, frame_length=400, hop_length=160)[0]
            out[f"pcm_{name}"] = pcm
            out[f"duration_{name}"] = np.float64(np.nan if dur is None else dur)
            out[f"rms_{name}"] = rms.astype(np.float32)
            summary[name] = None if dur is None else float(dur)
    np.savez_compressed(os.path.join(GOLDEN, "vad.npz"), **out)
    return summary


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    mod = H.import_reference()
    import soundfile as sf  # shim
    word64, sr = sf.read(REF_WAV)                     # float64 int16/32768
    assert sr == 16000
    word_i16 = np.rint(word64 * 32768.0).astype(np.int16)
    word = word_i16.astype(np.float32) / np.float32(32768.0)
    # the reference's own loader must give the same samples (wakeword.py:588)
    import librosa
    y, _ = librosa.load(REF_WAV, sr=16000)
    assert np.array_equal(y, word)
    np.savez_compressed(os.path.join(GOLDEN, "reference_word.npz"), pcm_i16=word_i16, sr=np.int64(sr))

    manifest = {
        "generated_by": "oracle/gen_golden.py",
        "reference_wakeword_py_sha256": hashlib.sha256(open(mod.__file__, "rb").read()).hexdigest(),
        "reference_word_wav_sha256": hashlib.sha256(open(REF_WAV, "rb").read()).hexdigest(),
        "numpy": np.__version__,
        "scipy": __import__("scipy").__version__,
        "librosa": "restated (oracle/librosa_restated.py) — real librosa not installable offline",
    }
    manifest["matcher_scores_vs_word"] = gen_matcher(mod, word)
    manifest["detect"] = gen_detect(word)
    manifest["dense"] = gen_dense(mod, word)
    manifest["vad_durations"] = gen_vad(mod, word)
    with open(os.path.join(GOLDEN, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1, default=str)
    print(json.dumps(manifest, indent=1, default=str))


if __name__ == "__main__":
    main()
