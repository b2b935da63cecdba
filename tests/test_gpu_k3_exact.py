"""GPU: K3 (segment_mfcc_match_kernel and both queue forms) equals, bit for bit, the exact float32 model of
oracle/frame_model.py: np.array_equal(device, model, equal_nan=True) for frames, features, template features, scores,
`matched`, queue events (score, template, matched) and, through oracle/dense_model.py fed with the model's frames, K4's
dense scores from PCM.  The model's log is the device's own __log2f (tests/k3_probe.cu: k3p_log_mel); everything else
is restated.  The probe also runs the frame pipeline on loaded frames, so that a difference is pinned to a stage."""
import numpy as np
import pytest

from easywakeword_b200 import synth
from helpers import K3Probe
from oracle import dense_model as D
from oracle import frame_model as M

pytestmark = pytest.mark.gpu

LENGTHS = [1, 2, 159, 160, 161, 255, 256, 257, 511, 512, 513, 4001, 7360, 15503, 23998, 47999, 48000, 48160]


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return K3Probe(tmp_path_factory.mktemp("k3_probe"))


@pytest.fixture(scope="module")
def tables(probe):
    return M.Tables.from_image(probe.tables()[0])


def assert_exact(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got, want, equal_nan=True):
        bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
        ex = [(tuple(int(v) for v in b), float(got[tuple(b)]), float(want[tuple(b)])) for b in bad[:4]]
        raise AssertionError(f"{what}: {len(bad)} of {got.size} values differ from the model, e.g. {ex}")


def signals(n, seed):
    """Named test signals of n samples (float32, int16-representable where the name says so)."""
    rng = np.random.default_rng(seed)
    out = {}
    x, _ = synth.stream(seed, max(n, 16000) / 16000 + 0.1, synth.synthetic_word(seed=seed, duration=0.6), gain=(1.5, 3.0))
    out["speech"] = synth.from_int16(synth.to_int16(x[:n]))
    q = rng.integers(-32768, 32768, n).astype(np.int16)
    q[:: 7] = -32768
    q[3:: 11] = 32767
    out["full scale"] = synth.from_int16(q)
    out["zero"] = np.zeros(n, np.float32)
    out["dc"] = np.full(n, np.float32(0.25))
    out["tiny noise"] = (rng.standard_normal(n) * 1e-6).astype(np.float32)
    loud = out["speech"].copy()
    loud[n // 3:] *= np.float32(1e-5)                            # frames below the top_db floor
    out["loud then silent"] = loud
    return out


def mid_range_features(mean, std, c0_scale):
    """Template features that score speech in the middle of the 0-100 range, where one ulp of a score is ~4e-6: the
    word's mean with coefficient 0 scaled down, and its std in reverse order."""
    m = np.asarray(mean, np.float32).copy()
    m[0] *= np.float32(c0_scale)
    return m, np.ascontiguousarray(np.asarray(std, np.float32)[::-1])


def make_ctx(**kw):
    from easywakeword_b200 import _lib
    return _lib.Context(device=0, n_streams=0, max_templates=4, **kw)


# ------------------------------------------------------------------------------------------------ stages
def test_probe_stages(probe, tables):
    """Power spectrum, un-floored log-mel and floored MFCC of loaded frames: impulses at every frame position mod 64
    (one lane / register / half each), full scale, zero, tiny noise, DC and random frames."""
    rng = np.random.default_rng(3)
    fr = []
    for p in range(64):
        for a in (0, 3, 7):
            f = np.zeros(512, np.float32)
            f[64 * a + p] = np.float32(0.7)
            fr.append(f)
    fr += [synth.from_int16(rng.integers(-32768, 32768, 512).astype(np.int16)), np.zeros(512, np.float32),
           (rng.standard_normal(512) * 1e-6).astype(np.float32), np.full(512, np.float32(-1.0))]
    fr += list((rng.standard_normal((40, 512)) * rng.uniform(1e-4, 1, (40, 1))).astype(np.float32))
    x = np.stack(fr)
    P = M.power_spectrum(x, tables)
    assert_exact(probe.power(x), P, "power spectrum")
    lm = M.log_mel(P, tables, probe.log_mel)
    for floor in (-np.inf, np.float32(-35.0)):
        mf, dlm = probe.frames(x, floor)
        assert_exact(dlm, lm, "log-mel")
        assert_exact(mf, M.dct20(np.maximum(lm, np.float32(floor)), tables), f"MFCC under floor {floor}")


# ------------------------------------------------------------------------------------------------ level 2
@pytest.mark.parametrize("pre,n_mfcc", [(0.0, 20), (0.97, 13), (0.5, 1)])
def test_extract_frames_and_features(probe, tables, pre, n_mfcc):
    """extract_mfcc(want_frames=True) at every length class (shared memory, 301 = the cap, 302 = the workspace spill)
    and signal, plus set_template / get_template."""
    ctx = make_ctx(preemphasis=pre, n_mfcc=n_mfcc)
    sig = signals(48160, 11)
    for L in LENGTHS:
        for name, s in sig.items():
            y = s[:L]
            mean, std, frames = ctx.extract_mfcc(y, want_frames=True)
            r = M.segment(y, tables, probe.log_mel, pre, n_mfcc)
            what = f"{name}, {L} samples, preemphasis {pre}, n_mfcc {n_mfcc}"
            assert_exact(frames, r["frames"], "frames: " + what)
            assert_exact(mean, r["mean"], "mean: " + what)
            assert_exact(std, r["std"], "std: " + what)
    for slot, L in enumerate((161, 15503, 48160)):
        y = sig["speech"][:L]
        ctx.set_template(slot, y)
        m, s, n = ctx.get_template(slot)
        r = M.segment(y, tables, probe.log_mel, pre, n_mfcc)
        assert n == L
        assert_exact(m, r["mean"], f"template mean ({L} samples)")
        assert_exact(s, r["std"], f"template std ({L} samples)")
    ctx.close()


@pytest.mark.parametrize("seg_lm", ["0", "1"])
def test_long_segment_block_max(probe, tables, monkeypatch, seg_lm):
    """More than 2048 frames: phase B's block-reduced max, and the floor over a loud-then-silent segment, with and
    without the log-mel workspace."""
    monkeypatch.setenv("EWK_SEG_LM", seg_lm)
    ctx = make_ctx()
    rng = np.random.default_rng(5)
    y = (rng.standard_normal(330001) * 0.1).astype(np.float32)
    y[200000:] *= np.float32(1e-6)
    assert 1 + len(y) // 160 > 2048
    mean, std, frames = ctx.extract_mfcc(y, want_frames=True)
    r = M.segment(y, tables, probe.log_mel)
    assert (r["lm"].min(axis=1) < r["floor"]).any()
    assert_exact(frames, r["frames"], "frames")
    assert_exact(mean, r["mean"], "mean")
    assert_exact(std, r["std"], "std")
    ctx.close()


def batch_model(probe, tables, pcm, offs, lens, tm, ts, pre=0.0):
    y = M.segment_values(pcm, "i16" if pcm.dtype == np.int16 else "f32")
    feats, scores = [], []
    for o, L in zip(offs, lens):
        r = M.segment(y[o:o + L], tables, probe.log_mel, pre)
        feats.append(np.concatenate([r["mean"], r["std"]]))
        scores.append(M.score(tm, ts, r["mean"], r["std"]))
    return np.stack(feats), np.asarray(scores, np.float32)


@pytest.mark.parametrize("seg_lm", ["0", "1"])
def test_similarity_batch(probe, tables, word, monkeypatch, seg_lm):
    """similarity_batch, float32 and int16, host and device input (the device input at an odd element offset: every
    frame through the scalar loader), even and odd offsets, every length class; features, scores, and `matched` with
    the threshold at the model's score and one ulp above it.  Loader branches reached are counted."""
    import torch
    monkeypatch.setenv("EWK_SEG_LM", seg_lm)
    from easywakeword_b200 import _lib
    ctx = make_ctx()
    ctx.set_template(0, word)
    ctx.set_template_features(0, *mid_range_features(*ctx.get_template(0)[:2], 0.2), len(word))
    tm, ts, _ = ctx.get_template(0)
    sig = signals(60000, 21)
    x = np.concatenate([sig["speech"], sig["loud then silent"][:20000], sig["full scale"][:3000], sig["zero"][:2000],
                        sig["speech"]])
    q = synth.to_int16(x)
    lens = [1, 2, 159, 160, 161, 255, 256, 257, 511, 512, 513, 16001, 30000, 48000, 48160, 5000, 2000]
    offs = [0, 1, 2, 3, 100, 101, 7, 8, 1000, 1001, 333, 12345, 60000, 12, 13, 80000, 83000]
    counts = np.zeros(5, np.int64)
    for pcm, fmt in ((x, "f32"), (q, "i16")):
        want_f, want_s = batch_model(probe, tables, pcm, offs, lens, tm, ts)
        assert 20 < np.nanmedian(want_s) < 90, want_s
        for o, L in zip(offs, lens):
            counts += np.bincount(M.loader_branch(o, L, 0, fmt, True, np.arange(1 + L // 160)), minlength=5)
        s, m, f = ctx.similarity_batch(0, pcm, offs, lens, threshold=75.0, want_features=True)
        assert_exact(f, want_f, f"{fmt} features")
        assert_exact(s, want_s, f"{fmt} scores")
        assert np.array_equal(m, want_s >= np.float32(75.0))
        for k in np.flatnonzero(~np.isnan(want_s))[:4]:
            thr = float(want_s[k])
            s1, m1 = ctx.similarity_batch(0, pcm, [offs[k]], [lens[k]], threshold=thr)
            assert_exact(s1, want_s[k:k + 1], "one segment at the threshold")
            assert bool(m1[0]), "score == threshold matches"
            _, m2 = ctx.similarity_batch(0, pcm, [offs[k]], [lens[k]], threshold=float(np.nextafter(want_s[k], np.float32(np.inf))))
            assert not bool(m2[0])
        # device input at an odd element offset: the base is misaligned, every frame takes the scalar loader
        dev = torch.from_numpy(np.concatenate([pcm[:1], pcm])).cuda()
        base = dev.data_ptr() + pcm.itemsize
        n = len(offs)
        s3 = np.empty(n, np.float32)
        m3 = np.empty(n, np.uint8)
        f3 = np.empty((n, 40), np.float32)
        off = np.asarray(offs, np.int64)
        ln = np.asarray(lens, np.int64)
        ctx._ck(ctx.lib.ewk_similarity_batch(ctx.h, 0, base, _lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, _lib.DEVICE,
                                             _lib.i64ptr(off), _lib.i64ptr(ln), n, 75.0, _lib.f32ptr(s3), _lib.u8ptr(m3),
                                             _lib.f32ptr(f3)))
        assert_exact(f3, want_f, f"{fmt} features, device input at an odd element offset")
        assert_exact(s3, want_s, f"{fmt} scores, device input at an odd element offset")
        for o, L in zip(offs, lens):
            counts += np.bincount(M.loader_branch(o, L, 0, fmt, False, np.arange(1 + L // 160)), minlength=5)
    print("linear-buffer loader branches: " + ", ".join(f"{n} {c}" for n, c in zip(M.BRANCH_NAMES, counts)))
    for b in (M.FAST, M.ODD, M.MASKED_LINEAR, M.SCALAR):
        assert counts[b] >= 3, (M.BRANCH_NAMES[b], counts)
    ctx.close()


# ------------------------------------------------------------------------------------------------ queue forms
@pytest.mark.parametrize("k3", ["0", "2"])
@pytest.mark.parametrize("seg_lm", ["0", "1"])
def test_queue_events(probe, tables, word, monkeypatch, k3, seg_lm):
    """Banks on small int16 and float32 rings (segments wrap), with and without pre-emphasis, under both queue forms of
    K3: every scored event's score, template and `matched` equal the model's over the segment read back from the ring.
    Loader branches of the scored segments are counted per ring format and pre-emphasis setting."""
    from easywakeword_b200.bank import WakeWordBank
    monkeypatch.setenv("EWK_K3", k3)
    monkeypatch.setenv("EWK_SEG_LM", seg_lm)
    tpls = [word, word, word]
    sets = [(0, 3), (1, 2), (2, 1)]                           # stream s scores templates [first, first + count)
    P = dict(speech_duration_min=0.5, speech_duration_max=2.8, timeout=30.0, frame_size=1600)
    report = []
    total = np.zeros(5, np.int64)
    for dt in (np.int16, np.float32):
        for pre in (0.0, 0.97):
            bank = WakeWordBank(3, tpls, buffer_seconds=4, pcm_dtype=dt, preemphasis=pre, similarity_threshold=60.0, **P)
            cfg = bank.ctx.cfg
            ring = ((cfg.ring_samples + cfg.slack_samples + 63) // 64) * 64
            fmt = "i16" if dt == np.int16 else "f32"
            wm, ws, _ = bank.ctx.get_template(0)
            for k, c0 in ((1, 0.2), (2, 0.1)):
                bank.ctx.set_template_features(k, *mid_range_features(wm, ws, c0), len(word))
            for st, (t0, nt) in enumerate(sets):
                bank.set_stream(st, template_first=t0, template_count=nt)
            feats = [bank.ctx.get_template(k)[:2] for k in range(len(tpls))]
            streams = [synth.stream(700 + 10 * i + int(pre * 7), 24.0, word, gain=(1.0, 4.0), inserts_per_10s=(3, 5))[0]
                       for i in range(3)]
            pcm = np.stack([synth.to_int16(s) if dt == np.int16 else synth.from_int16(synth.to_int16(s)) for s in streams])
            counts = np.zeros(5, np.int64)
            n_ev, mid = 0, 0
            for p0 in range(0, pcm.shape[1], 8000):
                bank.step(np.ascontiguousarray(pcm[:, p0:p0 + 8000]))
                for ev in bank.poll():
                    if ev["kind"] != 2:
                        continue
                    seg = bank.read_segment(ev)
                    r = M.segment(seg, tables, probe.log_mel, pre)
                    t0, nt = sets[int(ev["stream"])]
                    sc = np.asarray([M.score(tm, ts, r["mean"], r["std"]) for tm, ts in feats[t0:t0 + nt]], np.float32)
                    best, arg = M.best_template(sc, t0)
                    what = f"{fmt} ring, preemphasis {pre}, EWK_K3={k3}, EWK_SEG_LM={seg_lm}, event {ev}"
                    assert_exact(np.float32(ev["score"]), best, what)
                    assert int(ev["template_slot"]) == arg, (what, sc)
                    assert bool(ev["matched"]) == bool(best >= np.float32(60.0)), what
                    mid += int(((sc > 20) & (sc < 80)).sum())
                    n_ev += 1
                    F = 1 + int(ev["seg_len"]) // 160
                    counts += np.bincount(M.loader_branch(int(ev["seg_start"]) % ring, int(ev["seg_len"]), ring, fmt, True,
                                                          np.arange(F)), minlength=5)
            bank.ctx.close()
            report.append(f"{fmt} preemphasis {pre}: {n_ev} events ({mid} mid-range template scores); branches " +
                          ", ".join(f"{n} {c}" for n, c in zip(M.BRANCH_NAMES, counts)))
            assert n_ev >= 5 and mid >= 5, report[-1]
            total += counts
    print("\n".join(report))
    # segments start where the gate's float64 timing puts them, at even and odd ring positions
    for b in (M.FAST, M.ODD, M.MASKED_RING, M.SCALAR):
        assert total[b] >= 3, report


# ------------------------------------------------------------------------------------------------ K4 from PCM
def test_dense_from_pcm(probe, tables, word):
    """K4's dense scores equal dense_model fed with THIS model's frames (not the device's extract_mfcc): the dense chain is
    pinned from PCM.  Speech and decaying clicks, so that un-floored, way and edge-floored windows are all sampled."""
    from easywakeword_b200 import _lib
    tpls = [word, synth.synthetic_word(seed=5, duration=0.5)]
    ctx = _lib.Context(device=0, n_streams=2, ring_samples=200000, slack_samples=16000, pcm_format=_lib.PCM_I16,
                       max_templates=4)
    for i, t in enumerate(tpls):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, template_count=1)
    xs = [synth.stream(4100, 3.0, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0], np.zeros(48000, np.float32)]
    y = np.zeros(48000, np.float32)
    a = 0.9
    for m, p in enumerate(range(160, 48000, 320)):
        if m % 20 < 16:
            y[p] = a
            a *= 0.995
    xs[1] = y
    q = np.stack([synth.to_int16(x[:48000]) for x in xs])
    ctx.push(q)
    frames_fn = lambda pcm: M.segment_frames(pcm, tables, probe.log_mel)[0]          # noqa: E731
    hops = np.arange(0, 300, 3)
    got = ctx.dense_scores(0, 300, 0, 2)[:, hops]
    seen = set()
    for s in range(2):
        model = D.DenseModel(synth.from_int16(q[s]), tpls, frames_fn)
        assert_exact(got[s], model.scores(hops), f"stream {s}")
        for k in range(2):
            seen |= set(int(c) for c in model.classes(hops, k)[0] if c >= 0)
    assert seen == {D.UNFLOORED, D.WAY, D.EDGE}, seen
    ctx.close()
