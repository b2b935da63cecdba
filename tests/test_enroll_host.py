"""CPU: the host side of batched template enrolment (ewk_set_templates, ewk_set_templates_from_streams) — exported
symbols and prototypes, the published slot limits, and WakeWordBank.enroll's argument checks, which must refuse a bad
list before any call reaches the library (the library's own checks and every result need a device: test_gpu_enroll.py)."""
import os
import re

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_symbols_exported():
    from easywakeword_b200 import _lib
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    lib = _lib.load()
    for name in ("ewk_set_templates", "ewk_set_templates_from_streams"):
        assert re.search(r"\b" + name + r"\s*\(", hdr), name
        assert hasattr(lib, name) and name in lib._protos, name


def test_limits_published():
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    assert re.search(r"#define\s+EWK_MAX_TEMPLATE_SLOTS\s+4096\b", hdr)
    assert re.search(r"#define\s+EWK_MAX_STREAM_TEMPLATES\s+64\b", hdr)
    # the queue-form K3 keeps one score per template of a stream's range in shared memory
    src = open(os.path.join(REPO, "easywakeword_b200", "csrc", "ewk_streams.cuh")).read()
    assert "__shared__ float sc_s[EWK_MAX_STREAM_TEMPLATES];" in src


class _NoLibrary:
    """A context that fails the test if enroll reaches it."""

    def __getattr__(self, name):
        raise AssertionError(f"enroll reached the context ({name}) with a list it must refuse")


def _bank():
    from easywakeword_b200.bank import WakeWordBank
    b = WakeWordBank.__new__(WakeWordBank)
    b.ctx = _NoLibrary()
    b.params = dict(template_first=0, template_count=1)
    return b


def test_enroll_argument_errors_before_the_library():
    b = _bank()
    with pytest.raises(ValueError, match="consecutive"):            # stream 2 again, slot 7 after 5
        b.enroll(([1, 2, 2], [0, 0, 9000], [8000, 8000, 8000]), [4, 5, 7])
    with pytest.raises(ValueError, match="consecutive"):            # a repeated stream going backwards
        b.enroll(([3, 3], [0, 9000], [8000, 8000]), [10, 9])
    with pytest.raises(ValueError, match="consecutive"):            # the same slot twice for one stream
        b.enroll(([0, 0], [0, 9000], [8000, 8000]), [6, 6])
    with pytest.raises(ValueError, match="one of each"):            # mismatched lengths
        b.enroll(([0, 1], [0, 0], [8000, 8000]), [0, 1, 2])
    with pytest.raises(ValueError, match="one of each"):
        b.enroll(([0, 1], [0], [8000, 8000]), [0, 1])
    ev = np.zeros(3, dtype=[("stream", "<i4"), ("seg_start", "<i8"), ("seg_len", "<i4")])
    ev["stream"] = [5, 6, 5]
    with pytest.raises(ValueError, match="stream 5"):               # structured rows: stream 5 at slots 0 and 2
        b.enroll(ev, [0, 1, 2])
    with pytest.raises(ValueError, match="more than 64"):
        b.enroll(([0] * 65, list(range(65)), [800] * 65), list(range(65)))


def test_enroll_ranges():
    from easywakeword_b200.bank import enroll_ranges
    r = enroll_ranges([4, 1, 4, 4, 9], [0] * 5, [1] * 5, [20, 3, 21, 22, 0])
    assert r == {4: (20, 3, 0), 1: (3, 1, 1), 9: (0, 1, 4)}
    assert list(r) == [4, 1, 9]
    assert enroll_ranges([], [], [], []) == {}
    assert enroll_ranges([0] * 64, [0] * 64, [1] * 64, list(range(4032, 4096))) == {0: (4032, 64, 0)}


def test_enroll_calls_once_then_sets_each_stream():
    """a valid list: one library call for all segments, then set_stream per stream with its range and durations"""
    from easywakeword_b200 import _lib
    from easywakeword_b200.bank import WakeWordBank
    calls = []

    class Ctx:
        def set_templates_from_streams(self, slots, streams, starts, lens, want_vad=False):
            calls.append(("install", list(slots), list(streams), list(starts), list(lens), want_vad))
            v = np.zeros(len(slots), _lib.VAD_DTYPE)
            v["duration_s"] = [0.5, 0.7, 0.9][:len(slots)]
            v["voiced"] = [1, 0, 1][:len(slots)]
            return v

        def set_stream_params(self, stream, **p):
            calls.append(("params", stream, p["template_first"], p["template_count"], p["speech_duration_min"],
                          p["speech_duration_max"], p["similarity_threshold"]))

    b = WakeWordBank.__new__(WakeWordBank)
    b.ctx = Ctx()
    b.params = dict(template_first=0, template_count=1, similarity_threshold=70.0, speech_duration_min=0.4,
                    speech_duration_max=0.8)
    ev = np.zeros(3, dtype=_lib.EVENT_DTYPE)
    ev["stream"] = [7, 2, 7]
    ev["seg_start"] = [100, 200, 300]
    ev["seg_len"] = [8000, 9000, 10000]
    vad = b.enroll(ev, [40, 3, 41])
    assert calls[0] == ("install", [40, 3, 41], [7, 2, 7], [100, 200, 300], [8000, 9000, 10000], True)
    assert calls[1] == ("params", 7, 40, 2, 0.5, 1.0, 70.0)
    assert calls[2] == ("params", 2, 3, 1, 0.3, 2.0, 70.0)      # not voiced: the constructor's fallbacks
    assert len(calls) == 3 and len(vad) == 3
    calls.clear()
    b.enroll(([1], [0], [8000]), [9], set_durations=False)
    assert calls[0][-1] is False
    assert calls[1][:4] == ("params", 1, 9, 1) and calls[1][4:6] == (0.4, 0.8)


def test_template_slots_below_templates_refused():
    from easywakeword_b200.bank import WakeWordBank
    with pytest.raises(ValueError, match="template_slots"):
        WakeWordBank(2, [np.zeros(800, np.float32)] * 3, template_slots=2)
