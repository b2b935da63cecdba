"""CPU: the host side of stream migration — exported symbols, the blob header dtype against the C layout, the blob
size formula, the packing in Context.export_streams / import_streams, and the call order of WakeWordBank.move_streams."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("ewk_stream_blob_bytes", "ewk_export_streams", "ewk_import_streams")


def test_symbols_exported():
    from easywakeword_b200 import _lib, build
    build.build()
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    lib = _lib.load()
    for name in NAMES:
        assert re.search(r"\b" + name + r"\s*\(", hdr), name
        assert hasattr(lib, name) and name in lib._protos, name


def test_header_dtype_matches_c_layout(tmp_path):
    """STREAM_BLOB_HEADER_DTYPE has the size and field offsets gcc gives ewk_stream_blob"""
    from easywakeword_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    dt = _lib.STREAM_BLOB_HEADER_DTYPE
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "ewk.h"', "int main(void) {",
           '  printf("size %zu\\n", sizeof(ewk_stream_blob));',
           '  printf("MAGIC %u %d\\n", EWK_STREAM_BLOB_MAGIC, EWK_STREAM_BLOB_VERSION);']
    src += [f'  printf("{f} %zu %zu\\n", offsetof(ewk_stream_blob, {f}), sizeof(((ewk_stream_blob*)0)->{f}));'
            for f in dt.names]
    src += ["  return 0;", "}"]
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = str(tmp_path / "layout")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(REPO, "include"), str(c), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = dict((l.split()[0], l.split()[1:]) for l in subprocess.run([exe], capture_output=True, text=True).stdout.splitlines())
    assert int(out["size"][0]) == dt.itemsize == 96
    assert (int(out["MAGIC"][0]), int(out["MAGIC"][1])) == (_lib.STREAM_BLOB_MAGIC, _lib.STREAM_BLOB_VERSION)
    for f in dt.names:
        off, size = (int(v) for v in out[f])
        assert (off, size) == (dt.fields[f][1], dt.fields[f][0].itemsize), f


@pytest.mark.parametrize("ring,slack,fmt,n,nt,tail", [(160000, 19200, 1, 1, 1, 0), (160000, 19200, 1, 4096, 4, 188),
                                                     (80000, 32000, 0, 3, 2, 564), (16000, 0, 1, 0, 1, 0)])
def test_blob_bytes_formula(ring, slack, fmt, n, nt, tail):
    """the layout stated piece by piece: header, ids, 304-byte meta records, 176-byte template records, bulk rows of
    ring + block sums + chunk mean squares + K8 tail, every section and row part 16-byte aligned"""
    from easywakeword_b200 import _lib
    L = _lib.stream_blob_layout(ring, slack, fmt, n, nt, tail)
    P = -(-(ring + slack) // 64) * 64
    esz = 2 if fmt == _lib.PCM_I16 else 4
    row = P * esz + -(-(8 * (P // 1600)) // 16) * 16 + 16 * (ring // 160) + 4 * tail
    row = -(-row // 16) * 16
    meta = -(-(96 + 4 * n) // 16) * 16
    assert L["ids_offset"] == 96 and L["meta_offset"] == meta
    assert L["template_offset"] == meta + 304 * n and L["bulk_offset"] == meta + 304 * n + 176 * nt
    assert L["bulk_row_bytes"] == row and L["total_bytes"] == L["bulk_offset"] + n * row
    for k in ("meta_offset", "template_offset", "bulk_offset", "bulk_row_bytes", "ss_off", "ms_off", "tail_off"):
        assert L[k] % 16 == 0, k
    if (ring, slack, fmt, n) == (160000, 19200, 1, 4096):
        assert 1.4e9 < L["total_bytes"] < 1.6e9                       # a 4096-stream bank of 10 s int16 rings


class _FakeLib:
    """Writes a blob of `size` bytes whose header says so, and records every call."""

    def __init__(self, size=300):
        self.calls, self.size = [], size

    def ewk_stream_blob_bytes(self, h, n):
        self.calls.append(("bytes", n))
        return 1000 + n

    def ewk_export_streams(self, h, st, n, blob, cap, where):
        from easywakeword_b200 import _lib
        self.calls.append(("export", [st[i] for i in range(n)], cap, where))
        if where == _lib.HOST:
            buf = (C.c_uint8 * cap).from_address(blob)
            hdr = np.zeros(1, _lib.STREAM_BLOB_HEADER_DTYPE)
            hdr["magic"], hdr["total_bytes"], hdr["n_streams"] = _lib.STREAM_BLOB_MAGIC, self.size, n
            raw = hdr.view(np.uint8)
            for i in range(96):
                buf[i] = int(raw[i])
        return 0

    def ewk_import_streams(self, h, st, n, blob, length, where):
        self.calls.append(("import", [st[i] for i in range(n)], length, where, blob))
        return 0

    def ewk_reset_streams(self, h, st, n):
        self.calls.append(("reset", [st[i] for i in range(n)]))
        return 0

    def ewk_poll(self, h, out, cap, dropped):
        self.calls.append(("poll",))
        return 0

    rate = 0

    def ewk_stream_input(self, h, s, sr, n):
        sr._obj.value = self.rate
        return 0


def _ctx(lib, n_streams=6):
    from easywakeword_b200 import _lib
    ctx = object.__new__(_lib.Context)
    ctx.lib, ctx.h = lib, None
    ctx.cfg = _lib.Config(n_streams, 16000, 1600, _lib.PCM_I16, 4, 16, 0.0, 20, 0, 0)
    return ctx


def test_context_packing():
    from easywakeword_b200 import _lib
    lib = _FakeLib()
    ctx = _ctx(lib)
    blob = ctx.export_streams([4, 0, 2])
    assert lib.calls[0] == ("bytes", 3) and lib.calls[1][:4] == ("export", [4, 0, 2], 1003, _lib.HOST)
    assert blob.dtype == np.uint8 and blob.size == 300                 # cut to the header's total_bytes
    assert ctx.export_streams([1], where=_lib.DEVICE, out=(4096, 777)) is None
    assert lib.calls[-1] == ("export", [1], 777, _lib.DEVICE)
    with pytest.raises(ValueError):
        ctx.export_streams([1], where=_lib.DEVICE)
    with pytest.raises(ValueError):
        ctx.export_streams([1], out=(4096, 777))
    ctx.import_streams([5, 3, 1], blob)
    c = lib.calls[-1]
    assert c[:4] == ("import", [5, 3, 1], 300, _lib.HOST) and c[4] == blob.ctypes.data
    ctx.import_streams([2], (8192, 640), where=_lib.DEVICE)
    assert lib.calls[-1][:4] == ("import", [2], 640, _lib.DEVICE) and lib.calls[-1][4].value == 8192
    with pytest.raises(ValueError):
        ctx.import_streams([2**31], blob)


def _blob_with_rates(rates):
    from easywakeword_b200 import _lib
    n = len(rates)
    L = _lib.stream_blob_layout(16000, 1600, _lib.PCM_I16, n, 0, 0)
    b = np.zeros(L["bulk_offset"], np.uint8)
    h = b[:96].view(_lib.STREAM_BLOB_HEADER_DTYPE)
    h["magic"], h["version"], h["n_streams"], h["meta_bytes"] = _lib.STREAM_BLOB_MAGIC, 1, n, _lib.STREAM_META_BYTES
    h["meta_offset"] = L["meta_offset"]
    for i, r in enumerate(rates):
        o = L["meta_offset"] + i * _lib.STREAM_META_BYTES + 52
        b[o:o + 4].view(np.int32)[0] = r
    return b


def test_blob_rates():
    from easywakeword_b200.bank import stream_blob_rates
    assert stream_blob_rates(_blob_with_rates([8000, 0, 16000])).tolist() == [8000, 0, 16000]
    with pytest.raises(ValueError):
        stream_blob_rates(np.zeros(40, np.uint8))


def _bank(lib, rate=16000, n=6):
    from easywakeword_b200.bank import WakeWordBank
    b = object.__new__(WakeWordBank)
    b.ctx, b.sample_rate, b.n_streams = _ctx(lib, n), rate, n
    return b


def test_move_streams_order():
    """poll the destination, export, import (which polls again), poll the source, reset the source slots"""
    sl, dl = _FakeLib(), _FakeLib()
    src, dst = _bank(sl), _bank(dl)
    from easywakeword_b200 import bank as bank_mod
    real = bank_mod.stream_blob_rates
    bank_mod.stream_blob_rates = lambda blob: np.zeros(2, np.int32)
    try:
        s_ev, d_ev = src.move_streams([3, 1], dst, [0, 5])
    finally:
        bank_mod.stream_blob_rates = real
    assert [c[0] for c in dl.calls] == ["poll", "poll", "import"]
    assert dl.calls[-1][1] == [0, 5]
    assert [c[0] for c in sl.calls] == ["bytes", "export", "poll", "reset"]
    assert sl.calls[1][1] == [3, 1] and sl.calls[-1] == ("reset", [3, 1])
    assert len(s_ev) == 0 and len(d_ev) == 0
    # within one bank: slots that received a stream are not reset
    one = _FakeLib()
    b = _bank(one)
    bank_mod.stream_blob_rates = lambda blob: np.zeros(2, np.int32)
    try:
        b.move_streams([1, 2], b, [2, 4])
    finally:
        bank_mod.stream_blob_rates = real
    assert one.calls[-1] == ("reset", [1])
    with pytest.raises(ValueError):
        b.move_streams([1, 2], b, [3])


def test_import_refuses_other_rates():
    from easywakeword_b200 import bank as bank_mod
    lib = _FakeLib()
    b = _bank(lib, rate=16000)
    with pytest.raises(ValueError, match="takes 8000 Hz"):
        b.import_streams([0], _blob_with_rates([8000]))
    assert lib.calls == []                                             # refused before any library call
    b.import_streams([0, 1], _blob_with_rates([16000, 0]))
    assert [c[0] for c in lib.calls] == ["poll", "import"]
    assert bank_mod.stream_blob_rates(_blob_with_rates([0])).tolist() == [0]


def test_move_streams_refuses_other_rates_before_draining():
    """a source stream latched to another rate than the destination's: ValueError before any poll, export or import"""
    sl, dl = _FakeLib(), _FakeLib()
    sl.rate = 8000
    src, dst = _bank(sl, rate=8000), _bank(dl, rate=16000)
    with pytest.raises(ValueError, match="takes 8000 Hz"):
        src.move_streams([3], dst, [0])
    assert dl.calls == [] and sl.calls == []
