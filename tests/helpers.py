"""Shared test helpers (stream regeneration identical to oracle/gen_golden.py)."""
import hashlib

import numpy as np

from easywakeword_b200 import synth


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def detect_stream_for(case, word):
    if case.get("special") == "config1":     # SURVEY §8(d) config 1
        rng = np.random.default_rng(7)
        s = (rng.standard_normal(400000) * 0.002).astype(np.float32)
        s[224000:224000 + len(word)] += (3.0 * word).astype(np.float32)
        return s
    x, _ = synth.stream(case["seed"], case["seconds"], word, noise_sigma=case["noise"], gain=tuple(case["gain"]),
                        zero_gaps=case.get("zero_gaps", 0), distractor_prob=case.get("distractor_prob", 0.0),
                        inserts_per_10s=tuple(case.get("inserts", (1, 3))))
    return synth.from_int16(synth.to_int16(x))


def mfcc_rel_l2(a, b):
    """Per-frame relative L2 error of MFCC matrices [20, F] (SURVEY §7 'hard parts': the parity metric)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    num = np.linalg.norm(a - b, axis=0)
    den = np.linalg.norm(b, axis=0)
    return num / np.maximum(den, 1e-30)


class K3Probe:
    """tests/k3_probe.cu built with the library's nvcc flags into `out_dir` and loaded with ctypes.  tables() runs on
    the host only; log_mel / frames / power need a device."""

    def __init__(self, out_dir):
        import ctypes as C
        import os
        import subprocess
        from easywakeword_b200 import build
        here = os.path.dirname(os.path.abspath(__file__))
        so = os.path.join(str(out_dir), "k3_probe.so")
        cmd = [build._nvcc(), *build.NVCC_FLAGS, "-I", build.CSRC, "-o", so,
               os.path.join(here, "k3_probe.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed building the K3 probe:\n" + r.stdout + r.stderr)
        lib = C.CDLL(so)
        f32p, vp = C.POINTER(C.c_float), C.c_void_p
        lib.k3p_tables.restype, lib.k3p_tables.argtypes = C.c_longlong, [vp, C.c_longlong, C.POINTER(C.c_longlong)]
        lib.k3p_log_mel.restype, lib.k3p_log_mel.argtypes = C.c_int, [f32p, f32p, C.c_longlong]
        lib.k3p_frames.restype, lib.k3p_frames.argtypes = C.c_int, [f32p, C.c_int, C.c_float, f32p, f32p]
        lib.k3p_power.restype, lib.k3p_power.argtypes = C.c_int, [f32p, C.c_int, f32p]
        self.lib, self.C = lib, C

    def tables(self):
        """-> (image bytes, (sizeof(DeviceTables), FRAME_IMAGE_OFFSET, sizeof(FrameTables)))."""
        C = self.C
        sizes = (C.c_longlong * 3)()
        n = self.lib.k3p_tables(None, 0, sizes)
        buf = (C.c_ubyte * n)()
        assert self.lib.k3p_tables(buf, n, sizes) == n
        return bytes(buf), tuple(int(v) for v in sizes)

    def _p(self, a):
        return a.ctypes.data_as(self.C.POINTER(self.C.c_float))

    def log_mel(self, S):
        """TEN_LOG10_2 * __log2f(fmaxf(S, 1e-10f)) on the device (the model's log_fn)."""
        S = np.ascontiguousarray(S, np.float32)
        out = np.empty_like(S)
        if S.size:
            assert self.lib.k3p_log_mel(self._p(S), self._p(out), S.size) == 0
        return out

    def frames(self, x, floor_db=-np.inf):
        """warp_frame_mfcc on loaded frames [n, 512] -> (MFCC [n, 20], un-floored log-mel [n, 128])."""
        x = np.ascontiguousarray(x, np.float32).reshape(-1, 512)
        m = np.empty((len(x), 20), np.float32)
        lm = np.empty((len(x), 128), np.float32)
        assert self.lib.k3p_frames(self._p(x), len(x), float(floor_db), self._p(m), self._p(lm)) == 0
        return m, lm

    def power(self, x):
        """warp_power_spectrum on loaded frames [n, 512] -> P [n, 257]."""
        x = np.ascontiguousarray(x, np.float32).reshape(-1, 512)
        P = np.empty((len(x), 257), np.float32)
        assert self.lib.k3p_power(self._p(x), len(x), self._p(P)) == 0
        return P


def dense_geometry_sets(plan_fn):
    """Template-length sets (1-8 templates of 640 .. 48000 samples, remainders mod 160 on both sides of 96 so that
    windows have 1 and 2 right-edge frames) through K4's planner -> {(DH, threads, CTAs per SM): lengths}, one set per
    reachable geometry: the one with the fewest templates and samples, so that a device test of every geometry stays
    cheap.  plan_fn(lengths) -> (DH, threads, CTAs per SM, shared-memory bytes)."""
    grid = [640, 1001, 4097, 8000, 15503, 16000, 24013, 33406, 40111, 48000]
    sets = set()
    for T in range(1, 9):
        for a in grid:
            for b in grid:
                if a <= b:
                    sets.add(tuple(sorted([a] * (T - 1) + [b])))
        for i in range(len(grid)):
            sets.add(tuple(sorted((grid * 2)[i:i + T])))
    rng = np.random.default_rng(160)
    for _ in range(400):
        T = int(rng.integers(1, 9))
        sets.add(tuple(sorted(int(v) for v in rng.integers(640, 48001, T))))
    reach = {}
    for lens in sorted(sets, key=lambda s: (len(s), sum(s), s)):
        try:
            g = tuple(plan_fn(list(lens))[:3])
        except ValueError:                       # does not fit shared memory: ewk_dense_scores refuses it too
            continue
        reach.setdefault(g, list(lens))
    return reach
