"""K8 (resample_push_kernel, csrc/ewk_resample_push.cuh) against an exact float32 model of the arithmetic it documents:
output n is the sequential fmaf chain, from +0, over taps j = 0 .. 2W-1 of H[j][p] * x[k_c - W + 1 + j].  The model
(oracle.resample_restated.resample_chain) restates that chain with a correctly rounded fmaf, so every GPU test here
compares by np.array_equal: a wrong tap, phase, window slot, tail sample or ring index fails however small its effect.

The rate matrix reaches every kernel instance and plan branch of ewk_ctx::launch_fir (ewk_api.cu); the CPU tests
below restate that plan and assert so.  On the CPU the file also pins the model itself: fmaf32 against exact rational
arithmetic, the chain against float64 within Higham's bound, and the library's host-built table against the oracle's."""
import os
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from oracle import resample_restated as R

# sr -> (the K8 instance or plan branch it exercises)
RATES = {
    2000: "fast L8 M1", 4000: "fast L4 M1", 8000: "fast L2 M1", 32000: "fast L1 M2",
    6000: "fast L8 M3", 12000: "fast L4 M3", 24000: "fast L2 M3", 48000: "fast L1 M3",
    1000: "generic, L=16, tile raised by need",
    11025: "generic, table in global memory", 44100: "generic, table in global memory", 22050: "generic",
    3205: "generic, L=3200", 47995: "generic, L=3200",
    64000: "generic, L=1, table staged", 96000: "generic, L=1, table staged",
    192000: "generic, tile reduced by the span cap", 384000: "generic",
    768000: "generic, table in global memory, 8994-float tail",
}
FAST = [2000, 4000, 8000, 32000, 6000, 12000, 24000, 48000]

# ------------------------------------------------------------------------------------------------ launch plan
RSP_THREADS, RSP_TABLE_SMEM, RSP_GENERIC_TILE, SPAN_CAP = 256, 8192, 2048, 24576


def _rsp_k(m):
    return 11 if m == 3 else 15


def fir_plan(sr):
    """ewk_ctx::launch_fir's plan for sr, restated: the path, tile, staged input span and where the table lives."""
    d = R.design(sr)
    W, L, M = d["W"], d["L"], d["M"]
    taps = 2 * W
    table_smem = taps * L <= RSP_TABLE_SMEM
    plan = dict(W=W, L=L, M=M, table_smem=table_smem, reduced=False, raised=False)
    if L in (1, 2, 4, 8) and M <= 3 and table_smem and (RSP_THREADS // L) * _rsp_k(M) * M >= taps + M:
        plan.update(fast_m=M, tile=RSP_THREADS * _rsp_k(M), span=(RSP_THREADS // L) * _rsp_k(M) * M + taps + M + 1)
    else:
        def span(tile):
            return (tile * M + L - 1) // L + taps + 1
        tile = RSP_GENERIC_TILE
        while tile > RSP_THREADS and span(tile) > SPAN_CAP:
            tile //= 2
            plan["reduced"] = True
        need = (taps * L + M - 1) // M
        raised = (need + RSP_THREADS - 1) // RSP_THREADS * RSP_THREADS
        plan["raised"] = raised > tile
        tile = max(tile, raised)
        plan.update(fast_m=0, tile=tile, span=span(tile))
    plan["smem"] = 4 * (256 + taps + (taps * L if table_smem else 0) + plan["span"])
    return plan


def test_rate_matrix_reaches_every_plan_branch():
    plans = {sr: fir_plan(sr) for sr in RATES}
    fast = {(p["L"], p["M"]) for p in plans.values() if p["fast_m"]}
    # every instance (M = 1, 2, 3) at every phase count (L = 1, 2, 4, 8); L = M = 1 is 16 kHz, which is not resampled
    assert fast == {(L, M) for L in (2, 4, 8) for M in (1, 3)} | {(1, 2), (1, 3)}, fast
    assert {sr for sr, p in plans.items() if p["fast_m"]} == set(FAST)
    gen = {sr: p for sr, p in plans.items() if not p["fast_m"]}
    assert gen[1000]["raised"] and gen[1000]["L"] == 16
    assert all(not p["table_smem"] for sr, p in gen.items() if sr in (11025, 44100, 3205, 47995, 768000))
    assert gen[3205]["L"] == gen[47995]["L"] == 3200
    assert all(p["table_smem"] and p["L"] == 1 for sr, p in gen.items() if sr in (64000, 96000, 384000))
    assert gen[192000]["reduced"] and not gen[192000]["raised"]
    assert 2 * gen[768000]["W"] == 8994 and not gen[768000]["table_smem"]
    for sr, p in plans.items():
        assert p["smem"] <= 200 * 1024, sr                           # launch_fir refuses above this
    for sr in (2000, 4000, 8000, 6000, 12000, 24000, 32000, 48000):      # the fast path's windows fit its span
        p = plans[sr]
        b_max = (RSP_THREADS // p["L"] - 1) * _rsp_k(p["M"]) * p["M"] + p["M"] - 1
        assert b_max + 2 * p["W"] + _rsp_k(p["M"]) * p["M"] - 1 < p["span"], sr


# ------------------------------------------------------------------------------------------------ the model (CPU)
def _fma_exact(a, b, c):
    """float32 fmaf by rational arithmetic: the nearest float32 to a * b + c, ties to the even significand."""
    t = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    f = np.float32(float(t))
    cands = [f, np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))]
    return min(cands, key=lambda v: (abs(Fraction(float(v)) - t), int(np.float32(v).view(np.uint32)) & 1))


def test_fmaf32_rounds_once():
    rng = np.random.default_rng(11)
    n = 6000
    a = rng.standard_normal(n).astype(np.float32)
    b = (rng.standard_normal(n) * 1e-3).astype(np.float32)
    c = (rng.standard_normal(n) * rng.choice([1e-9, 1e-6, 1e-3, 1.0], n)).astype(np.float32)
    m = 1500                                                    # products at or near half an ulp of c: ties
    a[:m] = np.float32(2.0 ** -24)
    b[:m] = (1 + rng.integers(-3, 4, m) * 2.0 ** -23).astype(np.float32)
    c[:m] = np.float32(1.0)
    a[m:2 * m] = np.float32(3 * 2.0 ** -25)
    b[m:2 * m] = np.float32(1.0)
    c[m:2 * m] = (1 + rng.integers(0, 100, m) * 2.0 ** -23).astype(np.float32)
    got = R.fmaf32(a, b, c)
    want = np.array([_fma_exact(a[i], b[i], c[i]) for i in range(n)], np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # rounding the float64 sum to float32 rounds twice and misses this one: the exact value is just above the
    # midpoint between 1 + 2^-23 and 1 + 2^-22, the float64 sum lands on it and ties to even (1 + 2^-22)
    a1, b1, c1 = np.float32(1 + 2.0 ** -15), np.float32(2.0 ** -24 * (1 - 2.0 ** -15)), np.float32(1 + 2.0 ** -23)
    assert np.float32(np.float64(a1) * np.float64(b1) + np.float64(c1)) == np.float32(1 + 2.0 ** -22)
    assert R.fmaf32(a1, b1, c1) == _fma_exact(a1, b1, c1) == np.float32(1 + 2.0 ** -23)


def _square(n, sr, f=1000.3, amp=1.0):
    return (amp * np.sign(np.sin(2 * np.pi * f * (np.arange(n) + 0.5) / sr))).astype(np.float32)


def _chain64(x, sr, n_out):
    """float64 sum of the float32 table's products and sum |h x| for outputs [0, n_out) of x."""
    d = R.design(sr)
    W, L, M = d["W"], d["L"], d["M"]
    H = R.phase_table(d).astype(np.float32).astype(np.float64)
    n = np.arange(n_out, dtype=np.int64)
    kc, p = (n * M) // L, (n * M) % L
    xp = np.concatenate([np.zeros(2 * W), x.astype(np.float64), np.zeros(2 * W + M)])
    base = kc - W + 1 + 2 * W
    y, a = np.zeros(n_out), np.zeros(n_out)
    for j in range(2 * W):
        v = xp[base + j] * H[j, p]
        y += v
        a += np.abs(v)
    return y, a


@pytest.mark.parametrize("sr", sorted(RATES))
def test_chain_within_higham_bound_of_float64(sr):
    """|chain - exact| <= gamma_2W sum|h x|, gamma_k = k u / (1 - k u), u = 2^-24, on full-scale square waves."""
    W = R.design(sr)["W"]
    n_out = 400 if sr > 100000 else 1200
    x = _square(R.design(sr)["M"] * n_out // R.design(sr)["L"] + 2 * W + 8, sr)
    got = R.resample_chain(x, sr, n_out=n_out)
    y, a = _chain64(x, sr, n_out)
    u = 2.0 ** -24
    gamma = 2 * W * u / (1 - 2 * W * u)
    err = np.abs(got.astype(np.float64) - y)
    assert (err <= gamma * a).all(), float(np.max(err / (gamma * a)))
    print(f"{sr}: max |err| {err.max():.2e}, max |err| / (u sum|hx|) {np.max(err / (u * a)):.1f} (bound {2 * W})")


def test_chain_input_formats_and_ring_quantize():
    from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE
    q = np.array([-32768, -1, 0, 1, 32767], np.int16)
    assert np.array_equal(R.chain_input(q), np.array([-1, -2 ** -15, 0, 2 ** -15, 1 - 2 ** -15], np.float32))
    codes = np.arange(256, dtype=np.uint8)
    assert np.array_equal(R.chain_input(codes, "ulaw") * 32768, ULAW_TABLE.astype(np.float32))
    assert np.array_equal(R.chain_input(codes, "alaw") * 32768, ALAW_TABLE.astype(np.float32))
    y = np.array([1.5, 1.0, -1.0, -1.2, 0.5 / 32768, 1.5 / 32768, -2.5 / 32768, 32766.5 / 32768], np.float32)
    assert R.ring_quantize(y).tolist() == [32767, 32767, -32768, -32768, 0, 2, -2, 32766]
    # windows: the same outputs whichever buffer holds them
    x = _square(3000, 44100, 311.0, 0.7)
    whole = R.resample_chain(x, 44100)
    assert np.array_equal(R.resample_chain(x[500:], 44100, in_first=500, out_first=300, n_out=500),
                          R.resample_chain(np.concatenate([np.zeros(500, np.float32), x[500:]]), 44100)[300:800])
    assert np.array_equal(R.resample_chain(x, 44100, out_first=7, n_out=1), whole[7:8])


def _table_driver(tmp_path):
    """Compile a host-only program that prints the library's float32 table for each rate given."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    from easywakeword_b200 import build
    try:
        inc = [os.path.join(os.path.dirname(os.path.dirname(build._nvcc())), "include")]
    except RuntimeError:
        inc = []
    inc += [os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include"), "/usr/local/cuda/include"]
    inc = [p for p in inc if os.path.exists(os.path.join(p, "cuda_runtime.h"))]
    if not inc:
        pytest.skip("no cuda_runtime.h")
    src = tmp_path / "rs_table.cpp"
    src.write_text(
        '#include "ewk_resample.cuh"\n#include <cstdio>\n#include <cstdlib>\n'
        "int main(int argc, char** argv) {\n"
        "    for (int i = 1; i < argc; i++) {\n"
        "        ewk::ResampleDesign d;\n"
        "        if (!ewk::rs_design(atoi(argv[i]), d)) return 2;\n"
        "        std::vector<float> H;\n"
        "        ewk::rs_build_table(d, H);\n"
        "        int hdr[3] = {d.W, d.L, d.M};\n"
        "        fwrite(hdr, 4, 3, stdout);\n"
        "        fwrite(H.data(), 4, H.size(), stdout);\n"
        "    }\n    return 0;\n}\n")
    exe = str(tmp_path / "rs_table")
    csrc = os.path.join(os.path.dirname(build.__file__), "csrc")
    r = subprocess.run([gxx, "-std=c++17", "-O2", "-I", csrc, "-I", inc[0], str(src), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_host_table_equals_oracle_float32(tmp_path):
    """rs_design / rs_build_table (csrc/ewk_resample.cuh, what the device reads) against the oracle's table rounded
    to float32, by value: the entry at tau = -W is +0 in C++ and -0 in numpy, which no output can see."""
    exe = _table_driver(tmp_path)
    rates = sorted(RATES) + [88200, 176400]
    raw = subprocess.run([exe] + [str(sr) for sr in rates], capture_output=True, check=True).stdout
    off = 0
    for sr in rates:
        W, L, M = np.frombuffer(raw, np.int32, 3, off)
        off += 12
        d = R.design(sr)
        assert (W, L, M) == (d["W"], d["L"], d["M"]), sr
        H = np.frombuffer(raw, np.float32, 2 * W * L, off).reshape(2 * W, L)
        off += 4 * H.size
        want = R.phase_table(d).astype(np.float32)
        bad = np.argwhere(H != want)
        assert bad.size == 0, (sr, bad[:4].tolist())
    assert off == len(raw)


# ------------------------------------------------------------------------------------------------ GPU
def _first_diff(got, want):
    bad = np.argwhere(got != want)
    if bad.size == 0:
        return None
    i = tuple(bad[0])
    return f"{len(bad)} of {got.size} differ; first at {i}: device {got[i]!r}, model {want[i]!r}"


def _assert_equal(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    msg = _first_diff(got, want)
    assert msg is None, f"{what}: {msg}"


@pytest.fixture(scope="module")
def ctx():
    from easywakeword_b200 import _lib
    c = _lib.Context(device=0, n_streams=0, max_templates=1)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sr", FAST + [1000, 96000])
def test_taps_seen_through_the_kernel(ctx, sr):
    """A unit impulse at input k0 gives out[n] = H[k0 - k_c(n) + W - 1][p(n)] exactly (the other products are 0); rows
    with k0 = W .. 3W + M - 1 see every (j, p) of the table, at many CTA and lane positions."""
    d = R.design(sr)
    W, L, M = d["W"], d["L"], d["M"]
    H = R.phase_table(d).astype(np.float32)
    rows = M + 2 * W
    n_in = 4 * W + rows + M
    k0 = W + np.arange(rows)
    x = np.zeros((rows, n_in), np.float32)
    x[np.arange(rows), k0] = 1.0
    got = ctx.resample(x, sr)
    n = np.arange(got.shape[1], dtype=np.int64)
    kc, p = (n * M) // L, (n * M) % L
    j = k0[:, None] - kc[None, :] + W - 1
    inside = (j >= 0) & (j < 2 * W)
    want = np.where(inside, H[np.clip(j, 0, 2 * W - 1), np.broadcast_to(p, j.shape)], np.float32(0))
    seen = np.zeros((2 * W, L), bool)
    seen[j[inside], np.broadcast_to(p, j.shape)[inside]] = True
    assert seen.all(), "the impulses do not reach every tap"
    bad = np.argwhere(got != want)
    if bad.size:
        r, c = bad[0]
        pytest.fail(f"{sr} Hz: {len(bad)} outputs differ; first: row {r} output {c} = tap (j={j[r, c]}, p={p[c]}): "
                    f"device {got[r, c]!r}, table {want[r, c]!r}")


def _one_shot_cases(sr):
    """-> list of (label, input [rows, n] f32 or i16, in_first, out_first, n_out)."""
    plan = fir_plan(sr)
    W, L, M, tile = plan["W"], plan["L"], plan["M"], plan["tile"]
    rng = np.random.default_rng(sr)
    cases = []
    for n in (1, 2, W - 1, W, 2 * W + 1):                       # shorter than the filter .. just past it
        x = rng.uniform(-1, 1, (7, n)).astype(np.float32)
        x[3] = np.where(x[3] > 0, 1.0, -1.0)
        cases.append((f"len {n}", x, 0, 0, None))
        cases.append((f"len {n} i16", rng.integers(-32768, 32768, (7, n)).astype(np.int16), 0, 0, None))
    # across tile boundaries: up to 3 tiles + 1 of one row (outputs tile - 1, tile, tile + 1 ... are the same
    # samples whichever n_out asks for them; each call ends its last tile elsewhere)
    big = 3 * tile + 1
    n_in = big * M // L + 2 * W + 3
    sq = _square(n_in, sr, 997.1)
    sq[n_in // 2:] = (0.25 * rng.standard_normal(n_in - n_in // 2)).astype(np.float32)
    sq16 = np.where(np.arange(n_in) % 53 < 26, -32768, 32767).astype(np.int16)[None]
    sq16[0, n_in // 3:] = rng.integers(-32768, 32768, n_in - n_in // 3)
    for n_out in (tile - 1, tile, tile + 1, 3 * tile - 1, 3 * tile, big):
        cases.append((f"n_out {n_out} (tile {tile})", sq[None], 0, 0, n_out))
    cases.append(("int16 extremes, 3 tiles + 1", sq16, 0, 0, big))
    # windows: buffer starting at in_first > 0, out_first not a multiple of L, outputs before the buffer's reach and
    # past its end, a single output
    w_in = sq[W + 5:W + 5 + tile * M // L + 2 * W]
    first = (W + 5) * L // M
    cases.append(("in_first > 0", w_in[None], W + 5, first + (L > 1), tile // 2 + 3))
    cases.append(("before reach, past end", w_in[None], W + 5, max(0, first - 2 * W * L // M - 7),
                  len(w_in) * L // M + 4 * W * L // M + 9))
    cases.append(("n_out 1", w_in[None], W + 5, first + 2 * L + 1, 1))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("sr", sorted(RATES), ids=[f"{sr}-{RATES[sr].split(',')[0]}" for sr in sorted(RATES)])
def test_one_shot_equals_chain(ctx, sr):
    cases = _one_shot_cases(sr)
    longest = {}                                                # one model run per input for the n_out series
    for _, x, in_first, out_first, n_out in cases:
        if n_out is not None and in_first == out_first == 0:
            longest[id(x)] = max(longest.get(id(x), 0), n_out)
    models = {}
    for label, x, in_first, out_first, n_out in cases:
        got = ctx.resample(x, sr, in_first=in_first, out_first=out_first, n_out=n_out)
        if id(x) in longest and in_first == out_first == 0:
            if id(x) not in models:
                models[id(x)] = R.resample_chain(x, sr, n_out=longest[id(x)])
            want = models[id(x)][:, :n_out]
        else:
            want = R.resample_chain(x, sr, in_first=in_first, out_first=out_first, n_out=n_out)
        _assert_equal(got, want, f"{sr} Hz {RATES[sr]}, {label}")


@pytest.mark.gpu
@pytest.mark.parametrize("sr", sorted(RATES))
def test_device_error_against_float64(ctx, sr):
    """The device's float32 accumulation error on full-scale square waves stays within gamma_2W sum|h x| of the
    float64 sum of the same products (printed with -s: the figures include/ewk.h and DESIGN.md quote)."""
    W = R.design(sr)["W"]
    n_out = 400 if sr > 100000 else 1200
    x = _square(R.design(sr)["M"] * n_out // R.design(sr)["L"] + 2 * W + 8, sr)
    got = ctx.resample(x, sr, n_out=n_out)
    y, a = _chain64(x, sr, n_out)
    u = 2.0 ** -24
    err = np.abs(got.astype(np.float64) - y)
    assert (err <= 2 * W * u / (1 - 2 * W * u) * a).all()
    print(f"\n{sr} Hz: device max |err| vs float64 {err.max():.2e} ({20 * np.log10(err.max()):.1f} dBFS), "
          f"max |err| / (u sum|hx|) {np.max(err / (u * a)):.1f}, peak |y| {np.abs(y).max():.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [8000, 44100, 48000, 2000])
def test_one_shot_4096_rows(ctx, sr):
    """4096 short rows (grid.y): row y is pattern y % 61 scaled by 2^-(y % 5), which scales its outputs exactly."""
    W = R.design(sr)["W"]
    rng = np.random.default_rng(sr + 7)
    pat = rng.uniform(-1, 1, (61, W + 9)).astype(np.float32)
    pat[::4] = np.where(pat[::4] > 0, 1.0, -1.0)
    y = np.arange(4096)
    x = pat[y % 61] * (np.float32(2.0) ** -(y % 5)).astype(np.float32)[:, None]
    got = ctx.resample(x, sr)
    base = R.resample_chain(pat, sr)
    want = base[y % 61] * (np.float32(2.0) ** -(y % 5)).astype(np.float32)[:, None]
    _assert_equal(got, want, f"{sr} Hz, 4096 rows")


# ---- landing in the rings
RING_R, RING_SLACK = 16000, 4011          # about 1 s: landings wrap several times


def _bank(n, ring_fmt):
    from easywakeword_b200 import _lib
    c = _lib.Context(device=0, n_streams=n, ring_samples=RING_R, slack_samples=RING_SLACK, pcm_format=ring_fmt,
                     max_templates=1)
    c.set_stream_params(-1, live=1)          # reads see what has landed, and no push guard waits for a tick
    return c


def _overshooting_feed(n_rows, n, sr, kind, seed):
    """Full-scale square waves (band-limiting makes them overshoot 1.0) with stretches of noise -> (pushed, float)."""
    from easywakeword_b200 import synth
    rng = np.random.default_rng(seed)
    y = np.empty((n_rows, n))
    for r in range(n_rows):
        y[r] = np.sign(np.sin(2 * np.pi * (311.7 + 97 * r) * (np.arange(n) + 0.5) / sr))
        a = n // 3 + 401 * r
        y[r, a:a + n // 4] = np.clip(0.3 * rng.standard_normal(n // 4), -1, 1)[:len(y[r, a:a + n // 4])]
    if kind == "f32":
        return y.astype(np.float32), None
    q = synth.to_int16(y)
    q[:, ::7] = np.where(q[:, ::7] > 0, 32767, -32768)
    if kind == "i16":
        return q, None
    from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE
    table = (ULAW_TABLE if kind == "ulaw" else ALAW_TABLE).astype(np.int32)
    order = np.argsort(table, kind="stable")
    i = np.clip(np.searchsorted(table[order], q.astype(np.int32)), 0, 255)
    return order[i].astype(np.uint8), kind


def _push_sizes(sr, total):
    """1-sample pushes, pushes shorter than W that land nothing, and pushes landing several tiles."""
    plan = fir_plan(sr)
    W, L, M, tile = plan["W"], plan["L"], plan["M"], plan["tile"]
    several = min(3 * tile + 17, RING_R - 64) * M // L
    cyc = [1, W // 3, W - W // 3 - 2, 1, 7, sr // 50, several, 1, 997, W - 1, sr // 3 + 1, several // 2 + 5]
    out, pos, i = [], 0, 0
    while pos < total:
        k = min(cyc[i % len(cyc)], total - pos)
        out.append(k)
        pos += k
        i += 1
    return out


def _expect(xf_rows, sr, law, ring_fmt):
    """What the ring holds for each whole feed, read back as float32."""
    from easywakeword_b200 import _lib
    y = R.resample_chain(xf_rows, sr, law=law)
    if ring_fmt == _lib.PCM_I16:
        return R.ring_quantize(y).astype(np.float32) / np.float32(32768)
    return y


def _check_ring(c, s, written, want, what):
    n = min(written, RING_R)
    if n:
        _assert_equal(c.read_last(s, n), want[written - n:written], f"{what}, stream {s} after {written} outputs")


PUSH_CASES = [(8000, "ulaw", "i16"), (8000, "alaw", "f32"), (12000, "i16", "i16"), (12000, "alaw", "i16"),
              (24000, "f32", "i16"), (24000, "ulaw", "f32"), (44100, "f32", "i16"), (48000, "i16", "f32"),
              (48000, "f32", "i16"), (192000, "f32", "i16")]


@pytest.mark.gpu
@pytest.mark.parametrize("sr,kind,ring", PUSH_CASES, ids=[f"{a}-{b}-into-{c}" for a, b, c in PUSH_CASES])
def test_push_resampled_equals_chain(sr, kind, ring):
    from easywakeword_b200 import _lib
    ring_fmt = _lib.PCM_I16 if ring == "i16" else _lib.PCM_F32
    secs = 1.4 if sr > 100000 else 2.3
    n = int(secs * sr)
    x, law = _overshooting_feed(2, n, sr, kind, sr + len(kind))
    want = _expect(x, sr, law, ring_fmt)
    assert np.abs(R.resample_chain(x[:, :sr // 4], sr, law=law)).max() > 1.05      # the int16 clamp runs
    from easywakeword_b200.resample import ready_outputs
    W, L, M = _lib.resample_info(sr)
    c = _bank(2, ring_fmt)
    try:
        pos = written = 0
        for i, k in enumerate(_push_sizes(sr, n)):
            m = c.push_resampled(x[:, pos:pos + k], sr, fmt=law)
            pos += k
            assert written + m == ready_outputs(pos, W, L, M)
            written += m
            if i % 3 == 2 or pos == n:
                for s in range(2):
                    _check_ring(c, s, written, want[s], f"{sr} Hz {kind} into {ring}")
        assert c.status(1).written == written and written > RING_R + RING_SLACK      # wrapped
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,ring", [(12000, "i16"), (24000, "f32")])
def test_push_each_staggered_positions(sr, ring):
    """ewk_push_resampled_each with streams at positions 1 .. L-1 and W + 1 .. W + L inputs (rows that start at
    different output phases), one at 0 (landing nothing while the others land) and one several tiles ahead."""
    from easywakeword_b200 import _lib
    from easywakeword_b200.resample import landed_counts
    ring_fmt = _lib.PCM_I16 if ring == "i16" else _lib.PCM_F32
    plan = fir_plan(sr)
    W, L, M, tile = plan["W"], plan["L"], plan["M"], plan["tile"]
    offsets = [0] + list(range(1, L)) + [W + i for i in range(1, L + 1)] + [4 * tile * M // L + 3]
    ns = len(offsets)
    n = max(offsets) + int(2.2 * sr)
    x, law = _overshooting_feed(ns, n, sr, "f32" if ring == "f32" else "i16", sr + 3)
    want = _expect(x, sr, law, ring_fmt)
    c = _bank(ns, ring_fmt)
    try:
        pos = np.array(offsets, np.int64)
        written = np.zeros(ns, np.int64)
        for s, off in enumerate(offsets):
            if off:
                written[s] = c.push_resampled(x[s:s + 1, :off], sr, stream0=s)
        landed_zero_beside_work = False
        for i, k in enumerate(_push_sizes(sr, n - max(offsets))):
            block = np.stack([x[s, pos[s]:pos[s] + k] for s in range(ns)])
            landed = c.push_resampled_each(block, sr)
            assert np.array_equal(landed, landed_counts(pos, k, sr))
            landed_zero_beside_work |= bool((landed == 0).any() and landed.max() > 0)
            pos += k
            written += landed
            if i % 2 == 1 or i < 4:
                for s in range(ns):
                    _check_ring(c, s, int(written[s]), want[s], f"{sr} Hz each, offset {offsets[s]}")
        for s in range(ns):
            _check_ring(c, s, int(written[s]), want[s], f"{sr} Hz each, offset {offsets[s]}")
            assert c.stream_input(s) == (sr, int(pos[s]))
        assert landed_zero_beside_work
    finally:
        c.close()


@pytest.mark.gpu
def test_tail_growth_and_recycled_streams():
    """Streams 0-1 start at 8 kHz; stream 2 joins at 44.1 kHz and stream 3 at 192 kHz, each widening the tails
    (rs_tail_cap: 2W = 188, 518, 2250 floats) while the earlier streams keep pushing.  Then streams 0 and 3 are reset
    and restart at 48 kHz and 24 kHz.  Every stream equals the model of its own feed throughout."""
    from easywakeword_b200 import _lib
    c = _bank(4, _lib.PCM_I16)
    feeds = {}                                              # key -> (stream, rate, pushed, law, expected ring, pos, written)

    def start(key, s, sr, kind, secs, seed):
        x, law = _overshooting_feed(1, int(secs * sr), sr, kind, seed)
        feeds[key] = dict(s=s, sr=sr, x=x[0], law=law, want=_expect(x, sr, law, _lib.PCM_I16)[0], pos=0, written=0)

    def push(key, k):
        f = feeds[key]
        k = min(k, len(f["x"]) - f["pos"])
        if k <= 0:
            return
        f["written"] += c.push_resampled(f["x"][None, f["pos"]:f["pos"] + k], f["sr"], stream0=f["s"], fmt=f["law"])
        f["pos"] += k

    def check(keys):
        for key in keys:
            f = feeds[key]
            _check_ring(c, f["s"], f["written"], f["want"], f"{key} ({f['sr']} Hz)")

    try:
        start("a", 0, 8000, "ulaw", 4.0, 1)
        start("b", 1, 8000, "ulaw", 4.0, 2)
        for k in (1, 50, 700, 1603):                        # streams 0 and 1 in one call (same position)
            xa, xb = feeds["a"], feeds["b"]
            block = np.stack([xa["x"][xa["pos"]:xa["pos"] + k], xb["x"][xb["pos"]:xb["pos"] + k]])
            m = c.push_resampled(block, 8000, stream0=0, fmt="ulaw")
            for f in (xa, xb):
                f["pos"] += k
                f["written"] += m
        check("ab")
        start("c", 2, 44100, "i16", 2.0, 3)
        for k8, k44 in ((1, 100), (900, 300), (2001, 17777), (77, 1)):
            push("c", k44)
            push("a", k8)
            push("b", k8)
            check("abc")
        start("d", 3, 192000, "f32", 1.0, 4)
        for k8, k44, k192 in ((1, 1, 1000), (800, 4410, 2248), (3000, 20000, 61441), (1999, 3, 7), (5000, 9000, 60000)):
            push("d", k192)
            push("c", k44)
            push("a", k8)
            push("b", k8)
            check("abcd")
        assert len(c.poll()) == 0
        c.reset_streams([0, 3])
        assert c.stream_input(0) == (0, 0) and c.stream_input(3) == (0, 0)
        start("a2", 0, 48000, "f32", 1.0, 5)
        start("d2", 3, 24000, "i16", 1.5, 6)
        for k48, k24, k8 in ((1, 1, 1), (300, 170, 2), (24001, 12345, 4000), (9000, 4000, 1000)):
            push("a2", k48)
            push("d2", k24)
            push("b", k8)
            push("c", 11025)
            check(["a2", "d2", "b", "c"])
        assert c.stream_input(0) == (48000, feeds["a2"]["pos"]) and c.stream_input(3) == (24000, feeds["d2"]["pos"])
    finally:
        c.close()
