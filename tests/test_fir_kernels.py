"""Every sparse-FIR kernel on the route it is meant for, bit for bit against the oracle, on hand-built tap tables.

``sparse_fir_launch`` (vnd_fir.cu) hands a SEGMENTED float32 planar slab to up to three kernels in turn and everything
else to one of the general ones.  Outputs alone cannot tell which kernel produced them, so every GPU case here records
the kernels it launched (``launched``: ``torch.profiler`` with CUDA activity) and asserts the FIR kernels among them, and
a coverage test asserts that the catalogue as a whole launches every FIR kernel instance the library builds.  In a long
process the profiler now and then loses a session's GPU records, so ``routed`` runs a call again (up to three times)
until its record matches; a case whose profiles never match, or hold no CUDA kernel at all, fails.

The tables are built by hand (``build_table``), not drawn from the velvet-noise generator, whose lists are ascending,
log-distributed and start within 32 samples: the case splits of the kernels are reached on purpose, not by chance.  The
builder is checked on the CPU against a float64 sum of ``sign * gain * x[n + i]``, and a deliberately wrong sign or
offset must break that agreement.  The oracle is ``O.fir_class_order`` / ``O.vn_decorrelate`` on the same lists.

What each group covers, and why those inputs:

- ``fir_window_kernel<29, 32, 4, 4>`` (planar float32 slabs of at least one 3712-frame tile, halo up to ~23 400): taps at
  offsets 0, 1, 31 (the register window) against 32, 33 (shared memory); one, two and all segments with a register tap
  (two segments use the staging buffer while a bulk store may still read it), with an all-far middle segment;
  all-negative, all-positive, single-tap and empty lists; duplicate offsets; non-ascending lists mixing both kinds; a
  halo under 32; a channel stride that is not a multiple of four (no bulk store); more than 32 tiles (several runs).
- ``fir_tmem_kernel`` (at least four interior 12 288-frame tiles, halo up to ~2 000): offsets 0, 415, 416 (the last
  tensor-memory column) and 417 (the first far tap); far taps at every ``o & 3`` and across a 96-sample row; a near tap
  behind a far one; near prefixes of length 0, 1, 2, 3 and all; all-near, all-far and far / near / far programs; the
  largest halo it takes and that halo + 4 (window kernel); unfiltered channels and a filtered channel without segments;
  150 channels (more than one wave of CTAs); one 1.3 M-frame pair of channels compared in full, where runs start inside
  the channel.
- ``fir_ring_kernel`` (halo ~23 400 to 36 864, frames >= max(4 x halo, (8 + K) x 9216)): one, three and five segments
  (the single-stream pass), two of unequal length either way, the identity envelope, taps next to the largest offset
  (lanes read the mirror behind the ring), frames a whole number of steps, the minimum length and one frame less.
- ``fir_tile_kernel<float, 0, 1024, 16>`` (halo up to ~41 700 on long signals) and ``fir_tile_kernel<TIn, MODE, NT, 8>``
  (float64, ASCENDING, interleaved input, short signals, the tails of the above): every NT, every mode.
- ``fir_direct_kernel<TIn, MODE>`` (the halo does not fit in shared memory): all five instances.
- The halo ladder: the last halo on each side of every boundary between two kernels.
- Non-finite values on every kernel: gains inf, -inf, nan, 0 and -0 (an empty segment with an infinite gain is kept and
  turns its channel into NaN, ``0 * inf``), and inputs holding +-inf and NaN.  NaN positions must match and every other
  sample must match bit for bit.
- Forced routes: the SEGMENTED float32 cases again in a child process with ``VND_DISABLE_TMEM``, ``VND_DISABLE_WINDOW``
  or ``VND_DISABLE_RING`` set, so the kernels behind each one meet the same tables.
- The other SEGMENTED consumers: ``decorrelate`` (fused and unfused), ``decorrelate_batch``, ``BlockConvolver`` and
  ``BlockDecorrelator`` on a subset of the tables.

Expected routes come from ``predict_route``, a restatement of the launchers' conditions, and the catalogue names the
route of each default case as well; the two must agree, and the recorder must agree with both.
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from dataclasses import dataclass, field

import numpy as np
import pytest

from oracle import vnd_oracle as O
from vndecorrelate_b200.taps import IDENTITY_ENVELOPE, TapTable, segmented_program

gpu = pytest.mark.gpu
PAD = np.iinfo(np.int32).max  # the index of an impulse a channel does not use: past every signal, so the packer drops it

# ------------------------------------------------------------------ kernel names (as the profiler reports them)

TMEM = "fir_tmem_kernel"
WIN = "fir_window_kernel<29, 32, 4, 4>"
RING = "fir_ring_kernel"
LONG = "fir_tile_kernel<float, 0, 1024, 16>"


def TILE(t, mode, nt):
    return f"fir_tile_kernel<{t}, {mode}, {nt}, 8>"


def DIRECT(t, mode):
    return f"fir_direct_kernel<{t}, {mode}>"


ALL_FIR_KERNELS = {TMEM, WIN, RING, LONG, *(TILE("float", m, nt) for m in (0, 1, 2) for nt in (256, 512, 1024)),
                   *(TILE("double", m, nt) for m in (0, 2) for nt in (256, 512, 1024)),
                   DIRECT("float", 0), DIRECT("float", 1), DIRECT("float", 2), DIRECT("double", 0), DIRECT("double", 2)}

# ------------------------------------------------------------------ hand-built tap tables


def build_table(channels) -> TapTable:
    """``channels[c]`` is None (an unfiltered channel, copied through) or a list of S segments ``(negative, positive)``,
    each list in the order the kernel must add it.  S is the same for every filtered channel.  Impulse slots are shared
    across channels (``TapTable.segment``); a slot a channel does not use holds ``PAD``."""
    segs = [ch for ch in channels if ch is not None]
    S = len(segs[0]) if segs else 0
    assert all(len(ch) == S for ch in segs), "every filtered channel has the same number of segments"
    width = [max((len(ch[s][0]) + len(ch[s][1]) for ch in segs), default=0) for s in range(S)]
    N = sum(width)
    Cn = len(channels)
    index = np.full((Cn, N), PAD, dtype=np.int32)
    positive = np.zeros((Cn, N), dtype=bool)
    segment = np.repeat(np.arange(S), width).astype(np.int64)
    for c, ch in enumerate(channels):
        if ch is None:
            continue
        at = 0
        for s, (neg, pos) in enumerate(ch):
            k = len(neg) + len(pos)
            index[c, at:at + k] = list(neg) + list(pos)
            positive[c, at + len(neg):at + k] = True
            at += width[s]
    fir_length = max(1000, 5 * N + 5, int(index[index != PAD].max(initial=0)) + 1)
    return TapTable(fir_length, N, S, np.array([ch is not None for ch in channels]), index, positive, segment)


def nested(channels):
    """The oracle's view of the same table: unfiltered channels are ``[]``."""
    return [[] if ch is None else [(list(map(int, n)), list(map(int, p))) for n, p in ch] for ch in channels]


def oracle_convolve(x, channels, envelope):
    with np.errstate(invalid="ignore", over="ignore"):
        return O.fir_class_order(x, nested(channels), envelope, len(channels))


def float64_reference(x, channels, envelope):
    """``sum sign * gain * x[n + i]`` in float64, and the bound ``n_terms * 2^-24 * sum |terms|`` of each sample."""
    n, Cn = x.shape
    y = np.zeros((n, Cn))
    bound = np.zeros((n, Cn))
    identity = envelope == IDENTITY_ENVELOPE
    for c, ch in enumerate(channels):
        if ch is None:
            y[:, c] = x[:, c]
            continue
        terms = 0
        for s, (neg, pos) in enumerate(ch):
            g = 1.0 if identity else float(np.float32(envelope[s]))
            for sign, lst in ((-1.0, neg), (1.0, pos)):
                for i in lst:
                    if i < n:
                        t = sign * g * x[i:, c].astype(np.float64)
                        y[: n - i, c] += t
                        bound[: n - i, c] += np.abs(t)
                        terms += 1
        bound[:, c] *= max(terms, 1) * 2.0 ** -24
    return y, bound


# ------------------------------------------------------------------ CPU self-checks of the builder

_SELF_CHECK_TABLES = {
    "mixed": ([[([40, 3, 40], [0, 31, 900]), ([], [33, 2])], None, [([1000], []), ([5, 5], [7])]], (0.85, -0.55)),
    "identity": ([[([0, 17], [31, 32, 416, 417])], [([], [])]], IDENTITY_ENVELOPE),
    "three": ([[([100], [1]), ([2], []), ([], [9, 8, 7])]], (0.5, 2.0, -0.25)),
}


@pytest.mark.parametrize("name", sorted(_SELF_CHECK_TABLES))
def test_builder_packs_the_lists_it_was_given(name):
    """The packed program holds, per channel, each segment's negative then positive list in the given order; the oracle's
    output agrees with a float64 evaluation of the same taps."""
    chans, env = _SELF_CHECK_TABLES[name]
    table = build_table(chans)
    frames = 1200
    prog = segmented_program(table, env, frames)
    for c, ch in enumerate(chans):
        w = prog.words[prog.offsets[c]:prog.offsets[c + 1]]
        if ch is None:
            assert len(w) == 0
            continue
        kept = [(n, p, s) for s, (n, p) in enumerate(ch) if [i for i in n + p if i < frames]]
        assert w[0] == len(kept)
        taps = w[1 + 3 * len(kept):]
        want = []
        for k, (n, p, s) in enumerate(kept):
            n2, p2 = [i for i in n if i < frames], [i for i in p if i < frames]
            assert (w[1 + 3 * k], w[2 + 3 * k]) == (len(n2), len(p2))
            g = np.float32(1.0 if env == IDENTITY_ENVELOPE else env[s])
            assert w[3 + 3 * k] == g.view(np.int32)
            want += n2 + p2
        assert taps.tolist() == want
    x = np.random.default_rng(5).standard_normal((frames, len(chans))).astype(np.float32)
    got = oracle_convolve(x, chans, env)
    ref, bound = float64_reference(x, chans, env)
    assert np.all(np.abs(got - ref) <= bound + 1e-30)


@pytest.mark.parametrize("fault", ["sign", "offset"])
def test_builder_self_check_catches_a_wrong_table(fault):
    """A table with one sign flipped or one offset moved by a sample no longer agrees with the float64 sum of the lists
    that were meant: the self-check above can tell a wrong table from a right one."""
    chans, env = _SELF_CHECK_TABLES["mixed"]
    frames = 1200
    x = np.random.default_rng(6).standard_normal((frames, len(chans))).astype(np.float32)
    ref, bound = float64_reference(x, chans, env)
    neg, pos = chans[0][0]
    bad = ([*neg], [*pos])
    if fault == "sign":
        bad = (bad[0] + [bad[1][1]], [bad[1][0], bad[1][2]])
    else:
        bad = (bad[0], [bad[1][0], bad[1][1] + 1, bad[1][2]])
    wrong = [[bad, chans[0][1]], *chans[1:]]
    got = oracle_convolve(x, wrong, env)
    assert not np.all(np.abs(got - ref) <= bound + 1e-30)


# ------------------------------------------------------------------ route model (the launchers' conditions restated)

KMAX = 227 * 1024
WIN_STATIC_SMEM = 128  # fir_window_kernel's static shared memory (one int, 128-byte aligned), out of the same KMAX


def _tile_plan(halo, elem, mpw, frames):
    span_max = (KMAX - 32 - mpw * 4) // elem
    tile = 8192 if halo <= 4096 else (halo + 2047) // 2048 * 2048
    if tile + halo > span_max:
        tile = int((span_max - halo) / 256) * 256  # C++ division truncates toward zero
    if tile < 256:
        return 0, 0
    tile = min(tile, -(-frames // 256) * 256)
    smem = 16 + (((tile + halo) * elem + 15) & ~15) + mpw * 4
    ctas = (228 * 1024) // (smem + 1024)
    nt = 256 if ctas >= 4 else (512 if ctas >= 2 else 1024)
    while nt > 256 and tile // 256 < nt // 32:
        nt //= 2
    return tile, nt


def tmem_takes(frames, halo4, mpw):
    nblk = max(128 + (halo4 + 4 + 95) // 96, 128 + (512 + 95) // 96)
    opstride = (mpw + 4 + 3) & ~3
    smem = 384 + 3 * (((nblk * 100) + 31) & ~31) * 4 + 128 * 100 * 4 + 6 * opstride * 4
    if smem > KMAX or nblk > 256 or frames < nblk * 96 + 3 * 12288:
        return 0
    return ((frames - nblk * 96) // 12288 + 1) * 12288


def predict_route(frames, halo, mpw, *, f64=False, mode=0, bulk=True, y_ok=True, y_bulk=True, disable=()) -> set:
    """The FIR kernels ``sparse_fir_launch`` launches: ``bulk`` is the planar, 16-byte aligned input the bulk copies
    need, ``y_ok`` the planar output the tensor-memory kernel stores with, ``disable`` the VND_DISABLE_* switches set."""
    out = set()
    if frames == 0:
        return out
    halo = (min(max(halo, 0), frames) + 3) & ~3
    seg32 = not f64 and mode == 0
    if seg32 and "TMEM" not in disable and bulk and y_ok:
        done = tmem_takes(frames, halo, mpw)
        if done:
            out.add(TMEM)
            frames -= done
            if frames == 0:
                return out
            if halo > frames:
                halo = (frames + 3) & ~3
    if seg32 and "WINDOW" not in disable and bulk and y_bulk:
        if frames >= 3712 and 32 + 2 * (3712 + halo) * 4 + 4 * 928 * 4 + (mpw + 4) * 4 + WIN_STATIC_SMEM <= KMAX:
            return out | {WIN}
    if seg32 and halo > 4096 and frames >= 4 * halo and "RING" not in disable and bulk:
        K = (9216 + halo + 9215) // 9216 - 1
        steps = frames // 9216 - K
        if K + 2 <= 8 and 256 + ((K + 2) * 9216 + 32 * 24) * 4 + mpw * 4 + 16 <= KMAX and steps >= 8:
            out.add(RING)
            frames -= steps * 9216
            if halo > frames:
                halo = (frames + 3) & ~3
    if seg32 and halo > 4096 and frames >= 4 * halo:
        if ((KMAX - 32 - mpw * 4) // 4 - halo) // 16384 > 0:
            return out | {LONG}
    t = "double" if f64 else "float"
    tile, nt = _tile_plan(halo, 8 if f64 else 4, mpw, frames)
    m = mode if not f64 or mode == 0 else 2
    return out | ({TILE(t, m, nt)} if tile else {DIRECT(t, m)})


def tmem_max_halo(mpw):
    """The largest halo (max tap index + 1, a multiple of four) the tensor-memory kernel takes."""
    h = 4
    while tmem_takes(1 << 30, h + 4, mpw):
        h += 4
    return h


def window_max_halo(mpw):
    return ((KMAX - WIN_STATIC_SMEM - 32 - 4 * 928 * 4 - (mpw + 4) * 4) // 8 - 3712) & ~3


def long_max_halo(mpw):
    return ((KMAX - 32 - mpw * 4) // 4 - 16384) & ~3


def tile_max_halo(mpw, elem=4):
    return ((KMAX - 32 - mpw * 4) // elem - 256) & ~3


def test_route_model_boundaries():
    """The halo bands of the route model for a 53-word program (DESIGN.md section 4)."""
    mpw = 53
    assert tmem_max_halo(mpw) == 2012
    assert window_max_halo(mpw) == 23436
    assert long_max_halo(mpw) == 41664
    assert tile_max_halo(mpw) == 57792
    assert predict_route(1 << 20, 36864, mpw) == {RING, TILE("float", 0, 1024)}


# ------------------------------------------------------------------ the recorder and the GPU helpers


def launched(fn):
    """``(names, result)``: the names of the CUDA kernels ``fn()`` launched, as the profiler reports them with the return
    type, the namespace and the parameter list removed (``fir_tile_kernel<float, 0, 256, 8>``), and what it returned."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        n = e.name
        if n.startswith("void "):
            n = n[5:]
        n = n.replace("(anonymous namespace)::", "").replace("vnd::", "")
        depth = 0
        for k, ch in enumerate(n):  # drop the parameter list: the first '(' outside the template arguments
            depth += ch == "<"
            depth -= ch == ">"
            if ch == "(" and depth == 0:
                n = n[:k]
                break
        names.add(n)
    return names, result


def routed(fn, want, what="", attempts=3):
    """Runs ``fn()`` under the recorder and returns its result once the FIR kernels recorded are exactly ``want`` (a
    set of names, or a predicate on all recorded names).  In a long process the profiler now and then loses the GPU
    records of a whole session or part of one, so a call whose record does not match is run again, in a fresh
    session, up to ``attempts`` times; ``fn`` must give the same result every time.  Records are only ever lost, never
    made up, so a kernel that did not run cannot make a case pass.  Fails when no attempt matched, and says so when
    the profiler recorded no CUDA kernel at all."""
    ok = want if callable(want) else (lambda names: fir_kernels(names) == set(want))
    seen = []
    for _ in range(attempts):
        names, result = launched(fn)
        if ok(names):
            return result
        seen.append(sorted(names))
    if not any(seen):
        raise AssertionError(f"{what}: the profiler recorded no CUDA kernel in {attempts} attempts: the route is unknown")
    raise AssertionError(f"{what}: expected {want if callable(want) else sorted(want)}; FIR kernels launched: "
                         f"{[sorted(fir_kernels(n)) for n in seen]}; all kernels recorded: {seen}")


def fir_kernels(names):
    return {n for n in names if n.startswith(("fir_tmem", "fir_window", "fir_ring", "fir_tile", "fir_direct"))}


def same(got, want) -> bool:
    """Equal shapes and dtypes, NaN at the same places, every other sample equal bit for bit."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    if got.shape != want.shape or got.dtype != want.dtype:
        return False
    gn, wn = np.isnan(got), np.isnan(want)
    if not np.array_equal(gn, wn):
        return False
    bits = {4: np.uint32, 8: np.uint64}[got.dtype.itemsize]
    return np.array_equal(got.view(bits)[~gn], want.view(bits)[~wn])


def mismatch(got, want):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))) | (np.signbit(got) != np.signbit(want)) & ~np.isnan(want))
    return f"{len(bad)} samples differ; first at (frame, channel) {bad[0].tolist() if len(bad) else None}"


def _hand_vn_class():
    import vndecorrelate_b200.decorrelation as D

    class HandVelvetNoise(D.VelvetNoise):
        """A ``VelvetNoise`` whose table is the hand-built one, so that every public path uses the same table."""

        def __init__(self, table, envelope, **kw):
            self._hand = table
            kw.setdefault("mode", "LR")
            kw.setdefault("normalizer", None)
            super().__init__(sample_rate_hz=table.fir_length_samples, duration_seconds=1.0, num_impulses=table.num_impulses,
                             num_outs=table.num_outs, segment_envelope=envelope,
                             filtered_channels=tuple(int(c) for c in np.nonzero(table.filtered)[0]), **kw)

        def _generate(self):
            return self._hand

    return HandVelvetNoise


def hand_vn(channels, envelope, **kw):
    return _hand_vn_class()(build_table(channels), envelope, **kw)


# ------------------------------------------------------------------ the catalogue


@dataclass
class Case:
    name: str
    chans: list
    env: tuple
    frames: int
    route: set            # the FIR kernels of the default run
    layout: str = "planar"   # planar: (C, frames) slab, channel stride a multiple of 4 | interleaved: (frames, C) C-order
    dtype: str = "float32"
    signal: str = "randn"    # randn | nonfinite (with +-inf and NaN)
    plan_runs: int = 0       # assert the tensor-memory plan splits each channel into at least this many runs
    tags: tuple = field(default=())

    @property
    def seg32(self):
        return self.dtype == "float32"


def _far(a, b, step):
    return list(range(a, b, step))


def _signal(case: Case) -> np.ndarray:
    """(frames, C) float32 / float64 samples with runs of +0 and -0 (the sign of a zero sum) and, for ``nonfinite``,
    +-inf and NaN."""
    rng = np.random.default_rng(abs(hash(case.name)) % (1 << 32))
    Cn = len(case.chans)
    x = (rng.standard_normal((case.frames, Cn)) * 0.1).astype(np.float64 if case.dtype == "float64" else np.float32)
    n = case.frames
    x[n // 7: n // 7 + min(600, n // 9)] = 0.0
    x[n // 3: n // 3 + min(200, n // 20)] = -0.0
    if case.signal == "nonfinite":
        x[n // 2, 0] = np.inf
        x[n // 2 + 3, 0] = -np.inf
        x[(2 * n) // 3, -1] = np.nan
        x[5, :] = np.inf
    return x


def _device_input(x, layout):
    """The CUDA tensor the call gets: a planar slab whose channel stride is a multiple of four (bulk copies allowed) or a
    C-order interleaved array."""
    import torch

    n, Cn = x.shape
    if layout == "interleaved":
        return torch.from_numpy(np.ascontiguousarray(x)).cuda()
    pitch = (n + 3) & ~3
    buf = torch.zeros((Cn, pitch), dtype=torch.float64 if x.dtype == np.float64 else torch.float32, device="cuda")
    buf[:, :n] = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    return buf[:, :n].t()


def case_route(case: Case, mpw: int, halo: int, disable=()):
    planar = case.layout == "planar"
    y_ok = planar and case.frames % 4 == 0
    return predict_route(case.frames, halo, mpw, f64=case.dtype == "float64", bulk=planar and case.dtype == "float32",
                         y_ok=y_ok, y_bulk=True, disable=disable)


def run_case(case: Case, disable=()):
    """Runs one case through ``VelvetNoise.convolve`` on the GPU; asserts the route and the oracle's bits."""
    vn = hand_vn(case.chans, case.env)
    x = _signal(case)
    xt = _device_input(x, case.layout)
    prog = vn.tap_program(case.frames)
    predicted = case_route(case, prog.max_channel_words, prog.halo, disable)
    if not disable:
        assert predicted == case.route, f"{case.name}: the route model gives {sorted(predicted)}, the catalogue {sorted(case.route)}"
    got = routed(lambda: vn.convolve(xt), predicted, case.name).cpu().numpy()
    want = oracle_convolve(x, case.chans, case.env)
    assert same(got, want), f"{case.name}: {mismatch(got, want)}"
    if case.plan_runs:
        from vndecorrelate_b200 import _native as N

        lib = N.lib()
        lib.vnd_debug_fir_plan.restype = C.c_int
        plan = (C.c_int * 3)()
        assert lib.vnd_debug_fir_plan(C.c_longlong(case.frames), len(case.chans), prog.halo, plan) == 0
        assert plan[1] >= case.plan_runs, list(plan)


def _window_cases():
    env2 = (0.85, -0.55)
    return [
        Case("win-offsets-0-1-31-32-33", [[([1, 32], [0, 31, 33])], [([33, 0], [32, 1, 31])]], (0.7,), 3712 * 3, {WIN}),
        Case("win-s_win-2-all-far-middle", [[([5], [0, 40]), ([100, 200], [300]), ([7], [31])],
                                            [([2], [3]), ([1], []), ([], [30])],
                                            [([], [60]), ([500], [600]), ([700], [])]], (0.85, -0.55, 0.35), 3712 * 2 + 8, {WIN}),
        Case("win-all-negative-positive-single-empty", [[([3, 50, 7, 200], []), ([1], [])], [([], [3, 50, 7, 200]), ([], [90])],
                                                        [([], [17]), ([], [])], [([], []), ([], [])]], (0.6, 1.5), 3712 * 2, {WIN}),
        Case("win-duplicates-non-ascending", [[([40, 3, 40, 3], [900, 1, 31, 900, 32]), ([2, 2], [500, 0])],
                                              [([1000, 0, 999], [33, 31, 33]), ([], [5, 5, 5])]], (0.3, -1.25), 3712 + 4, {WIN}),
        Case("win-halo-under-32", [[([0, 5], [31, 2])], [([30], [0, 0])]], IDENTITY_ENVELOPE, 3712 * 4, {WIN}),
        Case("win-odd-stride-no-bulk-store", [[([40, 3], [0, 31, 32]), ([], [33])], [([2], [7]), ([600], [])]], env2, 3712 * 2 + 1, {WIN}),
        Case("win-33-tiles-several-runs", [[([3000, 2], [0, 31, 32]), ([1], [2999])], [([31], [1500]), ([], [0])]], env2,
             3712 * 34 + 8, {WIN}),
        Case("win-33-tiles-odd-frames", [[([300, 2], [0, 31, 32]), ([1], [299])], [([31], [150]), ([], [0])]], env2,
             3712 * 33 + 3, {WIN}),
    ]


def _tmem_cases():
    env = (0.9, -0.7)
    prefixes = [[([], [500, 600]), ([], [3])], [([], [5, 500]), ([], [3])], [([], [5, 9, 500]), ([], [3])],
                [([], [5, 9, 13, 500]), ([], [3])], [([], [5, 9, 13, 100, 200]), ([], [3])]]
    F = 5 * 12288 + 3716  # five interior tiles, a 3716-frame tail for the window kernel
    hmax = tmem_max_halo(1 + 3 * 2 + 3)
    cases = [
        Case("tmem-offsets-0-415-416-417", [[([416], [0, 417, 415]), ([1], [])], [([0, 417], [415, 416]), ([], [900])]], env, F, {TMEM, WIN}),
        Case("tmem-far-alignments-and-rows", [[(_far(417, 421, 1), _far(476, 484, 1)), ([1], _far(572, 580, 1))],
                                              [(_far(669, 675, 1), [1000, 1001, 1002, 1003]), (_far(956, 964, 1), [0])]],
             env, F, {TMEM, WIN}),
        Case("tmem-near-behind-far", [[([600, 10, 700, 20], [417, 3]), ([], [416, 0])], [([1], [2]), ([800, 4], [])]], env, F, {TMEM, WIN}),
        Case("tmem-near-prefixes-0-1-2-3-all", prefixes, env, F, {TMEM, WIN}),
        Case("tmem-all-near-all-far-far-near-far", [[([3], [400]), ([600], [1200]), ([], [7])],
                                                     [([500], [900]), ([2, 1], [0]), ([1500], [417])],
                                                     [([420], []), ([700], [800]), ([1300], [1800])]], (0.85, 0.55, 0.35), F, {TMEM, WIN}),
        Case("tmem-largest-halo", [[([hmax - 1], [0, 416, 417]), ([5], [])], [([9], [hmax - 2]), ([], [1])]], env, F, {TMEM, WIN}),
        Case("tmem-largest-halo-plus-4-window", [[([hmax + 3], [0, 416, 417]), ([5], [])], [([9], [hmax - 2]), ([], [1])]], env, F, {WIN}),
        Case("tmem-unfiltered-and-empty-channel", [None, [([416], [0, 1]), ([417], [])], [([], []), ([], [])], None], env, F, {TMEM, WIN}),
        Case("tmem-identity-envelope", [[([416, 3], [0, 417, 1000])], [([5], [415, 2000])]], IDENTITY_ENVELOPE, F, {TMEM, WIN}),
        Case("tmem-shortest-slab-tile-tail", [[([416], [0, 417]), ([5], [])], [([9], [40]), ([], [1])]], env, 4 * 12288 + 12864,
             {TMEM, TILE("float", 0, 256)}),
        Case("tmem-150-channels", [[([(7 * c) % 500], [c % 417, 417 + c]), ([c], [1000 - c])] for c in range(150)], env, F + 12288,
             {TMEM, WIN}),
        Case("tmem-1.3M-frames-in-full", [[([416, 2], [0, 417, 1500]), ([5], [33])], [([3], [7, 415]), ([1800], [])]], env,
             1_300_000, {TMEM, WIN}, plan_runs=2),
    ]
    return cases


def _ring_cases():
    K4 = 4 * 9216
    def ring_min(h):
        K = -(-h // 9216)
        return max(4 * h, (8 + K) * 9216)
    return [
        Case("ring-S1", [[([30000, 5], [0, 29999, 100])], [([3], [17000])]], (0.7,), ring_min(30004) + 777, {RING, TILE("float", 0, 1024)}),
        Case("ring-S3", [[([30000], [0]), ([12000, 31], [9]), ([1], [25000])], [([2], [3]), ([4], [5]), ([28000], [])]],
             (0.85, 0.55, 0.35), 160000, {RING, TILE("float", 0, 1024)}),
        Case("ring-S5", [[([30000], [0]), ([12000], [9]), ([1], []), ([], [25000]), ([7], [8])],
                         [([2], [3]), ([4], [5]), ([28000], []), ([6], []), ([], [29001])]], (0.85, 0.55, 0.35, 0.2, -1.5),
             160000, {RING, TILE("float", 0, 1024)}),
        Case("ring-S2-unequal-lengths", [[([30000, 1, 2, 3], [0, 4, 5]), ([6], [])], [([7], []), ([30001, 1, 2, 3], [0, 4, 5])]],
             (0.85, -0.55), 160000, {RING, TILE("float", 0, 1024)}),
        Case("ring-identity", [[([30000, 1], [0, 12345])], [([2], [29000])]], IDENTITY_ENVELOPE, 160000, {RING, TILE("float", 0, 1024)}),
        Case("ring-taps-at-the-mirror", [[(_far(K4 - 8, K4, 2), _far(K4 - 7, K4, 2)), ([0], [9215, 9216])],
                                         [([K4 - 1], [K4 - 2, 0]), ([18431], [18432])]], (0.85, -0.55), 4 * K4 + 9216 * 3, None),
        Case("ring-whole-steps", [[([30000, 5], [0, 29999])], [([3], [17000])]], (0.7,), 9216 * 15, None),
        Case("ring-minimum-frames", [[([23999, 5], [0, 100])], [([3], [17000])]], (0.7,), ring_min(24000), None),
        Case("ring-minimum-frames-less-one", [[([23999, 5], [0, 100])], [([3], [17000])]], (0.7,), ring_min(24000) - 1, None),
        Case("ring-unfiltered", [None, [([30000], [0, 1])], None, [([2], [29000])]], (0.7,), 160000, {RING, TILE("float", 0, 1024)}),
    ]


def _tile_cases():
    env = (0.85, -0.55)
    return [
        Case("long-tile-band", [[([39999, 5], [0, 31])], [([3], [20000])]], (0.7,), 160001, None),
        Case("stereo-c-order-long", [[([6000, 1], [0, 31]), ([2], [])], [([3], [4999]), ([], [7])]], env, 30000, None, layout="interleaved"),
        Case("stereo-c-order-short", [[([6000, 1], [0, 31]), ([2], [])], [([3], [4999]), ([], [7])]], env, 20000, None, layout="interleaved"),
        Case("tile-nt256", [[([1000, 1], [0, 31, 32]), ([2], [])], [([3], [999]), ([], [7])]], env, 9001, None, layout="interleaved"),
        Case("tile-nt512", [[([10000, 1], [0, 31, 32]), ([2], [])], [([3], [999]), ([], [7])]], env, 30000, None, layout="interleaved"),
        Case("tile-nt1024", [[([20000, 1], [0, 31, 32]), ([2], [])], [([3], [999]), ([], [7])]], env, 50000, None, layout="interleaved"),
        Case("tile-f64-segmented", [[([3000, 1], [0, 31, 32]), ([2], [])], [([3], [999]), ([], [7])]], env, 20000, None, dtype="float64"),
        Case("tile-f64-nt1024", [[([12000, 1], [0, 31, 32]), ([2], [])], [([3], [999]), ([], [7])]], env, 40000, None, dtype="float64"),
        Case("tile-short-signal", [[([100, 1], [0, 31, 32]), ([2], [])], [([3], [99]), ([], [7])]], env, 1000, None),
        Case("direct-float-seg", [[([60000, 1], [0, 31])], [([3], [7])]], (0.7,), 70000, None),
        Case("direct-double-seg", [[([30000, 1], [0, 31])], [([3], [7])]], (0.7,), 40000, None, dtype="float64"),
    ]


def _ladder_cases():
    """The last halo on each side of every boundary between two kernels: (name, halo-1 offset, frames)."""
    mpw = 1 + 3 * 1 + 3
    rows = [
        ("tmem|window", tmem_max_halo(mpw), lambda h: 4 * 12288 + 14400 + 8),
        ("window|ring", window_max_halo(mpw), lambda h: 4 * h + 4 * 9216),
        ("ring|long", 36864, lambda h: 4 * h + 4 * 9216),
        ("long|tile", long_max_halo(mpw), lambda h: 4 * h + 64),
        ("tile|direct", tile_max_halo(mpw), lambda h: h + 5000),
    ]
    out = []
    for name, h, frames in rows:
        for side, hh in (("last", h), ("first", h + 4)):
            out.append(Case(f"ladder-{name}-{side}-{hh}", [[([hh - 1], [0, 31, 417])], [([2], [hh - 3])]], (0.6,), frames(h), None,
                            tags=("ladder",)))
    return out


def _nonfinite_cases():
    """Every kernel with non-finite gains (the envelope) and non-finite inputs."""
    routes = [  # (label, offsets of the table, frames, layout, dtype)
        ("window", 300, 3712 * 2, "planar", "float32"),
        ("tmem", 1000, 4 * 12288 + 14400, "planar", "float32"),
        ("ring", 30000, 160000, "planar", "float32"),
        ("long", 40000, 160000, "planar", "float32"),
        ("tile", 300, 5000, "interleaved", "float32"),
        ("tile-f64", 300, 5000, "planar", "float64"),
        ("direct", 60000, 61000, "planar", "float32"),
    ]
    envs = {"inf": (0.5, np.inf, 0.25), "-inf": (-np.inf, 0.5, 0.25), "nan": (0.5, 0.25, np.nan), "zero": (0.0, 0.5, 0.25),
            "-zero": (0.5, -0.0, 0.25), "empty-inf": (0.5, np.inf, 0.25)}
    out = []
    for label, far, frames, layout, dtype in routes:
        chans = [[([far - 1, 3], [0, 31]), ([1], [far // 2, 32]), ([5], [7])], [([2], [far - 2]), ([], [33]), ([4, 4], [])]]
        for ename, env in envs.items():
            ch = chans
            if ename == "empty-inf":  # segment 1 empty in every channel (and one tap past the end): kept for its gain
                ch = [[c[0], ([frames + 5], []), c[2]] for c in chans]
            out.append(Case(f"nonfinite-{label}-gain-{ename}", ch, env, frames, None, layout=layout, dtype=dtype, tags=("nonfinite",)))
        out.append(Case(f"nonfinite-{label}-input", chans, (0.5, -0.75, 0.25), frames, None, layout=layout, dtype=dtype,
                        signal="nonfinite", tags=("nonfinite",)))
    return out


def catalogue():
    cases = _window_cases() + _tmem_cases() + _ring_cases() + _tile_cases() + _ladder_cases() + _nonfinite_cases()
    for c in cases:  # cases stated without a route take the route model's
        if c.route is None:
            prog = segmented_program(build_table(c.chans), c.env, c.frames)
            c.route = case_route(c, prog.max_channel_words, prog.halo)
    return cases


CATALOGUE = {c.name: c for c in catalogue()}


@gpu
@pytest.mark.parametrize("name", list(CATALOGUE))
def test_catalogue(name):
    run_case(CATALOGUE[name])


def _function_cases():
    """``convolve_velvet_noise`` with hand-made dense FIRs (ASCENDING programs), whose coefficients make products that
    are inexact in float32: (name, FIR length, nonzero offsets, FIR dtype, signal dtype, layout, frames).  Per FIR and
    signal dtype, one halo for each NT of the tile kernel and one past the shared memory (the direct kernel)."""
    out = []
    halos = {np.float32: {256: 2000, 512: 6200, 1024: 14400, "direct": 60001}, np.float64: {256: 1000, 512: 2100, 1024: 6300, "direct": 30001}}
    for fdt, xdt in ((np.float32, np.float32), (np.float64, np.float32), (np.float64, np.float64), (np.float32, np.float64)):
        for nt, m in halos[xdt].items():
            layout = "interleaved" if nt == 512 else "planar"
            out.append((f"fir-{np.dtype(fdt).name}-signal-{np.dtype(xdt).name}-{nt}", m, [0, 1, 31, 32, m // 2, m - 1], fdt, xdt, layout,
                        m + 3000))
    return out


FUNCTION_CASES = {c[0]: c for c in _function_cases()}


@gpu
@pytest.mark.parametrize("name", list(FUNCTION_CASES))
def test_function_order_kernels(name):
    import vndecorrelate_b200.decorrelation as D

    _, m, offs, fdt, xdt, layout, frames = FUNCTION_CASES[name]
    rng = np.random.default_rng(len(name))
    fir = np.zeros((m, 2), dtype=fdt)
    for k, i in enumerate(offs):
        fir[i] = [(0.1 + 0.7 * k) / 3.0 * (-1) ** k, 1.0 / (7 + k)]
    x = (rng.standard_normal((frames, 2)) * 0.3).astype(xdt)
    xt = _device_input(x, layout)
    prog = D.ascending_program(fir, frames)
    want_route = predict_route(frames, prog.halo, prog.max_channel_words, f64=xdt == np.float64, mode=prog.order, bulk=False)
    got = routed(lambda: D.convolve_velvet_noise(xt, fir), want_route, name).cpu().numpy()
    want = O.fir_function_order(x, fir)
    assert same(got, want), f"{name}: {mismatch(got, want)}"


def test_route_model_covers_every_fir_kernel():
    """The union of the catalogue's routes (default and forced) and the ASCENDING cases names every FIR kernel instance
    the library builds, and nothing else.  A kernel added to the dispatch, or one no longer reached, fails here."""
    seen = set()
    for c in CATALOGUE.values():
        seen |= c.route
        if c.seg32:
            prog = segmented_program(build_table(c.chans), c.env, c.frames)
            for sw in FORCED:
                seen |= case_route(c, prog.max_channel_words, prog.halo, FORCED[sw])
    for name, m, offs, fdt, xdt, layout, frames in FUNCTION_CASES.values():
        fir = np.zeros((m, 2), dtype=fdt)
        fir[offs] = 1.0
        from vndecorrelate_b200.taps import ascending_program

        prog = ascending_program(fir, frames)
        seen |= predict_route(frames, prog.halo, prog.max_channel_words, f64=xdt == np.float64, mode=prog.order, bulk=False)
    assert seen == ALL_FIR_KERNELS, (sorted(ALL_FIR_KERNELS - seen), sorted(seen - ALL_FIR_KERNELS))


# ------------------------------------------------------------------ forced routes (one child process per switch)

FORCED = {"VND_DISABLE_TMEM": ("TMEM",), "VND_DISABLE_WINDOW": ("WINDOW",), "VND_DISABLE_RING": ("RING",)}


def _forced_main(switch):
    """Child process: every SEGMENTED float32 case with ``switch`` set in the environment before the library loads."""
    failures = []
    for c in CATALOGUE.values():
        if not c.seg32:
            continue
        try:
            run_case(c, disable=FORCED[switch])
        except AssertionError as e:
            failures.append(f"{c.name}: {e}")
    print(f"{switch}: {len(failures)} failed")
    for f in failures:
        print(f)
    return 1 if failures else 0


@gpu
@pytest.mark.parametrize("switch", list(FORCED))
def test_forced_routes(switch):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, **{switch: "1"})
    env["PYTHONPATH"] = root + os.pathsep + env.get("PYTHONPATH", "")
    code = f"import sys; from tests import test_fir_kernels as T; sys.exit(T._forced_main({switch!r}))"
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-4000:]


# ------------------------------------------------------------------ the other SEGMENTED consumers

CONSUMER_TABLES = {
    # non-ascending lists, two segments with register taps, an empty segment with an infinite gain, a tap at the last
    # in-range offset (None: frames - 1).  Both channels have as many taps in each segment: the block consumers pack the
    # whole table for any length, so a PAD slot would be a real tap to them.
    "non-ascending-s_win": ([[([40, 3, 900], [0, 31, 32]), ([2], [33, 1])], [([1000, 0], [5, 999, 31, 2]), ([31], [7, 30])]],
                            (0.85, -0.55)),
    "empty-inf-segment": ([[([40, 3], [0, 31]), ([], []), ([5], [6])], [([7], [8, 1, 2]), ([], []), ([], [9, 10])]],
                          (0.85, np.inf, 0.35)),
    "last-offset": ([[([None], [0, 31])], [([2], [None, 5])]], (0.7,)),
    "long-halo": ([[([30000, 3], [0, 31])], [([2], [29000, 1, 7])]], (0.7,)),
}


def _consumer_table(name, frames):
    chans, env = CONSUMER_TABLES[name]
    chans = [[(tuple(frames - 1 if i is None else i for i in n), tuple(frames - 1 if i is None else i for i in p)) for n, p in ch]
             for ch in chans]
    return chans, env


@gpu
@pytest.mark.parametrize("ms", [False, True])
@pytest.mark.parametrize("name", sorted(CONSUMER_TABLES))
def test_decorrelate_fused_and_unfused(name, ms):
    import torch

    frames = 70000 if name == "long-halo" else 9001
    chans, env = _consumer_table(name, frames)
    x = (np.random.default_rng(3).standard_normal((frames, 2)) * 0.2).astype(np.float32)
    for norm in (None, "rms"):
        import vndecorrelate_b200.decorrelation as D

        vn = hand_vn(chans, env, mode="MS" if ms else "LR", normalizer=D.rms_normalize if norm else None)
        xt = torch.from_numpy(x).cuda()
        fused = name != "long-halo"  # the fused kernel when the halo fits its shared memory, else the unfused composition
        y = routed(lambda: vn.decorrelate(xt), lambda names: ("vn_stereo_kernel<float, 4>" in names) == fused and
                   bool(fir_kernels(names)) != fused, f"{name} ms={ms} norm={norm}")
        with np.errstate(invalid="ignore", over="ignore"):
            want = O.vn_decorrelate(x, nested(chans), envelope=env, ms_mode=ms, normalizer=norm)
        got = y.cpu().numpy()
        assert same(got, want), f"{name} ms={ms} norm={norm}: {mismatch(got, want)}"
        assert same(vn.decorrelate(x), want)


@gpu
@pytest.mark.parametrize("name", sorted(CONSUMER_TABLES))
def test_decorrelate_batch(name):
    import vndecorrelate_b200.decorrelation as D

    frames = 70000 if name == "long-halo" else 9001
    chans, env = _consumer_table(name, frames)
    rng = np.random.default_rng(4)
    clips = [(rng.standard_normal((L, 2)) * 0.2).astype(np.float32) for L in (frames, frames - 1000, 33)]
    vn = hand_vn(chans, env, mode="LR")
    if name != "long-halo":
        got = routed(lambda: D.decorrelate_batch(clips, vn), lambda names: "vn_batch_stereo_kernel<float, 4>" in names, name)
    else:
        got = D.decorrelate_batch(clips, vn)
    for k, (g, x) in enumerate(zip(got, clips)):
        with np.errstate(invalid="ignore", over="ignore"):
            want = O.vn_decorrelate(x, nested(chans), envelope=env, ms_mode=False, normalizer=None)
        assert same(g, want), f"{name} clip {k}: {mismatch(g, want)}"


def _blocks(x, sizes):
    out, at = [], 0
    for s in sizes:
        out.append(x[at:at + s])
        at += s
    out.append(x[at:])
    return out


@gpu
@pytest.mark.parametrize("kind", ["convolver", "decorrelator"])
@pytest.mark.parametrize("name", sorted(CONSUMER_TABLES))
def test_block_consumers(name, kind):
    import vndecorrelate_b200.decorrelation as D

    frames = 70000 if name == "long-halo" else 9001
    chans, env = _consumer_table(name, frames)
    x = (np.random.default_rng(5).standard_normal((frames, 2)) * 0.2).astype(np.float32)
    vn = hand_vn(chans, env, mode="LR")
    if kind == "decorrelator" and name == "long-halo":  # past the block-step kernel's shared memory: refused, not approximated
        with pytest.raises(NotImplementedError):
            D.BlockDecorrelator(vn, 1)
        return
    blocks = _blocks(x, [1, 700, 31, 5000, 0, 2000])

    def feed():  # a fresh object per attempt, and one profile over all steps: a step with an empty block may launch nothing
        b = D.BlockConvolver(vn, 1) if kind == "convolver" else D.BlockDecorrelator(vn, 1)
        return [b.process([blk], final=k == len(blocks) - 1)[0] for k, blk in enumerate(blocks)]

    kernel = "fir_block_step_kernel" if kind == "convolver" else "vn_block_step_kernel"
    parts = routed(feed, lambda names: any(n.startswith(kernel) for n in names), f"{name} {kind}")
    got = np.concatenate([np.asarray(p) for p in parts])
    with np.errstate(invalid="ignore", over="ignore"):
        want = oracle_convolve(x, chans, env) if kind == "convolver" else O.vn_decorrelate(x, nested(chans), envelope=env, ms_mode=False,
                                                                                            normalizer=None)
    assert same(got, want), f"{name} {kind}: {mismatch(got, want)}"
