"""Every objective kernel against a float64 reference of its partial sums, slot by slot.

``oracle.vnd_oracle.objective_partials`` / ``haas_partials`` compute the sums the objective is made of from the
decorrelated signal the oracle builds bit-exactly (correctly rounded ``math.fsum``, float64 angles, the exact
max-|d|/|s| frame).  The CPU tests pin that reference to the reference library's own values and check that every probe
below is sharp enough to see one frame dropped, counted twice or shifted.  The GPU tests compare every objective entry
point with it at the lengths, filters, candidate groups, chunk plans and signals where a kernel can go wrong, and check
that the sums do not depend on the chunk plan.

Tolerances (float32 velvet-noise slots 0-5, per candidate; ``mag`` is the sum of the terms' magnitudes):

* accumulation: ``K * 2**-24 * mag``.  A whole tile runs two chains of 64 frames per lane (63 roundings), one chain
  add and five warp levels (K ~ 72); the ragged last tile runs one chain of up to 128 frames per lane (127) and the
  five warp levels.  Each term itself is a product of up to three rounded factors (rad * th, * th, fma).  K = 140
  covers the larger; the float64 tile and chunk sums add nothing measurable.
* radius: ``sqrt.approx`` is within 2 float32 ulps, ``2 * 2**-23 * mag`` on the r-weighted slots 0-3 (the squares
  and their sum are the reference's own float32 operations, which the reference radius repeats).
* angle: the kernels' theta is within ``D_THETA`` = 3e-7 rad of the true folded angle (the minimax polynomial's 1e-7,
  the approximate reciprocal and the quotient's 1.5 ulps of t, the Horner and pi/2 - th roundings), so slot n (r
  theta^n) moves by at most ``n (pi/2)^(n-1) D_THETA sum r``.
* underflow: a float32 rounding of a subnormal result can be off by half the smallest subnormal (2**-150) whatever
  its relative bound says; four roundings per frame and slot give ``4 frames 2**-150``.

Haas slots (float64): ``(frames / 256 + 16) 2**-53 mag`` (a thread's chain of frames / 256 terms, eight reduction
levels, the rounded terms) plus ``5e-16 n sum r`` for the angle of r theta^n; max|theta| within 4 double ulps.

Exact slots: 6-9 must hold the reference's largest ratio (equal float64 cross products) and be |d|, |s| of a real
frame of that sign class (ties may pick any of the tied frames); slot 10 is the frame count, slot 11 is zero, Haas slot
7 is frames + delay.
"""

from __future__ import annotations

import math

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200 import optimization as opt
from vndecorrelate_b200.taps import IDENTITY_ENVELOPE, TapProgram, candidate_program

gpu = pytest.mark.gpu
KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
FS = 48000
TILE = 4096

K_F32 = 140
EPS_SQRT = 2 * 2.0**-23
D_THETA = 3e-7
HALF_PI = math.pi / 2

# largest error / bound seen per (kind, slot), reported at the end of the module
_RATIOS: dict = {}


@pytest.fixture(scope="module", autouse=True)
def _report_ratios(request):
    yield
    if not _RATIOS:
        return
    rep = request.config.pluginmanager.get_plugin("terminalreporter")
    lines = ["largest error / bound per slot:"] + [f"  {k[0]} slot {k[1]}: {v:.3g}" for k, v in sorted(_RATIOS.items())]
    for line in lines:
        rep.write_line(line) if rep is not None else print(line)


def _note(kind, slot, err, tol):
    r = err / tol if tol > 0 else (0.0 if err == 0 else math.inf)
    _RATIOS[(kind, slot)] = max(_RATIOS.get((kind, slot), 0.0), r)


# ------------------------------------------------------------------ tolerances and comparisons


def vn_tolerance(ref) -> np.ndarray:
    mag, n = ref["mag"], ref["frames"]
    tol = K_F32 * 2.0**-24 * mag + 4 * n * 2.0**-150
    tol[:4] += EPS_SQRT * mag[:4]
    for k in (1, 2, 3):
        tol[k] += k * HALF_PI ** (k - 1) * D_THETA * mag[0]
    return tol


def haas_tolerance(ref) -> np.ndarray:
    mag, n = ref["mag"], ref["frames"]
    tol = (n / 256 + 16) * 2.0**-53 * mag
    for k in (1, 2, 3):
        tol[k] += 5e-16 * k * mag[0]
    return tol


def check_vn(got, ref, what="", sums=True):
    got = np.asarray(got, dtype=np.float64)
    p = ref["p"]
    if sums:
        tol = vn_tolerance(ref)
        for k in range(6):
            err = abs(got[k] - p[k])
            _note("vn", k, err, tol[k])
            assert err <= tol[k], f"{what}: slot {k}: {got[k]!r} vs {p[k]!r} (error {err:.3g}, bound {tol[k]:.3g})"
    ad, as_ = np.abs(ref["d"]).astype(np.float64), np.abs(ref["s"]).astype(np.float64)
    for kd, ks, cls in ((6, 7, ref["s"] >= 0), (8, 9, ref["s"] < 0)):
        assert got[kd] * p[ks] == p[kd] * got[ks], f"{what}: ratio slots {kd},{ks}: {got[kd]!r}/{got[ks]!r} vs {p[kd]!r}/{p[ks]!r}"
        if p[kd] == 0.0:
            assert (got[kd], got[ks]) == (0.0, 1.0), f"{what}: slots {kd},{ks} should keep 0 / 1"
        else:
            assert np.any(cls & (ad == got[kd]) & (as_ == got[ks])), f"{what}: slots {kd},{ks}: no frame has |d|, |s| = {got[kd]!r}, {got[ks]!r}"
    assert got[10] == ref["frames"], f"{what}: frame count {got[10]} vs {ref['frames']}"
    assert got[11] == 0.0


def check_haas(got, ref, what=""):
    got = np.asarray(got, dtype=np.float64)
    p, tol = ref["p"], haas_tolerance(ref)
    for k in (0, 1, 2, 3, 5, 6):
        err = abs(got[k] - p[k])
        _note("haas", k, err, tol[k])
        assert err <= tol[k], f"{what}: slot {k}: {got[k]!r} vs {p[k]!r} (error {err:.3g}, bound {tol[k]:.3g})"
    err = abs(got[4] - p[4])
    _note("haas", 4, err, 4 * np.spacing(p[4]))
    assert err <= 4 * np.spacing(p[4]), f"{what}: max|theta| {got[4]!r} vs {p[4]!r}"
    assert got[7] == ref["frames"], f"{what}: frame count {got[7]} vs {ref['frames']}"


# ------------------------------------------------------------------ candidates and their oracle outputs


def identity_program(n=1) -> TapProgram:
    w = opt._IDENTITY_PROGRAM_WORDS
    return TapProgram(np.tile(w, n), (np.arange(n + 1) * w.size).astype(np.int32), n, N.ORDER_SEGMENTED, 0, 1, w.size)


def identity_output(x):
    y = np.array(x, dtype=np.float32)
    y[:, 0] = np.float32(0.0) + (np.float32(0.0) + y[:, 0])  # the program's segment sum and running output: -0 -> +0
    return y


class VnFamily:
    """Velvet-noise candidates of the reference's family (channel 0 filtered, LR, no normaliser), with their oracle
    taps: ``program(frames)`` for the kernels, ``output(x, j)`` for the reference."""

    def __init__(self, kappas, duration=0.03, num_impulses=30, envelope=O.DEFAULT_ENVELOPE, seed=1, fs=FS):
        self.kappas, self.envelope, self.fs = list(kappas), tuple(envelope), fs
        self.decs = [D.VelvetNoise(sample_rate_hz=fs, duration_seconds=duration, num_impulses=num_impulses, segment_envelope=envelope,
                                   log_distribution_strength=k, normalizer=None, filtered_channels=(0,), mode="LR", seed=seed) for k in self.kappas]
        self.taps = [O.class_taps(sample_rate_hz=fs, duration_seconds=duration, num_impulses=num_impulses, num_outs=2, num_segments=len(envelope),
                                  log_distribution_strength=k, filtered_channels=(0,), seed=seed) for k in self.kappas]
        self.max_tap = max(int(i) for t in self.taps for seg in t[0] for lst in seg for i in lst)

    def program(self, frames):
        return candidate_program([d.velvet_noise for d in self.decs], self.decs[0].segment_envelope, frames)

    def output(self, x, j):
        return O.vn_decorrelate(x, self.taps[j], envelope=self.envelope, ms_mode=False, normalizer=None)


_FAMILIES: dict = {}


def family(name) -> VnFamily:
    if name not in _FAMILIES:
        _FAMILIES[name] = {
            "std": lambda: VnFamily([0.0, 0.35, 0.7, 1.0]),
            "long": lambda: VnFamily([0.2, 0.9], duration=0.1, num_impulses=40),  # halo 4800 > one tile
            "identity_env": lambda: VnFamily([0.1, 0.6], envelope=IDENTITY_ENVELOPE),
            "seg150": lambda: VnFamily([0.5], num_impulses=150, envelope=tuple(np.linspace(1.0, 0.1, 150).tolist())),
            "one": lambda: VnFamily([0.7]),
        }[name]()
    return _FAMILIES[name]


def dense_clip(frames, seed=0, scale=0.3):
    return (np.random.default_rng(seed).standard_normal((frames, 2)) * scale).astype(np.float32)


# ------------------------------------------------------------------ probe signals

PROBE_FRAMES = 2 * TILE + 700  # two whole tiles and a ragged tile longer than one 512-frame pass
# frame 0 and its pair, lane 31's group, a pass boundary, a packed pair, the tile edge, the ragged tile's lane 31 / 32,
# its pass boundary and its last frame
POSITIONS = [0, 1, 2, 3, 124, 125, 126, 127, 511, 512, 1000, 1001, 4094, 4095, 4096, 4097, 4096 + 511, 4096 + 512, 8191, 8192,
             8192 + 31, 8192 + 32, 8192 + 511, 8192 + 512, PROBE_FRAMES - 1]
PLANTED = [0, 1, 127, 512, 1001, 4095, 4096, 4097, 8192 + 31, 8192 + 32, PROBE_FRAMES - 1]


def _pm(rng, n, lo=0.5, hi=1.0):
    return (rng.uniform(lo, hi, n) * rng.choice([-1.0, 1.0], n)).astype(np.float32)


def _sparse(frames, at, l, r):
    x = np.zeros((frames, 2), np.float32)
    x[at, 0] = l
    x[at, 1] = r
    return x


def _background(rng, frames, max_ratio=3.0):
    """Dense frames with |d| / |s| <= max_ratio, steep ones (|d| > |s|) included."""
    s = _pm(rng, frames).astype(np.float64)
    d = s * rng.uniform(0.0, max_ratio, frames) * rng.choice([-1.0, 1.0], frames)
    return np.column_stack(((s + d) / 2, (s - d) / 2)).astype(np.float32)


def _near_ties(kind, rng, n=300, frames=PROBE_FRAMES):
    """n frames whose |d| / |s| differ by a few float32 ulps or less, in random order over lanes, tiles and chunks."""
    k = rng.integers(0, 4, n)
    e = 2.0 ** rng.integers(-2, 3, n)
    if kind == "zero":  # d = 2**-20 exactly, s moves by k ulps: ratios ~ 2**-21 apart by k ulps; power-of-two copies tie
        L = (1.0 + k * 2.0**-23) * e
        R = L - 2.0**-20 * e
    elif kind == "one":  # R tiny of either sign: ratios on both sides of 1 (the key's steep switch), k ulps of R apart
        L = e
        R = rng.choice([-1.0, 1.0], n) * (3.0 + k) * 2.0**-24 * e
    else:  # subnormal: integers times the smallest subnormal (exact d and s, every frame below FLT_MIN)
        m = rng.integers(1000, 1004, n)
        L = m * 2.0**-149
        R = (m - 97 - k) * 2.0**-149
    at = np.sort(rng.choice(frames, n, replace=False))
    perm = rng.permutation(n)
    return _sparse(frames, at, np.asarray(L, np.float32)[perm], np.asarray(R, np.float32)[perm])


def _filtered_impulses(rng, fam: VnFamily, frames):
    """Impulses in the filtered channel near both ends and at the halo edge of tile 0 (the last input frame a tap of
    tile 0 reaches, and the first it does not); the passed-through channel holds a value wherever the output of the
    filtered one does, so that a shifted filtered channel moves sum L*R."""
    m = fam.max_tap
    at = [0, 1, 7, frames - 1, frames - 2, TILE - 1, TILE, TILE + m, TILE + m + 1, frames - m - 2]
    x = np.zeros((frames, 2), np.float32)
    x[at, 0] = _pm(rng, len(at))
    y = fam.output(x, 0)
    nz = np.flatnonzero(y[:, 0])
    x[nz, 1] = _pm(rng, nz.size)
    return x


def _make_probes():
    """name -> (input (frames, 2) float32, family name or 'identity', sums compared?, planted (frame, class) or None).

    ``sums`` marks the probes whose sums the sensitivity self-check covers (sparse signals: every frame carries a
    visible share of every sum).  The other probes check the exact slots: a planted max-ratio frame over a dense
    background, empty sign classes, ties, zeros."""
    rng = np.random.default_rng(20261021)
    F = PROBE_FRAMES
    pr = {}
    n = len(POSITIONS)
    pr["isolated"] = (_sparse(F, POSITIONS, _pm(rng, n), _pm(rng, n)), "identity", True, None)
    fam = family("one")
    pr["filtered_impulses"] = (_filtered_impulses(rng, fam, 3 * TILE + 5), "one", True, None)
    for p in PLANTED:
        for cls in ("pos", "neg"):
            x = _background(rng, F)
            sgn = 1.0 if cls == "pos" else -1.0
            x[p] = np.float32(sgn * 0.5005), np.float32(-sgn * 0.4995)  # |d| / |s| = 1000
            pr[f"max_ratio_{cls}_{p}"] = (x, "identity", False, (p, cls))
    x = -np.abs(_background(rng, F, max_ratio=0.9))
    pr["all_s_negative"] = (x, "identity", False, None)
    at = np.sort(rng.choice(F, 300, replace=False))
    v = _pm(rng, 300)
    pr["pure_side"] = (_sparse(F, at, v, -v), "identity", True, None)
    z = np.zeros((F, 2), np.float32)
    z[::3, 0] = -0.0
    z[1::3, 1] = -0.0
    z[2::5] = -0.0
    pr["zeros"] = (z, "identity", False, None)
    for kind in ("zero", "one"):
        pr[f"near_ties_{kind}"] = (_near_ties(kind, rng), "identity", True, None)
    pr["near_ties_subnormal"] = (_near_ties("subnormal", rng), "identity", False, None)
    at = np.sort(rng.choice(F, 300, replace=False))
    pr["quiet_1e-20"] = (_sparse(F, at, _pm(rng, 300) * np.float32(1e-20), _pm(rng, 300) * np.float32(1e-20)), "identity", True, None)
    pr["quiet_1e-41"] = (_sparse(F, at, _pm(rng, 300) * np.float32(1e-41), _pm(rng, 300) * np.float32(1e-41)), "identity", False, None)
    pr["loud_int16"] = (_sparse(F, at, np.round(_pm(rng, 300) * 32767), np.round(_pm(rng, 300) * 32767)), "identity", True, None)
    return pr


_PROBES: dict = {}


def probes():
    if not _PROBES:
        _PROBES.update(_make_probes())
    return _PROBES


def probe_output(name):
    x, fam, _, _ = probes()[name]
    return identity_output(x) if fam == "identity" else family(fam).output(x, 0)


def probe_program(name, frames):
    fam = probes()[name][1]
    return identity_program() if fam == "identity" else family(fam).program(frames)


_REFS: dict = {}


def probe_ref(name):
    if name not in _REFS:
        _REFS[name] = O.objective_partials(probe_output(name))
    return _REFS[name]


def loud_overflow_clip():
    """Values whose float32 squares overflow (|x| > 1.9e19) beside ordinary ones."""
    rng = np.random.default_rng(5)
    x = dense_clip(2 * TILE + 9, seed=5)
    x[rng.choice(len(x), 20, replace=False)] = np.float32(3e19)
    return x


# ------------------------------------------------------------------ CPU: the reference itself


def test_reference_pins_the_golden_viola_values():
    """The reference against the reference library's own intermediate values (tests/golden/objective.json)."""
    fs, x = G.wav("viola")
    for row in G.objective()["viola_vn"]:
        taps = O.vn_candidate_taps(row["kappa"], sample_rate_hz=fs, duration_seconds=0.03, num_impulses=30, seed=1)
        p = O.objective_partials(O.vn_candidate_signal(x, taps))["p"]
        assert abs(p[0] - row["sum_r"]) <= 2e-6 * row["sum_r"]  # the golden value is a float32 pairwise sum
        assert abs(p[2] / p[0] - row["spread"]) <= 2e-6
        assert abs(p[1] / p[0] - row["centroid"]) <= 2e-6
        assert abs(p[3] / p[0] - row["m3"]) <= 2e-6
        assert abs(p[4] - row["dot_lr"]) <= 1e-5 * max(1.0, abs(row["dot_lr"]))
        assert abs(np.sqrt(p[5]) - row["norm_l"]) <= 1e-5 * row["norm_l"]
        assert float(opt._max_abs_theta_f32(p)) == pytest.approx(row["max_abs_theta"], abs=1.2e-7)
        assert p[10] == x.shape[0] and p[11] == 0.0


def test_reference_partials_give_the_reference_scores():
    """The library's scalar chains applied to the reference partials reproduce O.objective."""
    fs, viola = G.wav("viola")
    sigs = [viola[40000:100000], O.coloured_clip(0, 3 * TILE + 5), dense_clip(TILE + 1, seed=3)]
    for x in sigs:
        for j in range(len(family("std").kappas)):
            y = family("std").output(x, j)
            got = opt._vn_scores_rows(O.objective_partials(y)["p"][None], **KW)[0]
            assert abs(float(got) - float(O.objective(y, **KW))) <= 5e-4
        for d in (0, 1, 300, len(x) + 5):
            y = O.haas(x, sample_rate_hz=1, delay_time_seconds=d)
            got = opt._haas_scores_rows(O.haas_partials(y)["p"][None], **KW)[0]
            want = O.objective(y, **KW)
            assert abs(got - want) <= 1e-9 * abs(want)
    for name in ("isolated", "filtered_impulses", "near_ties_one", "max_ratio_neg_4097", "quiet_1e-20", "loud_int16"):
        y = probe_output(name)
        got = opt._vn_scores_rows(probe_ref(name)["p"][None], **KW)[0]
        want = float(O.objective(y, **KW))
        assert abs(float(got) - want) <= 5e-4 + 1e-6 * abs(want), name  # the quiet probe's correlation makes a score of 1.6e6


def test_reference_tracker_is_exact_and_keeps_the_earliest_tie():
    d = np.array([1, 3, 2, 6, 0, 5], np.float32)
    s = np.array([2, 4, 1, 2, 0, 0], np.float32)
    assert O._best_ratio(d, s) == (5.0, 0.0, 5)  # s == 0 is an infinite ratio
    assert O._best_ratio(d[:4], s[:4]) == (6.0, 2.0, 3)  # 3 / 1 ... 6 / 2: the earlier 2 / 1 is smaller, 6 / 2 == 3 keeps frame 3
    assert O._best_ratio(np.array([2, 6], np.float32), np.array([1, 3], np.float32)) == (2.0, 1.0, 0)
    assert O._best_ratio(np.zeros(3, np.float32), np.ones(3, np.float32)) == (0.0, 1.0, -1)
    a, b = np.float32(1 + 2**-23), np.float32(1)  # ratios one float32 ulp apart, beyond float64 division's help
    assert O._best_ratio(np.array([b * a, a * a], np.float32), np.array([a, a], np.float32))[2] == 1


def test_tolerances_are_not_vacuous():
    """For dense clips the bound is a few parts in 1e5 of the terms' magnitudes, so a sum that lost or doubled a
    thousandth of its frames fails, and the penalty slots are exact."""
    ref = O.objective_partials(family("std").output(O.coloured_clip(1, 3 * TILE + 5), 2))
    tol = vn_tolerance(ref)
    assert np.all(tol[:6] <= 2e-5 * ref["mag"] + 1e-6 * ref["mag"][0])
    hr = O.haas_partials(O.haas(O.coloured_clip(1, 3 * TILE + 5), sample_rate_hz=1, delay_time_seconds=7))
    assert np.all(haas_tolerance(hr)[[0, 5, 6]] <= 1e-14 * hr["mag"][[0, 5, 6]])


@pytest.mark.parametrize("name", sorted(_make_probes()))
def test_probe_sensitivity(name):
    """Each compared slot's bound is at least 10x below what the reference shows when a probe frame is dropped or
    counted twice (the change is that frame's term) or when the filtered channel moves by one frame.  Probes that check
    only the exact slots must have their planted record frame as the unique maximum."""
    x, fam, sums, planted = probes()[name]
    y = probe_output(name)
    ref = probe_ref(name)
    if planted is not None:
        p, cls = planted
        assert ref["at"][0 if cls == "pos" else 1] == p
        d, s = ref["d"].astype(np.float64), ref["s"].astype(np.float64)
        in_cls = (s >= 0) if cls == "pos" else (s < 0)
        others = np.delete(np.abs(d) / np.abs(s), p)[np.delete(in_cls, p)]
        assert np.all(others * 1.01 < abs(d[p]) / abs(s[p]))  # dropping it moves the record
    if not sums:
        return
    tol = vn_tolerance(ref)
    l, r = y[:, 0].astype(np.float64), y[:, 1].astype(np.float64)
    th = ref["theta"]
    rad = np.sqrt((y[:, 0] * y[:, 0] + y[:, 1] * y[:, 1]).astype(np.float64))
    terms = np.stack([rad, rad * th, rad * th**2, rad * th**3, l * r, l * l])
    live = np.flatnonzero(np.any(terms != 0, axis=0))
    assert live.size > 0
    seen = np.max(np.abs(terms[:, live]) / tol[:6, None], axis=0)
    assert np.min(seen) >= 10, f"frame {live[np.argmin(seen)]} moves no slot by 10 bounds ({np.min(seen):.3g})"
    for step in (1, -1):
        z = y.copy()
        z[:, 0] = np.roll(y[:, 0], step)
        z[0 if step == 1 else -1, 0] = 0.0
        q = O.objective_partials(z)
        moved = np.max(np.abs(q["p"][:6] - ref["p"][:6]) / tol[:6])
        assert moved >= 10 or q["p"][6] * ref["p"][7] != ref["p"][6] * q["p"][7], (step, moved)


# ------------------------------------------------------------------ GPU: velvet-noise objective, every kernel

@pytest.fixture
def tpc_env(monkeypatch):
    """Sets VND_OBJ_TPC (the tiles per chunk of the objective's chunk plan; None: the planned chunks)."""

    def use(tpc=None):
        if tpc is None:
            monkeypatch.delenv("VND_OBJ_TPC", raising=False)
        else:
            monkeypatch.setenv("VND_OBJ_TPC", tpc)

    use(None)
    return use


def _lengths(halo):
    return sorted({1, 7, 300, TILE - 1, TILE, TILE + 1, 3 * TILE + 5, 9216, halo - 1, halo, halo + 1})


@gpu
@pytest.mark.parametrize("fam_name", ["std", "long", "identity_env", "seg150"])
def test_vn_partials_against_reference(tpc_env, fam_name):
    fam = family(fam_name)
    for frames in _lengths(fam.max_tap + 1):
        x = O.coloured_clip(frames % 7, frames) if frames > 1 else dense_clip(1)
        got = opt.vn_objective_partials(x, fam.program(frames))[0]
        for j in range(len(fam.kappas)):
            check_vn(got[j], O.objective_partials(fam.output(x, j)), f"{fam_name} frames={frames} cand={j}")


@gpu
def test_vn_partials_thirty_seconds(tpc_env):
    fam = family("std")
    x = O.coloured_clip(3, 30 * FS)
    got = opt.vn_objective_partials(x, fam.program(len(x)))[0]
    for j in range(len(fam.kappas)):
        check_vn(got[j], O.objective_partials(fam.output(x, j)), f"30 s cand={j}")


@gpu
def test_filter_beyond_shared_memory_is_refused(tpc_env):
    """A 1000-segment envelope's program does not fit the shared-memory budget of any objective kernel: an error, not a
    result."""
    fam = VnFamily([0.5], duration=0.03, num_impulses=1000 // 4, envelope=tuple(np.linspace(1.0, 0.1, 1000)))
    with pytest.raises(N.VndError) as e:
        opt.vn_objective_partials(dense_clip(5000), fam.program(5000))
    assert e.value.status == N.VND_EUNSUPPORTED


@gpu
@pytest.mark.parametrize("n_cand", [15, 16, 17, 40])
def test_candidate_groups_and_chunk_plans(tpc_env, n_cand):
    """Groups shrink to 16 candidates on a short clip; every chunk size must give the reference."""
    fam = VnFamily(np.linspace(0.0, 1.0, n_cand))
    frames = 3 * TILE + 5
    x = O.coloured_clip(n_cand, frames)
    prog = fam.program(frames)
    refs = [O.objective_partials(fam.output(x, j)) for j in range(n_cand)]
    first = None
    for tpc in ("1", "2", "3", None):
        tpc_env(tpc)
        got = opt.vn_objective_partials(np.stack([x.T, x.T[::-1]]), prog)
        for j in range(n_cand):
            check_vn(got[0, j], refs[j], f"tpc={tpc} cand={j}")
        first = got if first is None else first
        assert np.array_equal(got, first), tpc  # the chunk plan does not change a bit


@gpu
def test_vn_probes(tpc_env):
    for name, (x, fam, sums, _) in probes().items():
        got = opt.vn_objective_partials(x, probe_program(name, len(x)))[0, 0]
        check_vn(got, probe_ref(name), name, sums=True)


@gpu
def test_run_list_probes_and_ragged_batches(tpc_env):
    """Every probe and 1-frame and ordinary clips packed in one buffer, loud neighbours around each, with runs of count
    0: one run-list call, every row against the reference."""
    loud = dense_clip(TILE + 3, seed=9, scale=3e4)
    clips, fams = [], []
    for name, (x, fam, _, _) in probes().items():
        clips += [loud, x]
        fams += [None, name]
    extra = [("one_frame", dense_clip(1, seed=1)), ("seven", dense_clip(7, seed=2)), ("tile_plus_one", dense_clip(TILE + 1, seed=3))]
    for name, x in extra:
        clips += [x, loud]
        fams += [name, None]
    offs = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    xp = np.ascontiguousarray(np.concatenate(clips).T)
    std = family("std")
    progs, runs, refs = [], [[], [], [], []], []
    ch = row = 0
    for i, (c, name) in enumerate(zip(clips, fams)):
        if name is None:
            prog, ys = std.program(len(c)), None
            runs_count = 0  # a run that scores nothing
        elif name in probes():
            prog, ys = probe_program(name, len(c)), [probe_output(name)]
            runs_count = 1
        else:
            prog, ys = std.program(len(c)), [std.output(c, j) for j in range(len(std.kappas))]
            runs_count = len(std.kappas)
        progs.append(prog)
        for r, v in zip(runs, (i, ch, runs_count, row)):
            r.append(v)
        if ys:
            refs += [(name, O.objective_partials(y) if name not in probes() else probe_ref(name)) for y in ys]
        ch += prog.channels
        row += runs_count
    got = opt.vn_objective_run_partials(xp, offs, opt._concat_programs(progs), runs)
    assert got.shape[0] == len(refs)
    for k, (name, ref) in enumerate(refs):
        check_vn(got[k], ref, f"run row {k} ({name})")


@gpu
def test_loud_overflow_scores_are_non_finite_where_the_reference_is(tpc_env):
    x = loud_overflow_clip()
    fam = family("std")
    with np.errstate(all="ignore"):
        want = [O.objective(fam.output(x, j), **KW) for j in range(len(fam.kappas))]
        got = opt.vn_scores_from_partials(opt.vn_objective_partials(x, fam.program(len(x))), **KW)[0]
        assert [bool(np.isfinite(g)) for g in got] == [bool(np.isfinite(w)) for w in want]
        ok = dense_clip(len(x))
        got = opt.vn_scores_from_partials(opt.vn_objective_partials(ok, fam.program(len(ok))), **KW)[0]
        assert np.all(np.isfinite(got))


# ------------------------------------------------------------------ GPU: stereo-family velvet noise


@gpu
def test_vn_stereo_partials_against_reference(tpc_env):
    cases = [("LR", (0,), None), ("MS", (0, 1), None), ("MS", (0, 1), 0.3), ("LR", (0, 1), 1.0), ("MS", (), 0.7), ("LR", (), None)]
    for frames in (1, 7, 1000, TILE, TILE + 1, 3 * TILE + 5):
        x = O.coloured_clip(frames % 5, frames) if frames > 1 else dense_clip(1)
        decs, ys = [], []
        for k, (mode, fc, width) in enumerate(cases):
            decs.append(D.VelvetNoise(sample_rate_hz=FS, normalizer=None, mode=mode, filtered_channels=fc, width=width, log_distribution_strength=k / 5,
                                      seed=k + 1))
            taps = O.class_taps(sample_rate_hz=FS, log_distribution_strength=k / 5, filtered_channels=fc, seed=k + 1)
            ys.append(O.vn_decorrelate(x, taps, ms_mode=mode == "MS", width=width, normalizer=None))
        got = opt.vn_stereo_objective_partials(x, decs)
        for j, y in enumerate(ys):
            check_vn(got[j], O.objective_partials(y), f"stereo frames={frames} cand={j}")
    for name in ("isolated", "max_ratio_pos_4097", "near_ties_one", "quiet_1e-20"):
        x = probes()[name][0]
        d = D.VelvetNoise(sample_rate_hz=FS, normalizer=None, mode="LR", filtered_channels=(), seed=1)  # both channels passed through
        check_vn(opt.vn_stereo_objective_partials(x, [d])[0], O.objective_partials(identity_output(x)), f"stereo {name}")


# ------------------------------------------------------------------ GPU: Haas objective


def _haas_y64(x64, d):
    n = len(x64)
    y = np.zeros((n + d, 2))
    y[:n] = x64
    y[:, 0] = np.roll(y[:, 0], d)
    return y


@gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_haas_partials_against_reference(dtype):
    for frames in (1, 7, 255, 256, 257, 3 * TILE + 5):
        x = dense_clip(frames, seed=frames).astype(dtype)
        if dtype == np.float64:
            x = x + np.random.default_rng(1).standard_normal(x.shape) * 1e-9  # values no float32 holds
        delays = [0, 1, frames - 1, frames, frames + 3, 700]
        got = opt.haas_objective_partials(np.ascontiguousarray(x.T[None]), delays)[0]
        for j, d in enumerate(delays):
            y = O.haas(x, sample_rate_hz=1, delay_time_seconds=d) if dtype == np.float32 else _haas_y64(x, d)
            check_haas(got[j], O.haas_partials(y), f"{dtype.__name__} frames={frames} delay={d}")
    for name in ("isolated", "pure_side", "near_ties_subnormal", "quiet_1e-41", "loud_int16", "zeros", "all_s_negative"):
        x = probes()[name][0]
        got = opt.haas_objective_partials(np.ascontiguousarray(x.T[None]), [0, 3])[0]
        for j, d in enumerate((0, 3)):
            check_haas(got[j], O.haas_partials(O.haas(x, sample_rate_hz=1, delay_time_seconds=d)), f"{name} delay={d}")


@gpu
def test_haas_pair_partials_against_reference():
    loud = dense_clip(999, seed=4, scale=3e4)
    clips = [loud, dense_clip(1, seed=1), loud, dense_clip(7, seed=2), probes()["isolated"][0], loud, dense_clip(TILE + 1, seed=3)]
    offs = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    xp = np.ascontiguousarray(np.concatenate(clips).T)
    pairs = [(i, d) for i in (1, 3, 4, 6) for d in (0, 1, 5, 1200)]
    got = opt.haas_objective_pair_partials(xp, offs, [p[0] for p in pairs], [p[1] for p in pairs])
    for k, (i, d) in enumerate(pairs):
        check_haas(got[k], O.haas_partials(O.haas(clips[i], sample_rate_hz=1, delay_time_seconds=d)), f"pair clip={i} delay={d}")


@gpu
def test_haas_effect_partials_against_reference():
    settings = [(0.0, 0, False, None), (0.001, 0, False, None), (0.002, 1, True, None), (0.0005, -1, True, 0.4), (0.003, -2, False, 1.0)]
    for x in (dense_clip(3 * TILE + 5, seed=8), dense_clip(5, seed=8)[:, 0], probes()["isolated"][0]):
        hs = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=t, delayed_channel=ch, mode="MS" if ms else "LR", width=w) for t, ch, ms, w in settings]
        got = opt.haas_effect_objective_partials(x, hs)
        for j, (t, ch, ms, w) in enumerate(settings):
            y = O.haas(x, sample_rate_hz=FS, delay_time_seconds=t, delayed_channel=ch, ms_mode=ms, width=w)
            check_haas(got[j], O.haas_partials(y), f"effect frames={len(x)} cand={j}")


# ------------------------------------------------------------------ GPU: sums independent of the chunk plan


def hdr_clip(seed, frames=30 * FS, fade_db=-120.0):
    """A clip whose first half is near-mono (side channel at 1e-3 of the mid) and fades in from ``fade_db``: there theta
    is tiny and r small, so the tile sums of r theta^n, L*R and L*L span more binades than float64 adds exactly, and a
    plain float64 sum of them depended on the chunk plan."""
    from scipy.signal import lfilter

    rng = np.random.default_rng(7000 + seed)
    m = lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    s = lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    half = frames // 2
    side = np.full(frames, 0.3)
    side[:half] = 1e-3
    gain = np.ones(frames)
    gain[:half] = 10.0 ** (np.linspace(fade_db, 0.0, half) / 20)
    x = np.column_stack((m + side * s, m - side * s)) * gain[:, None]
    return (x / np.max(np.abs(x)) * 0.5).astype(np.float32)


# (seed, fade-in from dB).  -360 dB: the r-weighted tile sums span about 60 binades, close to the ~70 within which the
# double-double sums stay exact.
HDR = [(0, -120.0), (1, -120.0), (2, -120.0), (0, -200.0), (1, -200.0), (2, -200.0), (3, -360.0)]
HDR_FAMILY = np.linspace(0.0, 1.0, 16)


@gpu
def test_sums_do_not_depend_on_the_chunk_plan(tpc_env):
    import torch

    fam = VnFamily(HDR_FAMILY)
    frames = 30 * FS
    prog = fam.program(frames)
    for seed, fade in HDR:
        x = hdr_clip(seed, frames, fade)
        alone = opt.vn_objective_partials(x, prog)[0]
        for tpc in ("1", "2", "3", "7"):
            tpc_env(tpc)
            assert np.array_equal(opt.vn_objective_partials(x, prog)[0], alone), (seed, tpc)
        tpc_env(None)
        xt = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
        for others in (1, 3, 64):
            g = torch.Generator(device="cuda").manual_seed(others)
            batch = torch.randn((others + 1, 2, frames), device="cuda", generator=g) * 0.2
            batch[others // 2] = xt
            got = opt.vn_objective_partials(batch, prog)[others // 2].cpu().numpy()
            assert np.array_equal(got, alone), (seed, others)
            del batch
        # the run list, next to clips of other lengths
        clips = [dense_clip(10 * FS + 3, seed=1), x, dense_clip(7, seed=2), dense_clip(20 * FS, seed=3)]
        offs = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
        progs = [fam.program(len(c)) for c in clips]
        k = len(fam.kappas)
        runs = [[0, 1, 2, 3], [0, k, 2 * k, 3 * k], [k, k, k, k], [0, k, 2 * k, 3 * k]]
        got = opt.vn_objective_run_partials(np.ascontiguousarray(np.concatenate(clips).T), offs, opt._concat_programs(progs), runs)
        assert np.array_equal(got[k:2 * k], alone), seed
        if fade == -360.0:
            check_vn(alone[5], O.objective_partials(fam.output(x, 5)), "hdr -360 dB")


@gpu
def test_batch_optimiser_equals_clip_by_clip_on_high_dynamic_range_clips():
    kw = dict(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1, grid_size=48)
    clips = [hdr_clip(seed, 30 * FS, fade) for seed, fade in HDR[::2]] + [O.coloured_clip(4, 12 * FS)]
    both, info = opt.optimize_velvet_noise_batch(input_signals=clips, details=True, **kw)
    fam = opt._vn_family(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)
    kappas = np.linspace(0.0, 1.0, kw["grid_size"])
    for i, c in enumerate(clips):
        one = opt.vn_scores_from_partials(opt.vn_objective_partials(c, fam(kappas, len(c))), **KW)[0]
        assert np.array_equal(info["scores"][i], one), i
        assert float(both[i]) == float(opt.optimize_velvet_noise(input_signal=c, **kw)), i
