"""CPU oracle for the velvet-noise decorrelation hot path.  TEST INFRASTRUCTURE ONLY.

This module is a numpy restatement of the reference algorithm (ckonst/VNDecorrelate,
``src/vndecorrelate``).  It exists so that the CUDA path can be checked on a box where the
reference itself is not installed.  Nothing under ``vndecorrelate_b200/`` may import it; only
``tests/``, ``__graft_entry__.smoke()`` and the CPU-baseline legs of ``bench.py`` do.

Parity status: PINNED.  ``tests/test_oracle_golden.py`` checks every function here against
fixtures in ``tests/golden/`` that were produced by importing the unmodified reference in the
build container (``tests/golden/make_golden.py``), including the two golden outputs the reference
itself commits (``audio/viola_decorrelated.wav``, ``audio/vocal_decorrelated.wav``).

Each function cites the reference lines it restates (paths relative to the reference root).
The numpy operation order is kept where it decides the rounding (slice accumulation per tap,
separate multiply/add, axis-0 reductions); the code structure is otherwise our own.
"""

from __future__ import annotations

import math
from typing import Callable, Sequence

import numpy as np

EPS = 1e-10  # src/vndecorrelate/utils/dsp.py:6
DEFAULT_ENVELOPE = (0.85, 0.55, 0.35, 0.2)  # src/vndecorrelate/decorrelation.py:357


# --------------------------------------------------------------------------------------
# tap positions  (decorrelation.py:478-546 class path, :549-627 function path)
# --------------------------------------------------------------------------------------


def log_weights(strength: float, count: int) -> np.ndarray:
    """``count + 1`` exponentially growing weights; utils/dsp.py:194-201."""
    ramp = np.arange(count + 1.0) / count
    return (10.0 ** (2.0 * strength * ramp)) / (100.0 * ((1.0 + (strength * 99.0)) / 100.0))


def place_impulses(u: np.ndarray, weights: np.ndarray, starts: np.ndarray, jitter: float) -> np.ndarray:
    """int32 positions = round(u * max(0, w*jitter - 1) + start); utils/dsp.py:248-250."""
    return np.round(u * np.fmax(0.0, weights * jitter - 1) + starts).astype(np.int32)


def _draws(seed, n_imp: int, n_filters: int):
    """The two uniform draws, in the reference's order and shapes; decorrelation.py:488,510-521."""
    rng = np.random.default_rng(seed)
    sign_u = rng.uniform(low=0, high=1, size=(n_imp, n_filters))
    offs_u = rng.uniform(low=0, high=1, size=(n_imp + 1, n_filters))
    signs = (2 * np.round(sign_u)) - 1
    return signs, offs_u


def _interval_starts(strength: float, n_imp: int, fir_len: int):
    """decorrelation.py:494-506 (same in :580-590)."""
    w = log_weights(strength, n_imp)
    starts = np.cumsum(w)
    if strength == 0.0:
        starts -= 1.0
    starts *= fir_len / starts[-1]
    return w, starts


def class_fir_length(sample_rate_hz: int, duration_seconds: float) -> int:
    """decorrelation.py:449-452 (round, then int)."""
    return int(round(sample_rate_hz * duration_seconds))


def class_taps(
    *,
    sample_rate_hz: int,
    duration_seconds: float = 0.03,
    num_impulses: int = 30,
    num_outs: int = 2,
    num_segments: int = 4,
    log_distribution_strength: float = 1.0,
    filtered_channels: Sequence[int] = (0, 1),
    seed=None,
):
    """Tap structure of ``VelvetNoise._generate``: ``taps[channel][segment][0|1]`` is the list of
    int32 indices of negative (0) / positive (1) impulses in impulse order; ``[]`` for channels
    that are not filtered.  decorrelation.py:478-546.
    """
    fir_len = class_fir_length(sample_rate_hz, duration_seconds)
    w, starts = _interval_starts(log_distribution_strength, num_impulses, fir_len)
    n_filters = len(filtered_channels)
    signs, offs_u = _draws(seed, num_impulses, n_filters)
    density = num_impulses / duration_seconds  # decorrelation.py:444-447
    jitter = sample_rate_hz / density  # decorrelation.py:523
    out = []
    for ch in range(num_outs):
        if ch not in filtered_channels:
            out.append([])
            continue
        # NB: the draw column is the channel number itself (decorrelation.py:531), so a filtered
        # channel >= len(filtered_channels) raises IndexError exactly like the reference.
        pos = place_impulses(offs_u[:, ch], w, starts, jitter)
        segs = [([], []) for _ in range(num_segments)]
        for j in range(num_impulses):
            s = int(j / (num_impulses / num_segments))  # decorrelation.py:540
            which = int((signs[j, ch] + 1) / 2)  # decorrelation.py:541
            segs[s][which].append(pos[j])
        out.append(segs)
    return out


def dense_fir(
    *,
    duration_seconds: float,
    num_impulses: int,
    num_outs: int = 2,
    sample_rate_hz: int = 44100,
    segment_envelope: Sequence[float] = DEFAULT_ENVELOPE,
    log_distribution_strength: float = 1.0,
    seed=None,
) -> np.ndarray:
    """``generate_velvet_noise``: dense ``(int(dur*fs), num_outs)`` fp32 FIR, later impulses
    overwrite earlier ones on a collision.  decorrelation.py:549-627."""
    fir_len = int(duration_seconds * sample_rate_hz)  # decorrelation.py:575 (truncation!)
    fir = np.zeros((fir_len, num_outs), dtype=np.float32)
    env = tuple(segment_envelope) if len(segment_envelope) else (1.0,)
    w, starts = _interval_starts(log_distribution_strength, num_impulses, fir_len)
    signs, offs_u = _draws(seed, num_impulses, num_outs)
    jitter = sample_rate_hz / (num_impulses / duration_seconds)
    for ch in range(num_outs):
        pos = place_impulses(offs_u[:, ch], w, starts, jitter)
        for j in range(num_impulses):
            s = int(j / (num_impulses / len(env)))
            fir[pos[j], ch] = signs[j, ch] * env[s]
    return fir


def class_dense_fir(taps, envelope: Sequence[float], fir_len: int) -> np.ndarray:
    """``VelvetNoise.FIR``: float64 ``(fir_len, n_filters)``; decorrelation.py:454-472."""
    chans = [c for c in taps if c != []]
    fir = np.zeros((fir_len, len(chans)))
    for ci, segs in enumerate(chans):
        for si, (neg, pos) in enumerate(segs):
            for i in neg:
                fir[i, ci] = envelope[si] * -1
            for i in pos:
                fir[i, ci] = envelope[si] * 1
    return fir


# --------------------------------------------------------------------------------------
# sparse FIR  (decorrelation.py:393-415 and :630-660)
# --------------------------------------------------------------------------------------


def fir_class_order(x: np.ndarray, taps, envelope: Sequence[float], num_outs: int) -> np.ndarray:
    """``VelvetNoise.convolve``.  Per channel and segment: subtract the shifted input for each
    negative tap, add it for each positive tap (fp32 scratch), scale by the segment gain unless
    the envelope is exactly ``(1.0,)``, add into the output.  decorrelation.py:393-415."""
    n = len(x)
    scratch = np.zeros(n, dtype=np.float32)
    y = np.zeros((n, num_outs), dtype=np.float32)
    # the reference compares the attribute itself with the tuple (1.0,): a list [1.0] is != (1.0,)
    # and is multiplied through (by exactly 1.0, which changes nothing).
    identity = envelope == (1.0,)
    for ch in range(num_outs):
        if taps[ch] == []:
            y[:, ch] = x[:, ch]
    for ch, segs in enumerate(taps):
        for si, (neg, pos) in enumerate(segs):
            for i in neg:
                i = int(i)
                if i < n:
                    scratch[: n - i] -= x[i:, ch]
            for i in pos:
                i = int(i)
                if i < n:
                    scratch[: n - i] += x[i:, ch]
            if not identity:
                scratch *= envelope[si]
            y[:, ch] += scratch
            scratch.fill(0)
    return y


def fir_function_order(x: np.ndarray, fir: np.ndarray) -> np.ndarray:
    """``convolve_velvet_noise``: ascending non-zero index, ``y[:n-i] += x[i:] * v``.
    decorrelation.py:630-660.  (1-D input raises IndexError in the reference, :650.)"""
    n_ch = 1 if x.ndim == 1 else x.shape[1]
    if n_ch > 1 and x.shape[1] != fir.shape[1]:
        raise ValueError("channel mismatch")  # utils/dsp.py:305-310
    n = len(x)
    y = np.zeros(x.shape, dtype=np.float32)
    for ch in range(n_ch):
        col = fir[:, ch]
        nz = np.nonzero(col)[0]
        for i in nz:
            i = int(i)
            if i < n:
                y[: n - i, ch] += x[i:, ch] * col[i]
    return y


# --------------------------------------------------------------------------------------
# stereo helpers  (utils/dsp.py:21-167)
# --------------------------------------------------------------------------------------


def _need_stereo(a: np.ndarray) -> None:
    if a.ndim != 2 or a.shape[1] != 2:
        raise ValueError(f"expected (n, 2), got {a.shape}")  # utils/dsp.py:297-302


def lr_to_ms(a: np.ndarray) -> None:
    """utils/dsp.py:124-144."""
    _need_stereo(a)
    m = np.sum(a, axis=1) * 0.5
    s = (a[:, 0] - a[:, 1]) * 0.5
    a[:, 0] = m
    a[:, 1] = s


def ms_to_lr(a: np.ndarray) -> None:
    """utils/dsp.py:147-167."""
    _need_stereo(a)
    l = np.sum(a, axis=1)
    r = a[:, 0] - a[:, 1]
    a[:, 0] = l
    a[:, 1] = r


def stereo_width(a: np.ndarray, width: float) -> None:
    """utils/dsp.py:21-37."""
    lr_to_ms(a)
    a[:, 0] *= 1.0 - width
    a[:, 1] *= width
    ms_to_lr(a)


def side_encode(x: np.ndarray, y: np.ndarray) -> None:
    """``encode_signal_to_side_channel``: M from the dry input, S from the wet signal.
    utils/dsp.py:40-63."""
    _need_stereo(x)
    _need_stereo(y)
    m = np.sum(x, axis=1)
    s = (y[:, 0] - y[:, 1]) * 0.5
    y[:, 0] = (m + s) * 0.5
    y[:, 1] = (m - s) * 0.5


def rms_match(x: np.ndarray, y: np.ndarray, stereo_mode: bool = False, epsilon: float = EPS) -> None:
    """``rms_normalize``: y *= sqrt(mean(x^2)) / sqrt(mean(y^2) + eps), per channel (DUAL_MONO)
    or over the whole array (STEREO / 1-D).  utils/dsp.py:87-109."""
    ax_x = None if (x.ndim == 1 or stereo_mode) else 0
    ax_y = None if (y.ndim == 1 or stereo_mode) else 0
    y *= np.sqrt(np.mean(np.square(x), axis=ax_x)) / np.sqrt(np.mean(np.square(y), axis=ax_y) + epsilon)


def seq_sumsq_f32(col: np.ndarray) -> np.float32:
    """What numpy's axis-0 reduction of a C-order (n, C) fp32 array does per column: a strict
    left-to-right fp32 running sum of the fp32-rounded squares (SURVEY.md Appendix A.4)."""
    sq = np.square(col.astype(np.float32))
    return np.cumsum(sq, dtype=np.float32)[-1] if len(sq) else np.float32(0)


# --------------------------------------------------------------------------------------
# decorrelators  (decorrelation.py:417-442, :192-230, :137-144)
# --------------------------------------------------------------------------------------


def vn_decorrelate(
    x: np.ndarray,
    taps,
    *,
    envelope: Sequence[float] = DEFAULT_ENVELOPE,
    num_outs: int = 2,
    ms_mode: bool = True,
    width: float | None = None,
    normalizer: Callable | None | str = "rms",
) -> np.ndarray:
    """``VelvetNoise.decorrelate``; decorrelation.py:417-442."""
    x = x.astype(np.float32, copy=False)
    if x.ndim == 1:
        x = np.column_stack((x, x))
    y = fir_class_order(x, taps, envelope, num_outs)
    if ms_mode:
        side_encode(x, y)
    if width is not None:
        stereo_width(y, width)
    if normalizer == "rms":
        rms_match(x, y)
    elif normalizer:
        normalizer(x, y)
    return y


def haas(
    x: np.ndarray,
    *,
    sample_rate_hz: int,
    delay_time_seconds: float = 0.02,
    delayed_channel: int = 0,
    ms_mode: bool = False,
    width: float | None = None,
) -> np.ndarray:
    """``HaasEffect.decorrelate``: float64 ``(n + d, 2)``; decorrelation.py:192-230."""
    x = x.astype(np.float32, copy=False)
    d = round(delay_time_seconds * sample_rate_hz)
    n = len(x)
    out = np.zeros((n + d, 2))
    mono = x.ndim == 1
    if mono:
        x = np.column_stack((x, x))
    out[:n, :] = x
    if ms_mode and not mono:
        lr_to_ms(out)
    out[:, delayed_channel] = np.roll(out[:, delayed_channel], d, axis=0)
    if ms_mode:
        ms_to_lr(out)
        if mono:
            out *= 0.5
    if width is not None:
        stereo_width(out, width)
    return out


# --------------------------------------------------------------------------------------
# stereo-image objective and the sweep  (optimization.py:11-155, utils/dsp.py:374-422)
# --------------------------------------------------------------------------------------


def polar(left: np.ndarray, right: np.ndarray):
    """``polar_coordinates(left, right, normalize=False)`` with the default 'MS' angle and
    semicircular fold; returns (radii, thetas, weights).  utils/dsp.py:374-422."""
    th = np.arctan2(left - right, left + right)
    th = np.where(th < -np.pi / 2, th + np.pi, np.where(th > np.pi / 2, th - np.pi, th))
    r = np.sqrt(left**2 + right**2)
    w = r / (r.sum() + EPS)
    return r, th, w


def objective_terms(y: np.ndarray, angle_limit: float):
    """The five ingredients of ``symmetry_aware_objective`` with the reference's dtype chain.
    optimization.py:11-43, :71-95."""
    _, th, w = polar(y[:, 0], y[:, 1])
    spread = float(np.sum(w * th**2))
    cen = float(np.sum(w * th))
    skew = float(np.sum(w * th**3)) / (max(spread, EPS) ** 1.5)
    nl = np.linalg.norm(y[:, 0]) + EPS
    corr = np.dot(y[:, 0] / nl, y[:, 1] / nl)  # both channels normalised by ||L||, optimization.py:13-16
    exceed = max(0.0, float(np.max(np.abs(th)) - angle_limit))
    return spread, cen, skew, corr, exceed


def objective(
    y: np.ndarray,
    *,
    angle_limit: float = np.pi / 4,
    lambda_mean: float = 5.0,
    lambda_skew: float = 2.0,
    lambda_correlation: float = 15.0,
    lambda_penalty: float = 1e3,
):
    """``symmetry_aware_objective`` applied to an already decorrelated signal ``y``.
    optimization.py:46-105."""
    spread, cen, skew, corr, exceed = objective_terms(y, angle_limit)
    obj = spread - lambda_mean * cen**2 - lambda_skew * skew**2 - lambda_correlation * corr**2 - lambda_penalty * exceed**2
    return -obj


# --------------------------------------------------------------------------------------
# float64 references of the objective kernels' partial sums (include/vnd_b200.h layouts)
# --------------------------------------------------------------------------------------


def _folded_theta(d: np.ndarray, s: np.ndarray) -> np.ndarray:
    """float64 ``arctan2(d, s)`` folded into [-pi/2, pi/2] (utils/dsp.py:399-412)."""
    th = np.arctan2(d, s)
    return np.where(th < -np.pi / 2, th + np.pi, np.where(th > np.pi / 2, th - np.pi, th))


def _sums(terms) -> tuple[np.ndarray, np.ndarray]:
    """Correctly rounded sums (``math.fsum``) of each term array and of its magnitudes; ``np.sum`` where a term is not
    finite (the sum is then inf or nan either way)."""
    sums, mags = [], []
    for t in terms:
        if np.all(np.isfinite(t)):
            sums.append(math.fsum(t.tolist()))
            mags.append(math.fsum(np.abs(t).tolist()))
        else:
            sums.append(float(np.sum(t)))
            mags.append(float(np.sum(np.abs(t))))
    return np.array(sums), np.array(mags)


def _best_ratio(ad: np.ndarray, as_: np.ndarray) -> tuple[float, float, int]:
    """The frame with the largest ``ad / as`` as the kernels' tracker defines it: a frame replaces the record
    (initially 0 / 1) when ``ad * rs > rd * as``, decided on float64 products of float32 operands (exact), so ties keep
    the earliest frame.  Returns (|d|, |s|, frame index or -1)."""
    a = ad.astype(np.float64)
    b = as_.astype(np.float64)
    live = a > 0.0  # nothing else ever beats the initial record (a nan compares false)
    if not np.any(live):
        return 0.0, 1.0, -1
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(b > 0.0, a / b, np.inf)
    q = np.where(live, q, -1.0)
    qmax = np.nanmax(q)
    # float64 division rounds monotonically, so every frame of the largest exact ratio has q == qmax
    bd, bs, at = 0.0, 1.0, -1
    for i in np.flatnonzero(q == qmax):
        if a[i] * bs > bd * b[i]:
            bd, bs, at = float(a[i]), float(b[i]), int(i)
    return bd, bs, at


def objective_partials(y: np.ndarray) -> dict:
    """float64 reference of the 12 velvet-noise partials (``vn_objective_partials``) of a float32 stereo signal ``y``
    (frames, 2), e.g. ``vn_decorrelate(x, taps, ms_mode=..., width=..., normalizer=None)``.

    d = L - R and s = L + R are the float32 values the reference computes; theta is the float64 folded ``arctan2`` of
    them, and the radius the float64 root of the reference's float32 ``L*L + R*R`` (utils/dsp.py:413: each square and
    the sum rounded to float32, so its underflow and overflow are the reference's).  The six sums are correctly rounded
    (``math.fsum``); ``mag`` holds the sums of their terms' magnitudes, for tolerances.  Slots 6-9 are |d|, |s| of the
    largest-|d|/|s| frame with s >= 0 and with s < 0 (``_best_ratio``; 0 / 1 when there is none); ``at`` their frame
    indices."""
    y = np.asarray(y, dtype=np.float32)
    l, r = y[:, 0], y[:, 1]
    with np.errstate(over="ignore", invalid="ignore"):
        d, s = l - r, l + r
        th = _folded_theta(d.astype(np.float64), s.astype(np.float64))
        rad = np.sqrt((l * l + r * r).astype(np.float64))
        l64, r64 = l.astype(np.float64), r.astype(np.float64)
        terms = [rad, rad * th, rad * th * th, rad * th * th * th, l64 * r64, l64 * l64]
        sums, mag = _sums(terms)
    pos = s >= 0.0
    ad, as_ = np.abs(d), np.abs(s)
    dp, sp, ip = _best_ratio(np.where(pos, ad, 0.0), np.where(pos, as_, 1.0))
    neg = s < 0.0
    dn, sn, i_n = _best_ratio(np.where(neg, ad, 0.0), np.where(neg, as_, 1.0))
    p = np.zeros(12)
    p[:6] = sums
    p[6:10] = dp, sp, dn, sn
    p[10] = len(y)
    return {"p": p, "mag": mag, "at": (ip, i_n), "frames": len(y), "theta": th, "d": d, "s": s}


def haas_partials(y: np.ndarray) -> dict:
    """float64 reference of the 8 Haas partials (``haas_objective_partials``) of a float64 stereo signal ``y``
    (frames, 2), e.g. ``haas(x, ...)``: the sums of r, r*theta^n (n = 1..3), L*R and L*L correctly rounded, max|theta|,
    and the frame count.  d, s, theta and r are float64, as the kernel computes them; ``mag`` as in
    ``objective_partials``."""
    y = np.asarray(y, dtype=np.float64)
    l, r = y[:, 0], y[:, 1]
    th = _folded_theta(l - r, l + r)
    rad = np.sqrt(l * l + r * r)
    sums, mag = _sums([rad, rad * th, rad * th * th, rad * th * th * th, l * r, l * l])
    p = np.zeros(8)
    p[:4] = sums[:4]
    p[4] = float(np.max(np.abs(th))) if len(th) else 0.0
    p[5:7] = sums[4:]
    p[7] = len(y)
    return {"p": p, "mag": np.concatenate([mag[:4], [0.0], mag[4:]]), "frames": len(y), "theta": th}


def local_minima(scores: np.ndarray) -> list[int]:
    """Strict interior minima, else [argmin].  optimization.py:120-128."""
    g = len(scores)
    found = [i for i in range(1, g - 1) if scores[i] < scores[i - 1] and scores[i] < scores[i + 1]]
    return found if found else [int(np.argmin(scores))]


def vn_candidate_taps(kappa: float, *, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed: int):
    """Tap structure of the candidates ``optimize_velvet_noise`` builds; optimization.py:260-272."""
    return class_taps(
        sample_rate_hz=sample_rate_hz,
        duration_seconds=duration_seconds,
        num_impulses=num_impulses,
        num_outs=2,
        log_distribution_strength=kappa,
        filtered_channels=(0,),
        seed=seed,
    )


def vn_candidate_signal(x: np.ndarray, taps) -> np.ndarray:
    """Candidate output: LR mode, no normaliser, channel 0 filtered, channel 1 passed through."""
    return vn_decorrelate(x, taps, ms_mode=False, normalizer=None)


def vn_grid_scores(x: np.ndarray, kappas, *, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed: int = 1, **obj_kw):
    """``grid_scan`` over velvet-noise candidates; optimization.py:108-117, :258-282."""
    out = []
    for k in kappas:
        t = vn_candidate_taps(k, sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses, seed=seed)
        out.append(objective(vn_candidate_signal(x, t), **obj_kw))
    return np.array(out)


def haas_grid_scores(x: np.ndarray, taus, *, sample_rate_hz: int, **obj_kw):
    """``grid_scan`` over Haas candidates (float64); optimization.py:183-203."""
    return np.array([objective(haas(x, sample_rate_hz=sample_rate_hz, delay_time_seconds=t), **obj_kw) for t in taus])


def refine(minima: list[int], grid: np.ndarray, fn: Callable[[float], float]):
    """``optimize_local_minima``: bounded Brent (scipy) between the grid neighbours of each
    minimum, first strictly better result wins.  optimization.py:131-155."""
    from scipy.optimize import minimize_scalar

    best_x, best_f = 0.0, np.inf
    g = len(grid)
    for i in minima:
        res = minimize_scalar(fun=fn, bounds=(grid[max(0, i - 1)], grid[min(g - 1, i + 1)]), method="bounded", options={"xatol": 1e-4})
        if res.fun < best_f:
            best_f, best_x = res.fun, res.x
    return best_x


def optimize_vn(x: np.ndarray, *, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed: int = 1, grid_size: int = 400, **obj_kw):
    """``optimize_velvet_noise``; optimization.py:230-310.  Returns (kappa, scores, minima)."""
    kappas = np.linspace(0.0, 1.0, grid_size)
    kw = dict(sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses, seed=seed)
    scores = vn_grid_scores(x, kappas, **kw, **obj_kw)
    mins = local_minima(scores)
    best = refine(mins, kappas, lambda k: objective(vn_candidate_signal(x, vn_candidate_taps(k, **kw)), **obj_kw))
    return best, scores, mins


def optimize_haas(x: np.ndarray, *, sample_rate_hz: int, max_delay_seconds: float, grid_size: int = 400, **obj_kw):
    """``optimize_haas_delay``; optimization.py:158-227.  Returns (tau, scores, minima)."""
    taus = np.linspace(0.0, max_delay_seconds, grid_size)
    scores = haas_grid_scores(x, taus, sample_rate_hz=sample_rate_hz, **obj_kw)
    mins = local_minima(scores)
    best = refine(mins, taus, lambda t: objective(haas(x, sample_rate_hz=sample_rate_hz, delay_time_seconds=t), **obj_kw))
    return best, scores, mins


# --------------------------------------------------------------------------------------
# synthetic inputs named by the benchmark configs (SURVEY.md section 8d)
# --------------------------------------------------------------------------------------


def coloured_clip(index: int, frames: int) -> np.ndarray:
    """Config-5 clip: low-passed mid plus 0.3x low-passed side, peak 0.5, fp32 (frames, 2)."""
    from scipy.signal import lfilter

    rng = np.random.default_rng(1000 + index)
    m = lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    s = 0.3 * lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    x = np.column_stack((m + s, m - s))
    return (x / np.max(np.abs(x)) * 0.5).astype(np.float32)


def table_rows(taps) -> np.ndarray:
    """int32 rows (channel, segment, index, sign) in iteration order — the layout SURVEY.md
    Appendix C hashes."""
    rows = []
    for ch, segs in enumerate(taps):
        for si, (neg, pos) in enumerate(segs):
            rows += [(ch, si, int(i), -1) for i in neg]
            rows += [(ch, si, int(i), 1) for i in pos]
    return np.array(rows, dtype=np.int32).reshape(-1, 4)
