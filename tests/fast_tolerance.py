"""
The tolerance contract of the two fast trace modes (csrc/trace_fast.cu, DESIGN.md section 8), in one place.

``compare`` holds a fast-mode result to the fp64 reference ray by ray: every value before a ray's first departure must
be within tolerance, and that first departure -- a value out of tolerance, or a NaN where the reference has a number or
the other way round -- must be explained by a knife-edge decision of the reference (``edge_margins``) at a surface
between the last compared slab that agreed and the departing slab.  After its first departure a ray is not compared
any more: a different root or an aperture decision on the other side of the edge makes every later value differ.

Tolerances (L = 1000 mm, the length scale of the traced systems):

    mode       positions       directions   phase
    f32        2e-6 * L        2e-6         2e-6 * max(|phi|, 1)
    f64_fast   1e-11 * L       1e-12        1e-12 * max(|phi|, 1)

The hard class (``HARD``: high-NA perfect-lens systems, where the fp32 direction error is amplified by 1/cos(theta),
and the deliberately extreme edge-mix rays) is 10x looser in f32 and 100x looser in f64_fast; in f32 only, long trains of large
spheres take a 10x looser phase (``PHASE_F32``, derivation there).  The wavelength column
must be bit-equal wherever both values are finite.

trace_fast.cu is compiled with FMA contraction, and in f32 with the approximate division and square root
(-prec-div=false -prec-sqrt=false, about 2 ulp of fp32).  Nothing below depends on how the fast mode rounds: the
margins are the reference's own quantities, recomputed in fp64, compared with the mode's tolerance, which is orders
of magnitude above any single rounding of either precision.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

L_MM = 1000.0
MODES = {"f32": (2e-6, 2e-6, 2e-6, 10.0), "f64_fast": (1e-11, 1e-12, 1e-12, 100.0)}

# systems whose rays the stated tolerances hold only in the hard class (trace_fast.cu header, DESIGN.md section 8)
HARD = frozenset({"opm", "opm_system", "edge_mix"})

# f32 only, phase only: long trains of large spheres.  The sphere's quadratic is fp64 but its root is taken in fp32
# (sqrt_t((T)disc), approximate square root): root = sqrt(b^2 - cq) <= |R| carries an absolute error of up to ~4 ulp,
# |R| 2^-22, and t = root - b inherits it.  Each sphere adds k n1 |R| 2^-22 to the phase -- 1.5e-3 rad for R = 400 mm,
# n1 = 1.5 at 0.59 um -- against 2e-6 of a phase of ~1e2 rad after the first surface (2e-4 rad).  Positions take the same
# 1e-4 mm, well inside 2e-3 mm, and the normal (p - c) / R only |R| 2^-22 / |R|: positions and directions keep the
# ordinary class.  The 70-surface train (66 spheres, radii 400-720 mm) is this class.
# The same holds for perfect lenses of long focal length: a lens takes two plane steps with t in fp32 (to_plane_f, to
# its front focal plane and from its back focal plane, |t| ~ n f up to ~180 mm), each adding k n |t| 2^-23 to the
# phase -- ~2.5e-4 rad at 0.59 um, against 2e-6 of a phase of ~1e2 rad just after a lens near the launch plane.  The
# random systems (lenses of f = 20..100 mm in media up to n = 1.8) are this class too, and so are the bundles launched
# on a perfect lens (f = 20 mm), whose phase just behind the lens is only ~1e2 rad.
PHASE_F32 = frozenset({"long_train", "random_system", "launched_on_plane"})
# margin names, in the order they are tested
REASONS = ("aperture", "sphere_graze", "root_choice", "behind_flat", "plane_graze", "front_side", "critical_angle",
           "lens_na", "on_surface_1e-12")

# a departure at slab 0 (the launch rays), a wavelength that changed, or one without a margin is never explained
KIND_FLAT, KIND_SPHERE, KIND_MIRROR, KIND_LENS = 0, 1, 2, 3


@dataclass(frozen=True)
class Tolerance:
    pos: float
    dir: float
    phase: float

    def scaled(self, k: float) -> "Tolerance":
        return Tolerance(self.pos * k, self.dir * k, self.phase * k)


def tolerance(mode: str, hard: bool = False) -> Tolerance:
    if mode not in MODES:
        raise ValueError(f"no tolerance for mode {mode!r}")
    p, d, ph, k = MODES[mode]
    t = Tolerance(p * L_MM, d, ph)
    return t.scaled(k) if hard else t


def is_hard(name: str) -> bool:
    return name in HARD


def class_tolerance(name: str, mode: str) -> Tolerance:
    """the tolerance of a named system family in one mode: HARD, PHASE_F32 (phase 10x in f32) or the ordinary class"""
    t = tolerance(mode, name in HARD)
    if mode == "f32" and name in PHASE_F32:
        t = Tolerance(t.pos, t.dir, t.phase * MODES["f32"][3])
    return t


# ----------------------------------------------------------------------------------------------------------
# the reference's per-surface decisions, restated in NumPy (rt_oracle.c, surface_steps.cuh)
# ----------------------------------------------------------------------------------------------------------
def _surface_rows(surfaces):
    from oracle import oracle
    return oracle.pack_surfaces(surfaces)


def _indices(materials, wl):
    """(n_media, N) refractive indices of the rays' wavelengths, evaluated by the materials' own n()"""
    out = np.empty((len(materials), wl.size))
    with np.errstate(all="ignore"):
        for j, m in enumerate(materials):
            out[j] = np.broadcast_to(np.asarray(m.n(wl), dtype=float).reshape(-1), wl.shape)
    return out


def _dot(a, b):
    return (a * b).sum(axis=1)


def edge_margins(incoming: np.ndarray, surface_row: np.ndarray, n1: np.ndarray, n2: np.ndarray, tol: Tolerance):
    """
    The reference's decisions at one surface for the rays ``incoming`` (M, 8), which are the reference's own rays in the
    slab before that surface.  Returns (reasons, margins): ``reasons`` is a list of M strings ('' = no decision of the
    reference lies within tolerance), ``margins`` a dict name -> (M,) distance of each ray from that decision's edge in
    the decision's own unit (mm, direction cosine or 1 - sin^2), NaN where it does not apply.
    """
    s = surface_row
    kind = int(s[0])
    c, nrm, axis = s[1:4], s[4:7], s[7:10]
    aperture = s[13]
    o, d = incoming[:, 0:3], incoming[:, 3:6]
    m = incoming.shape[0]
    nan = np.full(m, np.nan)
    margins = {r: nan.copy() for r in REASONS}
    with np.errstate(all="ignore"):
        if kind in (KIND_FLAT, KIND_MIRROR):
            den = _dot(d, np.broadcast_to(nrm, d.shape))
            t = -_dot(o - c, np.broadcast_to(nrm, o.shape)) / den
            p = o + d * t[:, None]
            pc = p - c
            margins["behind_flat"] = np.abs(t)
            margins["plane_graze"] = np.abs(den)                        # t = -num / den: ill-conditioned as den -> 0
            margins["aperture"] = np.abs(np.linalg.norm(pc, axis=1) - aperture)
            on_plane = np.abs(_dot(pc, np.broadcast_to(nrm, pc.shape))) < 1e-12
            normal = np.broadcast_to(nrm, d.shape)
            in_aperture = np.linalg.norm(pc, axis=1) <= aperture
            alive_geo = t >= 0
        elif kind == KIND_SPHERE:
            radius = s[10]
            oc = o - c
            b = _dot(d, oc)
            h = np.linalg.norm(oc - d * b[:, None], axis=1)             # distance of the ray's line from the centre
            margins["sphere_graze"] = np.abs(h - abs(radius))
            disc = b * b - (_dot(oc, oc) - s[11])
            root = np.sqrt(disc)
            t1, t2 = -b + root, -b - root
            margins["root_choice"] = np.minimum(np.abs(t1), np.abs(t2))
            t = np.where(t2 >= 0, t2, np.where(t1 >= 0, t1, np.nan))
            p = o + d * t[:, None]
            along = _dot(p, np.broadcast_to(axis, p.shape))
            r_ax = np.linalg.norm(p - along[:, None] * axis, axis=1)  # from the axis through the origin, as the reference
            margins["aperture"] = np.abs(r_ax - aperture)
            normal = (p - c) / radius
            on_plane = np.abs(np.linalg.norm(p - c, axis=1) - abs(radius)) < 1e-12
            in_aperture = r_ax <= aperture
            alive_geo = np.isfinite(t)
        elif kind == KIND_LENS:
            s1n = _dot(d, np.broadcast_to(nrm, d.shape))
            sin1 = np.linalg.norm(d - s1n[:, None] * nrm, axis=1)
            ffp = c - s[15:18] * n1[:, None]
            den = s1n
            t = -_dot(o - ffp, np.broadcast_to(nrm, o.shape)) / den
            r1 = o + d * t[:, None] - ffp
            sin2 = np.linalg.norm(r1, axis=1) / s[14] / n2
            sin_alpha = s[18]
            margins["lens_na"] = np.minimum(np.abs(sin1 - sin_alpha), np.abs(np.abs(sin2) - sin_alpha))
            reasons = ["lens_na" if v <= tol.dir else "" for v in margins["lens_na"]]
            return reasons, margins
        else:
            raise ValueError(f"surface kind {kind}")

        if kind != KIND_MIRROR:
            margins["front_side"] = np.abs(_dot(d, np.broadcast_to(axis, d.shape)))
            cos_n = _dot(normal, d)
            sin2 = np.maximum(_dot(d, d) - cos_n * cos_n, 0.0)
            mu = n1 / n2
            margins["critical_angle"] = np.abs(1.0 - mu * mu * sin2)
            front_ok = _dot(d, np.broadcast_to(axis, d.shape)) >= 0
            tir = 1.0 - mu * mu * sin2 < 0
        else:
            front_ok = np.ones(m, bool)
            tir = np.zeros(m, bool)
        # culled by the absolute 1e-12 on-surface test and by nothing else
        only_1e12 = alive_geo & front_ok & ~tir & in_aperture & ~on_plane
        margins["on_surface_1e-12"] = np.where(only_1e12, 0.0, np.nan)
    return _first_reasons(margins, tol, m), margins


def _limits(tol: Tolerance) -> dict:
    return {"aperture": tol.pos, "sphere_graze": tol.pos, "root_choice": tol.pos, "behind_flat": tol.pos,
            "plane_graze": tol.dir, "front_side": tol.dir, "critical_angle": 2 * tol.dir, "lens_na": tol.dir,
            "on_surface_1e-12": 0.0}


def _first_reasons(margins: dict, tol: Tolerance, m: int, allowed=None) -> list:
    """per ray, the first reason of REASONS whose margin is within its limit ('' = none); ``allowed`` (M,) sets of
    names restrict each ray to the decisions that can produce its kind of departure"""
    limits = _limits(tol)
    reasons = []
    for i in range(m):
        why = ""
        for r in REASONS:
            if allowed is not None and r not in allowed[i]:
                continue
            if margins[r][i] <= limits[r]:
                why = r
                break
        reasons.append(why)
    return reasons


# which decisions can produce which kind of first departure.  The aperture, the front-side cull, a lens's NA and the
# 1e-12 on-surface test only ever kill a ray, so they explain a NaN flip and nothing else.  A value out of tolerance
# on a ray both sides keep needs a decision that selects or conditions the value itself: the root (the other root,
# the sign of t at a flat) or an intersection / refraction whose derivative diverges at its edge -- a sphere met at
# grazing incidence (dt ~ d(disc) / 2 sqrt(disc)), a plane met at grazing incidence (t = -num / den, den -> 0) and the
# critical angle (dw = d(sin^2) / 2 w, w = cos of the refracted angle -> 0).  The on-surface test only explains a ray
# the reference killed at that surface's after-slab and the fast mode kept.
_VALUE = frozenset({"root_choice", "behind_flat", "sphere_graze", "plane_graze", "critical_angle"})
_FAST_KILLED = frozenset(REASONS) - {"on_surface_1e-12"}
_REF_KILLED = frozenset(REASONS)


# ----------------------------------------------------------------------------------------------------------
# the comparison
# ----------------------------------------------------------------------------------------------------------
@dataclass
class Report:
    mode: str
    hard: object
    n_rays: int
    max_multiple: dict = field(default_factory=dict)      # column group -> largest |error| / tolerance before departures
    explained: dict = field(default_factory=dict)         # ray -> (slab, surface, reason)
    unexplained: list = field(default_factory=list)       # (ray, slab, worst column, got row, want row)

    def counts(self) -> dict:
        out = {}
        for _, _, why in self.explained.values():
            out[why] = out.get(why, 0) + 1
        return out

    def summary(self, what: str = "") -> str:
        mult = ", ".join(f"{k} {v:.3g}x" for k, v in self.max_multiple.items())
        return (f"{what} [{self.mode}{'' if self.hard is False else ' hard' if self.hard is True else ' ' + str(self.hard)}] {self.n_rays} rays: max error {mult}; "
                f"explained {len(self.explained)} {self.counts()}; unexplained {len(self.unexplained)}")

    def unexplained_report(self, limit: int = 6) -> str:
        lines = [f"{len(self.unexplained)} unexplained departure(s)"]
        for ray, slab, col, g, w in self.unexplained[:limit]:
            lines.append(f"  ray {ray} slab {slab} column {col}:\n    got  {np.array2string(g, precision=17)}\n"
                         f"    want {np.array2string(w, precision=17)}")
        return "\n".join(lines)


_GROUPS = (("position", slice(0, 3)), ("direction", slice(3, 6)), ("phase", slice(6, 7)))


def _departures(g: np.ndarray, w: np.ndarray, tol: Tolerance):
    """(N,) bool: ray departs at this slab; (N,) worst column; dict group -> (N,) error multiple where both finite"""
    with np.errstate(all="ignore"):
        gn, wn = np.isnan(g), np.isnan(w)
        nan_flip = gn != wn
        same = (g == w) | (gn & wn)                           # equal infinities included
        err = np.where(same, 0.0, np.abs(g - w))
        err = np.where(np.isnan(err), np.inf, err)            # +-inf against a number
        lim = np.empty_like(w)
        lim[:, 0:3] = tol.pos
        lim[:, 3:6] = tol.dir
        lim[:, 6] = tol.phase * np.maximum(np.abs(np.nan_to_num(w[:, 6], nan=1.0, posinf=1.0, neginf=1.0)), 1.0)
        mult = err[:, 0:7] / lim[:, 0:7]
        wl_bad = ~gn[:, 7] & ~wn[:, 7] & (g[:, 7].view(np.uint64) != w[:, 7].view(np.uint64))
        bad = nan_flip[:, 0:7] | (mult > 1.0)
        col_score = np.where(nan_flip[:, 0:7], np.inf, mult)
        worst = np.argmax(col_score, axis=1)
        worst = np.where(wl_bad, 7, worst)
        dep = bad.any(axis=1) | nan_flip[:, 7] | wl_bad
        multiples = {name: np.where(nan_flip[:, sl], 0.0, mult[:, sl]).max(axis=1) for name, sl in _GROUPS}
    return dep, worst, wl_bad, multiples


def compare(got, want_history, slabs, mode: str, hard, surfaces, materials, strict: bool = True) -> Report:
    """
    got: (len(slabs), N, 8) fast-mode slabs; want_history: (2S+1, N, 8) reference history of the same launch rays;
    slabs: the history index of each slab of ``got`` (ascending).  materials = [initial] + system.materials + [final].
    hard: False / True for the ordinary / hard class, or a Tolerance (a named class, see ``class_tolerance``).
    Raises AssertionError on an unexplained departure (``strict``) and returns the Report.
    """
    got = np.asarray(got, dtype=np.float64)
    want_history = np.asarray(want_history, dtype=np.float64)
    slabs = [int(j) + (want_history.shape[0] if int(j) < 0 else 0) for j in slabs]
    if got.shape[0] != len(slabs) or got.shape[1:] != want_history.shape[1:]:
        raise ValueError(f"got {got.shape} does not match slabs {slabs} of a history {want_history.shape}")
    if list(slabs) != sorted(set(slabs)):
        raise ValueError("slabs must be ascending and distinct")
    if want_history.shape[0] != 2 * len(surfaces) + 1:
        raise ValueError("want_history must be the whole reference history")
    tol = hard if isinstance(hard, Tolerance) else tolerance(mode, hard)
    n = got.shape[1]
    rep = Report(mode, hard, n, {name: 0.0 for name, _ in _GROUPS})
    active = np.ones(n, bool)
    rows = _surface_rows(surfaces)
    prev = -1
    for q, j in enumerate(slabs):
        dep, worst, wl_bad, multiples = _departures(got[q], want_history[j], tol)
        ok = active & ~dep
        for name, _ in _GROUPS:
            if ok.any():
                rep.max_multiple[name] = max(rep.max_multiple[name], float(multiples[name][ok].max()))
        new = np.flatnonzero(active & dep)
        if new.size:
            # surfaces whose slabs (2k+1, 2k+2) lie in (prev, j]: the decisions between the last agreeing slab and j
            ks = [k for k in range(len(surfaces)) if 2 * k + 2 > prev and 2 * k + 1 <= j]
            why = np.array([""] * new.size, dtype=object)
            where = np.full(new.size, -1)
            cand = new[~wl_bad[new]] if j > 0 else new[:0]
            if cand.size:
                g_dead = np.isnan(got[q][cand, 0:7]).any(axis=1)
                w_dead = np.isnan(want_history[j][cand, 0:7]).any(axis=1)
                kinds = np.where(g_dead == w_dead, 0, np.where(w_dead, 2, 1))     # value / fast killed / ref killed
                for k in ks:
                    incoming = want_history[2 * k][cand]
                    idx = _indices(materials, incoming[:, 7])
                    _, margins = edge_margins(incoming, rows[k], idx[k], idx[k + 1], tol)
                    # the on-surface test decided it only if the reference had the ray at that surface and lost it there
                    ref_lost_here = (~np.isnan(want_history[2 * k + 1][cand, 0]) &
                                     np.isnan(want_history[2 * k + 2][cand, 0]))
                    allowed = [_VALUE if kd == 0 else _FAST_KILLED if kd == 1 else
                               (_REF_KILLED if lost else _FAST_KILLED) for kd, lost in zip(kinds, ref_lost_here)]
                    reasons = _first_reasons(margins, tol, cand.size, allowed)
                    pos = np.searchsorted(new, cand)
                    for p, r in zip(pos, reasons):
                        if r and not why[p]:
                            why[p], where[p] = r, k
            for p, i in enumerate(new):
                if why[p]:
                    rep.explained[int(i)] = (j, int(where[p]), why[p])
                else:
                    rep.unexplained.append((int(i), j, int(worst[i]), got[q][i], want_history[j][i]))
        active &= ~dep
        prev = j
    if strict and rep.unexplained:
        raise AssertionError(rep.summary() + "\n" + rep.unexplained_report())
    return rep


def assert_minority(rep: Report, limit: float = 0.01, what: str = ""):
    """explained (knife-edge) rays are a small minority of an ordinary bundle"""
    frac = len(rep.explained) / max(rep.n_rays, 1)
    assert frac <= limit, f"{what}: {frac:.3%} of rays explained by knife edges (limit {limit:.0%}): {rep.counts()}"
