"""Every instance of the non-local-means filters against the f64 definition of include/rt_b200.h (an EXTENSION).

The colour-only, guided, cross and guided-cross filters are each compiled once per count of E locations per thread (NE,
chosen by the patch radius f).  Here every f in 0..7 runs against the restatement at search radii up to the largest, on
inputs whose far candidates keep weights of order 1, at the shapes where tiles and halos go wrong, plus the largest
height, the largest launch, the exact reductions, the glue at the bound and the edges of the accepted parameters.

CPU part: the full-image sweep below against the restatements of test_denoise.py, test_guided_denoise.py and
test_dual_denoise.py; the NE reached by the matrix; the sensitivity of every matrix case to a wrong search or patch
radius; the boundaries of the accepted parameters, restated in f32.  GPU part: the rest."""
import ctypes as C

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import test_denoise as TD
import test_dual_denoise as TDD
import test_guided_denoise as TG

FAMILIES = ("colour", "guided", "cross", "guided_cross")
PATCH_RADII = tuple(range(abi.RT_DENOISE_MAX_PATCH_RADIUS + 1))
SEARCH_RADII = (1, 2, 11, abi.RT_DENOISE_MAX_SEARCH_RADIUS)
SHAPES = ((1, 1), (1, 70), (70, 1), (15, 31), (16, 32), (17, 33), (48, 64))
PAIRS = ((abi.RT_DENOISE_DEFAULT_K, abi.RT_DENOISE_DEFAULT_ALPHA), (1.0, 0.0))  # (k, alpha)
GUIDE = dict(k_feature=0.6, tau=1e-3)
FLT_MIN = float(np.finfo(np.float32).tiny)


def locations_per_thread(f):
    """E locations per thread of the 32 x 16 tile and 256 threads (rt_denoise.cu)"""
    return ((32 + 2 * f) * (16 + 2 * f) + 255) // 256


# ------------------------------------------------------------------------------------------------------------- inputs
def live(H, W, seed):
    """smooth ramps under noise of high variance (1e-3.5 to 1e-2.5): far candidates keep weights of order 1, so a missing ring
    of offsets or a wrong patch radius moves the output"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    ramp = 0.4 + 0.15 * xx / max(W - 1, 1) + 0.1 * yy / max(H - 1, 1)
    v = 10.0 ** rng.uniform(-3.5, -2.5, (H, W, 3))
    mu = ramp[..., None] * np.array([1.0, 0.8, 0.6]) + rng.standard_normal((H, W, 3)) * np.sqrt(v)
    return mu.astype(np.float32), v.astype(np.float32)


def live_features(H, W, seed):
    """albedo and normal ramps with noise of variance 1e-4 to 1e-3 (some pixels exact): feature weights of order 1"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    ma = (0.5 + 0.1 * xx / max(W - 1, 1))[..., None] * np.array([1.0, 0.7, 0.4])
    mn = np.stack([0.3 + 0.1 * yy / max(H - 1, 1), np.full((H, W), 0.9), np.full((H, W), 0.3)], axis=-1)
    sa = 10.0 ** rng.uniform(-4, -3, (H, W, 3)) * (rng.random((H, W, 1)) > 0.1)
    sn = 10.0 ** rng.uniform(-4, -3, (H, W, 3)) * (rng.random((H, W, 1)) > 0.1)
    ma = ma + rng.standard_normal((H, W, 3)) * np.sqrt(sa)
    mn = mn + rng.standard_normal((H, W, 3)) * np.sqrt(sn)
    return tuple(a.astype(np.float32) for a in (ma, sa, mn, sn))


def inputs(family, kind, H, W):
    """(mu_a, v_a, mu_b, v_b, feats) of one case; mu_b, v_b only for the cross families, feats only for the guided ones"""
    seed = H * 1000 + W
    if kind == "live":
        a, b = live(H, W, seed), live(H, W, seed + 1)
        feats = live_features(H, W, seed + 2)
    else:  # zero variances and hard edges
        a, b = TD.synthetic(H, W, seed), TD.synthetic(H, W, seed + 1)
        feats = TG.synthetic_features(H, W, seed + 2)
    return (*a, *b, feats if "guided" in family else None)


# ---------------------------------------------------------------------------------------------------------- reference
def _box_mean(e, f):
    """the mean of e [n, H, W] over (2f + 1)^2 pixels, neighbours clamped: separable direct sums over the edge-padded image.
    (Running sums would cancel: zero-variance pixels give terms up to 1e22.)"""
    H, W = e.shape[1:]
    p = np.pad(e, ((0, 0), (f, f), (f, f)), mode="edge")
    h = p[:, :, 0:W].copy()
    for a in range(1, 2 * f + 1):
        h += p[:, :, a:a + W]
    s = h[:, 0:H].copy()
    for b in range(1, 2 * f + 1):
        s += h[:, b:b + H]
    return s / (2 * f + 1) ** 2


def sweep(mu_w, v_w, mu_val, rs, fs, k, alpha, feats=None, kf=1.0, tau=1e-2):
    """TDD.cross_ref for every (r, f) of rs x fs in one pass over the offsets (the weights from (mu_w, v_w) and the features,
    the values of mu_val; mu_val = mu_w is the colour-only or guided filter).  Returns {(r, f): out [H, W, 3]}, f64."""
    mu_w, v_w, mu_val = (np.asarray(a, np.float64) for a in (mu_w, v_w, mu_val))
    H, W, _ = mu_w.shape
    R = max(rs)
    yy, xx = np.mgrid[0:H, 0:W]
    dxs = np.arange(-R, R + 1)
    xs = np.clip(xx[None] + dxs[:, None, None], 0, W - 1)
    g2 = [TG.gradient2(feats[0]), TG.gradient2(feats[2])] if feats is not None else None
    wsum = {(r, f): np.ones((H, W)) for r in rs for f in fs}
    acc = {(r, f): mu_val.copy() for r in rs for f in fs}
    for dy in range(-R, R + 1):
        ys = np.broadcast_to(np.clip(yy + dy, 0, H - 1), xs.shape)
        e = TD.term_ref(mu_w[None], v_w[None], mu_w[ys, xs], v_w[ys, xs], k, alpha).sum(axis=-1)
        inside = ((yy + dy >= 0) & (yy + dy < H))[None] & (xx[None] + dxs[:, None, None] >= 0) & (xx[None] + dxs[:, None, None] < W)
        inside[dxs == 0] &= dy != 0  # d = 0 is the initial weight 1
        fw = None
        if feats is not None:
            for (m, s), g in zip(((feats[0], feats[1]), (feats[2], feats[3])), g2):
                wf = np.exp(-np.maximum(TG.distance_ref(m[None], s[None], g[None], m[ys, xs], s[ys, xs], kf, tau), 0.0))
                fw = wf if fw is None else np.minimum(fw, wf)
        vals = mu_val[ys, xs]
        ring = np.maximum(np.abs(dxs), abs(dy))
        for f in fs:
            w = np.exp(-np.maximum(_box_mean(e, f) / 3.0, 0.0))
            if fw is not None:
                w = np.minimum(w, fw)
            w = w * inside
            for r in rs:
                sel = ring <= r
                if sel.any():
                    wsum[(r, f)] += w[sel].sum(axis=0)
                    acc[(r, f)] += (w[sel][..., None] * vals[sel]).sum(axis=0)
    return {key: acc[key] / wsum[key][..., None] for key in acc}


def reference(family, case, rs, fs, k, alpha, kf=GUIDE["k_feature"], tau=GUIDE["tau"]):
    """{(r, f): out} of the colour-only and guided families; {(r, f): (F_A, F_B, out, eps)} of the cross families"""
    mu_a, v_a, mu_b, v_b, feats = case
    g = dict(feats=feats, kf=kf, tau=np.float32(tau))
    if "cross" not in family:
        return sweep(mu_a, v_a, mu_a, rs, fs, k, alpha, **g)
    fa, fb = sweep(mu_b, v_b, mu_a, rs, fs, k, alpha, **g), sweep(mu_a, v_a, mu_b, rs, fs, k, alpha, **g)
    return {key: (fa[key], fb[key], (fa[key] + fb[key]) / 2, TDD.box3_ref(((fa[key] - fb[key]) / 2) ** 2)) for key in fa}


def _rel(got, want):
    """the error measure of test_denoise.py: |got - want| / (|want| + 1e-3), its largest value"""
    return float((np.abs(got - want) / (np.abs(want) + 1e-3)).max())


# Largest error against the restatement, per family and input kind (colour-only and guided: _rel; cross: the larger of the
# two measures of TDD._check_against_ref), f32 kernels against the f64 restatement.  Each bound is four times the worst value
# measured on an NVIDIA B200 (1000 W power limit) over the matrix (test_matrix_against_restatement prints them): live
# 2.74e-6, 3.10e-6, 2.01e-6, 2.09e-6 and synthetic 5.22e-6, 7.62e-6, 2.46e-6, 5.95e-6 for colour, guided, cross and
# guided-cross.  The other GPU tests measured at most 2.2e-6 (parameter edges) and 1.3e-6 (the largest launch).
TOL = {"colour": {"live": 1.1e-5, "synthetic": 2.1e-5}, "guided": {"live": 1.25e-5, "synthetic": 3.05e-5},
       "cross": {"live": 8.1e-6, "synthetic": 9.9e-6}, "guided_cross": {"live": 8.4e-6, "synthetic": 2.4e-5}}
# how far (in units of the family's tolerance) a wrong search or patch radius must move each live case's output
SENSITIVITY = 50.0


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_sweep_matches_the_restatements():
    """the sweep equals TD.nlm_ref, TG.guided_ref, TDD.cross_ref and TDD.dual_ref, and the per-pixel restatements, to 1e-12"""
    H, W = 17, 33
    mu, v = live(H, W, 1)
    mu_b, v_b = live(H, W, 2)
    feats = live_features(H, W, 3)
    syn, syn_v = TD.synthetic(H, W, 4)
    sfeats = TG.synthetic_features(H, W, 5)
    pix = [(0, 0), (H - 1, W - 1), (8, 16), (0, W - 1), (16, 3)]
    idx = tuple(np.array(pix).T)
    close = lambda a, b: np.allclose(a, b, rtol=1e-12, atol=0)  # noqa: E731
    for m, vv, fe in ((mu, v, feats), (syn, syn_v, sfeats)):
        got = sweep(m, vv, m, (0, 3, 15), (0, 2, 7), 0.45, 1.0)
        got_g = sweep(m, vv, m, (3, 15), (2, 7), 0.45, 1.0, fe, 0.6, np.float32(1e-3))
        got_x = sweep(mu_b, v_b, m, (3, 15), (2, 7), 1.0, 0.0, fe, 0.6, np.float32(1e-3))
        for r, f in ((0, 0), (3, 2), (15, 7)):
            assert close(got[(r, f)], TD.nlm_ref(m, vv, r, f, 0.45, 1.0)), (r, f)
            assert close(got[(r, f)][idx], TD.nlm_ref_pixels(m, vv, pix, r, f, 0.45, 1.0)), (r, f)
        for r, f in ((3, 2), (15, 7)):
            assert close(got_g[(r, f)], TG.guided_ref(m, vv, fe, r, f, 0.45, 1.0, 0.6, np.float32(1e-3))), (r, f)
            assert close(got_g[(r, f)][idx], TG.guided_ref_pixels(m, vv, fe, pix, r, f, 0.45, 1.0, 0.6, np.float32(1e-3))), (r, f)
            assert close(got_x[(r, f)], TDD.cross_ref(mu_b, v_b, m, r, f, 1.0, 0.0, fe, 0.6, np.float32(1e-3))), (r, f)
            assert close(got_x[(r, f)][idx], TDD.cross_ref_pixels(mu_b, v_b, m, pix, r, f, 1.0, 0.0, fe, 0.6, np.float32(1e-3))), (r, f)
    case = (mu, v, mu_b, v_b, None)
    fa, fb, out, eps = reference("cross", case, (15,), (7,), 0.45, 1.0)[(15, 7)]
    want = TDD.dual_ref(mu, v, mu_b, v_b, 15, 7, 0.45, 1.0)
    for a, b in zip((fa, fb, out), want):
        assert close(a, b)
    # eps squares a difference of nearly equal values: compared as sqrt(eps) against the scale of F (_check_against_ref)
    assert np.abs(np.sqrt(eps) - np.sqrt(want[3])).max() <= 1e-12 * np.abs(fa).max()


def test_matrix_reaches_every_instance():
    """the patch radii of the matrix reach every NE instance (2 to 6) the filters are compiled for"""
    assert sorted({locations_per_thread(f) for f in PATCH_RADII}) == [2, 3, 4, 5, 6]
    assert [locations_per_thread(f) for f in PATCH_RADII] == [2, 3, 3, 4, 4, 5, 5, 6]
    assert max(SEARCH_RADII) == abi.RT_DENOISE_MAX_SEARCH_RADIUS and max(PATCH_RADII) == abi.RT_DENOISE_MAX_PATCH_RADIUS


def sensitivity(family, H, W, f, pair):
    """{(r, change): _rel(reference with the change, reference)} of one live matrix case, changes r - 1, f - 1 and f + 1"""
    case = inputs(family, "live", H, W)
    rs = sorted(set(SEARCH_RADII) | {r - 1 for r in SEARCH_RADII})
    fs = [x for x in (f - 1, f, f + 1) if x >= 0]
    ref = reference(family, case, rs, fs, *pair)
    out = (lambda x: x) if "cross" not in family else (lambda x: x[2])
    res = {}
    for r in SEARCH_RADII:
        want = out(ref[(r, f)])
        res[(r, "r-1")] = _rel(out(ref[(r - 1, f)]), want)
        for g in fs:
            if g != f:
                res[(r, f"f{g - f:+d}")] = _rel(out(ref[(r, g)]), want)
    return res


@pytest.mark.parametrize("family", FAMILIES)
def test_matrix_cases_see_a_wrong_radius(family):
    """for every live case of the matrix (but 1 x 1, whose output is its input), the restatement at (r - 1, f) and at (r, f +- 1)
    differs from that at (r, f) by at least SENSITIVITY times the family's tolerance: a kernel that skipped the outer ring
    of offsets or used a neighbouring patch radius (another NE instance) would fail the GPU matrix"""
    weakest = np.inf
    for H, W in SHAPES:
        if H * W == 1:
            continue
        for f in PATCH_RADII:
            for pair in PAIRS:
                for key, moved in sensitivity(family, H, W, f, pair).items():
                    weakest = min(weakest, moved)
                    assert moved >= SENSITIVITY * TOL[family]["live"], (family, H, W, f, pair, key, moved)
    print(f"{family}: the weakest wrong radius moves the output by {weakest:.3g} ({weakest / TOL[family]["live"]:.0f} tolerances)")


# ------------------------------------------------------------------------------------------------ the parameter bounds
def _f32_finite(x):
    with np.errstate(over="ignore"):
        return bool(np.isfinite(np.float32(x)))


def k_accepted(k):
    """check_denoise on k: > 0, and (float)(k * k) finite"""
    return k > 0 and _f32_finite(k * k)


def alpha_accepted(alpha):
    return alpha >= 0 and _f32_finite(alpha)


def guide_accepted(kf, tau):
    """check_guide: (float)(3 k_f^2), (float)tau and their f32 product at least FLT_MIN (the kernels flush subnormals to zero)"""
    if not (kf > 0 and 0 < tau < np.inf):
        return False
    with np.errstate(over="ignore", under="ignore"):
        kf2_3, t = np.float32(3.0 * kf * kf), np.float32(tau)
        return bool(kf2_3 >= FLT_MIN and t >= FLT_MIN and kf2_3 * t >= FLT_MIN)


def _bits(x):
    return int(np.float64(x).view(np.int64))


def _double(b):
    return float(np.int64(b).view(np.float64))


def boundary(accepted, lo, hi):
    """(last, first): neighbouring positive doubles between lo and hi with accepted(last) != accepted(first), by bisection
    over the bit patterns (ordered like the values); accepted(lo) != accepted(hi)"""
    a, b = _bits(lo), _bits(hi)
    assert accepted(lo) != accepted(hi)
    while b - a > 1:
        m = (a + b) // 2
        if accepted(_double(m)) == accepted(lo):
            a = m
        else:
            b = m
    return _double(a), _double(b)


def bounds():
    """{name: (last accepted, first rejected)}"""
    k_last, k_first = boundary(k_accepted, 1.0, 1e20)
    a_last, a_first = boundary(alpha_accepted, 1.0, 1e39)
    kf_first, kf_last = boundary(lambda kf: guide_accepted(kf, abi.RT_GUIDE_DEFAULT_TAU), 1e-25, 1.0)
    tau_first, tau_last = boundary(lambda t: guide_accepted(abi.RT_GUIDE_DEFAULT_K_FEATURE, t), 1e-45, 1.0)
    return {"k": (k_last, k_first), "alpha": (a_last, a_first), "k_feature": (kf_last, kf_first), "tau": (tau_last, tau_first)}


def test_parameter_bounds_are_where_f32_breaks():
    """the restated bounds: k^2 and alpha at most FLT_MAX after rounding, 3 k_f^2 tau and tau at least FLT_MIN"""
    b = bounds()
    fmax, mid = float(np.finfo(np.float32).max), 2.0 ** 128 - 2.0 ** 103  # (the f64 values from mid on round to +inf in f32)
    assert b["alpha"] == (np.nextafter(mid, 0.0), mid)
    assert b["k"][0] * b["k"][0] < mid <= b["k"][1] * b["k"][1] and b["k"][1] == np.nextafter(b["k"][0], np.inf)
    assert abs(b["k"][0] / np.sqrt(fmax) - 1) < 1e-7
    # with tau = 1e-2, 3 k_f^2 must reach FLT_MIN / (float)1e-2; with k_f = 1, tau must round to FLT_MIN or above
    assert abs(3 * b["k_feature"][0] ** 2 * np.float32(abi.RT_GUIDE_DEFAULT_TAU) / FLT_MIN - 1) < 1e-6
    assert b["tau"] == (FLT_MIN - 2.0 ** -150, np.nextafter(FLT_MIN - 2.0 ** -150, 0.0))
    assert guide_accepted(1e20, 1e-2) and guide_accepted(1e20, 1e300)  # 3 k_f^2 beyond f32: the feature is ignored


# ------------------------------------------------------------------------------------------------------------------ GPU
def run(family, case, **kw):
    """the device filter of the family: out, or (out, eps) for the cross families"""
    mu_a, v_a, mu_b, v_b, feats = case
    g = {k: kw.pop(k) for k in ("k_feature", "tau") if k in kw}
    if family == "colour":
        return TD._denoise_np(mu_a, v_a, **kw)
    if family == "guided":
        return TG._guided_np(mu_a, v_a, feats, **g, **kw)
    return TDD._cross_np(mu_a, v_a, mu_b, v_b, feats=feats, **g, **kw)


def error(family, got, want):
    """the family's error measure of a device result against the reference"""
    if "cross" not in family:
        return _rel(got, want)
    return max(TDD._check_against_ref(got[0], got[1], *want, None))


@pytest.mark.gpu
@pytest.mark.parametrize("f", PATCH_RADII)
@pytest.mark.parametrize("family", FAMILIES)
def test_matrix_against_restatement(family, f):
    """every shape, r in SEARCH_RADII and (k, alpha) in PAIRS on live inputs (the matrix), and on TD.synthetic (zero variances,
    hard edges), against the f64 restatement"""
    worst = {"live": 0.0, "synthetic": 0.0}
    for kind in ("live", "synthetic"):
        for H, W in SHAPES:
            case = inputs(family, kind, H, W)
            for k, alpha in PAIRS:
                ref = reference(family, case, SEARCH_RADII, (f,), k, alpha)
                for r in SEARCH_RADII:
                    got = run(family, case, search_radius=r, patch_radius=f, k=k, alpha=alpha, **GUIDE)
                    e = error(family, got, ref[(r, f)])
                    worst[kind] = max(worst[kind], e)
                    assert e < TOL[family][kind], (family, kind, H, W, r, f, k, alpha, e)
    print(f"{family} f={f} vs restatement: worst error live {worst['live']:.3g}, synthetic {worst['synthetic']:.3g}")


def _pixel_refs(family, case, pix, r, f, k, alpha, kf=GUIDE["k_feature"], tau=GUIDE["tau"]):
    """per-pixel restatement of out at pix, and for the cross families (out, eps, the scale of the eps measure)"""
    mu_a, v_a, mu_b, v_b, feats = case
    H, W, _ = mu_a.shape
    kw = (r, f, k, alpha, feats, kf, np.float32(tau))
    if "cross" not in family:
        return TDD.cross_ref_pixels(mu_a, v_a, mu_a, pix, *kw)
    nb = [(min(max(y + dy, 0), H - 1), min(max(x + dx, 0), W - 1)) for y, x in pix for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    fa = TDD.cross_ref_pixels(mu_b, v_b, mu_a, nb, *kw).reshape(len(pix), 9, 3)
    fb = TDD.cross_ref_pixels(mu_a, v_a, mu_b, nb, *kw).reshape(len(pix), 9, 3)
    return (fa[:, 4] + fb[:, 4]) / 2, (((fa - fb) / 2) ** 2).mean(axis=1), np.maximum(np.abs(fa), np.abs(fb)).max(axis=1) + 1e-3


def _pixel_error(family, got, pix, want):
    idx = tuple(np.array(pix).T)
    if "cross" not in family:
        return _rel(got[idx], want)
    out, eps, scale = want
    e_out = _rel(got[0][idx], out)
    e_err = float((np.abs(np.sqrt(got[1][idx].astype(np.float64)) - np.sqrt(eps)) / scale).max())
    return max(e_out, e_err)


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["colour", "cross"])
def test_largest_height(family):
    """W = 1, H = RT_DENOISE_MAX_HEIGHT (65 535 tile rows, the grid's limit), r = 15, f = 7: rows 0, 15, 16, 17, the last 17
    rows and random rows against the per-pixel restatement"""
    H, W = abi.RT_DENOISE_MAX_HEIGHT, 1
    case = (*live(H, W, 91), *live(H, W, 92), None)
    r, f = abi.RT_DENOISE_MAX_SEARCH_RADIUS, abi.RT_DENOISE_MAX_PATCH_RADIUS
    got = run(family, case, search_radius=r, patch_radius=f)
    rows = [0, 15, 16, 17] + list(range(H - 17, H)) + sorted(np.random.default_rng(93).integers(0, H, 20).tolist())
    pix = [(y, 0) for y in rows]
    e = _pixel_error(family, got, pix, _pixel_refs(family, case, pix, r, f, abi.RT_DENOISE_DEFAULT_K, abi.RT_DENOISE_DEFAULT_ALPHA))
    print(f"{family} {H}x{W} sampled rows: worst error {e:.3g}")
    assert e < TOL[family]["live"]


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["cross", "guided_cross"])
def test_largest_launch(family):
    """the cross kernel on 3840 x 2160 at r = 15, f = 7 (173 KB of shared memory): corners, tile seams and random pixels"""
    H, W = 2160, 3840
    case = inputs(family, "live", H, W)
    r, f = abi.RT_DENOISE_MAX_SEARCH_RADIUS, abi.RT_DENOISE_MAX_PATCH_RADIUS
    got = run(family, case, search_radius=r, patch_radius=f, **GUIDE)
    rng = np.random.default_rng(94)
    pix = [(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0), (15, 31), (16, 32), (15, 32), (16, 31), (H - 1, 32), (1087, 1919), (1088, 1920)]
    pix += list(zip(rng.integers(0, H, 20).tolist(), rng.integers(0, W, 20).tolist()))
    e = _pixel_error(family, got, pix, _pixel_refs(family, case, pix, r, f, abi.RT_DENOISE_DEFAULT_K, abi.RT_DENOISE_DEFAULT_ALPHA))
    print(f"{family} {W}x{H} r={r} f={f} sampled: worst error {e:.3g}")
    assert e < TOL[family]["live"]


@pytest.mark.gpu
@pytest.mark.parametrize("f", PATCH_RADII)
def test_exact_reductions_at_every_patch_radius(f):
    """r = 15: the cross filter with A = B is the colour-only (guided) filter bit for bit with eps = 0, and the guided filter with
    constant zero-variance features is the colour-only filter bit for bit"""
    H, W = 40, 70
    mu, v = live(H, W, 95)
    feats = live_features(H, W, 96)
    kw = dict(search_radius=abi.RT_DENOISE_MAX_SEARCH_RADIUS, patch_radius=f)
    bits = lambda x: x.view(np.uint32)  # noqa: E731
    colour = TD._denoise_np(mu, v, **kw)
    guided = TG._guided_np(mu, v, feats, **GUIDE, **kw)
    assert not np.array_equal(bits(colour), bits(guided))
    out, err = TDD._cross_np(mu, v, mu, v, **kw)
    assert np.array_equal(bits(out), bits(colour)) and not err.any()
    out, err = TDD._cross_np(mu, v, mu, v, feats=feats, **GUIDE, **kw)
    assert np.array_equal(bits(out), bits(guided)) and not err.any()
    zero = np.zeros_like(mu)
    const = (np.full_like(mu, 0.5), zero, np.broadcast_to(np.array([0, 1, 0], np.float32), mu.shape).copy(), zero)
    assert np.array_equal(bits(TG._guided_np(mu, v, const, **GUIDE, **kw)), bits(colour))


BOUND = dict(search_radius=abi.RT_DENOISE_MAX_SEARCH_RADIUS, patch_radius=abi.RT_DENOISE_MAX_PATCH_RADIUS)


@pytest.mark.gpu
def test_render_denoised_at_the_bound_is_the_chain():
    """rt_render_denoised at r = 15, f = 7: the moments, the numpy conversion and rt_denoise_device, bit for bit"""
    world, scene, cam = TD._setup("cornell_smoke")
    W, H, spp = 72, 56, 8
    rgb, den = TD._renderer(world, scene, cam, W, H, spp).render_denoised(**BOUND)
    mu, v = TD.mean_var_ref(*TD._moments(scene, cam, W, H, spp), spp)
    assert np.array_equal(den.view(np.uint32), TD._denoise_np(mu, v, **BOUND).view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


@pytest.mark.gpu
def test_render_denoised_dual_at_the_bound_is_the_chain():
    """rt_render_denoised_dual at r = 15, f = 7: the moments of the halves, the numpy conversion and rt_denoise_cross_device"""
    world, scene, cam = TD._setup("cornell_smoke")
    W, H, spp = 72, 56, 8
    rgb, den, err, n = TD._renderer(world, scene, cam, W, H, spp).render_denoised_dual(**BOUND)
    assert (n == spp).all()
    a = TD.mean_var_ref(*TDD._moments_range(scene, cam, W, H, 0, spp // 2), spp // 2)
    b = TD.mean_var_ref(*TDD._moments_range(scene, cam, W, H, spp // 2, spp // 2), spp // 2)
    want, want_err = TDD._cross_np(*a, *b, **BOUND)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32)) and np.array_equal(err.view(np.uint32), want_err.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


def _edge_cases():
    b = bounds()
    cases = [("colour", dict(k=k)) for k in (1e-6, 1e3, b["k"][0])] + [("colour", dict(alpha=a)) for a in (0.0, 1e3, b["alpha"][0])]
    cases += [("cross", dict(k=b["k"][0])), ("cross", dict(alpha=b["alpha"][0]))]
    for family in ("guided", "guided_cross"):
        # (each bound holds with the other guide parameter at its default)
        cases += [(family, dict(k_feature=kf, tau=abi.RT_GUIDE_DEFAULT_TAU)) for kf in (b["k_feature"][0], 1e20)]
        cases += [(family, dict(k_feature=abi.RT_GUIDE_DEFAULT_K_FEATURE, tau=b["tau"][0]))]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("family,param", _edge_cases(), ids=lambda x: x if isinstance(x, str) else ",".join(f"{k}={v:.9g}" for k, v in x.items()))
def test_parameter_edges_against_restatement(family, param):
    """the extreme accepted values follow the definition, on live and synthetic (zero-variance) inputs"""
    p = dict(k=abi.RT_DENOISE_DEFAULT_K, alpha=abi.RT_DENOISE_DEFAULT_ALPHA, **GUIDE)
    p.update(param)
    worst = 0.0
    for kind in ("live", "synthetic"):
        case = inputs(family, kind, 23, 37)
        for r, f in ((3, 1), (15, 7)):
            ref = reference(family, case, (r,), (f,), p["k"], p["alpha"], p["k_feature"], p["tau"])[(r, f)]
            got = run(family, case, search_radius=r, patch_radius=f, **p)
            e = error(family, got, ref)
            worst = max(worst, e)
            assert e < TOL[family][kind], (kind, r, f, e)
    print(f"{family} {param}: worst error {worst:.3g}")


@pytest.mark.gpu
def test_first_rejected_parameters():
    """the value next to each last accepted one is RT_ERR_INVALID with a message, from every filter entry point and a render"""
    import torch
    lib = abi.load()
    t = [torch.zeros(8, 8, 3, device="cuda") for _ in range(10)]
    ptr = [x.data_ptr() for x in t]
    b = bounds()
    fmax = float(np.finfo(np.float32).max)

    def calls(opt, guide):
        o, g = C.byref(rt.renderer.denoise_options_struct(**opt)), C.byref(rt.renderer.guide_struct(**guide))
        return [lib.rt_denoise_device(ptr[0], ptr[1], 8, 8, o, ptr[8], -1, None),
                lib.rt_denoise_guided_device(*ptr[:6], 8, 8, o, g, ptr[8], -1, None),
                lib.rt_denoise_cross_device(*ptr[:4], *(None,) * 4, 8, 8, o, None, ptr[8], ptr[9], -1, None),
                lib.rt_denoise_cross_device(*ptr[:8], 8, 8, o, g, ptr[8], ptr[9], -1, None)]

    assert calls({}, {}) == [abi.RT_OK] * 4
    assert calls(dict(k=b["k"][0], alpha=b["alpha"][0]), {}) == [abi.RT_OK] * 4
    assert calls({}, dict(k_feature=b["k_feature"][0]))[1::2] == [abi.RT_OK] * 2
    assert calls({}, dict(tau=b["tau"][0]))[1::2] == [abi.RT_OK] * 2
    assert calls({}, dict(k_feature=1e20, tau=1e300))[1::2] == [abi.RT_OK] * 2
    for opt in (dict(k=b["k"][1]), dict(k=float("inf")), dict(alpha=b["alpha"][1]), dict(alpha=fmax * 2), dict(alpha=float("inf"))):
        for rc in calls(opt, {}):
            assert rc == abi.RT_ERR_INVALID and b"finite in f32" in lib.rt_last_error(), opt
    for guide in (dict(k_feature=b["k_feature"][1]), dict(k_feature=1e-20), dict(tau=b["tau"][1]), dict(tau=1e-40),
                  dict(k_feature=1e-19, tau=1e-20)):
        for rc in calls({}, guide)[1::2]:
            assert rc == abi.RT_ERR_INVALID and b"FLT_MIN" in lib.rt_last_error(), guide
        assert calls({}, guide)[::2] == [abi.RT_OK] * 2  # (the colour-only entry points take no guide)
    world, scene, cam = TD._setup("cornell_smoke")
    p = TD._params(16, 16, 8)
    call = lambda opt, g=None: lib.rt_render_denoised_guided(scene.handle, C.byref(cam.c), C.byref(p), None,  # noqa: E731
                                                             C.byref(rt.renderer.denoise_options_struct(**opt)),
                                                             C.byref(rt.renderer.guide_struct(**(g or {}))), None, None, abi.RtProgressFn(),
                                                             None, None)
    assert call({}) == abi.RT_OK
    assert call(dict(k=b["k"][1])) == abi.RT_ERR_INVALID and b"rt_render_denoised_guided" in lib.rt_last_error()
    assert call({}, dict(tau=b["tau"][1])) == abi.RT_ERR_INVALID and b"FLT_MIN" in lib.rt_last_error()
    assert lib.rt_render_denoised_dual(scene.handle, C.byref(cam.c), C.byref(p), None, C.byref(rt.renderer.denoise_options_struct(alpha=b["alpha"][1])),
                                       None, None, None, None, None, abi.RtProgressFn(), None, None) == abi.RT_ERR_INVALID
    scene.close()
