"""SURE-based per-pixel selection among three strengths of the cross filter, with a bias-aware error estimate (an EXTENSION).

CPU part: the risk and the window selection of rt_denoise.cuh's host build against numpy restatements bit for bit; an f64
restatement of the whole definition of include/rt_b200.h, shown to be unbiased over many noise realisations and to reduce to
test_dual_denoise.cross_ref; the entry points and the CLI without a device.  GPU part: the kernels against the restatement,
the exact reductions, the selection on a synthetic image, the glue of rt_render_denoised_sure bit for bit (uniform, adaptive
through a Python replay of the rounds, the CLI), argument validation and measurement guards."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import mu_lambda_raytracer_b200 as rt
from mu_lambda_raytracer_b200 import abi
import support as S
import test_denoise as TD
import test_dual_denoise as TDD
import test_guided_denoise as TG

CLI = os.path.join(S.ROOT, "mu-lambda-raytracer_b200", "rt_main")


@pytest.fixture(scope="module")
def sure_emul(tmp_path_factory):
    """tests/emul/sure_emul.cpp: the SURE functions of rt_denoise.cuh built for the host"""
    path = str(tmp_path_factory.mktemp("sure_emul") / "libsure_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-w", "-ffp-contract=off", "-shared", "-o", path,
                           os.path.join(S.ROOT, "tests", "emul", "sure_emul.cpp")])
    L = C.CDLL(path)
    L.emul_sure_risk.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_void_p]
    L.emul_sure_out_risk.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.emul_sure_select.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3
    return L


# ------------------------------------------------------------------------------------------------- f32 restatements
def strengths(ratio):
    """s = (1, ratio^2, ratio^-2), computed in f64 and each rounded once to f32"""
    q = float(ratio) * float(ratio)
    return [np.float32(1.0), np.float32(q), np.float32(1.0 / q)]


def risk_ref(f, mu, v, w):
    """R = (f - mu)^2 + v (2 / w - 1), one f32 rounding per operation"""
    f, mu, v, w = (np.asarray(a, np.float32) for a in (f, mu, v, w))
    d = f - mu
    return (d * d + v * (np.float32(2.0) / w - np.float32(1.0))).astype(np.float32)


def out_risk_ref(ra, rb):
    return ((np.asarray(ra, np.float32) + np.asarray(rb, np.float32)) * np.float32(0.5)).astype(np.float32)


def select_ref(risk, fa, fb, b):
    """the selection in f32, one rounding per operation: risk [H, W, 9] (candidate-major), fa and fb [3, H, W, 3] -> out, err,
    choice"""
    H, W = risk.shape[:2]
    S_, E = np.zeros((3, H, W), np.float32), np.zeros((3, H, W, 3), np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    for dy in range(-b, b + 1):
        for dx in range(-b, b + 1):
            s = risk[np.clip(yy + dy, 0, H - 1), np.clip(xx + dx, 0, W - 1)].reshape(H, W, 3, 3)
            for j in range(3):
                S_[j] = S_[j] + ((s[..., j, 0] + s[..., j, 1]) + s[..., j, 2])
                E[j] = E[j] + s[..., j, :]
    n = np.float32((2 * b + 1) ** 2)
    S_, E = S_ / n, E / n
    choice = np.zeros((H, W), np.int32)
    best = S_[0].copy()
    for j in (1, 2):
        better = S_[j] < best
        choice[better], best[better] = j, S_[j][better]
    e = np.take_along_axis(E, choice[None, ..., None], axis=0)[0]
    err = np.where(e > 0, e, np.float32(0.0)).astype(np.float32)
    idx = choice[None, ..., None]
    out = TDD.dual_out_ref(np.take_along_axis(fa, idx, axis=0)[0], np.take_along_axis(fb, idx, axis=0)[0])
    return out, err, choice


# ------------------------------------------------------------------------------------------------- f64 restatement
def box_ref(x, b):
    """the mean over the (2b + 1)^2 window, neighbours clamped (f64, window over axes -2, -1)"""
    from numpy.lib.stride_tricks import sliding_window_view
    pad = [(0, 0)] * (x.ndim - 2) + [(b, b), (b, b)]
    return sliding_window_view(np.pad(x, pad, mode="edge"), (2 * b + 1, 2 * b + 1), axis=(-2, -1)).mean(axis=(-2, -1))


def sure_cross_ref(mu_w, v_w, mu_val, r, f, k, alpha, ss, feats=None, kf=1.0, tau=1e-2):
    """the candidates of strengths ss in f64: weights from (mu_w, v_w) (and the features), values of mu_val, arrays
    [..., H, W, 3].  Returns lists (F_j [..., H, W, 3], W_j [..., H, W])."""
    from numpy.lib.stride_tricks import sliding_window_view
    mu_w, v_w, mu_val = (np.asarray(a, np.float64) for a in (mu_w, v_w, mu_val))
    H, W = mu_w.shape[-3:-1]
    yy, xx = np.mgrid[0:H, 0:W]
    wsum, acc = [np.ones(mu_w.shape[:-1]) for _ in ss], [mu_val.copy() for _ in ss]
    g2 = [TG.gradient2(feats[0]), TG.gradient2(feats[2])] if feats is not None else None
    pad = [(0, 0)] * (mu_w.ndim - 3) + [(f, f), (f, f)]
    for dy in range(-r, r + 1):
        for dx in range(-r, r + 1):
            if dx == 0 and dy == 0:
                continue
            ys, xs = np.clip(yy + dy, 0, H - 1), np.clip(xx + dx, 0, W - 1)
            e = TD.term_ref(mu_w, v_w, mu_w[..., ys, xs, :], v_w[..., ys, xs, :], k, alpha).sum(axis=-1)
            D = sliding_window_view(np.pad(e, pad, mode="edge"), (2 * f + 1, 2 * f + 1), axis=(-2, -1)).mean(axis=(-2, -1)) / 3.0
            x = np.maximum(D, 0.0)
            wf = None
            if feats is not None:
                wf = np.ones((H, W))
                for (m, s), g in zip(((feats[0], feats[1]), (feats[2], feats[3])), g2):
                    wf = np.minimum(wf, np.exp(-np.maximum(TG.distance_ref(m, s, g, m[ys, xs], s[ys, xs], kf, tau), 0.0)))
            inside = (yy + dy >= 0) & (yy + dy < H) & (xx + dx >= 0) & (xx + dx < W)
            vals = mu_val[..., ys, xs, :]
            for j, s_j in enumerate(ss):
                w = np.exp(-float(s_j) * x)
                if wf is not None:
                    w = np.minimum(w, wf)
                w = w * inside
                wsum[j] = wsum[j] + w
                acc[j] = acc[j] + w[..., None] * vals
    return [a / ws[..., None] for a, ws in zip(acc, wsum)], wsum


def risk64(F, mu, v, Wsum):
    """R of one half in f64"""
    return (F - mu) ** 2 + np.asarray(v, np.float64) * (2.0 / Wsum[..., None] - 1.0)


def sure_ref(mu_a, v_a, mu_b, v_b, r, f, k, alpha, ratio, b, feats=None, kf=1.0, tau=1e-2):
    """the definition in f64 (images [H, W, 3]): F_A, F_B [3, H, W, 3], W_A, W_B [3, H, W], s_hat [3, H, W, 3], S [3, H, W],
    the choice, and out and err of every candidate [3, H, W, 3]"""
    ss = strengths(ratio)
    mu_a, v_a, mu_b, v_b = (np.asarray(a, np.float64) for a in (mu_a, v_a, mu_b, v_b))
    fa, wa = sure_cross_ref(mu_b, v_b, mu_a, r, f, k, alpha, ss, feats, kf, tau)
    fb, wb = sure_cross_ref(mu_a, v_a, mu_b, r, f, k, alpha, ss, feats, kf, tau)
    fa, fb, wa, wb = np.array(fa), np.array(fb), np.array(wa), np.array(wb)
    s_hat = (risk64(fa, mu_a, v_a, wa) + risk64(fb, mu_b, v_b, wb)) / 2
    S_ = box_ref(s_hat.sum(axis=-1), b)
    err = np.maximum(np.moveaxis(box_ref(np.moveaxis(s_hat, -1, -3), b), -3, -1), 0.0)
    return dict(fa=fa, fb=fb, wa=wa, wb=wb, s_hat=s_hat, S=S_, choice=np.argmin(S_, axis=0), out=(fa + fb) / 2, err=err)


def sure_cross_ref_pixels(mu_w, v_w, mu_val, pixels, r, f, k, alpha, ss, feats=None, kf=1.0, tau=1e-2):
    """sure_cross_ref for a list of pixels (y, x) only: F [n, 3 candidates, 3], W [n, 3 candidates]"""
    mu_w, v_w, mu_val = (np.asarray(a, np.float64) for a in (mu_w, v_w, mu_val))
    H, W, _ = mu_w.shape
    d = np.arange(-r, r + 1)
    dy, dx = [a.ravel() for a in np.meshgrid(d, d, indexing="ij")]
    o = np.arange(-f, f + 1)
    oy, ox = [a.ravel() for a in np.meshgrid(o, o, indexing="ij")]
    F, Ws = [], []
    for py, px in pixels:
        xy, xx = np.clip(py + oy, 0, H - 1), np.clip(px + ox, 0, W - 1)
        yy, yx = np.clip(xy[None, :] + dy[:, None], 0, H - 1), np.clip(xx[None, :] + dx[:, None], 0, W - 1)
        e = TD.term_ref(mu_w[xy, xx][None], v_w[xy, xx][None], mu_w[yy, yx], v_w[yy, yx], k, alpha).sum(axis=2)
        x = np.maximum(e.mean(axis=1) / 3.0, 0.0)
        inside = (py + dy >= 0) & (py + dy < H) & (px + dx >= 0) & (px + dx < W)
        qy, qx = np.clip(py + dy, 0, H - 1), np.clip(px + dx, 0, W - 1)
        wf = np.ones_like(x)
        if feats is not None:
            for m, s in ((feats[0], feats[1]), (feats[2], feats[3])):
                mm = m.astype(np.float64)
                gx = (mm[py, min(px + 1, W - 1)] - mm[py, max(px - 1, 0)]) / 2
                gy = (mm[min(py + 1, H - 1), px] - mm[max(py - 1, 0), px]) / 2
                wf = np.minimum(wf, np.exp(-np.maximum(TG.distance_ref(m[py, px], s[py, px], gx * gx + gy * gy, m[qy, qx], s[qy, qx], kf, tau), 0.0)))
        fj, wj = [], []
        for s_j in ss:
            w = np.minimum(np.exp(-float(s_j) * x), wf)
            w[(dy == 0) & (dx == 0)] = 1.0
            w = w[inside]
            fj.append((w[:, None] * mu_val[qy[inside], qx[inside]]).sum(axis=0) / w.sum())
            wj.append(w.sum())
        F.append(fj)
        Ws.append(wj)
    return np.array(F), np.array(Ws)


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_risk_matches_numpy_bit_for_bit(sure_emul):
    rng = np.random.default_rng(91)
    N = 300_000
    mu = (rng.choice([0.0, 1e-6, 0.02, 0.5, 3.0], N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)
    f = np.where(rng.random(N) < 0.2, mu, mu * (1 + rng.choice([1e-7, 1e-3, 0.3], N) * rng.standard_normal(N))).astype(np.float32)
    v = (rng.choice([0.0, 1e-10, 1e-6, 1e-3, 1.0], N) * rng.uniform(0.5, 1.5, N)).astype(np.float32)
    w = np.where(rng.random(N) < 0.2, 1.0, 1.0 + 10.0 ** rng.uniform(-7, 3, N)).astype(np.float32)
    got = np.zeros(N, np.float32)
    sure_emul.emul_sure_risk(f.ctypes.data, mu.ctypes.data, v.ctypes.data, w.ctypes.data, N, got.ctypes.data)
    assert np.array_equal(got.view(np.uint32), risk_ref(f, mu, v, w).view(np.uint32))
    # W = 1 and f = mu give v exactly; W > 2 with f = mu gives a negative risk
    one = w == 1.0
    sure_emul.emul_sure_risk(mu.ctypes.data, mu.ctypes.data, v.ctypes.data, w.ctypes.data, N, got.ctypes.data)
    assert np.array_equal(got[one].view(np.uint32), v[one].view(np.uint32))
    assert (got[(w > 2) & (v > 0)] < 0).all()
    rb = risk_ref(mu, f, v, w)
    s = np.zeros(N, np.float32)
    sure_emul.emul_sure_out_risk(got.ctypes.data, rb.ctypes.data, N, s.ctypes.data)
    assert np.array_equal(s.view(np.uint32), out_risk_ref(got, rb).view(np.uint32))


def _select_case(H, W, seed, ties):
    rng = np.random.default_rng(seed)
    risk = (rng.choice([1e-6, 1e-3, 0.1], (H, W, 1)) * rng.standard_normal((H, W, 9)) + rng.choice([0.0, 1e-3], (H, W, 1))).astype(np.float32)
    if ties:  # candidates equal pixel by pixel: ties to the smaller j, at every pair
        r3 = risk.reshape(H, W, 3, 3)
        pick = rng.integers(0, 4, (H, W))
        r3[pick == 1, 1] = r3[pick == 1, 0]
        r3[pick == 2, 2] = r3[pick == 2, 1]
        r3[pick == 3, 1:] = r3[pick == 3, 0][:, None]
    fa = rng.uniform(0, 2, (3, H, W, 3)).astype(np.float32)
    fb = (fa * rng.uniform(0.9, 1.1, fa.shape)).astype(np.float32)
    return np.ascontiguousarray(risk), fa, fb


@pytest.mark.parametrize("b", list(range(abi.RT_SURE_MAX_SMOOTH_RADIUS + 1)))
def test_selection_matches_numpy_bit_for_bit(sure_emul, b):
    for H, W, seed, ties in ((1, 1, 1, False), (7, 5, 2, False), (23, 37, 3, False), (16, 20, 4, True)):
        risk, fa, fb = _select_case(H, W, seed + 10 * b, ties)
        out, err, choice = np.zeros((H, W, 3), np.float32), np.zeros((H, W, 3), np.float32), np.zeros((H, W), np.int32)
        sure_emul.emul_sure_select(risk.ctypes.data, fa.ctypes.data, fb.ctypes.data, W, H, b, out.ctypes.data, err.ctypes.data, choice.ctypes.data)
        o, e, c = select_ref(risk, fa, fb, b)
        assert np.array_equal(choice, c), (H, W, b)
        assert np.array_equal(out.view(np.uint32), o.view(np.uint32)) and np.array_equal(err.view(np.uint32), e.view(np.uint32)), (H, W, b)
        assert (err >= 0).all()
        if (H, W) == (23, 37):
            assert len(np.unique(choice)) == 3 and (e == 0).any()  # (some window means are negative and clamped)
    # all three candidates equal: choice 0 everywhere
    risk, fa, fb = _select_case(9, 11, 5, False)
    risk.reshape(9, 11, 3, 3)[:, :, 1:] = risk.reshape(9, 11, 3, 3)[:, :, :1]
    _, _, c = select_ref(risk, fa, fb, b)
    assert not c.any()


def _halves_from_samples(t, n, N, rng, kind):
    """N independent realisations of two halves of n samples each around the truth t [H, W, 3]: (mu, v) per half, v the
    unbiased variance of the mean estimated from the samples"""
    shape = (N, n) + t.shape
    if kind == "gaussian":
        x = t + 0.15 * np.sqrt(t + 0.05) * rng.standard_normal(shape)
    else:  # skewed: exponential with mean t
        x = t * rng.exponential(1.0, shape)
    return x.mean(axis=1), x.var(axis=1, ddof=1) / n


def _truth(H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    return (np.where(xx < W // 2, 0.2, 0.8)[..., None] * np.array([1.0, 0.6, 0.3]) + 0.03 * yy[..., None] / H + 0.1 * ((xx + 2 * yy) % 5 == 0)[..., None])


@pytest.mark.parametrize("kind", ["gaussian", "exponential"])
def test_definition_is_unbiased(kind):
    """Over many noise realisations: the mean of R_A,j matches the mean of (F_A,j - t)^2 within 4 standard errors (frame sums
    per realisation, paired), and the mean of s_hat_j lies between the mean of (out_j - t)^2 and twice it"""
    rng = np.random.default_rng(101 if kind == "gaussian" else 102)
    H, W, n, N = 10, 12, 4, 3000
    t = _truth(H, W)
    mu_a, v_a = _halves_from_samples(t, n, N, rng, kind)
    mu_b, v_b = _halves_from_samples(t, n, N, rng, kind)
    ss = strengths(2.0)
    fa, wa = sure_cross_ref(mu_b, v_b, mu_a, 2, 1, 0.45, 1.0, ss)
    fb, wb = sure_cross_ref(mu_a, v_a, mu_b, 2, 1, 0.45, 1.0, ss)
    for j in range(3):
        ra, rb = risk64(fa[j], mu_a, v_a, wa[j]), risk64(fb[j], mu_b, v_b, wb[j])
        d = (ra - (fa[j] - t) ** 2).sum(axis=(1, 2, 3))
        z = d.mean() / (d.std(ddof=1) / np.sqrt(N))
        assert abs(z) < 4.0, (kind, j, z)
        assert (np.abs(fa[j] - t) ** 2).mean() > 1.5 * ((fa[j] - fa[j].mean(axis=0)) ** 2).mean() or j != 2  # (j = 2 carries a bias)
        s_hat = ((ra + rb) / 2).mean()
        e_out = (((fa[j] + fb[j]) / 2 - t) ** 2).mean()
        print(f"{kind} j={j}: z {z:.2f}, mean s_hat / mean (out - t)^2 {s_hat / e_out:.3f}")
        assert e_out < s_hat < 2 * e_out, (kind, j, s_hat, e_out)


def test_restatement_reduces_to_the_cross_filter():
    H, W = 14, 17
    mu_a, v_a, mu_b, v_b = TDD.synthetic_halves(H, W, 111)
    feats = TG.synthetic_features(H, W, 112)
    for r, f, fe in ((3, 1, None), (2, 0, feats), (4, 2, feats)):
        want = TDD.cross_ref(mu_b, v_b, mu_a, r, f, 0.45, 1.0, fe, 0.6, np.float32(1e-3))
        got, _ = sure_cross_ref(mu_b, v_b, mu_a, r, f, 0.45, 1.0, [1.0], fe, 0.6, np.float32(1e-3))
        assert np.abs(got[0] - want).max() <= 1e-12 * (np.abs(want).max() + 1), (r, f)
    # r = 0: every W = 1 and F = mu
    ref = sure_ref(mu_a, v_a, mu_b, v_b, 0, 2, 0.45, 1.0, 2.0, 1)
    assert (ref["wa"] == 1).all() and np.array_equal(ref["out"][1], (mu_a.astype(np.float64) + mu_b) / 2)
    # the pixel restatement is the image restatement
    pix = [(0, 0), (H - 1, W - 1), (5, 8), (13, 0)]
    F, Wp = sure_cross_ref_pixels(mu_b, v_b, mu_a, pix, 3, 1, 0.45, 1.0, strengths(2.0), feats, 0.6, np.float32(1e-3))
    Fi, Wi = sure_cross_ref(mu_b, v_b, mu_a, 3, 1, 0.45, 1.0, strengths(2.0), feats, 0.6, np.float32(1e-3))
    for i, (y, x) in enumerate(pix):
        for j in range(3):
            assert np.allclose(F[i, j], Fi[j][y, x], rtol=1e-12, atol=1e-14) and np.isclose(Wp[i, j], Wi[j][y, x], rtol=1e-12)


def test_rt_sure_struct_matches_header():
    assert C.sizeof(abi.RtSure) == 16
    hdr = open(os.path.join(S.ROOT, "include", "rt_b200.h")).read()
    for name in ("RT_SURE_DEFAULT_RATIO", "RT_SURE_DEFAULT_SMOOTH_RADIUS", "RT_SURE_MAX_SMOOTH_RADIUS"):
        line = next(x for x in hdr.split("\n") if x.startswith(f"#define {name} "))
        assert float(line.split()[2]) == getattr(abi, name), name


def test_sure_entry_points_without_a_device():
    lib = abi.load()
    if lib.rt_device_count() > 0:
        pytest.skip("a CUDA device is present")
    p, opt, sure = abi.RtParams(), rt.renderer.denoise_options_struct(), rt.renderer.sure_struct()
    assert lib.rt_denoise_sure_device(*[None] * 8, 0, 0, C.byref(opt), None, C.byref(sure), None, None, None, -1, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_denoised_sure(None, None, C.byref(p), None, C.byref(opt), None, C.byref(sure), None, None, None, None, None,
                                       abi.RtProgressFn(), None, None) == abi.RT_ERR_NO_DEVICE
    assert lib.rt_render_denoised_sure(None, None, C.byref(p), None, C.byref(opt), None, None, None, None, None, None, None,
                                       abi.RtProgressFn(), None, None) == abi.RT_ERR_NO_DEVICE
    assert b"no CPU path" in lib.rt_last_error()


@pytest.mark.parametrize("extra", [["--gpus=2"], ["--samples_per_pixel=31"], ["--min_samples=7", "--noise_threshold=0.02"],
                                   ["--denoise_guided", "--samples_per_pixel=9"]])
def test_cli_rejects_denoise_sure_arguments(extra):
    r = subprocess.run([CLI, "--world=cornell_smoke", "--denoise_sure", *extra], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1 and "--denoise_sure" in r.stderr and r.stdout == ""


def test_cli_usage_lists_denoise_sure():
    r = subprocess.run([CLI, "--help"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 0 and "--denoise_sure" in r.stdout


# ------------------------------------------------------------------------------------------------------------------ GPU
def _sure_np(mu_a, v_a, mu_b, v_b, feats=None, **kw):
    import torch
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    out, err, choice = rt.denoise_sure(t(mu_a), t(v_a), t(mu_b), t(v_b), features=None if feats is None else [t(x) for x in feats], **kw)
    torch.cuda.synchronize()
    return out.cpu().numpy(), err.cpu().numpy(), choice.cpu().numpy()


def _risk_scale(F, mu, v):
    """the size of the f32 error of R per unit of relative error of F: |d| (|F| + |mu| + 1e-3) 2 + 2 v"""
    return 2 * np.abs(F - mu) * (np.abs(F) + np.abs(mu) + 1e-3) + 2 * np.asarray(v, np.float64)


def _check_sure(got, ref, mu_a, v_a, mu_b, v_b, b, tol):
    """(worst out, worst err, share of pixels whose choice is decided, worst decided mismatch).  out and err are compared at the
    device's choice; the choice wherever the restated gap between the best and the second S exceeds tol times the scale of S."""
    out, err, choice = got
    scale = (_risk_scale(ref["fa"], mu_a, v_a) + _risk_scale(ref["fb"], mu_b, v_b)) / 2  # [3, H, W, 3]
    scale_S = box_ref(scale.sum(axis=-1), b).max(axis=0) + 1e-30
    S_sorted = np.sort(ref["S"], axis=0)
    decided = (S_sorted[1] - S_sorted[0]) > tol * scale_S
    mismatch = int((decided & (choice != ref["choice"])).sum())
    idx = choice[None, ..., None]
    want_out = np.take_along_axis(ref["out"], idx, axis=0)[0]
    want_err = np.take_along_axis(ref["err"], idx, axis=0)[0]
    scale_err = np.take_along_axis(np.moveaxis(box_ref(np.moveaxis(scale, -1, -3), b), -3, -1), idx, axis=0)[0] + 1e-30
    e_out = float((np.abs(out - want_out) / (np.abs(want_out) + 1e-3)).max())
    e_err = float((np.abs(err - want_err) / scale_err).max())
    return e_out, e_err, float(decided.mean()), mismatch


# out: |device - restatement| / (|restatement| + 1e-3) at the device's choice, as DUAL_REL_TOL of test_dual_denoise; err and the
# choice gap: relative to the propagated scale of the f32 error of R (_risk_scale).  The candidate filters run the arithmetic of
# the cross filter (worst measured error 2.5e-6 in test_denoise_instances.py).
SURE_REL_TOL = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(1, 1), (3, 5), (23, 37), (48, 64)])
def test_sure_matches_numpy_restatement(H, W):
    mu_a, v_a, mu_b, v_b = TDD.synthetic_halves(H, W, H * 1000 + W + 5)
    feats = TG.synthetic_features(H, W, H * 7 + W + 5)
    worst = [0.0, 0.0, 1.0]
    for (r, f), b in zip(((0, 0), (1, 1), (3, 0), (10, 3), (15, 7)), (0, 1, 2, abi.RT_SURE_DEFAULT_SMOOTH_RADIUS, 7)):
        for guided in (False, True):
            kw = dict(search_radius=r, patch_radius=f, k=0.45, alpha=1.0, smooth_radius=b)
            g = dict(feats=feats, k_feature=0.6, tau=1e-3) if guided else {}
            got = _sure_np(mu_a, v_a, mu_b, v_b, **g, **kw)
            ref = sure_ref(mu_a, v_a, mu_b, v_b, r, f, 0.45, 1.0, abi.RT_SURE_DEFAULT_RATIO, b, feats if guided else None, 0.6, np.float32(1e-3))
            e_out, e_err, decided, mismatch = _check_sure(got, ref, mu_a, v_a, mu_b, v_b, b, SURE_REL_TOL)
            worst = [max(worst[0], e_out), max(worst[1], e_err), min(worst[2], decided)]
            assert e_out < SURE_REL_TOL and e_err < SURE_REL_TOL and mismatch == 0, (r, f, b, guided, e_out, e_err, mismatch)
            if r > 0 and H * W > 100:  # (measured: at least 0.875 decided, at r = 15 on 23 x 37 where windows span the image)
                assert decided > 0.75 and (b > 2 or len(np.unique(got[2])) >= 2), (r, f, guided, decided)
    print(f"sure vs restatement {H}x{W}: worst out {worst[0]:.3g}, worst err {worst[1]:.3g}, least decided share {worst[2]:.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_sure_large_image_sampled_pixels(guided):
    H, W = 2160, 3840
    b = 2  # (the f64 restatement of every neighbour of a window is slow; other radii are checked on the smaller images)
    mu_a, v_a, mu_b, v_b = TDD.synthetic_halves(H, W, 121)
    feats = TG.synthetic_features(H, W, 123) if guided else None
    g = dict(feats=feats, k_feature=0.6, tau=1e-3) if guided else {}
    out, err, choice = _sure_np(mu_a, v_a, mu_b, v_b, smooth_radius=b, **g)
    rng = np.random.default_rng(122)
    pix = [(0, 0), (H - 1, W - 1), (0, W - 1), (H - 1, 0)] + list(zip(rng.integers(0, H, 6), rng.integers(0, W, 6)))
    side = 2 * b + 1
    nb = [(min(max(y + dy, 0), H - 1), min(max(x + dx, 0), W - 1)) for y, x in pix for dy in range(-b, b + 1) for dx in range(-b, b + 1)]
    kw = (10, 3, 0.45, 1.0, strengths(abi.RT_SURE_DEFAULT_RATIO), feats, 0.6, np.float32(1e-3))
    fa, wa = sure_cross_ref_pixels(mu_b, v_b, mu_a, nb, *kw)
    fb, wb = sure_cross_ref_pixels(mu_a, v_a, mu_b, nb, *kw)
    ny, nx = np.array(nb).T
    ma, va_, mb, vb_ = (a[ny, nx][:, None, :].astype(np.float64) for a in (mu_a, v_a, mu_b, v_b))
    s_hat = (risk64(fa, ma, va_, wa) + risk64(fb, mb, vb_, wb)) / 2  # [n * side^2, 3 candidates, 3]
    scale = (_risk_scale(fa, ma, va_) + _risk_scale(fb, mb, vb_)) / 2
    s_hat, scale = s_hat.reshape(len(pix), side * side, 3, 3), scale.reshape(len(pix), side * side, 3, 3)
    S_ = s_hat.sum(axis=-1).mean(axis=1)  # [n, 3]
    centre = side * side // 2
    py, px = np.array(pix).T
    got_c = choice[py, px]
    S_sorted = np.sort(S_, axis=1)
    decided = (S_sorted[:, 1] - S_sorted[:, 0]) > SURE_REL_TOL * scale.sum(axis=-1).mean(axis=1).max(axis=1)
    assert (got_c[decided] == np.argmin(S_, axis=1)[decided]).all() and decided.mean() > 0.8
    sel = np.arange(len(pix))
    want_out = (fa.reshape(len(pix), side * side, 3, 3)[sel, centre, got_c] + fb.reshape(len(pix), side * side, 3, 3)[sel, centre, got_c]) / 2
    want_err = np.maximum(s_hat[sel, :, got_c].mean(axis=1), 0.0)
    e_out = np.abs(out[py, px] - want_out) / (np.abs(want_out) + 1e-3)
    e_err = np.abs(err[py, px] - want_err) / (scale[sel, :, got_c].mean(axis=1) + 1e-30)
    print(f"sure 3840x2160 sampled (guided {guided}): worst out {e_out.max():.3g}, worst err {e_err.max():.3g}, decided {decided.mean():.2f}")
    assert e_out.max() < SURE_REL_TOL and e_err.max() < SURE_REL_TOL


@pytest.mark.gpu
def test_sure_exact_reductions_and_swap_symmetry():
    """ratio = 1: rt_denoise_cross_device's out bit for bit and choice 0; r = 0: out = (mu_A + mu_B) / 2 and err the window mean
    of (v_A + v_B) / 2 (the f32 restatement, bit for bit); A and B swapped, and a second call: the same bits"""
    H, W = 70, 90
    mu_a, v_a, mu_b, v_b = TDD.synthetic_halves(H, W, 131)
    feats = TG.synthetic_features(H, W, 132)
    g = dict(k_feature=0.6, tau=1e-3)
    for r, f in ((10, 3), (3, 0), (15, 7)):
        kw = dict(search_radius=r, patch_radius=f)
        for fe in (None, feats):
            gk = g if fe is not None else {}
            out, _, choice = _sure_np(mu_a, v_a, mu_b, v_b, feats=fe, ratio=1.0, **gk, **kw)
            want, _ = TDD._cross_np(mu_a, v_a, mu_b, v_b, feats=fe, **gk, **kw)
            assert np.array_equal(out.view(np.uint32), want.view(np.uint32)) and not choice.any(), (r, f)
            o1, e1, c1 = _sure_np(mu_a, v_a, mu_b, v_b, feats=fe, **gk, **kw)
            o2, e2, c2 = _sure_np(mu_b, v_b, mu_a, v_a, feats=fe, **gk, **kw)
            o3, e3, c3 = _sure_np(mu_a, v_a, mu_b, v_b, feats=fe, **gk, **kw)
            for o, e, c in ((o2, e2, c2), (o3, e3, c3)):
                assert np.array_equal(o1.view(np.uint32), o.view(np.uint32)) and np.array_equal(e1.view(np.uint32), e.view(np.uint32))
                assert np.array_equal(c1, c)
            assert len(np.unique(c1)) == 3
    for b in (0, 2, 7):
        for fe in (None, feats):
            out, err, choice = _sure_np(mu_a, v_a, mu_b, v_b, feats=fe, search_radius=0, patch_radius=3, smooth_radius=b, **(g if fe is not None else {}))
            s = out_risk_ref(v_a, v_b)
            risk = np.ascontiguousarray(np.concatenate([s, s, s], axis=-1))
            mu3 = np.stack([mu_a] * 3), np.stack([mu_b] * 3)
            o, e, c = select_ref(risk, *mu3, b)
            assert not c.any() and not choice.any()
            assert np.array_equal(out.view(np.uint32), TDD.dual_out_ref(mu_a, mu_b).view(np.uint32))
            assert np.array_equal(err.view(np.uint32), e.view(np.uint32)), b


@pytest.mark.gpu
def test_selection_follows_the_image():
    """flat and noisy on the left, a fine i.i.d. texture of low noise on the right (contrast of a few noise deviations, so the
    candidates' weights differ there): most of the flat side picks the stronger filter (j = 2) and most of the textured side
    the weaker one (j = 1), at the default ratio and smooth radius.  Shares (j = 0, 1, 2) of the f64 restatement: flat
    0.047 / 0.187 / 0.766, textured 0.015 / 0.985 / 0.000; measured on the device: the same."""
    H, W = 48, 96
    rng = np.random.default_rng(141)
    yy, xx = np.mgrid[0:H, 0:W]
    left = xx < W // 2
    texture = 0.5 + 0.002 * rng.standard_normal((H, W))
    t = np.where(left, 0.5, texture)[..., None] * np.array([1.0, 0.8, 0.6])
    v = np.where(left, 1e-2, 1e-5)[..., None] * np.ones(3)
    halves = [(t + np.sqrt(v) * rng.standard_normal(t.shape)).astype(np.float32) for _ in range(2)]
    _, _, choice = _sure_np(halves[0], v.astype(np.float32), halves[1], v.astype(np.float32))
    inner = (xx > 12) & (xx < W - 12) & (np.abs(xx - W // 2) > 12)
    flat = [float((choice[left & inner] == j).mean()) for j in range(3)]
    textured = [float((choice[~left & inner] == j).mean()) for j in range(3)]
    print(f"selection shares (j = 0, 1, 2): flat {flat}; textured {textured}")
    assert flat[2] > 0.5 and textured[1] > 0.5, (flat, textured)


@pytest.mark.gpu
def test_denoise_sure_rejects_bad_arguments():
    import torch
    lib = abi.load()
    t = [torch.zeros(8, 8, 3, device="cuda") for _ in range(10)]
    ch = [torch.zeros(8, 8, dtype=torch.int32, device="cuda") for _ in range(1)]
    ptr = [x.data_ptr() for x in t]
    opt = C.byref(rt.renderer.denoise_options_struct())

    def call(bufs=None, feats=(None,) * 4, guide=None, o=ptr[8], e=ptr[9], c=ch[0].data_ptr(), W=8, H=8, sure=None):
        b = list(ptr[:4]) if bufs is None else bufs
        g = C.byref(rt.renderer.guide_struct(**guide)) if guide is not None else None
        s = C.byref(rt.renderer.sure_struct(**(sure or {})))
        return lib.rt_denoise_sure_device(*b, *feats, W, H, opt, g, s, o, e, c, -1, None)

    assert call() == abi.RT_OK and call(e=None) == abi.RT_OK and call(c=None) == abi.RT_OK and call(e=None, c=None) == abi.RT_OK
    assert call(feats=ptr[4:8], guide={}) == abi.RT_OK
    for good in (dict(ratio=1.0), dict(ratio=1e18), dict(smooth_radius=0), dict(smooth_radius=abi.RT_SURE_MAX_SMOOTH_RADIUS)):
        assert call(sure=good) == abi.RT_OK, good
    for bad in (dict(ratio=0.999), dict(ratio=float("nan")), dict(ratio=float("inf")), dict(ratio=-2.0), dict(ratio=2e19), dict(ratio=1e20),
                dict(smooth_radius=-1), dict(smooth_radius=abi.RT_SURE_MAX_SMOOTH_RADIUS + 1)):
        assert call(sure=bad) == abi.RT_ERR_INVALID, bad
    for i in range(4):
        assert call(bufs=ptr[:i] + [None] + ptr[i + 1:4]) == abi.RT_ERR_INVALID, i
        assert call(o=ptr[i]) == abi.RT_ERR_INVALID and call(e=ptr[i]) == abi.RT_ERR_INVALID and call(c=ptr[i]) == abi.RT_ERR_INVALID, i
        assert call(feats=ptr[4:8][:i] + [None] + ptr[4:8][i + 1:], guide={}) == abi.RT_ERR_INVALID, i
        assert call(feats=[ptr[4 + i] if j == i else None for j in range(4)]) == abi.RT_ERR_INVALID, i
        assert call(feats=ptr[4:8], guide={}, c=ptr[4 + i] + 4 * 100) == abi.RT_ERR_INVALID, i
    assert call(feats=ptr[4:8]) == abi.RT_ERR_INVALID and call(guide={}) == abi.RT_ERR_INVALID
    for bad in (dict(o=None), dict(e=ptr[8]), dict(c=ptr[8]), dict(c=ptr[9] + 4 * 3 * 64 - 4), dict(o=ptr[9] + 4 * 3 * 8 * 7), dict(W=0), dict(H=-1),
                dict(H=abi.RT_DENOISE_MAX_HEIGHT + 1, W=1), dict(feats=ptr[4:8], guide=dict(tau=0.0))):
        assert call(**bad) == abi.RT_ERR_INVALID, bad
    assert call(c=ptr[9] + 4 * 3 * 64) == abi.RT_OK  # (right after err)
    assert lib.rt_denoise_sure_device(*ptr[:4], *(None,) * 4, 8, 8, opt, None, None, ptr[8], ptr[9], None, -1, None) == abi.RT_ERR_INVALID
    assert lib.rt_denoise_sure_device(*ptr[:4], *(None,) * 4, 8, 8, None, None, C.byref(rt.renderer.sure_struct()), ptr[8], ptr[9], None, -1,
                                      None) == abi.RT_ERR_INVALID
    with pytest.raises(ValueError):
        rt.denoise_sure(*[x.double() for x in t[:4]])


# ------------------------------------------------------------------------------------------------------------ the glue
GUIDE = TDD.GUIDE


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_render_denoised_sure_uniform_is_the_chain(guided):
    """two moments renders of the halves, the numpy conversion with n/2, rt_denoise_sure_device, to_rgb"""
    world, scene, cam = TD._setup("cornell_smoke")
    W, H, spp = 72, 56, 24
    rows = []
    r = TD._renderer(world, scene, cam, W, H, spp)
    kw = dict(search_radius=5, patch_radius=2, ratio=1.5, smooth_radius=3)
    rgb, den, err, n, choice = r.render_denoised_sure(logger=lambda j, total: rows.append((j, total)), guide=GUIDE if guided else None, **kw)
    assert rows == [(j, H) for j in range(H)]
    assert r.stats["paths"] == W * H * spp and r.stats["device_ms"] > 0 and (n == spp).all()
    a, b = TDD._moments_range(scene, cam, W, H, 0, spp // 2), TDD._moments_range(scene, cam, W, H, spp // 2, spp // 2)
    mu_a, v_a = TD.mean_var_ref(*a, spp // 2)
    mu_b, v_b = TD.mean_var_ref(*b, spp // 2)
    feats = TG._features(scene, cam, W, H, GUIDE["feature_samples"])[0] if guided else None
    g = dict(k_feature=GUIDE["k_feature"], tau=GUIDE["tau"]) if guided else {}
    want, want_err, want_c = _sure_np(mu_a, v_a, mu_b, v_b, feats=feats, **g, **kw)
    assert np.array_equal(den.view(np.uint32), want.view(np.uint32)) and np.array_equal(err.view(np.uint32), want_err.view(np.uint32))
    assert np.array_equal(choice, want_c) and len(np.unique(choice)) >= 2
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


def _replay(scene, cam, W, H, cap, t, m, feats=None, guide=None):
    """the rounds of rt_render_denoised_sure in Python: TDD._replay with rt_denoise_sure_device and its err in the rule"""
    sums = [np.zeros((H, W, 3), np.uint64) for _ in range(4)]
    half = np.zeros((H, W), np.int64)
    active = np.ones((H, W), bool)
    n_done = 0
    while active.any():
        count = m if n_done == 0 else min(n_done, cap - n_done)
        h = count // 2
        for j, begin in ((0, n_done), (2, n_done + h)):
            s1, s2 = TDD._moments_range(scene, cam, W, H, begin, h)
            sums[j][active] += s1[active]
            sums[j + 1][active] += s2[active]
        n_done += count
        half[active] = n_done // 2
        mu_a, v_a = TD.mean_var_ref(sums[0], sums[1], half[..., None])
        mu_b, v_b = TD.mean_var_ref(sums[2], sums[3], half[..., None])
        out, err, choice = _sure_np(mu_a, v_a, mu_b, v_b, feats=feats, **(guide or {}))
        idx = np.nonzero(active)
        active[idx] = ~TDD.filtered_done_ref(n_done, cap, out[idx], err[idx], t)
    return 2 * half, out, err, choice


@pytest.mark.gpu
@pytest.mark.parametrize("guided", [False, True])
def test_render_denoised_sure_adaptive_is_the_replay(guided):
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 64
    r = TD._renderer(world, scene, cam, W, H, 128)
    rows = []
    rgb, den, err, n, choice = r.render_denoised_sure(0.02, 8, logger=lambda j, total: rows.append((j, total)), guide={} if guided else None)
    assert sorted(rows) == [(j, H) for j in range(H)]
    feats = TG._features(scene, cam, W, H, abi.RT_GUIDE_DEFAULT_FEATURE_SAMPLES)[0] if guided else None
    n_ref, out_ref, err_ref, c_ref = _replay(scene, cam, W, H, 128, 0.02, 8, feats)
    assert len(np.unique(n)) >= 3 and r.stats["paths"] == int(n.sum())
    assert np.array_equal(n, n_ref) and np.array_equal(choice, c_ref)
    assert np.array_equal(den.view(np.uint32), out_ref.view(np.uint32)) and np.array_equal(err.view(np.uint32), err_ref.view(np.uint32))
    assert np.array_equal(rgb, TD.to_rgb_ref(den.astype(np.float64)))
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("adaptive", [False, True])
def test_cli_denoise_sure_ppm_matches_the_library(adaptive):
    args = ["--world=cornell_smoke", "--seed=42", "--aspect_ratio=1:1", "--image_width=48", "--samples_per_pixel=32", "--denoise_sure", "--stats"]
    if adaptive:
        args += ["--noise_threshold=0.02", "--min_samples=8", "--denoise_guided"]
    r = subprocess.run([CLI, *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "Done!" in r.stderr and '"mean_spp": ' in r.stderr
    world, scene, cam = TD._setup("cornell_smoke")
    rd = TD._renderer(world, scene, cam, 48, 48, 32)
    rgb, _, _, n, _ = rd.render_denoised_sure(0.02 if adaptive else None, 8, guide={} if adaptive else None)
    assert rt.to_ppm(rgb) == r.stdout
    assert f'"paths": {rd.stats["paths"]},' in r.stderr and f'"mean_spp": {n.mean():.3f}' in r.stderr
    scene.close()


@pytest.mark.gpu
def test_render_denoised_sure_rejects_bad_arguments():
    world, scene, cam = TD._setup("cornell_smoke")
    lib = abi.load()

    def call(p, ad=None, guide=None, sure=None, **kw):
        g = C.byref(rt.renderer.guide_struct(**guide)) if guide is not None else None
        return lib.rt_render_denoised_sure(scene.handle, C.byref(cam.c), C.byref(p), C.byref(ad) if ad else None,
                                           C.byref(rt.renderer.denoise_options_struct(**kw)), g, C.byref(rt.renderer.sure_struct(**(sure or {}))),
                                           None, None, None, None, None, abi.RtProgressFn(), None, None)

    def adaptive(t=0.01, m=4):
        ad = abi.RtAdaptive()
        ad.noise_threshold, ad.min_samples = t, m
        return ad

    assert call(TD._params(16, 16, 8)) == abi.RT_OK and call(TD._params(16, 16, 8), adaptive()) == abi.RT_OK
    assert call(TD._params(16, 16, 4), guide={}) == abi.RT_OK and call(TD._params(16, 16, 12), adaptive(m=6)) == abi.RT_OK
    for spp in (2, 3, 7, 9):
        assert call(TD._params(16, 16, spp)) == abi.RT_ERR_INVALID, spp
    for m in (2, 3, 5):
        assert call(TD._params(16, 16, 8), adaptive(m=m)) == abi.RT_ERR_INVALID, m
    assert call(TD._params(16, 16, 9), adaptive(m=4)) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8, begin=2)) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8, count=4), adaptive()) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), adaptive(t=float("nan"))) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), k=0.0) == abi.RT_ERR_INVALID
    assert call(TD._params(16, 16, 8), guide=dict(feature_samples=0)) == abi.RT_ERR_INVALID
    for bad in (dict(ratio=0.5), dict(ratio=float("inf")), dict(smooth_radius=-1), dict(smooth_radius=abi.RT_SURE_MAX_SMOOTH_RADIUS + 1)):
        assert call(TD._params(16, 16, 8), sure=bad) == abi.RT_ERR_INVALID, bad
    assert lib.rt_render_denoised_sure(scene.handle, C.byref(cam.c), C.byref(TD._params(16, 16, 8)), None, C.byref(rt.renderer.denoise_options_struct()),
                                       None, None, None, None, None, None, None, abi.RtProgressFn(), None, None) == abi.RT_ERR_INVALID
    assert lib.rt_render_denoised_sure(scene.handle, C.byref(cam.c), C.byref(TD._params(16, 16, 8)), None, None, None,
                                       C.byref(rt.renderer.sure_struct()), None, None, None, None, None, abi.RtProgressFn(), None, None) == abi.RT_ERR_INVALID
    for pipeline in (abi.RT_PIPELINE_MEGAKERNEL, abi.RT_PIPELINE_WAVEFRONT):
        assert call(TD._params(16, 16, 8, pipeline=pipeline)) == abi.RT_ERR_UNSUPPORTED
        assert call(TD._params(16, 16, 8, pipeline=pipeline), adaptive()) == abi.RT_ERR_UNSUPPORTED
    scene.close()


# ---------------------------------------------------------------------------------------------------------- measurement guards
# These bound measurements (DESIGN.md section 5h); they guard the measured behaviour and are not quality claims.  Measured on an
# NVIDIA B200 (1000 W); the sums are integers and the filters deterministic, so the values repeat exactly on the same build.
# Measured sum (out - gt)^2 / sum err, cornell_smoke 128^2, 64 spp: 0.61 (the dual filter's eps: 26.6 as a mean ratio).
SURE_CALIBRATION_BAND = (0.3, 1.5)
# Measured frame-mean shift against the noisy image at 64 spp: -1.90 %, -1.90 %, -1.81 % (r, g, b); dual 2.20 %, colour-only 1.21 %.
SURE_SHIFT_BOUND = 0.025
# Measured share of the early-stopped pixels off by more than 3 t: 57.6 % of the 57.4 % stopped before the cap (mean spp 469);
# the section 5d rule: 51.8 % of 30.5 %.  The goal (below 51.8 %) is missed.
SURE_TAIL_SHARE_BOUND = 0.65


@pytest.mark.gpu
def test_sure_error_estimate_calibration():
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    _, out, err, _, choice = TD._renderer(world, scene, cam, W, H, 64).render_denoised_sure()
    gt = TDD._ground_truth(scene, cam, W, H)
    ratio = float(((out.astype(np.float64) - gt) ** 2).sum() / err.astype(np.float64).sum())
    print("calibration: sum (out - gt)^2 / sum err", ratio, "choice shares", [float((choice == j).mean()) for j in range(3)])
    assert SURE_CALIBRATION_BAND[0] < ratio < SURE_CALIBRATION_BAND[1], ratio
    scene.close()


@pytest.mark.gpu
def test_sure_frame_mean_shift():
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    _, out, _, _, _ = TD._renderer(world, scene, cam, W, H, 64).render_denoised_sure()
    s1, s2 = TD._moments(scene, cam, W, H, 64)
    noisy, _ = TD.mean_var_ref(s1, s2, 64)
    shift = out.astype(np.float64).mean(axis=(0, 1)) / noisy.astype(np.float64).mean(axis=(0, 1)) - 1.0
    print("frame-mean shift: sure", shift.tolist())
    assert np.abs(shift).max() < SURE_SHIFT_BOUND, shift
    scene.close()


@pytest.mark.gpu
def test_sure_rule_early_stop_tail():
    """cornell_smoke 128^2, cap 1024, t = 0.01, min_samples 16: among the pixels stopped before the cap, the share whose display
    error exceeds 3 t, for the SURE rule judged on the SURE filter's output"""
    world, scene, cam = TD._setup("cornell_smoke")
    W = H = 128
    t = 0.01
    gt = TDD.display(TDD._ground_truth(scene, cam, W, H))
    _, out, _, n, _ = TD._renderer(world, scene, cam, W, H, 1024).render_denoised_sure(t, 16)
    stopped = n < 1024
    share = float((np.abs(TDD.display(out) - gt).max(axis=2)[stopped] > 3 * t).mean())
    print("early-stop tail: SURE rule", share, "stopped", float(stopped.mean()), "mean spp", float(n.mean()))
    assert stopped.mean() > 0.05 and share < SURE_TAIL_SHARE_BOUND, share
    scene.close()
