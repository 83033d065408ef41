"""An f64 path tracer that traces the device's own paths (TEST infrastructure; the product never loads it).

The device's randomness is fully specified: the uniforms of camera path (pixel, sample) are Philox4x32-10 blocks with
counter (pixel, sample, draw, RTB_PHILOX_TAG + block) and key = seed (rt_device.cuh: rng_block), draw 0 is the camera,
draw 1 + 2k the media of segment k and draw 2 + 2k its scatter (extend_and_shade), and every sampler is a direct function
of its uniforms.  So for a small class of scenes this module restates, in f64 and vectorised over paths, exactly the path
the device traces for any (pixel, sample), and returns its radiance, its segment count and how close it came to a branch.

Scene class (anything else raises): spheres of any radius (|r| >= 100 takes the device's f64 quadratic), xy / xz / yz
rects, Lambertian, metal (fuzz 0 or > 0) and diffuse-light materials whose texture is solid or a checker whose leaves all
have one colour, constant-density media with one sphere as boundary, black or gradient background.  No instances,
dielectrics, motion or non-constant textures: their oracle tests stay the check for them.

Each restatement cites the device function it restates (mu-lambda-raytracer_b200/csrc/rt_device.cuh unless named).
Transcendentals are exact here (the device uses MUFU approximations); the per-path tolerance of the tests absorbs that.

Robustness margin: for each path the smallest relative distance of any branch decision from its threshold (closest hit
against the runner-up and against t_min, a rect hit against the rect's edges, a sphere's discriminant, the face-forward
test, the Lambertian flip, metal's absorption test, a medium event against the boundary exit).  Only a path whose margin
is below the tests' threshold ("fragile") may legitimately take another branch on the f32 device.
"""
import numpy as np

from mu_lambda_raytracer_b200 import abi

TAG = 0x52544232  # RTB_PHILOX_TAG
T_MIN = float(np.float32(0.001))  # RTB_T_MIN
M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)
BIG_MARGIN = 1.0  # "no decision near a threshold"


def f32(x):
    """a value as the device stores it (f32), widened again to f64"""
    return np.asarray(x, dtype=np.float32).astype(np.float64)


# ---------------------------------------------------------------------------------------------------------- Philox
def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (philox_rounds) on arrays of 32-bit words held in uint64; returns the four output words"""
    c = [np.asarray(x, dtype=np.uint64) & MASK32 for x in (c0, c1, c2, c3)]
    c0, c1, c2, c3 = np.broadcast_arrays(*c)
    k0, k1 = np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)
    m0, m1 = np.uint64(M0), np.uint64(M1)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2  # 32 x 32 -> 64 bits: exact in uint64
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK32, p1 >> np.uint64(32), p1 & MASK32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + np.uint64(W0)) & MASK32, (k1 + np.uint64(W1)) & MASK32
    return c0, c1, c2, c3


def u32_to_unit(x):
    """__uint2float_rz(x) * 2^-32: the 24 leading significant bits of x, truncated, times 2^-32 (exact in f64)"""
    x = np.asarray(x, dtype=np.uint64)
    _, e = np.frexp(x.astype(np.float64))  # x < 2^32: exact; e = bit length
    drop = np.maximum(e - 24, 0).astype(np.uint64)
    return ((x >> drop) << drop).astype(np.float64) * 2.0 ** -32


def uniforms(pixel, sample, draw, block, seed):
    """rng_block: the four uniforms of Philox block `block` of draw `draw` of paths (pixel, sample), shape (n, 4)"""
    out = philox(pixel, sample, draw, TAG + block, seed & 0xFFFFFFFF, seed >> 32)
    return np.stack([u32_to_unit(w) for w in out], axis=-1)


# ---------------------------------------------------------------------------------------------------------- camera
def device_camera(cam):
    """make_camera (flatten.cpp) on an RtCamera: f64, then narrowed to f32 as the device stores it"""
    theta = cam.vfov_deg * np.pi / 180.0
    h = np.tan(theta / 2.0)
    vh = 2.0 * h
    vw = cam.aspect_ratio * vh
    lookfrom, lookat, vup = (np.array(list(v), dtype=np.float64) for v in (cam.lookfrom, cam.lookat, cam.vup))
    w = lookfrom - lookat
    w /= np.sqrt(w @ w)
    u = np.cross(vup, w)
    u /= np.sqrt(u @ u)
    v = np.cross(w, u)
    hor, ver = cam.focus_dist * vw * u, cam.focus_dist * vh * v
    llc = lookfrom - hor / 2.0 - ver / 2.0 - cam.focus_dist * w
    return {"origin": f32(lookfrom), "horizontal": f32(hor), "vertical": f32(ver), "lower_left": f32(llc - lookfrom),
            "u": f32(u), "v": f32(v), "lens_radius": float(f32(cam.aperture / 2.0))}


def camera_rays(dc, width, height, pixel, u):
    """generate_camera_ray for pixels `pixel` (py * W + px) with their draw-0 uniforms u (n, 4): origins, directions"""
    px, py = (pixel % width).astype(np.float64), (pixel // width).astype(np.float64)
    inv_wm1, inv_hm1 = float(f32(1.0 / (float(np.float32(width)) - 1.0))), float(f32(1.0 / (float(np.float32(height)) - 1.0)))
    s, t = (px + u[:, 0]) * inv_wm1, (py + u[:, 1]) * inv_hm1
    off = np.zeros((len(pixel), 3))
    if dc["lens_radius"] > 0.0:  # random_in_unit_disk without rejection: radius sqrt(u2), angle 2 pi u3
        r = dc["lens_radius"] * np.sqrt(u[:, 2])
        dx, dy = r * np.cos(2 * np.pi * u[:, 3]), r * np.sin(2 * np.pi * u[:, 3])
        off = dx[:, None] * dc["u"] + dy[:, None] * dc["v"]
    o = dc["origin"] + off
    d = dc["lower_left"] + s[:, None] * dc["horizontal"] + t[:, None] * dc["vertical"] - off
    return o, d


def unit_ball(u):
    """sample_unit_ball(u0, u1, u2): z = 1 - 2 u0, angle 2 pi u1, radius cbrt(u2)"""
    z = 1.0 - 2.0 * u[:, 0]
    rxy = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    r = np.cbrt(u[:, 2])
    a = 2 * np.pi * u[:, 1]
    return np.stack([r * rxy * np.cos(a), r * rxy * np.sin(a), r * z], axis=1)


# ---------------------------------------------------------------------------------------------------------- fixed point
def radiance_fixed(x):
    """radiance_fixed on f32 samples, exactly: clamp to [0, 2^20] (NaN -> 0), then (uint64) f32(x * 2^32 + 0.5)"""
    x = np.asarray(x, dtype=np.float32)
    x = np.where(np.isnan(x), np.float32(0), np.minimum(np.maximum(x, np.float32(0)), np.float32(2 ** 20)))
    v = x.astype(np.float64) * 2.0 ** 32  # exact: a power-of-two scaling of an f32
    return np.floor((v.astype(np.float32) + np.float32(0.5)).astype(np.float64)).astype(np.uint64)  # fmaf: one rounding of an exact sum


def moment2_fixed(q):
    """moment2_fixed: (min(q, 2^44))^2 >> 40, in exact integers"""
    q = min(int(q), 1 << 44)
    return (q * q) >> 40


# ---------------------------------------------------------------------------------------------------------- the scene
class UnsupportedScene(ValueError):
    pass


class Scene:
    """The restricted scene class, read from a finished support.DescBuilder (the description the device flattens)."""

    def __init__(self, builder):
        d = builder.desc
        self.bg = int(d.background_kind)
        self.bg_top, self.bg_bottom = f32(list(d.background_top)), f32(list(d.background_bottom))
        self.b = builder
        self.spheres, self.rects, self.media = [], [], []  # (c, r, mat), (axis k, (a0, a1, b0, b1), plane, mat), (c, r, neg_inv_density, colour)
        self._walk(d.root)
        self.mats = [self._material(i) for i in range(len(builder.materials))]
        self.n_prims = len(self.spheres) + len(self.rects)

    def _walk(self, i):
        n = self.b.nodes[i]
        f = [float(x) for x in n.f]
        if n.kind in (abi.RT_NODE_LIST, abi.RT_NODE_BVH):
            for k in range(n.child_count):
                self._walk(self.b.children[n.first_child + k])
        elif n.kind == abi.RT_NODE_SPHERE:
            self.spheres.append((f32(f[0:3]), float(f32(f[3])), n.material))
        elif n.kind in (abi.RT_NODE_XYRECT, abi.RT_NODE_XZRECT, abi.RT_NODE_YZRECT):
            k = {abi.RT_NODE_XYRECT: 2, abi.RT_NODE_XZRECT: 1, abi.RT_NODE_YZRECT: 0}[n.kind]
            self.rects.append((k, tuple(float(f32(x)) for x in f[0:4]), float(f32(f[4])), n.material))
        elif n.kind == abi.RT_NODE_MEDIUM:
            bnd = self.b.nodes[n.first_child]
            if bnd.kind != abi.RT_NODE_SPHERE:
                raise UnsupportedScene("a medium's boundary must be one sphere")
            m = self.b.materials[n.material]
            self.media.append((f32([bnd.f[0], bnd.f[1], bnd.f[2]]), float(f32(bnd.f[3])), float(f32(-1.0 / f[0])), self._colour(m.texture)))
        else:
            raise UnsupportedScene(f"node kind {n.kind}")

    def _colour(self, t):
        """a texture whose value is one colour everywhere: solid, or a checker whose leaves are all that colour"""
        tex = self.b.textures[t]
        if tex.kind == abi.RT_TEX_SOLID:
            return f32(list(tex.color))
        if tex.kind == abi.RT_TEX_CHECKER:
            a, b = self._colour(tex.a), self._colour(tex.b)
            if np.array_equal(a, b):
                return a
        raise UnsupportedScene("texture is not one colour")

    def _material(self, i):
        m = self.b.materials[i]
        if m.kind == abi.RT_MAT_METAL:  # metal reads its albedo, never a texture (flatten.cpp: tables)
            return (m.kind, f32(list(m.albedo)), float(f32(m.fuzz)))
        if m.kind in (abi.RT_MAT_LAMBERTIAN, abi.RT_MAT_DIFFUSE_LIGHT, abi.RT_MAT_ISOTROPIC):
            return (m.kind, self._colour(m.texture), 0.0)
        raise UnsupportedScene(f"material kind {m.kind}")


# ---------------------------------------------------------------------------------------------------------- tracing
def _dot(a, b):
    return np.einsum("ij,ij->i", a, b)


def _sphere_roots(c, r, o, d):
    """both roots of the sphere quadratic over (-inf, inf) (sphere_roots, exact), the discriminant over r^2, the mid-point t"""
    oc = o - c
    a = _dot(d, d)
    hb = _dot(oc, d)
    l = oc - (hb / a)[:, None] * d  # perpendicular offset, as the device computes it
    disc_rel = (r * r - _dot(l, l)) / (r * r)
    sq = np.sqrt(np.maximum(disc_rel, 0.0) * r * r * a)
    return (-hb - sq) / a, (-hb + sq) / a, disc_rel, -hb / a


def _rel(x, scale):
    return np.abs(x) / np.maximum(np.abs(scale), 1e-300)


class PathResult:
    def __init__(self, radiance, segments, margin):
        self.radiance, self.segments, self.margin = radiance, segments, margin


def trace(scene, cam, width, height, pixel, sample, seed, max_depth):
    """the path of every (pixel[i], sample[i]): radiance (n, 3) f64, segment count (rays traced) and robustness margin"""
    cam = getattr(cam, "c", cam)  # a renderer.Camera or its RtCamera
    pixel = np.asarray(pixel, dtype=np.int64)
    sample = np.asarray(sample, dtype=np.int64)
    n = len(pixel)
    rad = np.zeros((n, 3))
    segs = np.zeros(n, dtype=np.int64)
    margin = np.full(n, BIG_MARGIN)
    if max_depth <= 0 or n == 0:  # every path returns Color::ZERO before tracing (raytrace.rs:87-89)
        return PathResult(rad, segs, margin)
    dc = device_camera(cam)
    o, d = camera_rays(dc, width, height, pixel, uniforms(pixel, sample, 0, 0, seed))
    beta = np.ones((n, 3))
    origin = np.full(n, -1, dtype=np.int64)  # primitive the ray starts on: spheres 0.., rects after them
    idx = np.arange(n)  # the live paths
    ns = len(scene.spheres)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for seg in range(max_depth):
            if len(idx) == 0:
                break
            m = len(idx)
            po, pd = o[idx], d[idx]
            segs[idx] += 1
            mg = np.full(m, BIG_MARGIN)
            pix, smp = pixel[idx], sample[idx]
            # ---- media first (sample_media / sample_media_general: medium m uses uniform m & 3 of block m >> 2)
            t_best = np.full(m, np.inf)
            medium = np.full(m, -1, dtype=np.int64)
            if scene.media:
                length = np.sqrt(_dot(pd, pd))
                ublocks = {}
                for k, (c, r, nid, _) in enumerate(scene.media):
                    if k >> 2 not in ublocks:
                        ublocks[k >> 2] = uniforms(pix, smp, 1 + 2 * seg, k >> 2, seed)
                    um = ublocks[k >> 2][:, k & 3]
                    te, tx, disc, _ = _sphere_roots(c, r, po, pd)
                    mg = np.minimum(mg, np.abs(disc))
                    ok = (disc >= 0) & (tx >= te + T_MIN)  # medium_interval: the second boundary hit must exist
                    t1, t2 = np.maximum(te, T_MIN), np.minimum(tx, t_best)
                    ok &= t1 < t2
                    inside = (t2 - t1) * length
                    dist = nid * np.log(um)
                    mg = np.where(ok, np.minimum(mg, _rel(dist - inside, inside)), mg)
                    ev = ok & (dist <= inside)
                    t_best = np.where(ev, t1 + dist / length, t_best)
                    medium = np.where(ev, k, medium)
            # ---- surfaces (closest_hit over [t_min, t_best]; the origin primitive's rule of hit_sphere / box_slabs)
            cand = []  # every surface's hit distance in [t_min, inf) (inf: none) and its primitive number
            for j, (c, r, _) in enumerate(scene.spheres):
                t0, t1_, disc, tmid = _sphere_roots(c, r, po, pd)
                from_surface = origin[idx] == j
                oc = po - c
                t_fs = -2.0 * _dot(oc, pd) / _dot(pd, pd)
                t0 = np.where(from_surface, t_fs, t0)
                t1_ = np.where(from_surface, t_fs, t1_)
                real = from_surface | (disc >= 0)
                mg = np.where(~from_surface & (tmid > T_MIN), np.minimum(mg, np.abs(disc)), mg)
                for tr in (t0, t1_):
                    mg = np.where(real & (tr > 0), np.minimum(mg, _rel(tr - T_MIN, np.maximum(tr, T_MIN))), mg)
                th = np.where(real & (t0 >= T_MIN), t0, np.where(real & (t1_ >= T_MIN), t1_, np.inf))
                cand.append(th)
            rect_edge = []
            for j, (k, (a0, a1, b0, b1), plane, _) in enumerate(scene.rects):
                ax = [a for a in range(3) if a != k]  # (x, y) for xy, (x, z) for xz, (y, z) for yz: the node's (a, b) order
                tp = (plane - po[:, k]) / pd[:, k]
                pa = po[:, ax[0]] + tp * pd[:, ax[0]]
                pb = po[:, ax[1]] + tp * pd[:, ax[1]]
                inside = (pa >= a0) & (pa <= a1) & (pb >= b0) & (pb <= b1) & (origin[idx] != ns + j)
                edge = np.minimum(np.minimum(np.abs(pa - a0), np.abs(pa - a1)) / np.maximum(1.0, np.maximum(abs(a0), abs(a1))),
                                  np.minimum(np.abs(pb - b0), np.abs(pb - b1)) / np.maximum(1.0, np.maximum(abs(b0), abs(b1))))
                near = (origin[idx] != ns + j) & (tp > 0)
                mg = np.where(near, np.minimum(mg, _rel(tp - T_MIN, np.maximum(tp, T_MIN))), mg)
                rect_edge.append((tp, edge, near))
                cand.append(np.where(inside & (tp >= T_MIN), tp, np.inf))
            if cand:
                T = np.stack(cand, axis=1)
                prim = np.argmin(T, axis=1)
                t_surf = T[np.arange(m), prim]
                T_sorted = np.sort(np.concatenate([T, t_best[:, None]], axis=1), axis=1)
                gap = _rel(T_sorted[:, 1] - T_sorted[:, 0], T_sorted[:, 0])
                mg = np.where(np.isfinite(T_sorted[:, 1]), np.minimum(mg, gap), mg)
                t_lim = np.minimum(t_surf, t_best)
                for tp, edge, near in rect_edge:  # an edge decides only for rects whose plane lies before the event
                    mg = np.where(near & (tp <= t_lim * (1 + 1e-3)), np.minimum(mg, edge), mg)
                surf = np.isfinite(t_surf) & (t_surf <= t_best)  # closest_hit's t_max is the media event: a surface at it still wins
                prim = np.where(surf, prim, -1)
                t = np.where(surf, t_surf, t_best)
                medium = np.where(surf, -1, medium)
            else:
                prim, t = np.full(m, -1, dtype=np.int64), t_best
            # ---- miss: background (background_color)
            miss = (prim < 0) & (medium < 0)
            if miss.any():
                bg = np.zeros((int(miss.sum()), 3))
                if scene.bg != abi.RT_BG_BLACK:
                    dm = pd[miss]
                    tt = 0.5 * (dm[:, 1] / np.sqrt(_dot(dm, dm)) + 1.0)
                    bg = (1.0 - tt)[:, None] * scene.bg_bottom + tt[:, None] * scene.bg_top
                rad[idx[miss]] = beta[idx[miss]] * bg
            # ---- scatter (scatter_event / scatter) with the uniforms of draw 2 + 2k
            u = uniforms(pix, smp, 2 + 2 * seg, 0, seed)
            ball = unit_ball(u)
            p = po + t[:, None] * pd
            normal = np.zeros((m, 3))
            kind = np.zeros(m, dtype=np.int64)
            colour = np.zeros((m, 3))
            fuzz = np.zeros(m)
            for j, (c, r, mat) in enumerate(scene.spheres):
                s = prim == j
                normal[s] = (p[s] - c) * (1.0 / r)  # signed radius flips the normal
                kind[s], colour[s], fuzz[s] = scene.mats[mat]
            for j, (k, _, plane, mat) in enumerate(scene.rects):
                s = prim == ns + j
                p[s, k] = plane  # the hit point lies on the plane exactly
                normal[s] = np.eye(3)[k]
                kind[s], colour[s], fuzz[s] = scene.mats[mat]
            for k, (_, _, _, col) in enumerate(scene.media):
                s = medium == k
                kind[s], colour[s] = abi.RT_MAT_ISOTROPIC, col
            is_surf = prim >= 0
            dn = _dot(normal, pd)
            mg = np.where(is_surf, np.minimum(mg, _rel(dn, np.sqrt(_dot(pd, pd)))), mg)
            n_ff = np.where((dn < 0)[:, None], normal, -normal)  # face-forward (surface_at)
            dirn = ball.copy()  # isotropic: the raw in-ball direction
            alive = ~miss
            term = np.zeros((m, 3))
            lam = (kind == abi.RT_MAT_LAMBERTIAN) & alive
            if lam.any():
                nb = _dot(n_ff, ball)
                mg = np.where(lam, np.minimum(mg, _rel(nb, np.sqrt(_dot(ball, ball)))), mg)
                b = np.where((nb > 0)[:, None], ball, -ball)
                dl = n_ff + b
                tiny = np.all(np.abs(dl) < 1e-8, axis=1)
                dl[tiny] = n_ff[tiny]
                dirn[lam] = dl[lam]
            met = (kind == abi.RT_MAT_METAL) & alive
            if met.any():
                ud = pd / np.sqrt(_dot(pd, pd))[:, None]
                refl = ud - (2.0 * _dot(ud, n_ff))[:, None] * n_ff
                dm = refl + fuzz[:, None] * ball
                dmn = _dot(dm, n_ff)
                mg = np.where(met, np.minimum(mg, _rel(dmn, np.sqrt(_dot(dm, dm)))), mg)
                dirn[met] = dm[met]
                absorbed = met & ~(dmn > 0)
                alive &= ~absorbed  # scatter -> None: the path ends with 0
            light = (kind == abi.RT_MAT_DIFFUSE_LIGHT) & alive
            term[light] = colour[light]  # emits from both faces
            alive &= ~light
            ended = ~miss & ~alive
            rad[idx[ended]] = beta[idx[ended]] * term[ended]
            margin[idx] = np.minimum(margin[idx], mg)
            # ---- survivors: beta *= attenuation, new ray from the event; the depth check of extend_and_shade
            beta[idx[alive]] *= colour[alive]
            o[idx[alive]] = p[alive]
            d[idx[alive]] = dirn[alive]
            origin[idx[alive]] = prim[alive]  # -1 after a medium event
            idx = idx[alive]
            if seg + 1 == max_depth:  # depth exhausted after this segment's scatter: Color::ZERO
                rad[idx] = 0.0
    return PathResult(rad, segs, margin)
