"""Scenes of tests/path_reference.py's class that select each kernel instance of the persistent pipeline by their content,
and the exact-valued scenes (every path's radiance is one f32 emission).  Shared by test_render_paths.py's CPU guards and
GPU tests."""
import support as S
from mu_lambda_raytracer_b200 import abi

# rt_types.h
F_BOX, F_INSTBOX, F_INSTANCE, F_MOVING, F_BIG, F_MEDIA, F_BOXMEDIA, F_CHECKER, F_NOISE, F_IMAGE, F_SPHERE = (1 << k for k in range(11))
# rt_persist.cu: the feature masks of the specialised instances
MASK_SPHERES = F_SPHERE | F_BIG
MASK_BOXES = F_BOX | F_INSTBOX | F_INSTANCE | F_MEDIA | F_BOXMEDIA
MASK_FINAL = F_SPHERE | F_BOX | F_INSTANCE | F_BIG | F_MEDIA | F_NOISE | F_IMAGE


def _lam(b, r, g, bl):
    return b.lambertian(b.solid(r, g, bl))


def _light(b, e):
    return b.material(abi.RT_MAT_DIFFUSE_LIGHT, b.solid(e, e, e))


def _metal(b, albedo, fuzz):
    return b.material(abi.RT_MAT_METAL, albedo=albedo, fuzz=fuzz)


def spheres_scene():
    """spheres only, a ground of radius 1000 (F_BIG), gradient sky: the "spheres" instance"""
    b = S.DescBuilder()
    items = [b.sphere((0, -1000, 0), 1000.0, _lam(b, 0.5, 0.5, 0.5)),
             b.sphere((0, 1, 0), 1.0, _lam(b, 0.7, 0.3, 0.3)),
             b.sphere((-2.25, 1, 0.5), 1.0, _metal(b, (0.8, 0.8, 0.8), 0.0)),
             b.sphere((2.25, 1, 0.5), 1.0, _metal(b, (0.8, 0.6, 0.25), 0.375)),
             b.sphere((0.5, 2.75, -1.5), 0.5, _light(b, 4.0))]
    b.finish(b.group(abi.RT_NODE_BVH, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 2, 8), lookat=(0, 1, 0), vfov=40.0)


def boxes_scene():
    """rects only, plus a medium bounded by a sphere (which sets no surface bit): the "boxes" instance"""
    b = S.DescBuilder()
    white, red, green = _lam(b, 0.73, 0.73, 0.73), _lam(b, 0.65, 0.05, 0.05), _lam(b, 0.12, 0.45, 0.15)
    items = [b.rect(abi.RT_NODE_XZRECT, -3, 3, -3, 3, 0.0, white),
             b.rect(abi.RT_NODE_XYRECT, -3, 3, 0, 3, -3.0, white),
             b.rect(abi.RT_NODE_YZRECT, 0, 3, -3, 3, -3.0, red),
             b.rect(abi.RT_NODE_YZRECT, 0, 3, -3, 1, 3.0, green),
             b.rect(abi.RT_NODE_XYRECT, -1, 1.5, 0, 1.25, -1.0, _metal(b, (0.9, 0.9, 0.9), 0.0)),
             b.rect(abi.RT_NODE_XZRECT, -1, 1, -2, -1, 2.5, _light(b, 6.0)),
             b.medium(b.sphere((1.5, 0.75, 0.75), 0.75, white), 0.75, (0.9, 0.9, 0.9))]
    b.finish(b.group(abi.RT_NODE_LIST, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 1.5, 7), lookat=(0, 1, 0), vfov=50.0)


def final_scene(checker=False):
    """spheres, rects, a big sphere and a clear sphere medium: the "final" instance; with a checker texture whose two
    colours are equal (F_CHECKER, a constant value) the F_ALL instance"""
    b = S.DescBuilder()
    ground = _lam(b, 0.48, 0.83, 0.53)
    if checker:
        ground = b.lambertian(b.checker(b.solid(0.48, 0.83, 0.53), b.solid(0.48, 0.83, 0.53)))
    items = [b.sphere((0, -1000, 0), 1000.0, ground),
             b.sphere((-1.5, 1, 0), 1.0, _lam(b, 0.8, 0.8, 0.1)),
             b.sphere((1.5, 1, -0.5), 1.0, _metal(b, (0.7, 0.7, 0.9), 0.125)),
             b.rect(abi.RT_NODE_XYRECT, -4, 4, 0, 3, -3.0, _lam(b, 0.4, 0.4, 0.6)),
             b.rect(abi.RT_NODE_XZRECT, -1, 1, -1, 1, 4.0, _light(b, 5.0)),
             b.medium(b.sphere((0.25, 0.75, 2.0), 0.75, ground), 1.5, (0.2, 0.4, 0.9))]
    b.finish(b.group(abi.RT_NODE_BVH, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 2, 9), lookat=(0, 1, 0), vfov=40.0)


def general_media_scene():
    """five sphere media (more than the fast sampler's four, so the block of uniforms m >> 2 = 1 is drawn): the
    general-media instance"""
    b = S.DescBuilder()
    grey = _lam(b, 0.5, 0.5, 0.5)
    items = [b.sphere((0, -1000, 0), 1000.0, grey),
             b.sphere((0, 1, -2), 1.0, _lam(b, 0.3, 0.5, 0.7)),
             b.sphere((0, 4, -2), 0.75, _light(b, 4.0))]
    for k, (x, z) in enumerate([(-2.5, 0.5), (-1.25, 1.5), (0, 1.0), (1.25, 1.5), (2.5, 0.5)]):
        items.append(b.medium(b.sphere((x, 0.6, z), 0.55, grey), 1.0 + 0.5 * k, (0.9 - 0.1 * k, 0.5, 0.3 + 0.1 * k)))
    b.finish(b.group(abi.RT_NODE_LIST, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 2, 8), lookat=(0, 1, 0), vfov=45.0)


# name -> (builder function, the feature bits it must have, which instance those pick)
MATRIX = {
    "spheres": (spheres_scene, F_SPHERE | F_BIG, "spheres"),
    "boxes": (boxes_scene, F_BOX | F_MEDIA, "boxes"),
    "final": (final_scene, F_SPHERE | F_BOX | F_BIG | F_MEDIA, "final"),
    "all": (lambda: final_scene(checker=True), F_SPHERE | F_BOX | F_BIG | F_MEDIA | F_CHECKER, "all"),
    "general": (general_media_scene, F_SPHERE | F_BIG | F_MEDIA, "general"),
}


def instance_of(features, n_media):
    """the instance pick_feature_instance launches for a scene (the general-media form first)"""
    if n_media > 4:
        return "general"
    for name, mask in (("spheres", MASK_SPHERES), ("boxes", MASK_BOXES), ("final", MASK_FINAL)):
        if features & ~mask == 0:
            return name
    return "all"


def camera(view, width, height):
    return S.make_camera(view["lookfrom"], view["lookat"], view["vfov"], width / height)


def exact_scene(emission, variant):
    """Every camera path hits a diffuse light first and ends there, so its radiance is exactly `emission` (an f32 value).
    "boxes": a light rect fills the view.  Otherwise a light sphere of radius 500 around the camera (F_BIG), with decoys
    outside it that only select the instance: a rect ("final"), a checker ("all"), five media ("general").  A medium is
    sampled before the surface search, so an event beyond the shell is cut off by the shell hit."""
    b = S.DescBuilder()
    light = _light(b, emission)
    grey = _lam(b, 0.5, 0.5, 0.5)
    if variant == "boxes":
        items = [b.rect(abi.RT_NODE_XYRECT, -1000, 1000, -1000, 1000, -1.0, light)]
    else:
        items = [b.sphere((0, 0, 0), 500.0, light)]
        if variant in ("final", "all"):
            items += [b.rect(abi.RT_NODE_XYRECT, -1, 1, -1, 1, -600.0, grey), b.medium(b.sphere((0, 0, 700), 50.0, grey), 0.5, (1, 1, 1))]
        if variant == "all":
            items.append(b.sphere((0, 800, 0), 10.0, b.lambertian(b.checker(b.solid(0.5, 0.5, 0.5), b.solid(0.5, 0.5, 0.5)))))
        if variant == "general":
            items += [b.medium(b.sphere((0, 0, 700 + 120 * k), 50.0, grey), 0.5, (1, 1, 1)) for k in range(5)]
    b.finish(b.group(abi.RT_NODE_LIST, items), background=abi.RT_BG_GRADIENT)
    return b, dict(lookfrom=(0, 0, 0), lookat=(0, 0, -1), vfov=60.0)
