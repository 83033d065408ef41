//! FFI over include/rt_b200.h (ABI version 3): the GPU replacement of `Renderer::new_with_rng(..).render(..)`
//! (src/raytrace.rs:151-186), plus `SceneSink`, the recorder a Rust host fills while it builds a world.
//!
//! NOT compiled in this repository (there is no Rust toolchain in the build image or on the GPU box); kept in step
//! with the header by hand.  The same ABI is exercised by the C++ host (mu-lambda-raytracer_b200/csrc/main.cpp), a C99
//! client (tests/c_abi/abi_check.c) and Python ctypes (mu-lambda-raytracer_b200/abi.py).
#![allow(non_camel_case_types, dead_code)]
use std::ffi::{CStr, CString};
use std::os::raw::{c_char, c_int, c_void};

pub const RT_NODE_SPHERE: i32 = 1;
pub const RT_NODE_XYRECT: i32 = 2;
pub const RT_NODE_XZRECT: i32 = 3;
pub const RT_NODE_YZRECT: i32 = 4;
pub const RT_NODE_BLOCK: i32 = 5;
pub const RT_NODE_TRANSLATE: i32 = 6;
pub const RT_NODE_ROTATE: i32 = 7;
pub const RT_NODE_MEDIUM: i32 = 8;
pub const RT_NODE_BVH: i32 = 9;
pub const RT_NODE_LIST: i32 = 10;
pub const RT_NODE_MOVING_SPHERE: i32 = 11; // extension of the library (The Next Week's MovingSphere); the reference has none
pub const RT_MAT_LAMBERTIAN: i32 = 1;
pub const RT_MAT_METAL: i32 = 2;
pub const RT_MAT_DIELECTRIC: i32 = 3;
pub const RT_MAT_DIFFUSE_LIGHT: i32 = 4;
pub const RT_MAT_ISOTROPIC: i32 = 5;
pub const RT_TEX_SOLID: i32 = 1;
pub const RT_TEX_CHECKER: i32 = 2;
pub const RT_TEX_NOISE: i32 = 3;
pub const RT_TEX_IMAGE: i32 = 4;
pub const RT_BG_BLACK: i32 = 0;
pub const RT_BG_GRADIENT: i32 = 1;
pub const RT_PERLIN_POINTS: usize = 1024;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtNode {
    pub kind: i32,
    pub material: i32,
    pub first_child: i32,
    pub child_count: i32,
    pub axis: i32,
    pub reserved: i32,
    pub f: [f64; 8],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtMaterial {
    pub kind: i32,
    pub texture: i32,
    pub albedo: [f64; 3],
    pub fuzz: f64,
    pub ior: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtTexture {
    pub kind: i32,
    pub a: i32,
    pub b: i32,
    pub reserved: i32,
    pub color: [f64; 3],
    pub scale: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtPerlin {
    pub ranvec: [[f64; 3]; RT_PERLIN_POINTS],
    pub perm_x: [i32; RT_PERLIN_POINTS],
    pub perm_y: [i32; RT_PERLIN_POINTS],
    pub perm_z: [i32; RT_PERLIN_POINTS],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtImage {
    pub width: i32,
    pub height: i32,
    pub rgb: *const u8,
}
#[repr(C)]
pub struct RtSceneDesc {
    pub root: i32,
    pub background_kind: i32,
    pub background_top: [f64; 3],
    pub background_bottom: [f64; 3],
    pub n_nodes: i32,
    pub n_children: i32,
    pub n_materials: i32,
    pub n_textures: i32,
    pub n_perlins: i32,
    pub n_images: i32,
    pub nodes: *const RtNode,
    pub children: *const i32,
    pub materials: *const RtMaterial,
    pub textures: *const RtTexture,
    pub perlins: *const RtPerlin,
    pub images: *const RtImage,
}
#[repr(C)]
pub struct RtCamera {
    pub lookfrom: [f64; 3],
    pub lookat: [f64; 3],
    pub vup: [f64; 3],
    pub vfov_deg: f64,
    pub aspect_ratio: f64,
    pub aperture: f64,
    pub focus_dist: f64,
    /// shutter interval of the library's motion-blur extension; 0.0, 0.0 = the reference's camera
    pub time0: f64,
    pub time1: f64,
}
#[repr(C)]
pub struct RtParams {
    pub width: i32,
    pub height: i32,
    pub samples_per_pixel: i32,
    pub max_depth: i32,
    pub seed: u64,
    pub sample_begin: i32,
    pub sample_count: i32,
    pub pipeline: i32,
    pub device: i32,
    pub samples_per_item: i32,
    pub bvh_layout: i32,
}
#[repr(C)]
#[derive(Default)]
pub struct RtStats {
    pub paths: u64,
    pub rays: u64,
    pub device_ms: f64,
    pub kernel_launches: i32,
    pub pipeline_used: i32,
    pub bvh_layout_used: i32,
    pub reserved: i32,
}
/// EXTENSION: noise-threshold adaptive sampling (rt_render_adaptive)
#[repr(C)]
#[derive(Default)]
pub struct RtAdaptive {
    pub noise_threshold: f64,
    pub min_samples: i32,
    pub reserved: i32,
}
pub const RT_MOMENT2_FIXED_ONE: f64 = 16777216.0;
/// EXTENSION: variance-guided non-local-means denoiser (rt_denoise_device, rt_render_denoised)
#[repr(C)]
pub struct RtDenoise {
    pub k: f64,
    pub alpha: f64,
    pub search_radius: i32,
    pub patch_radius: i32,
}
pub const RT_DENOISE_DEFAULT_SEARCH_RADIUS: i32 = 10;
pub const RT_DENOISE_DEFAULT_PATCH_RADIUS: i32 = 3;
pub const RT_DENOISE_DEFAULT_K: f64 = 0.45;
pub const RT_DENOISE_DEFAULT_ALPHA: f64 = 1.0;
pub const RT_DENOISE_MAX_SEARCH_RADIUS: i32 = 15;
pub const RT_DENOISE_MAX_PATCH_RADIUS: i32 = 7;
pub const RT_DENOISE_MAX_HEIGHT: i32 = 1048560;
impl Default for RtDenoise {
    fn default() -> RtDenoise {
        RtDenoise {
            k: RT_DENOISE_DEFAULT_K,
            alpha: RT_DENOISE_DEFAULT_ALPHA,
            search_radius: RT_DENOISE_DEFAULT_SEARCH_RADIUS,
            patch_radius: RT_DENOISE_DEFAULT_PATCH_RADIUS,
        }
    }
}
/// EXTENSION: feature-guided denoising (rt_render_features_device, rt_denoise_guided_device, rt_render_denoised_guided)
#[repr(C)]
pub struct RtGuide {
    pub k_feature: f64,
    pub tau: f64,
    pub feature_samples: i32,
    pub reserved: i32,
}
pub const RT_GUIDE_DEFAULT_K_FEATURE: f64 = 1.0;
pub const RT_GUIDE_DEFAULT_TAU: f64 = 1e-2;
pub const RT_GUIDE_DEFAULT_FEATURE_SAMPLES: i32 = 16;
impl Default for RtGuide {
    fn default() -> RtGuide {
        RtGuide {
            k_feature: RT_GUIDE_DEFAULT_K_FEATURE,
            tau: RT_GUIDE_DEFAULT_TAU,
            feature_samples: RT_GUIDE_DEFAULT_FEATURE_SAMPLES,
            reserved: 0,
        }
    }
}
/// EXTENSION: SURE selection among three strengths of the cross filter (rt_denoise_sure_device, rt_render_denoised_sure)
#[repr(C)]
pub struct RtSure {
    pub ratio: f64,
    pub smooth_radius: i32,
    pub reserved: i32,
}
pub const RT_SURE_DEFAULT_RATIO: f64 = 1.5;
pub const RT_SURE_DEFAULT_SMOOTH_RADIUS: i32 = 5;
pub const RT_SURE_MAX_SMOOTH_RADIUS: i32 = 7;
impl Default for RtSure {
    fn default() -> RtSure {
        RtSure { ratio: RT_SURE_DEFAULT_RATIO, smooth_radius: RT_SURE_DEFAULT_SMOOTH_RADIUS, reserved: 0 }
    }
}
/// EXTENSION: neighbourhood variance prior of the stop rules (rt_render_adaptive_prior, rt_render_denoised_sure_prior)
#[repr(C)]
pub struct RtPrior {
    pub prior_samples: f64,
    pub radius: i32,
    pub reserved: i32,
}
pub const RT_PRIOR_DEFAULT_SAMPLES: f64 = 16.0;
pub const RT_PRIOR_DEFAULT_RADIUS: i32 = 7;
pub const RT_PRIOR_MAX_RADIUS: i32 = 7;
impl Default for RtPrior {
    fn default() -> RtPrior {
        RtPrior { prior_samples: RT_PRIOR_DEFAULT_SAMPLES, radius: RT_PRIOR_DEFAULT_RADIUS, reserved: 0 }
    }
}
pub enum RtScene {}
/// Called once per image row j = 0 .. total-1, in increasing order, on the calling thread (include/rt_b200.h).
pub type RtProgressFn = Option<extern "C" fn(row: c_int, total: c_int, user: *mut c_void)>;

extern "C" {
    pub fn rt_last_error() -> *const c_char;
    pub fn rt_abi_version() -> c_int;
    pub fn rt_device_count() -> c_int;
    pub fn rt_scene_hash(desc: *const RtSceneDesc, out: *mut u8) -> c_int;
    pub fn rt_scene_create(desc: *const RtSceneDesc, device: c_int, out: *mut *mut RtScene) -> c_int;
    pub fn rt_scene_destroy(scene: *mut RtScene);
    pub fn rt_release_cached_memory();
    pub fn rt_render(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, accum_rgb: *mut f32, rgb: *mut i32,
                     cb: RtProgressFn, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_multi(scenes: *const *mut RtScene, n_scenes: i32, cam: *const RtCamera, params: *const RtParams, accum_rgb: *mut f32,
                           rgb: *mut i32, cb: RtProgressFn, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_moments_fixed_device(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, d_accum_fixed: *mut u64,
                                          d_moment2_fixed: *mut u64, stream: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_adaptive(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive, rgb: *mut i32,
                              samples: *mut i32, accum_fixed: *mut u64, moment2_fixed: *mut u64, cb: RtProgressFn, user: *mut c_void,
                              stats: *mut RtStats) -> c_int;
    pub fn rt_denoise_device(d_mean_rgb: *const f32, d_var_rgb: *const f32, width: i32, height: i32, opt: *const RtDenoise, d_out_rgb: *mut f32,
                             device: c_int, stream: *mut c_void) -> c_int;
    pub fn rt_render_denoised(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive, opt: *const RtDenoise,
                              rgb: *mut i32, denoised_rgb: *mut f32, cb: RtProgressFn, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_features_device(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, d_albedo: *mut f32, d_albedo_var: *mut f32,
                                     d_normal: *mut f32, d_normal_var: *mut f32, stream: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_denoise_guided_device(d_mean_rgb: *const f32, d_var_rgb: *const f32, d_albedo: *const f32, d_albedo_var: *const f32,
                                    d_normal: *const f32, d_normal_var: *const f32, width: i32, height: i32, opt: *const RtDenoise,
                                    guide: *const RtGuide, d_out_rgb: *mut f32, device: c_int, stream: *mut c_void) -> c_int;
    pub fn rt_render_denoised_guided(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive,
                                     opt: *const RtDenoise, guide: *const RtGuide, rgb: *mut i32, denoised_rgb: *mut f32, cb: RtProgressFn,
                                     user: *mut c_void, stats: *mut RtStats) -> c_int;
    // EXTENSION: dual-buffer cross-filtered denoising with an error estimate (guide null: colour-only)
    pub fn rt_denoise_cross_device(d_mean_a: *const f32, d_var_a: *const f32, d_mean_b: *const f32, d_var_b: *const f32, d_albedo: *const f32,
                                   d_albedo_var: *const f32, d_normal: *const f32, d_normal_var: *const f32, width: i32, height: i32,
                                   opt: *const RtDenoise, guide: *const RtGuide, d_out_rgb: *mut f32, d_err_rgb: *mut f32, device: c_int,
                                   stream: *mut c_void) -> c_int;
    pub fn rt_render_denoised_dual(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive,
                                   opt: *const RtDenoise, guide: *const RtGuide, rgb: *mut i32, denoised_rgb: *mut f32, error_rgb: *mut f32,
                                   samples: *mut i32, cb: RtProgressFn, user: *mut c_void, stats: *mut RtStats) -> c_int;
    // EXTENSION: SURE selection among three strengths of the cross filter, with a risk estimate (guide null: colour-only)
    pub fn rt_denoise_sure_device(d_mean_a: *const f32, d_var_a: *const f32, d_mean_b: *const f32, d_var_b: *const f32, d_albedo: *const f32,
                                  d_albedo_var: *const f32, d_normal: *const f32, d_normal_var: *const f32, width: i32, height: i32,
                                  opt: *const RtDenoise, guide: *const RtGuide, sure: *const RtSure, d_out_rgb: *mut f32, d_err_rgb: *mut f32,
                                  d_choice: *mut i32, device: c_int, stream: *mut c_void) -> c_int;
    pub fn rt_render_denoised_sure(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive,
                                   opt: *const RtDenoise, guide: *const RtGuide, sure: *const RtSure, rgb: *mut i32, denoised_rgb: *mut f32,
                                   error_rgb: *mut f32, samples: *mut i32, choice: *mut i32, cb: RtProgressFn, user: *mut c_void,
                                   stats: *mut RtStats) -> c_int;
    // EXTENSION: the stop rules with a neighbourhood variance prior (adaptive must be non-null)
    pub fn rt_render_adaptive_prior(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive,
                                    prior: *const RtPrior, rgb: *mut i32, samples: *mut i32, accum_fixed: *mut u64, moment2_fixed: *mut u64,
                                    cb: RtProgressFn, user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_render_denoised_sure_prior(scene: *const RtScene, cam: *const RtCamera, params: *const RtParams, adaptive: *const RtAdaptive,
                                         opt: *const RtDenoise, guide: *const RtGuide, sure: *const RtSure, prior: *const RtPrior, rgb: *mut i32,
                                         denoised_rgb: *mut f32, error_rgb: *mut f32, samples: *mut i32, choice: *mut i32, cb: RtProgressFn,
                                         user: *mut c_void, stats: *mut RtStats) -> c_int;
    pub fn rt_world_build(name: *const c_char, seed: u64, earth_rgb: *const u8, earth_w: i32, earth_h: i32, out: *mut *mut RtSceneDesc,
                          n_draws: *mut u64) -> c_int;
    pub fn rt_scene_desc_free(desc: *mut RtSceneDesc);
}

fn check(code: c_int) {
    if code != 0 {
        // the reference panics on misuse (unwrap); so does the shim, with the library's message
        panic!("rt_b200: {}", unsafe { CStr::from_ptr(rt_last_error()) }.to_string_lossy());
    }
}

/// What a world recipe fills while it runs: one entry per constructor call of the reference, in call order, values
/// exactly as the Rust code holds them (f64).  Indices play the role of the reference's moved / cloned values: using
/// an index twice is `.clone()`.  `worlds_gpu.rs` is `worlds.rs` written against this sink.
#[derive(Default)]
pub struct SceneSink {
    pub nodes: Vec<RtNode>,
    pub children: Vec<i32>,
    pub materials: Vec<RtMaterial>,
    pub textures: Vec<RtTexture>,
    pub perlins: Vec<RtPerlin>,
    pub images: Vec<(i32, i32, Vec<u8>)>,
}

impl SceneSink {
    pub fn new() -> SceneSink {
        SceneSink::default()
    }

    fn node(&mut self, kind: i32, material: i32, first_child: i32, child_count: i32, axis: i32, f: &[f64]) -> i32 {
        let mut a = [0.0; 8];
        a[..f.len()].copy_from_slice(f);
        self.nodes.push(RtNode { kind, material, first_child, child_count, axis, reserved: 0, f: a });
        self.nodes.len() as i32 - 1
    }
    fn texture(&mut self, kind: i32, a: i32, b: i32, color: [f64; 3], scale: f64) -> i32 {
        self.textures.push(RtTexture { kind, a, b, reserved: 0, color, scale });
        self.textures.len() as i32 - 1
    }
    fn material(&mut self, kind: i32, texture: i32, albedo: [f64; 3], fuzz: f64, ior: f64) -> i32 {
        self.materials.push(RtMaterial { kind, texture, albedo, fuzz, ior });
        self.materials.len() as i32 - 1
    }

    // ---- textures (src/textures.rs, src/image_texture.rs)
    pub fn solid(&mut self, r: f64, g: f64, b: f64) -> i32 {
        self.texture(RT_TEX_SOLID, -1, -1, [r, g, b], 0.0)
    }
    pub fn checker(&mut self, odd: i32, even: i32) -> i32 {
        self.texture(RT_TEX_CHECKER, odd, even, [0.0; 3], 0.0)
    }
    /// `NoiseTexture::new(scale, rng)`: the Perlin tables are drawn HERE, with the calls of `Perlin::new`
    /// (textures.rs:62-74: 1024 x `Vec3::random(-1, 1).unit()`, then three `permute`s, textures.rs:136-148), because the
    /// reference keeps them in private fields.
    pub fn noise(&mut self, scale: f64, rng: &mut dyn rand::RngCore) -> i32 {
        use rand::Rng;
        let mut p = RtPerlin {
            ranvec: [[0.0; 3]; RT_PERLIN_POINTS],
            perm_x: [0; RT_PERLIN_POINTS],
            perm_y: [0; RT_PERLIN_POINTS],
            perm_z: [0; RT_PERLIN_POINTS],
        };
        for i in 0..RT_PERLIN_POINTS {
            p.ranvec[i] = crate::vec::Vec3::random(-1.0, 1.0, rng).unit().e;
        }
        let mut permute = |perm: &mut [i32; RT_PERLIN_POINTS]| {
            for i in 0..RT_PERLIN_POINTS {
                perm[i] = i as i32;
            }
            for i in (1..RT_PERLIN_POINTS).rev() {
                let j: usize = rng.gen_range(0..i);
                perm.swap(i, j);
            }
        };
        permute(&mut p.perm_x);
        permute(&mut p.perm_y);
        permute(&mut p.perm_z);
        self.perlins.push(p);
        self.texture(RT_TEX_NOISE, self.perlins.len() as i32 - 1, -1, [0.0; 3], scale)
    }
    /// `image_texture::Image::new(img.to_rgb8())`: rows top to bottom, 3 bytes per pixel
    pub fn image(&mut self, img: &image::RgbImage) -> i32 {
        let (w, h) = img.dimensions();
        self.images.push((w as i32, h as i32, img.as_raw().clone()));
        self.texture(RT_TEX_IMAGE, self.images.len() as i32 - 1, -1, [0.0; 3], 0.0)
    }

    // ---- materials (src/materials.rs, src/volumes.rs:67-83)
    pub fn lambertian(&mut self, tex: i32) -> i32 {
        self.material(RT_MAT_LAMBERTIAN, tex, [0.0; 3], 0.0, 0.0)
    }
    pub fn metal(&mut self, albedo: [f64; 3], fuzz: f64) -> i32 {
        self.material(RT_MAT_METAL, -1, albedo, fuzz, 0.0)
    }
    pub fn dielectric(&mut self, ior: f64) -> i32 {
        self.material(RT_MAT_DIELECTRIC, -1, [0.0; 3], 0.0, ior)
    }
    pub fn diffuse_light(&mut self, tex: i32) -> i32 {
        self.material(RT_MAT_DIFFUSE_LIGHT, tex, [0.0; 3], 0.0, 0.0)
    }
    pub fn isotropic(&mut self, tex: i32) -> i32 {
        self.material(RT_MAT_ISOTROPIC, tex, [0.0; 3], 0.0, 0.0)
    }

    // ---- shapes, transforms, volumes, containers
    pub fn sphere(&mut self, c: [f64; 3], r: f64, mat: i32) -> i32 {
        self.node(RT_NODE_SPHERE, mat, -1, 0, 0, &[c[0], c[1], c[2], r])
    }
    pub fn xy_rect(&mut self, x0: f64, x1: f64, y0: f64, y1: f64, z: f64, mat: i32) -> i32 {
        self.node(RT_NODE_XYRECT, mat, -1, 0, 0, &[x0, x1, y0, y1, z])
    }
    pub fn xz_rect(&mut self, x0: f64, x1: f64, z0: f64, z1: f64, y: f64, mat: i32) -> i32 {
        self.node(RT_NODE_XZRECT, mat, -1, 0, 0, &[x0, x1, z0, z1, y])
    }
    pub fn yz_rect(&mut self, y0: f64, y1: f64, z0: f64, z1: f64, x: f64, mat: i32) -> i32 {
        self.node(RT_NODE_YZRECT, mat, -1, 0, 0, &[y0, y1, z0, z1, x])
    }
    pub fn block(&mut self, p0: [f64; 3], p1: [f64; 3], mat: i32) -> i32 {
        self.node(RT_NODE_BLOCK, mat, -1, 0, 0, &[p0[0], p0[1], p0[2], p1[0], p1[1], p1[2]])
    }
    pub fn translate(&mut self, off: [f64; 3], child: i32) -> i32 {
        self.node(RT_NODE_TRANSLATE, -1, child, 0, 0, &off)
    }
    /// axis: 0 = X, 1 = Y, 2 = Z (transforms.rs `Axis`)
    pub fn rotate(&mut self, axis: i32, degrees: f64, child: i32) -> i32 {
        self.node(RT_NODE_ROTATE, -1, child, 0, axis, &[degrees])
    }
    /// `ConstantMedium::from_color(boundary, d, color)` (volumes.rs:19-23): the boundary is any node (a list or BVH too)
    pub fn medium(&mut self, boundary: i32, density: f64, color: [f64; 3]) -> i32 {
        let tex = self.solid(color[0], color[1], color[2]);
        let iso = self.isotropic(tex);
        self.node(RT_NODE_MEDIUM, iso, boundary, 0, 0, &[density])
    }
    fn group(&mut self, kind: i32, items: &[i32]) -> i32 {
        let first = self.children.len() as i32;
        self.children.extend_from_slice(items);
        self.node(kind, -1, first, items.len() as i32, 0, &[])
    }
    pub fn list(&mut self, items: &[i32]) -> i32 {
        self.group(RT_NODE_LIST, items)
    }
    /// `bhv::BHV::new(&mut builder, rng)`: `Node::new` draws one axis per inner node, pre-order, and splits at len / 2
    /// (bhv.rs:122-145) — the split sizes depend on the count alone, so the draws are replayed here without building
    /// the reference's tree; whatever is built next sees the same stream.  Only the member list is recorded (the device
    /// builds its own BVH).
    pub fn bvh(&mut self, items: &[i32], rng: &mut dyn rand::RngCore) -> i32 {
        fn draw_axes(count: usize, rng: &mut dyn rand::RngCore) {
            use rand::Rng;
            if count < 2 {
                return;
            }
            let _axis: usize = rng.gen_range(0..3);
            draw_axes(count / 2, rng);
            draw_axes(count - count / 2, rng);
        }
        draw_axes(items.len(), rng);
        self.group(RT_NODE_BVH, items)
    }

    /// The description over this sink's arrays.  `images` must outlive the returned struct (it holds the RtImage
    /// records whose pixel pointers point into `self.images`).
    pub fn seal(&self, root: i32, background_kind: i32, images: &mut Vec<RtImage>) -> RtSceneDesc {
        images.clear();
        for (w, h, px) in self.images.iter() {
            images.push(RtImage { width: *w, height: *h, rgb: px.as_ptr() });
        }
        let gradient = background_kind == RT_BG_GRADIENT; // GradientBackground::default() (raytrace.rs:21-26)
        RtSceneDesc {
            root,
            background_kind,
            background_top: if gradient { [0.5, 0.7, 1.0] } else { [0.0; 3] },
            background_bottom: if gradient { [1.0, 1.0, 1.0] } else { [0.0; 3] },
            n_nodes: self.nodes.len() as i32,
            n_children: self.children.len() as i32,
            n_materials: self.materials.len() as i32,
            n_textures: self.textures.len() as i32,
            n_perlins: self.perlins.len() as i32,
            n_images: images.len() as i32,
            nodes: self.nodes.as_ptr(),
            children: self.children.as_ptr(),
            materials: self.materials.as_ptr(),
            textures: self.textures.as_ptr(),
            perlins: self.perlins.as_ptr(), // Vec<RtPerlin>: contiguous, as the ABI wants it
            images: images.as_ptr(),
        }
    }

    /// canonical SHA-256 of the description: must equal tests/golden/scene_hashes.json of the B200 repository
    pub fn hash(&self, root: i32, background_kind: i32) -> [u8; 32] {
        let mut images = Vec::new();
        let desc = self.seal(root, background_kind, &mut images);
        let mut out = [0u8; 32];
        check(unsafe { rt_scene_hash(&desc, out.as_mut_ptr()) });
        out
    }
}

pub struct GpuJob<'a> {
    pub camera: RtCamera,
    pub width: usize,
    pub height: usize,
    pub samples_per_pixel: i32,
    pub max_depth: i32,
    pub seed: u64,
    pub gpus: usize,
    /// the closure `Renderer::render` takes (raytrace.rs:172-174): called as logger(j, H) once per row
    pub logger: &'a mut dyn FnMut(usize, usize),
}

extern "C" fn logger_trampoline(row: c_int, total: c_int, user: *mut c_void) {
    let f = unsafe { &mut *(user as *mut &mut dyn FnMut(usize, usize)) };
    f(row as usize, total as usize);
}

fn render_desc(desc: *const RtSceneDesc, job: &mut GpuJob) -> Vec<Vec<(i32, i32, i32)>> {
    assert_eq!(unsafe { rt_abi_version() }, 3, "librt_b200.so speaks another ABI version than src/gpu.rs");
    let gpus = job.gpus.max(1).min(unsafe { rt_device_count() }.max(1) as usize);
    let mut scenes: Vec<*mut RtScene> = vec![std::ptr::null_mut(); gpus];
    for (g, s) in scenes.iter_mut().enumerate() {
        check(unsafe { rt_scene_create(desc, g as c_int, s) }); // flatten + BVH build + upload, one copy per device
    }
    let prm = RtParams {
        width: job.width as i32,
        height: job.height as i32,
        samples_per_pixel: job.samples_per_pixel,
        max_depth: job.max_depth,
        seed: job.seed,
        sample_begin: 0,
        sample_count: 0,
        pipeline: 0,
        device: -1,
        samples_per_item: 0,
        bvh_layout: 0,
    };
    let (w, h) = (job.width, job.height);
    let mut rgb = vec![0i32; 3 * w * h];
    let mut stats = RtStats::default();
    let mut logger: &mut dyn FnMut(usize, usize) = &mut *job.logger;
    let user = &mut logger as *mut &mut dyn FnMut(usize, usize) as *mut c_void;
    check(unsafe {
        rt_render_multi(scenes.as_ptr(), gpus as i32, &job.camera, &prm, std::ptr::null_mut(), rgb.as_mut_ptr(), Some(logger_trampoline), user,
                        &mut stats)
    });
    for s in scenes {
        unsafe { rt_scene_destroy(s) };
    }
    // Vec<Vec<RGB>> with row 0 at the BOTTOM, exactly what Renderer::render returns (raytrace.rs:172-186)
    (0..h).map(|j| (0..w).map(|i| { let k = 3 * (j * w + i); (rgb[k], rgb[k + 1], rgb[k + 2]) }).collect()).collect()
}

/// The GPU arm of do_tracing for a world described by the Rust host (`worlds_gpu::describe`).
pub fn render_sink(sink: &SceneSink, root: i32, background_kind: i32, job: &mut GpuJob) -> Vec<Vec<(i32, i32, i32)>> {
    let mut images = Vec::new();
    let desc = sink.seal(root, background_kind, &mut images);
    render_desc(&desc, job)
}

/// The same with the library's own restatement of worlds.rs (rt_world_build: bit-identical descriptions, see
/// tests/test_scene_and_abi.py of the B200 repository) — for hosts that do not want to carry `worlds_gpu.rs`.
pub fn render_named_world(name: &str, seed: u64, earthmap: Option<&image::RgbImage>, job: &mut GpuJob) -> Vec<Vec<(i32, i32, i32)>> {
    let cname = CString::new(name).unwrap();
    let (ptr, w, h) = match earthmap {
        Some(img) => (img.as_raw().as_ptr(), img.width() as i32, img.height() as i32),
        None => (std::ptr::null(), 0, 0),
    };
    let mut desc: *mut RtSceneDesc = std::ptr::null_mut();
    check(unsafe { rt_world_build(cname.as_ptr(), seed, ptr, w, h, &mut desc, std::ptr::null_mut()) });
    let image = render_desc(desc, job);
    unsafe { rt_scene_desc_free(desc) };
    image
}
