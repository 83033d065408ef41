// Device-side path tracing: everything between "a (pixel, sample) index" and "a radiance sample".
//
// This is the B200 re-design of the reference's hot path (SURVEY §8a):
//   Camera::get_ray             src/camera.rs:40-48        -> generate_camera_ray
//   Hittable::hit dispatch      src/hittable.rs:53-68,
//                               src/bhv.rs:147-165         -> closest_hit (flat 32-byte-node BVH, short stack)
//   Sphere / AARect / Block     src/shapes.rs:57-82,
//                               src/aarects.rs:45-64       -> hit_sphere / hit_box (rects are flat boxes)
//   Translate / Rotate          src/transforms.rs:31-42,
//                               :127-142                   -> DInstance (composed rigid transform)
//   ConstantMedium::hit         src/volumes.rs:25-65       -> sample_media
//   Material::scatter / emit    src/materials.rs:25-127,
//                               src/volumes.rs:77-83       -> shade_hit
//   Texture::value              src/textures.rs:22-167,
//                               src/image_texture.rs:16-28 -> texture_value
//   trace_internal              src/raytrace.rs:79-101     -> the iterative loop in integrate_item
// Arithmetic is f32 (f64 only for spheres with |r| >= 100, whose quadratic cancels catastrophically in f32);
// random numbers are counter-based Philox4x32-10 keyed by (seed; pixel, sample, draw).
//
// The file also compiles as plain C++ (RTB_HOST_EMULATION) so that tests/ can run the very same functions on
// the CPU against the oracle; that build is test infrastructure only and is never part of librt_b200.so.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/rt_b200.h"
#include "rt_types.h"

#if defined(__CUDACC__) && !defined(RTB_HOST_EMULATION)
#define RTB_DEV __device__ __forceinline__
#define RTB_DEV_NOINLINE static __device__ __noinline__
namespace rtb {
RTB_DEV float4 ld4(const void* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// one 256-bit load (sm_100: LDG.E.256) of a 32-byte-aligned record: half the load instructions and L1 requests of 2 x 128 bit
struct F8 {
    float4 lo, hi;
};
RTB_DEV F8 ld8(const void* p) {
    F8 v;
    asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=f"(v.lo.x), "=f"(v.lo.y), "=f"(v.lo.z), "=f"(v.lo.w), "=f"(v.hi.x), "=f"(v.hi.y), "=f"(v.hi.z), "=f"(v.hi.w)
        : "l"(p));
    return v;
}
RTB_DEV uint32_t mulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
RTB_DEV float u32_to_unit(uint32_t x) { return __uint2float_rz(x) * 2.3283064365386963e-10f; }
// sin / cos of 2 pi x for x in [0, 1): the hardware approximations (MUFU.SIN / MUFU.COS, abs. error 2^-21.4 on [-pi, pi])
// of the angle shifted into [-pi, pi), negated back.  Explicit intrinsics: the library is built WITHOUT --use_fast_math
// (build.py), so that the libm names elsewhere (the checker's and the marble's sinf, acosf, atan2f) stay accurate.
RTB_DEV void sincos_2pi(float x, float* s, float* c) {
    float sn, cs;
    __sincosf(fmaf(x, 6.2831853071795865f, -3.1415926535897932f), &sn, &cs);
    *s = -sn, *c = -cs;
}
RTB_DEV float fast_cbrt(float x) { return __powf(x, 0.33333334f); }
RTB_DEV float sin_small(float x) { return __sinf(x); }  // |x| <= pi: MUFU.SIN, abs. error 2^-21.4
RTB_DEV float fast_log(float x) { return __logf(x); }
RTB_DEV float as_float(uint32_t u) { return __uint_as_float(u); }
RTB_DEV uint32_t as_uint(float f) { return __float_as_uint(f); }
RTB_DEV void image_fetch(const DImage& im, int i, int j, float rgb[3]) {
    uchar4 px = tex2D<uchar4>((cudaTextureObject_t)im.tex, (float)i + 0.5f, (float)j + 0.5f);
    rgb[0] = (float)px.x / 255.0f, rgb[1] = (float)px.y / 255.0f, rgb[2] = (float)px.z / 255.0f;
}
}  // namespace rtb
#else
#include <string.h>
#define RTB_DEV inline
#define RTB_DEV_NOINLINE inline
namespace rtb {
struct float4 {
    float x, y, z, w;
};
inline float4 ld4(const void* p) {
    float4 v;
    memcpy(&v, p, 16);
    return v;
}
struct F8 {
    float4 lo, hi;
};
inline F8 ld8(const void* p) {
    F8 v;
    memcpy(&v, p, 32);
    return v;
}
inline uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
inline float u32_to_unit(uint32_t x) {  // == __uint2float_rz(x) * 2^-32: keep the 24 leading significant bits
    int drop = x ? 8 - __builtin_clz(x) : 0;
    if (drop > 0) x = (x >> drop) << drop;
    return (float)x * 2.3283064365386963e-10f;
}
inline void sincos_2pi(float x, float* s, float* c) {
    *s = sinf(6.283185307179586f * x), *c = cosf(6.283185307179586f * x);
}
inline float fast_cbrt(float x) { return cbrtf(x); }
inline float sin_small(float x) { return sinf(x); }
inline float fast_log(float x) { return logf(x); }
inline float as_float(uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
}
inline uint32_t as_uint(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
inline void image_fetch(const DImage& im, int i, int j, float rgb[3]) {
    const uint8_t* px = (const uint8_t*)(uintptr_t)im.tex + 4 * ((size_t)j * im.width + i);
    rgb[0] = (float)px[0] / 255.0f, rgb[1] = (float)px[1] / 255.0f, rgb[2] = (float)px[2] / 255.0f;
}
}  // namespace rtb
#endif

namespace rtb {

#ifndef RTB_USE_FFMA2
#define RTB_USE_FFMA2 1
#endif
#define RTB_INF as_float(0x7f800000u)
#define RTB_T_MIN 0.001f  // raytrace.rs:90, in units of the (unnormalised) direction

// ------------------------------------------------------------------ small vector type
struct V3 {
    float x, y, z;
};
RTB_DEV V3 v3(float x, float y, float z) { return V3{x, y, z}; }
RTB_DEV V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
RTB_DEV V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
RTB_DEV V3 operator-(V3 a) { return V3{-a.x, -a.y, -a.z}; }
RTB_DEV V3 operator*(V3 a, V3 b) { return V3{a.x * b.x, a.y * b.y, a.z * b.z}; }
RTB_DEV V3 operator*(float s, V3 a) { return V3{a.x * s, a.y * s, a.z * s}; }
RTB_DEV V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
RTB_DEV float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
RTB_DEV float comp(V3 a, int k) { return k == 0 ? a.x : (k == 1 ? a.y : a.z); }
RTB_DEV V3 normalize(V3 a) {
    float inv = 1.0f / sqrtf(dot(a, a));
    return a * inv;
}
RTB_DEV V3 mul33(const float* m, V3 v) {  // row-major 3x3 times vector
    return V3{m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z};
}
RTB_DEV V3 mul33t(const float* m, V3 v) {  // transpose(m) times vector
    return V3{m[0] * v.x + m[3] * v.y + m[6] * v.z, m[1] * v.x + m[4] * v.y + m[7] * v.z, m[2] * v.x + m[5] * v.y + m[8] * v.z};
}

struct Ray {
    V3 o, d;
};

// ------------------------------------------------------------------ Philox4x32-10 (Salmon et al., SC'11)
// Out of line on the device: three call sites per path segment (camera, media, scatter) share one copy of the ten
// rounds AND of the conversion to uniforms, which keeps the instruction footprint of the shade stage inside the
// instruction cache.
struct U4 {
    uint32_t x, y, z, w;
};
struct F4 {
    float x, y, z, w;
};
RTB_DEV void philox_rounds(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
        uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
        k0 += W0, k1 += W1;
    }
}
// the raw block (known-answer tests)
RTB_DEV void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    philox_rounds(c0, c1, c2, c3, k0, k1);
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}
// the block as four uniforms in [0, 1)
RTB_DEV_NOINLINE F4 philox_uniforms(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    philox_rounds(c0, c1, c2, c3, k0, k1);
    return F4{u32_to_unit(c0), u32_to_unit(c1), u32_to_unit(c2), u32_to_unit(c3)};
}

// one stream per camera path: counter = (pixel, sample, draw, tag), key = seed
struct PathRng {
    uint32_t pixel, sample, draw, k0, k1;
};
#define RTB_PHILOX_TAG 0x52544232u
// block `block` of draw g.draw: four uniforms.  Block 0 is what rng_next4 returns; further blocks serve the media
// beyond the fourth (sample_media).
RTB_DEV void rng_block(const PathRng& g, uint32_t block, float u[4]) {
    const F4 r = philox_uniforms(g.pixel, g.sample, g.draw, RTB_PHILOX_TAG + block, g.k0, g.k1);
    u[0] = r.x, u[1] = r.y, u[2] = r.z, u[3] = r.w;
}
RTB_DEV void rng_next4(PathRng& g, float u[4]) {
    rng_block(g, 0u, u);
    g.draw += 1;
}

// Uniform point inside the unit ball, drawn directly instead of by the rejection loop of
// Vec3::random_in_unit_sphere (vec.rs:23-30): same distribution, fixed cost.
RTB_DEV V3 sample_unit_ball(float u0, float u1, float u2) {
    float z = 1.0f - 2.0f * u0;
    float rxy = sqrtf(fmaxf(0.0f, 1.0f - z * z));
    float s, c;
    sincos_2pi(u1, &s, &c);
    float r = fast_cbrt(u2);
    return V3{r * rxy * c, r * rxy * s, r * z};
}

// ------------------------------------------------------------------ camera (camera.rs:40-48, raytrace.rs:191-192)
#define WF_TIME_SHIFT 19
#define WF_TIME_MASK 0xFFF80000u
RTB_DEV float time_of_flags(uint32_t flags) { return (float)(flags >> WF_TIME_SHIFT) * (1.0f / 8191.0f); }
RTB_DEV uint32_t flags_of_time(float time) { return (uint32_t)(fminf(fmaxf(time, 0.0f), 1.0f) * 8191.0f + 0.5f) << WF_TIME_SHIFT; }
// EXTENSION: the ray time of camera path (pixel, sample), uniform in the shutter interval, as the upper flag bits; drawn from
// block 1 of the path's draw 0 (block 0 is the pixel jitter and the lens sample), only when the camera has a shutter
RTB_DEV uint32_t camera_time_flags(const DCamera& cam, const PathRng& g0) {
    if (!(cam.time1 > cam.time0)) return flags_of_time(cam.time0);
    float ut[4];
    rng_block(g0, 1u, ut);
    return flags_of_time(cam.time0 + ut[0] * (cam.time1 - cam.time0));
}

RTB_DEV Ray generate_camera_ray(const DCamera& cam, const DRenderParams& P, int px, int py, const float u[4]) {
    float s = ((float)px + u[0]) * P.inv_wm1;
    float t = ((float)py + u[1]) * P.inv_hm1;
    V3 off = v3(0.f, 0.f, 0.f);
    if (cam.lens_radius > 0.0f) {  // random_in_unit_disk (vec.rs:45-52) without the rejection loop
        float r = cam.lens_radius * sqrtf(u[2]);
        float sn, cs;
        sincos_2pi(u[3], &sn, &cs);
        float dx = r * cs, dy = r * sn;
        off = v3(cam.u[0] * dx + cam.v[0] * dy, cam.u[1] * dx + cam.v[1] * dy, cam.u[2] * dx + cam.v[2] * dy);
    }
    Ray r;
    r.o = v3(cam.origin[0], cam.origin[1], cam.origin[2]) + off;
    r.d = v3(cam.lower_left[0] + s * cam.horizontal[0] + t * cam.vertical[0], cam.lower_left[1] + s * cam.horizontal[1] + t * cam.vertical[1],
             cam.lower_left[2] + s * cam.horizontal[2] + t * cam.vertical[2]) -
          off;
    return r;
}

// ------------------------------------------------------------------ primitives
struct PrimRec {  // a DPrim in registers
    float v0, v1, v2, v3, v4, v5;
    uint32_t meta;
    int32_t mat;
};
RTB_DEV PrimRec prim_from(const float4& a, const float4& b) {
    PrimRec r;
    r.v0 = a.x, r.v1 = a.y, r.v2 = a.z, r.v3 = a.w, r.v4 = b.x, r.v5 = b.y;
    r.meta = as_uint(b.z), r.mat = (int32_t)as_uint(b.w);
    return r;
}
RTB_DEV PrimRec load_prim(const DPrim* p) {  // an element of the 32-byte-aligned primitive array
    const F8 v = ld8(p);
    return prim_from(v.lo, v.hi);
}
// two 128-bit loads: records that are only 16-byte aligned (DMedium.boundary), and the out-of-line compound-boundary
// loop, where ptxas 12.9 crashes on the 256-bit form
RTB_DEV PrimRec load_prim16(const DPrim* p) { return prim_from(ld4(p), ld4(reinterpret_cast<const char*>(p) + 16)); }
RTB_DEV int prim_instance(const PrimRec& p) { return (int)((p.meta >> PRIM_INST_SHIFT) & PRIM_INST_MASK); }

// EXTENSION (RT_NODE_MOVING_SPHERE; the reference has no ray time): a path carries ONE time for all its segments, quantised
// to 13 bits in the upper bits of its flags word; a moving sphere is its record with the centre advanced to that time.
template <class SV>
RTB_DEV void apply_motion(const SV& S, PrimRec& p, float time) {
    if ((SV::feat & F_MOVING) && (p.meta & PRIM_MOVING)) {
        const float4 dc = ld4(S.moving + 4 * as_uint(p.v4));
        p.v0 = fmaf(time, dc.x, p.v0), p.v1 = fmaf(time, dc.y, p.v1), p.v2 = fmaf(time, dc.z, p.v2);
    }
}

// Sphere::hit (shapes.rs:57-82).  `from_surface`: the ray starts on this very sphere, so one root is
// analytically zero (the reference rejects it through t_min) and the other is -2*half_b/a.
// f32 loses the quadratic's constant term c = |oc|^2 - r^2 only when the origin sits close to the surface of a
// large sphere (|c| << r^2); those cases (the r = 1000 ground of `random` seen from just above it) take the f64 path.
RTB_DEV bool sphere_needs_f64(const PrimRec& p, float c) { return (p.meta & PRIM_BIG) && fabsf(c) < 0.05f * p.v3 * p.v3; }

struct Roots {
    float t0, t1;
    int real;
};
// out of line: rare (only next to the surface of an |r| >= 100 sphere) and large (f64 divide and square root)
RTB_DEV_NOINLINE Roots sphere_roots_f64(double cx, double cy, double cz, double radius, float ox, float oy, float oz, float ddx, float ddy, float ddz) {
    double ocx = (double)ox - cx, ocy = (double)oy - cy, ocz = (double)oz - cz;
    double dx = ddx, dy = ddy, dz = ddz;
    double a = dx * dx + dy * dy + dz * dz;
    double hb = ocx * dx + ocy * dy + ocz * dz;
    double c = ocx * ocx + ocy * ocy + ocz * ocz - radius * radius;
    double disc = hb * hb - a * c;
    Roots out;
    out.real = !(disc < 0.0);
#ifdef RTB_HOST_EMULATION
    double sq = sqrt(out.real ? disc : 0.0);
    out.t0 = (float)((-hb - sq) / a), out.t1 = (float)((-hb + sq) / a);
#else
    // 1/a and sqrt(disc) by two Newton steps from f32 seeds (relative error < 1e-12; the roots are narrowed to f32 anyway)
    // instead of the IEEE division and square root, whose ~250 instructions of slow paths the instruction cache pays for
    double ra = (double)(1.0f / (float)a);
    ra = ra * (2.0 - a * ra), ra = ra * (2.0 - a * ra);  // 2^-22 -> 2^-44 -> 2^-88
    double sq = 0.0;
    if (out.real && disc > 1e-30) {
        double y = (double)rsqrtf((float)disc);
        y = y * (1.5 - 0.5 * disc * y * y), y = y * (1.5 - 0.5 * disc * y * y);
        sq = disc * y;
    }
    out.t0 = (float)((-hb - sq) * ra), out.t1 = (float)((-hb + sq) * ra);
#endif
    return out;
}

// both roots of the sphere quadratic, t0 <= t1 (shapes.rs:57-68); false when the discriminant is negative
template <class SV>
RTB_DEV bool sphere_roots(const SV& S, const PrimRec& p, const Ray& r, float& t0, float& t1) {
    V3 oc = r.o - v3(p.v0, p.v1, p.v2);
    float a = dot(r.d, r.d), hb = dot(oc, r.d), inv_a = 1.0f / a;
    float c = dot(oc, oc) - p.v3 * p.v3;
    if ((SV::feat & F_BIG) && sphere_needs_f64(p, c)) {
        const DBigSphere& b = S.big[as_uint(p.v4)];
        Roots q = sphere_roots_f64(b.c[0], b.c[1], b.c[2], b.r, r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z);
        t0 = q.t0, t1 = q.t1;
        return q.real != 0;
    }
    // discriminant from the perpendicular offset |oc - (hb/a) d|^2: no cancellation for distant origins
    V3 l = oc - (hb * inv_a) * r.d;
    float disc_a = p.v3 * p.v3 - dot(l, l);
    if (disc_a < 0.0f) return false;
    float sq = sqrtf(a * disc_a);
    float q = -(hb + copysignf(sq, hb));
    float ta = q * inv_a, tb = c / q;
    t0 = fminf(ta, tb), t1 = fmaxf(ta, tb);
    return true;
}

// Sphere::hit (shapes.rs:57-82).  `from_surface`: the ray starts on this very sphere, so one root is
// analytically zero (the reference rejects it through t_min) and the other is -2*half_b/a.
template <class SV>
RTB_DEV bool hit_sphere(const SV& S, const PrimRec& p, const Ray& r, float tmin, float tmax, bool from_surface, float& t_out) {
    float t0, t1;
    if (from_surface) {
        V3 oc = r.o - v3(p.v0, p.v1, p.v2);
        t0 = t1 = -2.0f * dot(oc, r.d) / dot(r.d, r.d);
    } else if (!sphere_roots(S, p, r, t0, t1)) {
        return false;
    }
    if (t0 >= tmin && t0 <= tmax) {
        t_out = t0;
        return true;
    }
    if (t1 >= tmin && t1 <= tmax) {
        t_out = t1;
        return true;
    }
    return false;
}

// both crossings of a sphere boundary over (-inf, +inf): what ConstantMedium asks of its boundary
template <class SV>
RTB_DEV bool sphere_interval(const SV& S, const PrimRec& p, const Ray& r, float& t0, float& t1) {
    if (!sphere_roots(S, p, r, t0, t1)) return false;
    return t0 == t0 && t1 == t1;
}

template <class SV>
RTB_DEV Ray to_object_space(const SV& S, int inst, const Ray& r) {
    if (inst == 0) return r;
    const DInstance& I = S.inst[inst - 1];
    Ray o;
    o.o = mul33t(I.rot, r.o - v3(I.trans[0], I.trans[1], I.trans[2]));
    o.d = mul33t(I.rot, r.d);
    return o;
}

// slab crossings of an object-space box; `origin_face` (axis | side << 2, or -1) pins the plane the ray
// starts on to t = 0 exactly, which is what f64 gives the reference for a ray leaving that face.
// One axis of it.  Scalars on purpose: with lo[3] / hi[3] arrays the compiler turned the pinning test into dynamically
// indexed loads and kept the arrays in LOCAL memory — 4 stores and 6 loads per box test in the hottest leaf path.
RTB_DEV void box_axis(int k, float lo, float hi, float o, float d, int pin, int side, float& t_enter, float& t_exit, int& face_enter, int& face_exit) {
    float inv = 1.0f / d;
    float a = lo - o, b = hi - o;
    if (pin == k) {
        if (side) b = 0.0f;
        else a = 0.0f;
        if (lo == hi) a = b = 0.0f;  // a rect: both "sides" are the one plane
    }
    float ta = a * inv, tb = b * inv;
    float tn = fminf(ta, tb), tf = fmaxf(ta, tb);  // fminf/fmaxf drop the NaN of 0 * inf
    bool neg = d < 0.0f;
    if (tn > t_enter) t_enter = tn, face_enter = k | ((neg ? 1 : 0) << 2);
    if (tf < t_exit) t_exit = tf, face_exit = k | ((neg ? 0 : 1) << 2);
}
RTB_DEV bool box_slabs(const PrimRec& p, const Ray& r, int origin_face, float& t_enter, float& t_exit, int& face_enter, int& face_exit) {
    t_enter = -RTB_INF, t_exit = RTB_INF;
    face_enter = 0, face_exit = 0;
    const int pin = origin_face >= 0 ? (origin_face & 3) : -1, side = origin_face >> 2;
    box_axis(0, p.v0, p.v3, r.o.x, r.d.x, pin, side, t_enter, t_exit, face_enter, face_exit);
    box_axis(1, p.v1, p.v4, r.o.y, r.d.y, pin, side, t_enter, t_exit, face_enter, face_exit);
    box_axis(2, p.v2, p.v5, r.o.z, r.d.z, pin, side, t_enter, t_exit, face_enter, face_exit);
    return t_enter <= t_exit;
}

// AARect::hit / Block::hit (aarects.rs:45-64, shapes.rs:188-191): closest side with t in [tmin, tmax]
template <class SV>
RTB_DEV bool hit_box(const SV& S, const PrimRec& p, const Ray& r_world, float tmin, float tmax, int origin_face, float& t_out, int& face_out) {
    Ray r = (SV::feat & F_INSTBOX) ? to_object_space(S, prim_instance(p), r_world) : r_world;
    float te, tx;
    int fe, fx;
    if (!box_slabs(p, r, origin_face, te, tx, fe, fx)) return false;
    int rect = (int)((p.meta >> PRIM_RECT_SHIFT) & PRIM_RECT_MASK);
    if (rect) {  // a flat box: both crossings are the plane; report the plane's own axis
        int k = rect - 1;
        float dk = comp(r.d, k);
        fe = fx = k | ((dk < 0.0f ? 1 : 0) << 2);
    }
    if (te >= tmin && te <= tmax) {
        t_out = te, face_out = fe;
        return true;
    }
    if (tx >= tmin && tx <= tmax) {
        t_out = tx, face_out = fx;
        return true;
    }
    return false;
}

template <class SV>
RTB_DEV bool hit_prim(const SV& S, const PrimRec& p, const Ray& r, float tmin, float tmax, bool is_origin, int origin_face, float& t, int& face) {
    if (!(SV::feat & F_BOX) || ((SV::feat & F_SPHERE) && (p.meta & PRIM_KIND_MASK) == PRIM_SPHERE)) {
        face = 0;
        return hit_sphere(S, p, r, tmin, tmax, is_origin, t);
    }
    return hit_box(S, p, r, tmin, tmax, is_origin ? origin_face : -1, t, face);
}

// ------------------------------------------------------------------ BVH traversal
// Per-ray constants of the node test.  The slab distances are evaluated as fma(n, inv, -o*inv): 6 FFMA per box instead
// of 6 FADD + 6 FMUL.  That form rounds o*inv before the subtraction, so a crossing carries an absolute error of about
// ulp(o*inv); `pad` (4 ulp of the largest |o*inv|) widens the far side by that much, which keeps the test conservative:
// a box the exact slabs would keep is never culled (leaf primitives are tested exactly, with the ray itself).
// Zero direction components are replaced by +-2^-80 (as in Aila & Laine's kernels) so that inv stays finite.
struct NodeRay {
    V3 inv, noi;  // 1/d and -o/d
    float pad;
};
RTB_DEV NodeRay node_ray(const Ray& r) {
    const float tiny = 8.271806e-25f;  // 2^-80
    NodeRay n;
    n.inv = v3(1.0f / (fabsf(r.d.x) > tiny ? r.d.x : copysignf(tiny, r.d.x)), 1.0f / (fabsf(r.d.y) > tiny ? r.d.y : copysignf(tiny, r.d.y)),
               1.0f / (fabsf(r.d.z) > tiny ? r.d.z : copysignf(tiny, r.d.z)));
    n.noi = v3(-r.o.x * n.inv.x, -r.o.y * n.inv.y, -r.o.z * n.inv.z);
    n.pad = 4.7683716e-7f * fmaxf(fmaxf(fabsf(n.noi.x), fabsf(n.noi.y)), fabsf(n.noi.z));  // 2^-21
    return n;
}
RTB_DEV bool slab_node(const float4& n0, const float4& n1, const NodeRay& q, float tmin, float tmax, float& tn_out) {
#if defined(__CUDA_ARCH__) && !defined(RTB_HOST_EMULATION) && RTB_USE_FFMA2
    // sm_100 packed FP32: one FFMA2 issues the x and y slabs of a box corner together (same roundings as two FFMA)
    const float2 ixy = make_float2(q.inv.x, q.inv.y), nxy = make_float2(q.noi.x, q.noi.y);
    const float2 a2 = __ffma2_rn(make_float2(n0.x, n0.y), ixy, nxy), b2 = __ffma2_rn(make_float2(n1.x, n1.y), ixy, nxy);
    const float ax = a2.x, ay = a2.y, bx = b2.x, by = b2.y;
#else
    float ax = fmaf(n0.x, q.inv.x, q.noi.x), bx = fmaf(n1.x, q.inv.x, q.noi.x);
    float ay = fmaf(n0.y, q.inv.y, q.noi.y), by = fmaf(n1.y, q.inv.y, q.noi.y);
#endif
    float az = fmaf(n0.z, q.inv.z, q.noi.z), bz = fmaf(n1.z, q.inv.z, q.noi.z);
    float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), tmin));
    float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), tmax));
    tn_out = tn;
    return tn <= fmaf(tf, 1.0000004f, q.pad);  // conservative: relative slack for the roundings of t, `pad` for those of o*inv
}

// Traversal stack entry: a node link and the entry distance of its box.  A popped entry whose box starts beyond the
// closest hit found since it was pushed is dropped without fetching the node (same conservative bound as slab_node).
#define RTB_TRAVERSAL_DONE ((int)0x80000000)
struct alignas(8) StackEntry {
    int node;
    float tn;
};
RTB_DEV int stack_pop(const StackEntry* stack, int& sp, float t_best, float pad) {
    const float limit = fmaf(t_best, 1.0000004f, pad);
    while (sp > 0) {
        const StackEntry e = stack[--sp];
        if (e.tn <= limit) return e.node;
    }
    return RTB_TRAVERSAL_DONE;
}

// Closest surface hit with t in [tmin, +inf): replaces HittableList::hit + BHV::hit + the shapes.
// origin_prim/origin_face identify the primitive the ray starts on (-1 for camera and medium rays).
template <class SV>
RTB_DEV void closest_hit(const SV& S, const Ray& r, float tmin, float tmax, int origin_prim, int origin_face, float& t_best, int& prim_best,
                         int& face_best, float time = 0.0f) {
    t_best = tmax, prim_best = -1, face_best = 0;
    if (S.n_prims == 0) return;
    const NodeRay nr = node_ray(r);
    StackEntry stack[RTB_BVH_STACK];
    int sp = 0;
    int cur = (int)as_uint(ld4(S.nodes).w);  // link of the root (its own box is never tested)
    while (cur != RTB_TRAVERSAL_DONE) {
        if (cur < 0) {
            int v = ~cur;
            int first = v & 0xFFFFFF, count = v >> 24;
            for (int i = first; i < first + count; ++i) {
                PrimRec p = load_prim(S.prims + i);
                apply_motion(S, p, time);
                float t;
                int face;
                if (hit_prim(S, p, r, tmin, t_best, i == origin_prim, origin_face, t, face)) t_best = t, prim_best = i, face_best = face;
            }
            cur = stack_pop(stack, sp, t_best, nr.pad);
        } else {
            const char* base = reinterpret_cast<const char*>(S.nodes + cur);
            const F8 ln = ld8(base), rn = ld8(base + 32);
            const float4 l0 = ln.lo, l1 = ln.hi, r0 = rn.lo, r1 = rn.hi;
            float tl, tr;
            bool hl = slab_node(l0, l1, nr, tmin, t_best, tl);
            bool hr = slab_node(r0, r1, nr, tmin, t_best, tr);
            int ll = (int)as_uint(l0.w), lr = (int)as_uint(r0.w);
            if (hl && hr) {
                bool left_first = tl <= tr;
                stack[sp].node = left_first ? lr : ll, stack[sp].tn = left_first ? tr : tl;
                sp += 1;
                cur = left_first ? ll : lr;
            } else if (hl) {
                cur = ll;
            } else if (hr) {
                cur = lr;
            } else {
                cur = stack_pop(stack, sp, t_best, nr.pad);
            }
        }
    }
}

// ------------------------------------------------------------------ 4-wide BVH traversal (DNode4, rt_types.h)
// One step fetches a 128-byte node (seven 128-bit loads) and tests its four child boxes with the same conservative
// FMA-form slabs as slab_node.  Every child yields ONE 32-bit key: (bits(entry distance) & 0xFFFF0000) | 16-bit link,
// or RTB_KEY_MISS.  Entry distances are >= t_min > 0, so keys order like distances (to bf16 resolution, rounded
// down = conservative): a five-exchange network on the keys sorts the children, the nearest becomes the cursor and the
// others are pushed farthest first — as 4-byte stack entries that still carry the distance for the pop-time cull.
#define RTB_KEY_MISS 0xFFFFFFFFu
RTB_DEV uint32_t child_key(const float4& ch, float cz, float hz, uint32_t link, const NodeRay& q, float tmin, float tmax) {
    // slab interval of an axis = t_centre -+ half * |1/d|: multiply-adds only (FMA pipe), no per-axis min/max (ALU pipe)
#if defined(__CUDA_ARCH__) && !defined(RTB_HOST_EMULATION) && RTB_USE_FFMA2
    const float2 c2 = __ffma2_rn(make_float2(ch.x, ch.y), make_float2(q.inv.x, q.inv.y), make_float2(q.noi.x, q.noi.y));
    const float tcx = c2.x, tcy = c2.y;
#else
    const float tcx = fmaf(ch.x, q.inv.x, q.noi.x), tcy = fmaf(ch.y, q.inv.y, q.noi.y);
#endif
    const float tcz = fmaf(cz, q.inv.z, q.noi.z);
    const float ax = fabsf(q.inv.x), ay = fabsf(q.inv.y), az = fabsf(q.inv.z);
    const float nx = fmaf(-ch.z, ax, tcx), ny = fmaf(-ch.w, ay, tcy), nz = fmaf(-hz, az, tcz);
    const float fx = fmaf(ch.z, ax, tcx), fy = fmaf(ch.w, ay, tcy), fz = fmaf(hz, az, tcz);
    float tn = fmaxf(fmaxf(nx, ny), fmaxf(nz, tmin));
    float tf = fminf(fminf(fx, fy), fminf(fz, tmax));
    bool hit = tn <= fmaf(tf, 1.0000004f, q.pad);
    return hit ? ((as_uint(tn) & 0xFFFF0000u) | link) : RTB_KEY_MISS;  // an empty slot's link is all ones: MISS either way
}
RTB_DEV void key_exchange(uint32_t& a, uint32_t& b) {
    const uint32_t lo = a < b ? a : b, hi = a < b ? b : a;
    a = lo, b = hi;
}
// a DNode4 in registers
struct Node4Regs {
    float4 c0, c1, c2, c3, lz, hz, lk;
};
RTB_DEV Node4Regs node4_fetch(const DNode4* nodes4, uint32_t node) {
    const char* base = reinterpret_cast<const char*>(nodes4 + node);
    const F8 a = ld8(base), b = ld8(base + 32), c = ld8(base + 64), d = ld8(base + 96);  // 128-byte aligned
    Node4Regs n;
    n.c0 = a.lo, n.c1 = a.hi, n.c2 = b.lo, n.c3 = b.hi, n.lz = c.lo, n.hz = c.hi, n.lk = d.lo;
    return n;
}
// the four child keys of a node, ascending (misses last)
RTB_DEV void node4_sorted_keys(const Node4Regs& n, const NodeRay& q, float tmin, float tmax, uint32_t& k0, uint32_t& k1, uint32_t& k2, uint32_t& k3) {
    k0 = child_key(n.c0, n.lz.x, n.hz.x, as_uint(n.lk.x), q, tmin, tmax);
    k1 = child_key(n.c1, n.lz.y, n.hz.y, as_uint(n.lk.y), q, tmin, tmax);
    k2 = child_key(n.c2, n.lz.z, n.hz.z, as_uint(n.lk.z), q, tmin, tmax);
    k3 = child_key(n.c3, n.lz.w, n.hz.w, as_uint(n.lk.w), q, tmin, tmax);
    key_exchange(k0, k1), key_exchange(k2, k3), key_exchange(k0, k2), key_exchange(k1, k3), key_exchange(k1, k2);
}
// largest key that can still matter once the closest hit is t_best (same conservative bound as slab_node)
RTB_DEV uint32_t key_limit(float t_best, float pad) { return as_uint(fmaf(t_best, 1.0000004f, pad)) | 0xFFFFu; }

RTB_DEV uint32_t stack4_pop(const uint32_t* stack, int& sp, float t_best, float pad) {
    const uint32_t limit = key_limit(t_best, pad);
    while (sp > 0) {
        const uint32_t k = stack[--sp];
        if (k <= limit) return k & 0xFFFFu;
    }
    return RTB_LINK4_DONE;
}

// closest_hit over the 4-wide tree (t_min must be > 0: keys compare as unsigned integers)
template <class SV>
RTB_DEV void closest_hit4(const SV& S, const Ray& r, float tmin, float tmax, int origin_prim, int origin_face, float& t_best, int& prim_best,
                          int& face_best, float time = 0.0f) {
    t_best = tmax, prim_best = -1, face_best = 0;
    if (S.n_prims == 0) return;
    const NodeRay nr = node_ray(r);
    uint32_t stack[RTB_WIDE_STACK];
    int sp = 0;
    uint32_t cur = 0u;  // the root node
    while (cur != RTB_LINK4_DONE) {
        if (cur & RTB_LINK4_LEAF) {
            const int i = (int)(cur & 0x7FFFu);
            PrimRec p = load_prim(S.prims + i);
            apply_motion(S, p, time);
            float t;
            int face;
            if (hit_prim(S, p, r, tmin, t_best, i == origin_prim, origin_face, t, face)) t_best = t, prim_best = i, face_best = face;
            cur = stack4_pop(stack, sp, t_best, nr.pad);
        } else {
            uint32_t k0, k1, k2, k3;
            node4_sorted_keys(node4_fetch(S.nodes4, cur), nr, tmin, t_best, k0, k1, k2, k3);
            if (k0 == RTB_KEY_MISS) {
                cur = stack4_pop(stack, sp, t_best, nr.pad);
            } else {
                if (k3 != RTB_KEY_MISS) stack[sp++] = k3;
                if (k2 != RTB_KEY_MISS) stack[sp++] = k2;
                if (k1 != RTB_KEY_MISS) stack[sp++] = k1;
                cur = k0 & 0xFFFFu;
            }
        }
    }
}

// brute force over a primitive range (test entry point; also cross-checks the BVH)
template <class SV>
RTB_DEV void closest_hit_linear(const SV& S, const Ray& r, float tmin, float tmax, float& t_best, int& prim_best, int& face_best, float time = 0.0f) {
    t_best = tmax, prim_best = -1, face_best = 0;
    for (int i = 0; i < S.n_prims; ++i) {
        PrimRec p = load_prim(S.prims + i);
        apply_motion(S, p, time);
        float t;
        int face;
        if (hit_prim(S, p, r, tmin, t_best, false, -1, t, face)) t_best = t, prim_best = i, face_best = face;
    }
}

// ------------------------------------------------------------------ media (volumes.rs:25-65)
// both crossings of one boundary primitive over (-inf, +inf), t0 <= t1 (a rect has one: t0 == t1)
template <class SV>
RTB_DEV bool boundary_crossings(const SV& S, const PrimRec& b, const Ray& r, float& t0, float& t1) {
    if (!(SV::feat & F_BOXMEDIA) || (b.meta & PRIM_KIND_MASK) == PRIM_SPHERE) return sphere_interval(S, b, r, t0, t1);
    Ray ro = to_object_space(S, prim_instance(b), r);
    int fe, fx;
    return box_slabs(b, ro, -1, t0, t1, fe, fx);
}
// A boundary made of several primitives (ConstantMedium<O: Hittable>, volumes.rs:7-11): h1 = the closest hit of the
// whole boundary over (-inf, inf), h2 = its closest hit from h1.t + 0.001 on (volumes.rs:27-34).  Every primitive
// answers a range query with its first crossing inside the range, the list with the smallest of those.
RTB_DEV_NOINLINE V3 compound_boundary(const DSceneView& S, int first, int count, float ox, float oy, float oz, float dx, float dy, float dz) {
    Ray r;
    r.o = v3(ox, oy, oz), r.d = v3(dx, dy, dz);
    float h1 = RTB_INF, h2 = RTB_INF;
    for (int i = first; i < first + count; ++i) {
        float t0, t1;
        if (boundary_crossings(S, load_prim16(S.media_prims + i), r, t0, t1)) h1 = fminf(h1, t0);
    }
    if (h1 < RTB_INF) {
        const float from = h1 + 0.001f;
        for (int i = first; i < first + count; ++i) {
            float t0, t1;
            if (!boundary_crossings(S, load_prim16(S.media_prims + i), r, t0, t1)) continue;
            const float t = t0 >= from ? t0 : t1;
            if (t >= from) h2 = fminf(h2, t);
        }
    }
    return v3(h1, h2, 0.f);
}

// deterministic part: the boundary interval clipped to [tmin, tmax]
RTB_DEV bool clip_interval(float te, float tx, float tmin, float tmax, float& t1, float& t2) {
    t1 = fmaxf(te, tmin), t2 = fminf(tx, tmax);
    if (t1 >= t2) return false;
    t1 = fmaxf(t1, 0.0f);
    return true;
}
// single-primitive boundary (every shipped world): entry and exit of that primitive
template <class SV>
RTB_DEV bool medium_interval(const SV& S, const PrimRec& b, const Ray& r, float tmin, float tmax, float& t1, float& t2) {
    float te, tx;
    if (!boundary_crossings(S, b, r, te, tx)) return false;
    if (!(tx >= te + 0.001f)) return false;  // second boundary.hit(h1.t + 0.001, inf) finds nothing
    return clip_interval(te, tx, tmin, tmax, t1, t2);
}
template <class SV>
RTB_DEV bool medium_interval_any(const SV& S, const DMedium* M, const Ray& r, float tmin, float tmax, float& t1, float& t2) {
    if (M->count <= 1) return medium_interval(S, load_prim16(&M->boundary), r, tmin, tmax, t1, t2);
    const V3 h = compound_boundary(S, M->first, M->count, r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z);
    if (!(h.y < RTB_INF)) return false;
    return clip_interval(h.x, h.y, tmin, tmax, t1, t2);
}

// free-flight sampling in every medium; keeps the closest event.  Medium m uses uniform m & 3 of Philox block
// (pixel, sample, draw, tag + (m >> 2)): scenes with up to four media draw exactly one block per segment.
// The general form — any number of media, boundaries of several primitives — is out of line: the kernels take it only
// for scenes that need it (DSceneView.media_general), so that the common case keeps its registers.
struct MediaEvent {
    float t;
    int medium;
};
RTB_DEV_NOINLINE MediaEvent sample_media_general(const DSceneView& S, float ox, float oy, float oz, float dx, float dy, float dz, float tmin, uint32_t pixel,
                                                 uint32_t sample, uint32_t draw, uint32_t k0, uint32_t k1, float t_best) {
    Ray r;
    r.o = v3(ox, oy, oz), r.d = v3(dx, dy, dz);
    PathRng rng;
    rng.pixel = pixel, rng.sample = sample, rng.draw = draw, rng.k0 = k0, rng.k1 = k1;
    MediaEvent ev;
    ev.t = t_best, ev.medium = -1;
    const float len = sqrtf(dot(r.d, r.d));
    float u[4] = {0.f, 0.f, 0.f, 0.f};
    for (int m = 0; m < S.n_media; ++m) {
        if ((m & 3) == 0) rng_block(rng, (uint32_t)(m >> 2), u);
        const DMedium* M = S.media + m;
        float t1, t2;
        if (!medium_interval_any(S, M, r, tmin, ev.t, t1, t2)) continue;
        const float um = (m & 3) == 0 ? u[0] : ((m & 3) == 1 ? u[1] : ((m & 3) == 2 ? u[2] : u[3]));
        const float dist = M->neg_inv_density * fast_log(um);
        if (dist > (t2 - t1) * len) continue;
        ev.t = t1 + dist / len, ev.medium = m;
    }
    return ev;
}
// MODE: MEDIA_FAST = the caller knows the scene is not "general" (no call site for the out-of-line form: a call in the
// persistent kernel's shade phase costs it 240 B of stack frame and 150 B of spills), MEDIA_GENERAL = it knows it is,
// MEDIA_ANY = decide here from the scene's flag.
enum { MEDIA_FAST = 0, MEDIA_GENERAL = 1, MEDIA_ANY = 2 };
template <int MODE = MEDIA_ANY, class SV = DSceneView>
RTB_DEV void sample_media(const SV& S, const Ray& r, float tmin, const PathRng& rng, float& t_best, int& medium_best) {
    if (MODE == MEDIA_GENERAL || (MODE == MEDIA_ANY && S.media_general)) {
        const MediaEvent ev = sample_media_general(S, r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z, tmin, rng.pixel, rng.sample, rng.draw, rng.k0, rng.k1, t_best);
        t_best = ev.t, medium_best = ev.medium;
        return;
    }
    medium_best = -1;
    float len = sqrtf(dot(r.d, r.d));
    float u[4];
    rng_block(rng, 0u, u);
    for (int m = 0; m < S.n_media; ++m) {  // <= 4 media, one primitive per boundary
        const DMedium* M = S.media + m;
        PrimRec b = load_prim16(&M->boundary);
        float4 tail = ld4(reinterpret_cast<const char*>(M) + 32);
        float t1, t2;
        if (!medium_interval(S, b, r, tmin, t_best, t1, t2)) continue;
        float inside = (t2 - t1) * len;
        const float um = m == 0 ? u[0] : (m == 1 ? u[1] : (m == 2 ? u[2] : u[3]));  // (u[m] would put the array in local memory)
        float dist = tail.x * fast_log(um);  // neg_inv_density * ln(U)
        if (dist > inside) continue;
        t_best = t1 + dist / len;
        medium_best = m;
    }
}

// ------------------------------------------------------------------ textures
struct UV {
    float u, v;
};
// out of line: only image-textured spheres need it, and acosf / atan2f are long
RTB_DEV_NOINLINE UV sphere_uv_v(float nx, float ny, float nz) {  // shapes.rs:44-55
    const float pi = 3.14159265358979f;
    float theta = acosf(fminf(fmaxf(-ny, -1.0f), 1.0f));
    float phi = atan2f(-nz, nx) + pi;
    return UV{phi / (2.0f * pi), theta / pi};
}
RTB_DEV void sphere_uv(V3 n, float& u, float& v) {
    UV r = sphere_uv_v(n.x, n.y, n.z);
    u = r.u, v = r.v;
}

RTB_DEV float perlin_noise(const float* vec, const unsigned short* perm, V3 p) {  // textures.rs:90-134
    float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    float u = p.x - fx, v = p.y - fy, w = p.z - fz;
    int i = (int)fx, j = (int)fy, k = (int)fz;
    float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
    float accum = 0.0f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                int idx = perm[(i + di) & 1023] ^ perm[1024 + ((j + dj) & 1023)] ^ perm[2048 + ((k + dk) & 1023)];
                float4 g = ld4(vec + 4 * idx);
                float wx = u - (float)di, wy = v - (float)dj, wz = w - (float)dk;
                float bi = di ? uu : 1.0f - uu, bj = dj ? vv : 1.0f - vv, bk = dk ? ww : 1.0f - ww;
                accum += bi * bj * bk * (wx * g.x + wy * g.y + wz * g.z);
            }
    return accum;
}

RTB_DEV float perlin_turbulence(const float* vec, const unsigned short* perm, V3 p) {  // textures.rs:76-88, depth 7
    float accum = 0.0f, weight = 1.0f;
    for (int i = 0; i < 7; ++i) {
        accum += weight * perlin_noise(vec, perm, p);
        weight *= 0.5f;
        p = 2.0f * p;
    }
    return fabsf(accum);
}

// A NoiseTexture::value the caller evaluates itself (the persistent kernel does it warp-cooperatively: the 56
// gradient terms of the 7-octave turbulence are spread over the lanes).  tex < 0: nothing pending.
struct NoiseReq {
    int tex;  // DTexture index of the NOISE leaf
    V3 p;     // the hit point (unscaled)
};

// Accurate sine for the two textures whose LOOK depends on it: the checker's sin(5x) at |5x| up to thousands of radians
// (the hardware sine alone loses the phase out there: its error grows with |x|) and the marble's phase.  Two-term
// Cody-Waite reduction to [-pi/2, pi/2] with FMAs (exact to the input's own rounding for |x| < 2^23), then the hardware
// sine where it is good to 2^-21.4 absolute: ~8 instructions instead of libm's ~100 (four inlined copies of which cost
// the persistent kernel 8 % through its instruction footprint; profiles/r2_fastmath_ab.txt).
RTB_DEV float sin_accurate(float x) {
    const float k = rintf(x * 0.318309886183790672f);
    float r = fmaf(k, -3.14159274101257324f, x);  // pi = 3.14159274101257324 - 8.74227765734758577e-8 - ...
    r = fmaf(k, 8.74227765734758577e-8f, r);
    const float s = sin_small(r);
    return ((int)k & 1) ? -s : s;
}

RTB_DEV float noise_value(const DTexture& T, V3 p, float turbulence) {  // NoiseTexture::value, textures.rs:163-166 — marble phase on z
    return 0.5f * (1.0f + sin_accurate(T.scale * p.z + 10.0f * turbulence));
}

// req == nullptr: evaluate everything here.  Otherwise a NOISE leaf is left pending in *req and white is returned.
template <class SV>
RTB_DEV V3 texture_leaf(const SV& S, int tex, float u, float v, V3 p, NoiseReq* req) {
    const DTexture& T = S.texs[tex];
    if ((SV::feat & F_NOISE) && T.kind == TEX_NOISE) {
        if (req) {
            req->tex = tex, req->p = p;
            return v3(1.f, 1.f, 1.f);
        }
        const float* vec = S.perlin_vec + (size_t)T.a * RTB_PERLIN_POINTS * 4;
        const unsigned short* perm = S.perlin_perm + (size_t)T.a * RTB_PERLIN_POINTS * 3;
        float g = noise_value(T, p, perlin_turbulence(vec, perm, T.scale * p));
        return v3(g, g, g);
    }
    if ((SV::feat & F_IMAGE) && T.kind == TEX_IMAGE) {  // image_texture.rs:16-28 — nearest texel, v flipped
        const DImage& im = S.images[T.a];
        u = fminf(fmaxf(u, 0.0f), 1.0f);
        v = fminf(fmaxf(1.0f - v, 0.0f), 1.0f);
        int i = (int)(u * (float)im.width), j = (int)(v * (float)im.height);
        i = i > im.width - 1 ? im.width - 1 : i;
        j = j > im.height - 1 ? im.height - 1 : j;
        float rgb[3];
        image_fetch(im, i, j, rgb);
        return v3(rgb[0], rgb[1], rgb[2]);
    }
    return v3(T.color[0], T.color[1], T.color[2]);
}

template <class SV>
RTB_DEV V3 texture_value(const SV& S, int tex, float u, float v, V3 p, NoiseReq* req = nullptr) {
    if ((SV::feat & F_CHECKER) && S.texs[tex].kind == TEX_CHECKER) {  // textures.rs:40-49; nested checkers see the same p, hence the same side
        const float sines = sin_accurate(5.0f * p.x) * sin_accurate(5.0f * p.y) * sin_accurate(5.0f * p.z);
        for (int level = 0; level < RTB_CHECKER_DEPTH && S.texs[tex].kind == TEX_CHECKER; ++level) tex = sines < 0.0f ? S.texs[tex].a : S.texs[tex].b;
    }
    return texture_leaf(S, tex, u, v, p, req);
}

template <class SV>
RTB_DEV bool texture_needs_uv(const SV& S, int tex) { return (SV::feat & F_IMAGE) && S.texs[tex].needs_uv != 0; }

// ------------------------------------------------------------------ hit attributes (hittable.rs:18-30 + transforms)
struct Surface {
    V3 p, n;
    float u, v;
    bool front;
};

template <class SV>
RTB_DEV void surface_at(const SV& S, const PrimRec& P, const Ray& r, float t, int face, bool want_uv, Surface& s) {
    const int inst = (SV::feat & F_INSTANCE) ? prim_instance(P) : 0;
    V3 ng;         // geometric normal in world space (the reference's "outward" one)
    V3 n_obj_out;  // outward normal in object space (for sphere uv)
    s.p = r.o + t * r.d;
    s.u = 0.0f, s.v = 0.0f;
    if (!(SV::feat & F_BOX) || ((SV::feat & F_SPHERE) && (P.meta & PRIM_KIND_MASK) == PRIM_SPHERE)) {
        float inv_r = 1.0f / P.v3;  // signed radius flips the normal (shapes.rs:78)
        ng = (s.p - v3(P.v0, P.v1, P.v2)) * inv_r;
        n_obj_out = inst ? mul33t(S.inst[inst - 1].rot, ng) : ng;
        if (want_uv) sphere_uv(n_obj_out, s.u, s.v);
    } else {
        int k = face & 3, side = face >> 2;
        V3 e = v3(k == 0 ? 1.0f : 0.0f, k == 1 ? 1.0f : 0.0f, k == 2 ? 1.0f : 0.0f);  // rects always report +axis
        float plane = side ? (k == 0 ? P.v3 : (k == 1 ? P.v4 : P.v5)) : (k == 0 ? P.v0 : (k == 1 ? P.v1 : P.v2));
        if (inst) {
            ng = mul33(S.inst[inst - 1].rot, e);
        } else {
            ng = e;
            if (k == 0) s.p.x = plane;  // the hit point lies on the plane exactly
            else if (k == 1) s.p.y = plane;
            else s.p.z = plane;
        }
        if (want_uv) {  // (a feature bit for "no box reads (u, v)" was tried: 56 instructions less and 32 B more spills, -3.5 %)
            Ray ro = to_object_space(S, inst, r);
            V3 po = ro.o + t * ro.d;
            int a0 = k == 0 ? 1 : 0, a1 = k == 2 ? 1 : 2;
            float lo0 = a0 == 0 ? P.v0 : P.v1, hi0 = a0 == 0 ? P.v3 : P.v4;
            float lo1 = a1 == 1 ? P.v1 : P.v2, hi1 = a1 == 1 ? P.v4 : P.v5;
            s.u = (comp(po, a0) - lo0) / (hi0 - lo0);
            s.v = (comp(po, a1) - lo1) / (hi1 - lo1);
        }
    }
    if (inst == 0) {
        s.front = dot(ng, r.d) < 0.0f;
        s.n = s.front ? ng : -ng;
    } else {
        const DInstance& I = S.inst[inst - 1];
        float d1 = dot(ng, mul33(I.m1, r.d));  // outermost wrapper's face-forward test
        float d2 = dot(ng, mul33(I.m2, r.d));  // the one below it
        s.n = d1 < 0.0f ? ng : -ng;
        // the normal handed up by the inner level is +ng if d2 < 0 else -ng; front_face = it already faced the ray
        s.front = (d2 < 0.0f) == (d1 < 0.0f);
    }
}

// ------------------------------------------------------------------ shading
struct PathState {
    Ray ray;
    V3 beta;          // product of attenuations so far (raytrace.rs:93)
    int origin_prim;  // primitive the ray starts on, -1 if none
    int origin_face;
    int depth;        // rays still allowed (raytrace.rs:87-89)
    float time;       // EXTENSION: the path's time in [0, 1] (moving spheres); 0 without a shutter
};

template <class SV>
RTB_DEV V3 background_color(const SV& S, const Ray& r) {  // raytrace.rs:29-35, :44-48
    if (S.bg_kind == 0) return v3(0.f, 0.f, 0.f);
    float t = 0.5f * (normalize(r.d).y + 1.0f);
    return v3((1.0f - t) * S.bg_bottom[0] + t * S.bg_top[0], (1.0f - t) * S.bg_bottom[1] + t * S.bg_top[1],
              (1.0f - t) * S.bg_bottom[2] + t * S.bg_top[2]);
}

template <class SV>
RTB_DEV V3 material_color(const SV& S, const DMaterial& M, const Surface& s, NoiseReq* req = nullptr) {
    if (M.tex < 0) return v3(M.albedo[0], M.albedo[1], M.albedo[2]);
    return texture_value(S, M.tex, s.u, s.v, s.p, req);
}

// Material::scatter / emit at a surface or medium event.  Returns true when the path goes on (ps updated);
// otherwise `radiance` is the terminal term (emission, or 0 for an absorbed metal reflection).
// With `req`, a noise texture is left pending: the caller multiplies ps.beta (alive) or radiance (emitter) by it.
template <class SV>
RTB_DEV bool scatter(const SV& S, const DMaterial& M, const Surface& s, const float u[4], PathState& ps, int prim, int face, V3& radiance,
                     NoiseReq* req = nullptr) {
    // Branch-light: what several material kinds need is computed once by every lane (the lanes of a warp shade
    // different materials side by side), the kinds then differ by a few selects.
    const int kind = M.kind;
    const V3 ball = sample_unit_ball(u[0], u[1], u[2]);  // Lambertian, fuzzy metal, isotropic
    const V3 ud = normalize(ps.ray.d);                   // metal, dielectric
    const float udn = dot(ud, s.n);
    const V3 refl = ud - (2.0f * udn) * s.n;             // reflect(), materials.rs:47-49
    const V3 color = material_color(S, M, s, req);       // albedo / texture value / emission
    V3 dir = ball, att = color;                          // MAT_ISOTROPIC, volumes.rs:77-83: raw in-ball direction
    bool scattered = true;
    if (kind == MAT_LAMBERTIAN) {  // materials.rs:25-34: normal + in-ball point flipped into the hemisphere
        V3 b = dot(s.n, ball) > 0.0f ? ball : -ball;
        dir = s.n + b;
        if (fabsf(dir.x) < 1e-8f && fabsf(dir.y) < 1e-8f && fabsf(dir.z) < 1e-8f) dir = s.n;
    } else if (kind == MAT_METAL) {  // materials.rs:51-61 (fuzz == 0 adds nothing)
        dir = refl + M.fuzz * ball;
        scattered = dot(dir, s.n) > 0.0f;  // otherwise scatter -> None, emit -> 0
    } else if (kind == MAT_DIELECTRIC) {  // materials.rs:88-106
        float ratio = s.front ? 1.0f / M.ior : M.ior;
        float cos_t = fminf(-udn, 1.0f);
        float sin_t = sqrtf(fmaxf(0.0f, 1.0f - cos_t * cos_t));
        float r0 = (1.0f - ratio) / (1.0f + ratio);
        r0 = r0 * r0;
        float x = 1.0f - cos_t;
        float x2 = x * x;
        float reflectance = r0 + (1.0f - r0) * (x * x2 * x2);
        V3 perp = ratio * (ud + cos_t * s.n);
        V3 par = -sqrtf(fabsf(1.0f - dot(perp, perp))) * s.n;
        dir = (ratio * sin_t > 1.0f || reflectance > u[3]) ? refl : perp + par;
        att = v3(1.f, 1.f, 1.f);
    } else if (kind == MAT_DIFFUSE_LIGHT) {  // materials.rs:119-127: emits from both faces, never scatters
        radiance = color;
        return false;
    }
    if (!scattered) {
        radiance = v3(0.f, 0.f, 0.f);
        return false;
    }
    ps.beta = ps.beta * att;
    ps.ray.o = s.p;
    ps.ray.d = dir;
    ps.origin_prim = prim;
    ps.origin_face = face;
    return true;
}

// Material::scatter / emit for the event the extend stage found: a medium event (volumes.rs:55-63: normal (1,0,0),
// front_face, u = v = 0) or a surface hit.  ONE scatter call site for both.
template <class SV>
RTB_DEV bool scatter_event(const SV& S, int medium, int prim, int face, float t, const float u[4], PathState& ps, V3& radiance, NoiseReq* req) {
    Surface sf;
    int mat_index;
    if ((SV::feat & F_MEDIA) && medium >= 0) {
        mat_index = (int)as_uint(ld4(reinterpret_cast<const char*>(S.media + medium) + 32).y);
        sf.p = ps.ray.o + t * ps.ray.d;
        sf.n = v3(1.f, 0.f, 0.f), sf.u = 0.f, sf.v = 0.f, sf.front = true;
        prim = -1, face = 0;
    } else {
        PrimRec Pr = load_prim(S.prims + prim);
        apply_motion(S, Pr, ps.time);
        mat_index = Pr.mat;
        int tex = (int)as_uint(ld4(S.mats + mat_index).y);
        bool want_uv = tex >= 0 && texture_needs_uv(S, tex);
        surface_at(S, Pr, ps.ray, t, face, want_uv, sf);
    }
    return scatter(S, S.mats[mat_index], sf, u, ps, prim, face, radiance, req);
}

// One path segment: nearest surface, media, then scatter.  Returns true while the path is alive; when it
// ends, `radiance` holds beta * terminal term.
template <class SV>
RTB_DEV bool extend_and_shade(const SV& S, PathState& ps, PathRng& rng, int segment, V3& radiance) {
    if (ps.depth <= 0) {  // depth exhausted: Color::ZERO (raytrace.rs:87-89)
        radiance = v3(0.f, 0.f, 0.f);
        return false;
    }
    ps.depth -= 1;
    // Media first: the free-flight event of ConstantMedium::hit (volumes.rs:44-53) does not depend on the surfaces,
    // only its acceptance does (event before the nearest surface), so the closest event is drawn up front and
    // bounds the surface search.  Philox draw indices are a function of the segment number k alone (camera = 0,
    // media = 1 + 2k, scatter = 2 + 2k), so the megakernel and the wavefront pipeline consume identical streams.
    float t = RTB_INF;
    int medium = -1;
    rng.draw = 1u + 2u * (uint32_t)segment;
    if ((SV::feat & F_MEDIA) && S.n_media > 0) {
        sample_media(S, ps.ray, RTB_T_MIN, rng, t, medium);
    }
    int prim, face;
    closest_hit(S, ps.ray, RTB_T_MIN, t, ps.origin_prim, ps.origin_face, t, prim, face, ps.time);
    if (prim >= 0) medium = -1;
    rng.draw = 2u + 2u * (uint32_t)segment;
    if (prim < 0 && medium < 0) {
        radiance = ps.beta * background_color(S, ps.ray);
        return false;
    }
    float us[4];
    rng_next4(rng, us);
    V3 term;
    bool alive = scatter_event(S, medium, prim, face, t, us, ps, term, nullptr);
    if (!alive) {
        radiance = ps.beta * term;
    } else if (ps.depth <= 0) {  // the next trace_internal call would return Color::ZERO at once
        radiance = v3(0.f, 0.f, 0.f);
        alive = false;
    }
    return alive;
}

// ------------------------------------------------------------------ accumulation in fixed point (AccumFx, rt_types.h)
// One radiance sample -> 2^-32 units, rounded to nearest.  Samples are >= 0 (albedos, emission and noise values are);
// NaN counts as 0 and a sample is capped at 2^20 so that a 64-bit sum holds 2^11 such extremes (2^31 ordinary ones).
RTB_DEV AccumFx radiance_fixed(float x) {
    x = x == x ? fminf(fmaxf(x, 0.0f), 1048576.0f) : 0.0f;
    return (AccumFx)fmaf(x, 4294967296.0f, 0.5f);
}

// EXTENSION: the square of one fixed-point sample q = radiance_fixed(x), exactly, in 2^-24 units of radiance^2
// (RT_MOMENT2_FIXED_ONE): (min(q, 2^44))^2 >> 40.  A sample above 4096 is capped in the square, so one sample adds at
// most 2^48 and a 64-bit sum holds 2^16 - 1 such extremes (about 2^40 ordinary ones).
RTB_DEV AccumFx moment2_fixed(AccumFx q) {
    q = q < (1ull << 44) ? q : (1ull << 44);
#if defined(__CUDACC__) && !defined(RTB_HOST_EMULATION)
    const AccumFx hi = __umul64hi(q, q);
#else
    const AccumFx hi = (AccumFx)(((unsigned __int128)q * q) >> 64);
#endif
    return (hi << 24) | ((q * q) >> 40);  // q^2 < 2^88: hi < 2^24
}

// to_rgb (raytrace.rs:59-68): gamma 2, clamp, x255.999, truncate.  Done in f64 so that, given the same sums, the
// bytes are the reference's.
RTB_DEV int32_t to_rgb_f64(double mean) {
    double x = sqrt(mean);
    x = x < 0.0 ? 0.0 : (x > 0.99999999 ? 0.99999999 : x);  // f64::clamp keeps NaN; `as i32` maps NaN to 0
    double y = 255.999 * x;
    return (y != y) ? 0 : (int32_t)y;
}

// EXTENSION: the stop rule of noise-threshold adaptive sampling (rt_render_adaptive) for one pixel that has received
// samples [0, n) of at most n_max, from its fixed-point sums S1 (radiance_fixed) and S2 (moment2_fixed) per channel:
//   mu = S1 2^-32 / n,  s^2 = max(0, (S2 2^-24 - n mu^2) / (n - 1)),  se = sqrt(s^2 / n),
//   e = se / (2 sqrt(max(mu, 2^-16)))   (the standard error carried through the gamma-2 tonemap),
// done when n == n_max or, for every channel, e <= threshold or mu - 3 se >= 1 (the channel saturates in to_rgb).
// f64 with every operation rounded on its own (no contraction), so that a restatement in numpy agrees on every pixel.
#if defined(__CUDACC__) && !defined(RTB_HOST_EMULATION)
#define RTB_DMUL __dmul_rn
#define RTB_DSUB __dsub_rn
#define RTB_DDIV __ddiv_rn
#define RTB_DSQRT __dsqrt_rn
#else
#define RTB_DMUL(a, b) ((double)(a) * (double)(b))
#define RTB_DSUB(a, b) ((double)(a) - (double)(b))
#define RTB_DDIV(a, b) ((double)(a) / (double)(b))
#define RTB_DSQRT(a) sqrt((double)(a))
#endif
RTB_DEV bool adaptive_pixel_done(uint32_t n, uint32_t n_max, const AccumFx s1[3], const AccumFx s2[3], double threshold) {
    if (n >= n_max) return true;
    const double dn = (double)n;
    for (int c = 0; c < 3; ++c) {
        const double mu = RTB_DDIV(RTB_DMUL((double)s1[c], 2.3283064365386963e-10), dn);
        const double m2 = RTB_DMUL((double)s2[c], 5.9604644775390625e-08);
        double var = RTB_DDIV(RTB_DSUB(m2, RTB_DMUL(dn, RTB_DMUL(mu, mu))), RTB_DSUB(dn, 1.0));
        var = var > 0.0 ? var : 0.0;
        const double se = RTB_DSQRT(RTB_DDIV(var, dn));
        const double e = RTB_DDIV(se, RTB_DMUL(2.0, RTB_DSQRT(mu > 1.52587890625e-05 ? mu : 1.52587890625e-05)));
        if (!(e <= threshold || RTB_DSUB(mu, RTB_DMUL(3.0, se)) >= 1.0)) return false;
    }
    return true;
}
#undef RTB_DMUL
#undef RTB_DSUB
#undef RTB_DDIV
#undef RTB_DSQRT

// ------------------------------------------------------------------ one work item = one pixel x a run of samples
// item -> (tile, lane): a warp covers an 8x4 pixel tile so that its 32 camera rays start coherent.
RTB_DEV bool item_to_pixel(const DRenderParams& P, long long item, int& px, int& py, int& chunk) {
    long long per_chunk = (long long)P.tiles_x * P.tiles_y * 32;
    chunk = (int)(item / per_chunk);
    int rest = (int)(item - (long long)chunk * per_chunk);
    int tile = rest >> 5, lane = rest & 31;
    int tx = tile % P.tiles_x, ty = tile / P.tiles_x;
    px = tx * 8 + (lane & 7), py = ty * 4 + (lane >> 3);
    return px < P.width && py < P.height && chunk < P.items_per_pixel;
}

// render_pixel's sample loop (raytrace.rs:188-198) for samples [first, first + count) of one pixel.
// Paths are regenerated in place: every loop iteration advances whatever path the thread currently holds by
// one segment, so the lanes of a warp stay busy until their whole run of samples is finished.
template <class SV>
RTB_DEV void integrate_item(const SV& S, const DCamera& cam, const DRenderParams& P, int px, int py, int first, int count, AccumFx sum[3],
                            uint32_t& n_rays) {
    PathRng rng;
    rng.pixel = (uint32_t)(py * P.width + px);
    rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    rng.sample = 0, rng.draw = 0;
    PathState ps;
    ps.depth = 0, ps.origin_prim = -1, ps.origin_face = 0, ps.time = 0.0f;
    ps.beta = v3(0.f, 0.f, 0.f);
    ps.ray.o = ps.ray.d = v3(0.f, 0.f, 0.f);
    AccumFx acc[3] = {0ull, 0ull, 0ull};
    bool alive = false;
    int next = 0;
    for (;;) {
        if (!alive) {
            if (next == count) break;
            rng.sample = (uint32_t)(first + next), rng.draw = 0;
            next += 1;
            ps.time = time_of_flags(camera_time_flags(cam, rng));
            float u[4];
            rng_next4(rng, u);
            ps.ray = generate_camera_ray(cam, P, px, py, u);
            ps.beta = v3(1.f, 1.f, 1.f);
            ps.origin_prim = -1, ps.origin_face = 0;
            ps.depth = P.max_depth;
            alive = true;
        }
        V3 radiance;
        n_rays += ps.depth > 0 ? 1u : 0u;
        alive = extend_and_shade(S, ps, rng, P.max_depth - ps.depth, radiance);
        if (!alive) acc[0] += radiance_fixed(radiance.x), acc[1] += radiance_fixed(radiance.y), acc[2] += radiance_fixed(radiance.z);
    }
    sum[0] = acc[0], sum[1] = acc[1], sum[2] = acc[2];
}

// ------------------------------------------------------------------ wavefront path state (rt_wavefront.cu)
// One pool slot = four 128-bit words:
//   A = origin.xyz, pixel            B = direction.xyz, flags (depth left | origin face << 16)
//   C = beta.rgb, sample index       D = t, code, origin primitive, -
// D.t / D.code enter the extend stage as the pre-sampled medium event (t_max of the surface search; +inf / -1 if
// none) and leave it as the final hit.
// hit code: -1 miss, prim | face << 24 for a surface, WF_MEDIUM | m for a medium event.
enum { WF_MISS = 0, WF_LAMBERTIAN = 1, WF_METAL = 2, WF_DIELECTRIC = 3, WF_LIGHT = 4, WF_ISOTROPIC = 5, WF_TEXTURED = 6, WF_CLASSES = 7 };
#define WF_MEDIUM 0x40000000
#define WF_DEPTH_MASK 0xFFFF
#define WF_FACE_SHIFT 16

struct WfSlot {
    float4 A, B, C, D;
};
RTB_DEV float4 f4(float x, float y, float z, float w) {
    float4 v;
    v.x = x, v.y = y, v.z = z, v.w = w;
    return v;
}

// the closest medium event along the slot's (new) ray, drawn with the media uniforms of segment `segment`; it
// becomes the t_max (and fallback hit code) of the surface search in the extend stage
template <int MODE = MEDIA_ANY, class SV = DSceneView>
RTB_DEV void wf_presample_media(const SV& S, const DRenderParams& P, WfSlot& s, int segment) {
    float t = RTB_INF;
    int medium = -1;
    if ((SV::feat & F_MEDIA) && S.n_media > 0) {
        Ray r;
        r.o = v3(s.A.x, s.A.y, s.A.z), r.d = v3(s.B.x, s.B.y, s.B.z);
        PathRng rng;
        rng.pixel = as_uint(s.A.w), rng.sample = as_uint(s.C.w), rng.draw = 1u + 2u * (uint32_t)segment, rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
        sample_media<MODE>(S, r, RTB_T_MIN, rng, t, medium);
    }
    s.D.x = t;
    s.D.y = as_float(medium >= 0 ? (uint32_t)(WF_MEDIUM | medium) : 0xFFFFFFFFu);
}

// a fresh camera path for (pixel, sample)
template <class SV>
RTB_DEV void wf_init_pixel_sample(const SV& S, const DCamera& cam, const DRenderParams& P, uint32_t pixel, uint32_t sample, WfSlot& s);

// a fresh camera path: global path number -> (pixel, sample); sample-major so that consecutive paths are
// neighbouring pixels of one sample index
template <class SV>
RTB_DEV void wf_init_path(const SV& S, const DCamera& cam, const DRenderParams& P, unsigned long long path, WfSlot& s) {
    unsigned long long npix = (unsigned long long)P.width * (unsigned long long)P.height;
    wf_init_pixel_sample(S, cam, P, (uint32_t)(path % npix), (uint32_t)P.sample_begin + (uint32_t)(path / npix), s);
}

// the camera ray alone (the caller pre-samples the media of segment 0)
template <uint32_t FEAT = F_ALL>
RTB_DEV void wf_init_camera(const DCamera& cam, const DRenderParams& P, uint32_t pixel, uint32_t sample, WfSlot& s) {
    PathRng rng;
    rng.pixel = pixel, rng.sample = sample, rng.draw = 0, rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    const uint32_t time_bits = (FEAT & F_MOVING) ? camera_time_flags(cam, rng) : 0u;  // nothing moves: nothing reads the path's time
    float u[4];
    rng_next4(rng, u);
    Ray r = generate_camera_ray(cam, P, (int)(pixel % (uint32_t)P.width), (int)(pixel / (uint32_t)P.width), u);
    s.A = f4(r.o.x, r.o.y, r.o.z, as_float(pixel));
    s.B = f4(r.d.x, r.d.y, r.d.z, as_float((uint32_t)P.max_depth | time_bits));
    s.C = f4(1.f, 1.f, 1.f, as_float(sample));
    s.D = f4(0.f, 0.f, as_float(0xFFFFFFFFu), 0.f);
}

template <class SV>
RTB_DEV void wf_init_pixel_sample(const SV& S, const DCamera& cam, const DRenderParams& P, uint32_t pixel, uint32_t sample, WfSlot& s) {
    wf_init_camera(cam, P, pixel, sample, s);
    wf_presample_media(S, P, s, 0);
}

// end of the extend stage for one ray: final hit code and the queue class the shade stage picks the path up from.
// prim/face/mat describe the closest surface found below the incoming t_max (prim < 0: none, the incoming code
// — a medium event or a miss — stands).
template <class SV>
RTB_DEV int wf_classify(const SV& S, int prim, int face, int mat, int code_in, int& code_out) {
    if (prim >= 0) {
        code_out = prim | (face << 24);
    } else {
        code_out = code_in;
        if (code_in < 0) return WF_MISS;
        mat = (int)as_uint(ld4(reinterpret_cast<const char*>(S.media + (code_in & 0xFFFF)) + 32).y);
    }
    float4 m = ld4(S.mats + mat);  // kind, tex, fuzz, ior
    if ((int)as_uint(m.y) >= 0) return WF_TEXTURED;
    return (int)as_uint(m.x);  // MAT_* == WF_* for the five material kinds
}

// the shade stage for one path: scatter or terminate.  Returns true while alive (slot updated in place, media
// event of the new ray pre-sampled); otherwise `radiance` is the path's contribution to its pixel.
// wf_shade_core: everything but the media pre-sampling of the new ray; `segment_next` = its segment number.
template <class SV>
RTB_DEV bool wf_shade_core(const SV& S, const DRenderParams& P, WfSlot& s, V3& radiance, NoiseReq* req, int& segment_next) {
    PathState ps;
    ps.ray.o = v3(s.A.x, s.A.y, s.A.z), ps.ray.d = v3(s.B.x, s.B.y, s.B.z);
    ps.beta = v3(s.C.x, s.C.y, s.C.z);
    uint32_t flags = as_uint(s.B.w);
    ps.depth = (int)(flags & WF_DEPTH_MASK);
    int segment = P.max_depth - ps.depth;
    ps.depth -= 1;  // this segment's ray has been traced
    segment_next = segment + 1;
    ps.origin_prim = -1, ps.origin_face = 0;
    ps.time = time_of_flags(flags);
    int code = (int)as_uint(s.D.y);
    float t = s.D.x;
    if (code < 0) {
        radiance = ps.beta * background_color(S, ps.ray);
        return false;
    }
    PathRng rng;
    rng.pixel = as_uint(s.A.w), rng.sample = as_uint(s.C.w), rng.draw = 2u + 2u * (uint32_t)segment, rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    float us[4];
    rng_next4(rng, us);
    V3 term;
    const bool is_medium = (code & WF_MEDIUM) != 0;
    bool alive = scatter_event(S, is_medium ? (code & 0xFFFF) : -1, code & 0xFFFFFF, (code >> 24) & 7, t, us, ps, term, req);
    if (!alive) {
        radiance = ps.beta * term;
        return false;
    }
    if (ps.depth <= 0) {
        radiance = v3(0.f, 0.f, 0.f);
        if (req) req->tex = -1;
        return false;
    }
    s.A = f4(ps.ray.o.x, ps.ray.o.y, ps.ray.o.z, s.A.w);
    s.B = f4(ps.ray.d.x, ps.ray.d.y, ps.ray.d.z, as_float((uint32_t)ps.depth | ((uint32_t)ps.origin_face << WF_FACE_SHIFT) | (flags & WF_TIME_MASK)));
    s.C = f4(ps.beta.x, ps.beta.y, ps.beta.z, s.C.w);
    s.D.z = as_float((uint32_t)ps.origin_prim);
    return true;
}

template <class SV>
RTB_DEV bool wf_shade(const SV& S, const DRenderParams& P, WfSlot& s, V3& radiance) {
    int segment_next;
    if (!wf_shade_core(S, P, s, radiance, nullptr, segment_next)) return false;
    wf_presample_media(S, P, s, segment_next);
    return true;
}

// Event-to-event advance inside a CLEAR medium (DSceneView.clear_media, flatten.cpp: find_clear_media).  The slot holds a
// path whose ray starts inside medium m's boundary and whose pre-sampled event (D.x, D.y = WF_MEDIUM | m) lies inside it
// as well: the boundary is one convex primitive with nothing else inside, so the surface search of the extend stage
// cannot find anything closer and is skipped.  One step = exactly what wf_shade does for such a slot (isotropic scatter,
// volumes.rs:77-83, then the media pre-sampling of the new ray) with the same Philox counters, minus everything a
// medium event never needs (surface attributes, textures, the other material kinds).
// Returns 0: the path ended (depth exhausted, contributes Color::ZERO), 1: the new ray's event is again inside medium m
// (the slot is ready for another step), 2: it is not (the slot is an ordinary ready path for the extend stage).
template <class SV>
RTB_DEV bool wf_chain_eligible(const SV& S, int code_shaded, const WfSlot& s_next) {
    return code_shaded >= 0 && (code_shaded & WF_MEDIUM) != 0 && (code_shaded & 0xFFFF) < 32 && ((S.clear_media >> (code_shaded & 31)) & 1u) != 0u &&
           (int)as_uint(s_next.D.y) == code_shaded;
}
template <int MODE = MEDIA_ANY, class SV = DSceneView>
RTB_DEV int wf_chain_step(const SV& S, const DRenderParams& P, WfSlot& s) {
    const uint32_t flags = as_uint(s.B.w);
    int depth = (int)(flags & WF_DEPTH_MASK);
    const int segment = P.max_depth - depth;
    depth -= 1;
    const int code = (int)as_uint(s.D.y);
    PathRng rng;
    rng.pixel = as_uint(s.A.w), rng.sample = as_uint(s.C.w), rng.draw = 2u + 2u * (uint32_t)segment, rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    float us[4];
    rng_next4(rng, us);
    const int mat_index = (int)as_uint(ld4(reinterpret_cast<const char*>(S.media + (code & 0xFFFF)) + 32).y);
    const float4 albedo = ld4(reinterpret_cast<const char*>(S.mats + mat_index) + 16);  // albedo.rgb, pad
    const float t = s.D.x;
    const V3 p = v3(s.A.x, s.A.y, s.A.z) + t * v3(s.B.x, s.B.y, s.B.z);
    const V3 dir = sample_unit_ball(us[0], us[1], us[2]);
    const V3 beta = v3(s.C.x, s.C.y, s.C.z) * v3(albedo.x, albedo.y, albedo.z);
    if (depth <= 0) return 0;
    s.A = f4(p.x, p.y, p.z, s.A.w);
    s.B = f4(dir.x, dir.y, dir.z, as_float((uint32_t)depth | (flags & WF_TIME_MASK)));
    s.C = f4(beta.x, beta.y, beta.z, s.C.w);
    s.D.z = as_float(0xFFFFFFFFu);
    wf_presample_media<MODE>(S, P, s, segment + 1);
    return (int)as_uint(s.D.y) == code ? 1 : 2;
}

// ------------------------------------------------------------------ test entry points (rt_intersect_batch etc.)
enum { QUERY_BVH = 0, QUERY_LINEAR = 1, QUERY_MEDIUM = 2, QUERY_BVH4 = 3 };

// Hittable::hit for one ray given as 8 floats (origin, direction, t_min, t_max) -> RtHit
template <class SV>
RTB_DEV void intersect_query(const SV& S, int mode, const float* q, RtHit& out, float time = 0.0f) {
    Ray r;
    r.o = v3(q[0], q[1], q[2]), r.d = v3(q[3], q[4], q[5]);
    float tmin = q[6], tmax = q[7];
    out.t = 0.f, out.u = 0.f, out.v = 0.f, out.front_face = 0, out.material = -1, out.prim = -1;
    out.p[0] = out.p[1] = out.p[2] = 0.f;
    out.normal[0] = out.normal[1] = out.normal[2] = 0.f;
    if (mode == QUERY_MEDIUM) {
        float t1, t2;
        if (medium_interval_any(S, S.media, r, tmin, tmax, t1, t2)) out.t = t1, out.u = t2, out.material = S.media[0].mat;
        return;
    }
    float t;
    int prim, face;
    if (mode == QUERY_BVH4 && S.nodes4 && tmin > 0.0f) closest_hit4(S, r, tmin, tmax, -1, 0, t, prim, face, time);
    else if (mode == QUERY_BVH || mode == QUERY_BVH4) closest_hit(S, r, tmin, tmax, -1, 0, t, prim, face, time);
    else closest_hit_linear(S, r, tmin, tmax, t, prim, face, time);
    if (prim < 0) return;
    PrimRec P = load_prim(S.prims + prim);
    apply_motion(S, P, time);
    Surface s;
    surface_at(S, P, r, t, face, true, s);
    out.t = t, out.u = s.u, out.v = s.v, out.front_face = s.front ? 1 : 0, out.material = P.mat, out.prim = prim;
    out.p[0] = s.p.x, out.p[1] = s.p.y, out.p[2] = s.p.z;
    out.normal[0] = s.n.x, out.normal[1] = s.n.y, out.normal[2] = s.n.z;
}

// Material::scatter / emit for one caller-supplied hit (rt_scatter_batch): the very `scatter` the pipelines call
template <class SV>
RTB_DEV void scatter_query(const SV& S, const RtScatterIn& in, RtScatterOut& out) {
    Surface sf;
    sf.p = v3(in.p[0], in.p[1], in.p[2]), sf.n = v3(in.normal[0], in.normal[1], in.normal[2]);
    sf.u = in.u, sf.v = in.v, sf.front = in.front_face != 0;
    PathState ps;
    ps.ray.o = v3(in.ray_origin[0], in.ray_origin[1], in.ray_origin[2]), ps.ray.d = v3(in.ray_dir[0], in.ray_dir[1], in.ray_dir[2]);
    ps.beta = v3(1.f, 1.f, 1.f), ps.origin_prim = -1, ps.origin_face = 0, ps.depth = 1;
    V3 radiance = v3(0.f, 0.f, 0.f);
    const bool alive = scatter(S, S.mats[in.material], sf, in.uniform, ps, -1, 0, radiance, nullptr);
    out.scattered = alive ? 1 : 0;
    out.attenuation[0] = alive ? ps.beta.x : 0.f, out.attenuation[1] = alive ? ps.beta.y : 0.f, out.attenuation[2] = alive ? ps.beta.z : 0.f;
    out.dir[0] = alive ? ps.ray.d.x : 0.f, out.dir[1] = alive ? ps.ray.d.y : 0.f, out.dir[2] = alive ? ps.ray.d.z : 0.f;
    out.emitted[0] = alive ? 0.f : radiance.x, out.emitted[1] = alive ? 0.f : radiance.y, out.emitted[2] = alive ? 0.f : radiance.z;
}

// the camera ray of (pixel, sample) exactly as integrate_item generates it
RTB_DEV void camera_query(const DCamera& cam, const DRenderParams& P, int pixel, int sample, float* ray6, float* u4) {
    PathRng rng;
    rng.pixel = (uint32_t)pixel, rng.sample = (uint32_t)sample, rng.draw = 0, rng.k0 = P.seed_lo, rng.k1 = P.seed_hi;
    rng_next4(rng, u4);
    Ray r = generate_camera_ray(cam, P, pixel % P.width, pixel / P.width, u4);
    ray6[0] = r.o.x, ray6[1] = r.o.y, ray6[2] = r.o.z, ray6[3] = r.d.x, ray6[4] = r.d.y, ray6[5] = r.d.z;
}

}  // namespace rtb
