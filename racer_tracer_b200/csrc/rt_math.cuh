// rt_math.cuh — small vector type templated on the scalar (float for the
// renderer, double for the f64 instantiation of the primary-visibility AOV),
// Philox4x32 and the uniform conversions of DESIGN.md "RNG streams".
#pragma once
#ifdef __CUDACC_RTC__
// NVRTC (scene-specialised kernels, rc_spec.cuh): no host headers
typedef unsigned char uint8_t;
typedef unsigned int uint32_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
#else
#include <cuda_runtime.h>
#include <stdint.h>
#endif

#define RT_HD __host__ __device__ __forceinline__
#define RT_D __device__ __forceinline__

template <typename T>
struct Vec3T {
    T x, y, z;
};
typedef Vec3T<float> vec3f;

template <typename T> RT_HD Vec3T<T> mk3(T x, T y, T z) { Vec3T<T> v; v.x = x; v.y = y; v.z = z; return v; }
template <typename T> RT_HD Vec3T<T> operator+(Vec3T<T> a, Vec3T<T> b) { return mk3<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename T> RT_HD Vec3T<T> operator-(Vec3T<T> a, Vec3T<T> b) { return mk3<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename T> RT_HD Vec3T<T> operator-(Vec3T<T> a) { return mk3<T>(-a.x, -a.y, -a.z); }
template <typename T> RT_HD Vec3T<T> operator*(Vec3T<T> a, Vec3T<T> b) { return mk3<T>(a.x * b.x, a.y * b.y, a.z * b.z); }
template <typename T> RT_HD Vec3T<T> operator*(T s, Vec3T<T> a) { return mk3<T>(s * a.x, s * a.y, s * a.z); }
template <typename T> RT_HD Vec3T<T> operator*(Vec3T<T> a, T s) { return mk3<T>(s * a.x, s * a.y, s * a.z); }
template <typename T> RT_HD T dot(Vec3T<T> a, Vec3T<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> RT_HD T length_squared(Vec3T<T> a) { return dot(a, a); }
template <typename T> RT_HD T axis_of(Vec3T<T> a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

RT_D float rt_sqrt(float v) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
RT_D double rt_sqrt(double v) { return sqrt(v); }
RT_D float rt_rsqrt(float v) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
RT_D double rt_rsqrt(double v) { return 1.0 / sqrt(v); }
// single-instruction SFU approximations (<= 2 ulp); the render path does not
// need IEEE-rounded reciprocals / square roots
RT_D float fast_rcp(float v) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
RT_D float fast_sqrt(float v) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
RT_D float fast_rsqrt(float v) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }
RT_D float rt_rcp(float v) { return fast_rcp(v); }
RT_D double rt_rcp(double v) { return 1.0 / v; }

// Packed FP32 (sm_100a: FFMA2 / FMUL2, two fp32 lanes per instruction and per issue slot; a scalar operand is
// broadcast).  Same rounding as the scalar instructions (RN, fused), so results do not change; what changes is
// the number of issue slots, which is what bounds the render kernel (profiles/).
RT_D void fma2_bcast(float s, float a0, float a1, float b0, float b1, float& r0, float& r1) {   // s * (a0, a1) + (b0, b1)
    asm("{\n\t.reg .b64 ss, aa, bb, rr;\n\t"
        "mov.b64 ss, {%2, %2};\n\tmov.b64 aa, {%3, %4};\n\tmov.b64 bb, {%5, %6};\n\t"
        "fma.rn.f32x2 rr, ss, aa, bb;\n\t"
        "mov.b64 {%0, %1}, rr;\n\t}" : "=f"(r0), "=f"(r1) : "f"(s), "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
RT_D void mul2_bcast(float s, float a0, float a1, float& r0, float& r1) {   // s * (a0, a1)
    asm("{\n\t.reg .b64 ss, aa, rr;\n\t"
        "mov.b64 ss, {%2, %2};\n\tmov.b64 aa, {%3, %4};\n\t"
        "mul.f32x2 rr, ss, aa;\n\t"
        "mov.b64 {%0, %1}, rr;\n\t}" : "=f"(r0), "=f"(r1) : "f"(s), "f"(a0), "f"(a1));
}
RT_D void mul2(float a0, float a1, float b0, float b1, float& r0, float& r1) {   // (a0, a1) * (b0, b1)
    asm("{\n\t.reg .b64 aa, bb, rr;\n\t"
        "mov.b64 aa, {%2, %3};\n\tmov.b64 bb, {%4, %5};\n\t"
        "mul.f32x2 rr, aa, bb;\n\t"
        "mov.b64 {%0, %1}, rr;\n\t}" : "=f"(r0), "=f"(r1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
RT_D void fma2(float a0, float a1, float b0, float b1, float c0, float c1, float& r0, float& r1) {   // (a0, a1) * (b0, b1) + (c0, c1)
    asm("{\n\t.reg .b64 aa, bb, cc, rr;\n\t"
        "mov.b64 aa, {%2, %3};\n\tmov.b64 bb, {%4, %5};\n\tmov.b64 cc, {%6, %7};\n\t"
        "fma.rn.f32x2 rr, aa, bb, cc;\n\t"
        "mov.b64 {%0, %1}, rr;\n\t}" : "=f"(r0), "=f"(r1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}

template <typename T> RT_D Vec3T<T> unit_vector(Vec3T<T> a) { return a * rt_rsqrt(length_squared(a)); }

// vec3.rs:412-414
template <typename T> RT_D Vec3T<T> reflect(Vec3T<T> v, Vec3T<T> n) { return v - (T(2) * dot(v, n)) * n; }

// ---------------------------------------------------------------------------
// Philox2x32-R (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3",
// SC'11): 64-bit counter, 32-bit key, 64 random bits per call.  One call costs
// R x (IMAD.WIDE.U32 + LOP3) with the key schedule in uniform registers, and
// 64 bits is exactly what one path event consumes, so nothing has to be cached
// between bounces.
// ---------------------------------------------------------------------------
#define PHILOX2_M 0xD256D193u
#define PHILOX2_W 0x9E3779B9u

// The key schedule (key + r*W, r = 0..9) is precomputed by the host into the kernel parameters:
// every round is IMAD.WIDE.U32 + one LOP3 with a constant-bank operand.
template <int ROUNDS>
RT_D uint2 philox2x32_ks(uint32_t c0, uint32_t c1, const uint32_t* ks) {
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint64_t p = (uint64_t)PHILOX2_M * c0;
        c0 = (uint32_t)(p >> 32) ^ ks[r] ^ c1;
        c1 = (uint32_t)p;
    }
    return make_uint2(c0, c1);
}

// The same block with round 0's multiplication hoisted: c0 is the pixel index, constant over all the blocks a
// lane draws for one pixel.  philox2x32_from(philox2x32_pre(c0, ks), c1, ks) == philox2x32_ks(c0, c1, ks).
struct PhiloxPre { uint32_t hi_k0, lo; };
RT_D PhiloxPre philox2x32_pre(uint32_t c0, const uint32_t* ks) {
    const uint64_t p = (uint64_t)PHILOX2_M * c0;
    PhiloxPre q;
    q.hi_k0 = (uint32_t)(p >> 32) ^ ks[0];
    q.lo = (uint32_t)p;
    return q;
}
template <int ROUNDS>
RT_D uint2 philox2x32_from(PhiloxPre q, uint32_t c1, const uint32_t* ks) {
    uint32_t c0 = q.hi_k0 ^ c1;
    c1 = q.lo;
#pragma unroll
    for (int r = 1; r < ROUNDS; ++r) {
        const uint64_t p = (uint64_t)PHILOX2_M * c0;
        c0 = (uint32_t)(p >> 32) ^ ks[r] ^ c1;
        c1 = (uint32_t)p;
    }
    return make_uint2(c0, c1);
}

// Counter layout (DESIGN.md "RNG streams"):
//   c0 = pixel index (24 bits) | iteration j of a rejection loop << 24
//   c1 = sample index (24 bits) | segment or bounce (6 bits) << 24 | stream tag << 30
//   key = low 32 bits of the seed XOR its high 32 bits
// ONE PATH block per path segment: block e of a sample belongs to segment e (e = 0 is the primary
// ray) and is drawn before the segment is intersected, by every lane of the warp together.  Its
// upper 24 bits per word feed the scattering event at the END of that segment (hit number e + 1);
// the low byte of each word is spare, and in block 0 the two spare bytes are the NEXT sample's v jitter
// (rt_vjit_sample).
#define RT_TAG_PATH   0u   // segment e: scatter bits of hit e + 1; e = 0 also: low bytes -> 16-bit v jitter of the next sample (cpu.rs:39-40)
#define RT_TAG_PIXEL  1u   // sample = segment = 0: x -> per-pixel u jitter (cpu.rs:35-36)
#define RT_TAG_LENS   2u   // j = 0: (x, y) -> direct lens sample, low bytes -> 16-bit ray time; j >= 1: rejection iteration j
#define RT_TAG_REJECT 3u   // (hit number b, iteration j): three 21-bit uniforms of a rejection iteration

RT_HD uint32_t rt_ctr1(uint32_t sample, uint32_t bounce, uint32_t tag) { return sample | (bounce << 24) | (tag << 30); }
// The sample whose PATH block 0 carries, in its two spare bytes, the v jitter of sample `s`: the one before it
// (24-bit wrap for s = 0).  A sample's own block is therefore not needed before its first hit is shaded.
RT_HD uint32_t rt_vjit_sample(uint32_t s) { return (s - 1u) & 0xFFFFFFu; }

// 24-bit and 21-bit uniforms in [0,1): exactly representable in fp32 and f64
RT_HD float u24(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }
RT_HD float u21(uint32_t w) { return (float)w * (1.0f / 2097152.0f); }  // w < 2^21
// three 21-bit uniforms out of 64 bits (REJECT blocks: all 64 bits belong to the iteration)
RT_HD void u21x3(uint2 w, float& a, float& b, float& c) {
    a = u21(w.x >> 11); b = u21(w.y >> 11); c = u21(((w.x & 0x7FFu) << 10) | (w.y & 0x3FFu));
}
// 16-bit uniform from the spare low byte of each word of a PATH / LENS block (v jitter, ray time).
// fp32 cannot hold more of the jitter anyway: (float)py + jitter keeps 2^-13 at py >= 1024.
RT_HD float u16lo(uint2 w) { return (float)(((w.x & 0xFFu) << 8) | (w.y & 0xFFu)) * (1.0f / 65536.0f); }
// the same 16 bits as a float integer in [0, 65536): one byte permute + one conversion
RT_D float u16lo_int(uint2 w) { return (float)(unsigned short)__byte_perm(w.y, w.x, 0x0040); }
// three 16-bit uniforms from the upper 24 bits of each word of a PATH block (metal fuzz, direct)
RT_HD void u16x3(uint2 w, float& a, float& b, float& c) {
    a = (float)(w.x >> 16) * (1.0f / 65536.0f);
    b = (float)(w.y >> 16) * (1.0f / 65536.0f);
    c = (float)(((w.x >> 8) & 0xFFu) << 8 | ((w.y >> 8) & 0xFFu)) * (1.0f / 65536.0f);
}
