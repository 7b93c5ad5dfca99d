// rt_denoise.cuh — the edge-avoiding à-trous filter of rc_render_denoised / rc_denoise_filter (include/racer_cuda.h
// states the filter exactly; tests/test_gpu_denoise.py restates it in f64).
//
//   denoise_moments_kernel   mean radiance and variance of the mean of y from one moments round
//   denoise_prepare_kernel   f64 inputs -> fp32, demodulated: float4 (c.rgb, var), float4 (n.xyz, z), albedo
//   denoise_level_kernel     one à-trous level (step 2^k), with the 3x3 blur of var fused in
//   denoise_finish_kernel    remodulate and gamma: sqrt(max(0, a c)) in f64
#pragma once
#include <cstdint>

#define RT_DENOISE_BX 32
#define RT_DENOISE_BY 8

// after a moments round of n samples over every pixel: mean = sum / n (as finalize_to_f64_kernel scales it) and the
// variance of the mean of y = (r + g + b) / 3, s^2 / n with s^2 = max(0, (S2 - S1^2 / n) / (n - 1))
__global__ void denoise_moments_kernel(const float* __restrict__ accum, const float* __restrict__ m2, double* __restrict__ mean,
                                       double* __restrict__ var, size_t n_pixels, int n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    const double scale = 1.0 / (double)n;
    mean[3 * i] = scale * (double)accum[3 * i];
    mean[3 * i + 1] = scale * (double)accum[3 * i + 1];
    mean[3 * i + 2] = scale * (double)accum[3 * i + 2];
    const double S1 = ((double)accum[3 * i] + (double)accum[3 * i + 1] + (double)accum[3 * i + 2]) / 3.0;
    const double S2 = (double)m2[i];
    var[i] = fmax(0.0, (S2 - S1 * S1 / n) / (n - 1)) / n;
}

// every input rounded to fp32, then demodulated: a = max(albedo, 1e-3), c = mean / a, var / mean(a)^2
__global__ void denoise_prepare_kernel(const double* __restrict__ mean, const double* __restrict__ var,
                                       const double* __restrict__ albedo, const double* __restrict__ normal,
                                       const double* __restrict__ depth, float4* __restrict__ cv, float4* __restrict__ nz,
                                       float4* __restrict__ alb, size_t n_pixels) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    const float ar = fmaxf((float)albedo[3 * i], 1e-3f), ag = fmaxf((float)albedo[3 * i + 1], 1e-3f),
                ab = fmaxf((float)albedo[3 * i + 2], 1e-3f);
    const float abar = (ar + ag + ab) / 3.0f;
    cv[i] = make_float4((float)mean[3 * i] / ar, (float)mean[3 * i + 1] / ag, (float)mean[3 * i + 2] / ab,
                        (float)var[i] / (abar * abar));
    nz[i] = make_float4((float)normal[3 * i], (float)normal[3 * i + 1], (float)normal[3 * i + 2], (float)depth[i]);
    alb[i] = make_float4(ar, ag, ab, 0.0f);
}

// One level: for q = p + step (i, j), i, j in -2..2, inside the image and with q's id equal to p's,
//   w = h(i) h(j) w_l w_n w_z,  w_l = exp(-|l_p - l_q| / (sigma_l sqrt(g_p) + 1e-3)),  w_n = max(0, n_p.n_q)^sigma_n,
//   w_z = exp(-|z_p - z_q| / (sigma_z z_p |(i, j)| step / H)),  w_n = w_z = 1 for q = p and for id 0,
// where g_p is the 3x3 [1/4 1/2 1/4]^2 blur of var over in-image pixels (renormalised, no id test); then
// c' = sum w c / sum w, var' = sum w^2 var / (sum w)^2.  The blur is fused in (its 9 reads hit lines the 25 taps read
// anyway); a separate blur pass was not built, so that choice is not measured.
__global__ void __launch_bounds__(RT_DENOISE_BX * RT_DENOISE_BY)
denoise_level_kernel(const float4* __restrict__ cv_in, float4* __restrict__ cv_out, const float4* __restrict__ nz,
                     const uint32_t* __restrict__ ids, int width, int height, int step, float sigma_l, float sigma_n,
                     float sigma_z) {
    const int x = blockIdx.x * RT_DENOISE_BX + threadIdx.x, y = blockIdx.y * RT_DENOISE_BY + threadIdx.y;
    if (x >= width || y >= height) return;
    const float h5[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
    const float h3[3] = {0.25f, 0.5f, 0.25f};
    const size_t p = (size_t)y * width + x;
    const float4 cp = cv_in[p], gp = nz[p];
    const uint32_t idp = ids[p];
    float gs = 0.0f, gw = 0.0f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qx >= width || qy < 0 || qy >= height) continue;
            const float w = h3[dx + 1] * h3[dy + 1];
            gs += w * cv_in[(size_t)qy * width + qx].w;
            gw += w;
        }
    const float lp = (cp.x + cp.y + cp.z) / 3.0f;
    const float l_den = sigma_l * sqrtf(gs / gw) + 1e-3f;
    const float z_den = sigma_z * gp.w * (float)step / (float)height;   // times |(i, j)| per tap
    float sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f, sw = 0.0f;
#pragma unroll
    for (int j = -2; j <= 2; ++j) {
        const int qy = y + j * step;
        if (qy < 0 || qy >= height) continue;
#pragma unroll
        for (int i = -2; i <= 2; ++i) {
            const int qx = x + i * step;
            if (qx < 0 || qx >= width) continue;
            const size_t q = (size_t)qy * width + qx;
            if (ids[q] != idp) continue;
            const float4 cq = cv_in[q];
            const float lq = (cq.x + cq.y + cq.z) / 3.0f;
            float w = h5[i + 2] * h5[j + 2] * expf(-fabsf(lp - lq) / l_den);
            if ((i != 0 || j != 0) && idp != 0) {
                const float4 gq = nz[q];
                const float wn = powf(fmaxf(0.0f, gp.x * gq.x + gp.y * gq.y + gp.z * gq.z), sigma_n);
                const float wz = expf(-fabsf(gp.w - gq.w) / (z_den * sqrtf((float)(i * i + j * j))));
                w *= wn * wz;
            }
            sr += w * cq.x; sg += w * cq.y; sb += w * cq.z;
            sv += w * w * cq.w;
            sw += w;
        }
    }
    cv_out[p] = make_float4(sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}

// out = sqrt(max(0, a c)) per channel, in f64 (the units rc_render returns)
__global__ void denoise_finish_kernel(const float4* __restrict__ cv, const float4* __restrict__ alb, double* __restrict__ rgb,
                                      size_t n_pixels) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pixels) return;
    const float4 c = cv[i], a = alb[i];
    rgb[3 * i] = sqrt(fmax(0.0, (double)a.x * (double)c.x));
    rgb[3 * i + 1] = sqrt(fmax(0.0, (double)a.y * (double)c.y));
    rgb[3 * i + 2] = sqrt(fmax(0.0, (double)a.z * (double)c.z));
}
