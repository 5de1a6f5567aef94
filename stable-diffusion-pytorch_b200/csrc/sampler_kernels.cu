// Fused CFG blend + scheduler latent update (SURVEY.md §8(a) rows S1, S2, S4, S5, S6).
//
// One elementwise pass: reads x_t and the UNet output (uncond and cond halves), writes x_{t-1}.
// Bandwidth-bound: 16-byte vector loads/stores, grid sized in multiples of the SM count, no
// shared memory (no reuse).  Per-timestep scalars come from a device-resident [T][8] fp32 table
// built by the host sampler, indexed by a timestep that may itself live in device memory, so a
// sampling loop has no host sync and is CUDA-graph capturable.
//
// Arithmetic is the reference's op sequence with one fp32 rounding per op (explicit _rn
// intrinsics, no FMA contraction), which makes the result bit-identical to the reference's
// CPU eager path for the same inputs:
//   CFG   (models/diffusion.py:234-235)  e  = u + s*(c - u)
//   DDIM  (models/scheduler/ddim.py:65-81)
//     eps-pred:  x0 = (x - s1*e)/s2 ; ee = e
//     v-pred:    x0 = s2*x - s1*e   ; ee = s2*e + s1*x
//     x' = sqrt_prev*x0 + dir*ee   (+ noise*std when eta > 0)
//   DDPM  (models/scheduler/ddpm.py:72-81)   x' = inv*(x - ce*e) + std*z
//   DPM-Solver++(2M) (diffusers' DPMSolverMultistepScheduler, algorithm_type="dpmsolver++", solver_type="midpoint")
//     m0 = x0 exactly as DDIM computes it (columns 0-1), m1 = history (the previous step's m0)
//     x' = (A*x + B*m0) + C*(m0 - m1)     the C term only when the row's flag (column 7) and hist_valid are set;
//                                         otherwise m1 is not read at all (history may hold garbage or NaN)
//     history = m0                        same thread reads m1, then writes m0: in place without a race
#define SDK_PDL_CAT 6
#include "common.cuh"

namespace {

constexpr int COEF_COLS = 8;

struct Coef { float c[COEF_COLS]; };

__device__ __forceinline__ bool load_coef(const float* __restrict__ table, int T,
                                          const long long* __restrict__ t_dev, long long t_host, Coef& k) {
    long long t = t_dev ? t_dev[0] : t_host;
    if (t < 0 || t >= T) return false;     // the reference raises IndexError; we poison the output with NaN
    const float4* p = reinterpret_cast<const float4*>(table + t * COEF_COLS);
    float4 a = __ldg(p), b = __ldg(p + 1);
    k.c[0] = a.x; k.c[1] = a.y; k.c[2] = a.z; k.c[3] = a.w;
    k.c[4] = b.x; k.c[5] = b.y; k.c[6] = b.z; k.c[7] = b.w;
    return true;
}

__device__ __forceinline__ float cfg_one(float u, float c, float s) {
    return __fadd_rn(u, __fmul_rn(s, __fsub_rn(c, u)));
}

template <int PRED>
__device__ __forceinline__ float ddim_one(float x, float e, const Coef& k, bool has_noise, float z) {
    const float s1 = k.c[0], s2 = k.c[1], sp = k.c[2], dir = k.c[3], sd = k.c[4];
    float x0, ee;
    if (PRED == 0) {
        x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(s1, e)), s2);
        ee = e;
    } else {
        x0 = __fsub_rn(__fmul_rn(s2, x), __fmul_rn(s1, e));
        ee = __fadd_rn(__fmul_rn(s2, e), __fmul_rn(s1, x));
    }
    float r = __fadd_rn(__fmul_rn(sp, x0), __fmul_rn(dir, ee));
    if (has_noise) r = __fadd_rn(r, __fmul_rn(z, sd));
    return r;
}

// x0 prediction of DDIM (columns 0-1), shared by the DPM-Solver++ update
template <int PRED>
__device__ __forceinline__ float x0_one(float x, float e, const Coef& k) {
    return PRED == 0 ? __fdiv_rn(__fsub_rn(x, __fmul_rn(k.c[0], e)), k.c[1])
                     : __fsub_rn(__fmul_rn(k.c[1], x), __fmul_rn(k.c[0], e));
}

// DPM-Solver++(2M): columns 2-4 = A, B, C; m1 is only used when `second`
__device__ __forceinline__ float dpmpp_one(float x, float m0, float m1, const Coef& k, bool second) {
    float r = __fadd_rn(__fmul_rn(k.c[2], x), __fmul_rn(k.c[3], m0));
    if (second) r = __fadd_rn(r, __fmul_rn(k.c[4], __fsub_rn(m0, m1)));
    return r;
}

__device__ __forceinline__ float ddpm_one(float x, float e, const Coef& k, float z) {
    float mu = __fmul_rn(k.c[0], __fsub_rn(x, __fmul_rn(k.c[1], e)));
    return __fadd_rn(mu, __fmul_rn(k.c[2], z));
}

// MODE 0/1: DDIM eps / v ; MODE 2: DDPM
template <int MODE>
__global__ void __launch_bounds__(256)
step_kernel(const float* x, const float* __restrict__ eu, const float* __restrict__ ec, float scale,
            const float* __restrict__ noise, float* out, long long n,      // x and out may alias (in-place latent state)
            const float* __restrict__ table, int T, const long long* __restrict__ t_dev, long long t_host, int vec_ok) {
    pdl_trigger();
    pdl_wait();
    Coef k;
    const bool ok = load_coef(table, T, t_dev, t_host, k);
    const float qnan = __int_as_float(0x7fc00000);
    const long long nvec = vec_ok ? (n >> 2) : 0;      // 16-byte path only when every pointer is 16-byte aligned
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float4 xv = reinterpret_cast<const float4*>(x)[i];
        float4 uv = __ldg(reinterpret_cast<const float4*>(eu) + i);
        float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (noise) zv = __ldg(reinterpret_cast<const float4*>(noise) + i);
        float ev[4] = {uv.x, uv.y, uv.z, uv.w};
        if (ec) {
            float4 cv = __ldg(reinterpret_cast<const float4*>(ec) + i);
            ev[0] = cfg_one(uv.x, cv.x, scale); ev[1] = cfg_one(uv.y, cv.y, scale);
            ev[2] = cfg_one(uv.z, cv.z, scale); ev[3] = cfg_one(uv.w, cv.w, scale);
        }
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
        const float zs[4] = {zv.x, zv.y, zv.z, zv.w};
        float r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (MODE == 2) r[j] = ddpm_one(xs[j], ev[j], k, zs[j]);
            else r[j] = ddim_one<MODE>(xs[j], ev[j], k, noise != nullptr, zs[j]);
            if (!ok) r[j] = qnan;
        }
        reinterpret_cast<float4*>(out)[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
    // scalar tail (n % 4)
    for (long long i = (nvec << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float e = eu[i];
        if (ec) e = cfg_one(e, ec[i], scale);
        float z = noise ? noise[i] : 0.f;
        float r = (MODE == 2) ? ddpm_one(x[i], e, k, z) : ddim_one<(MODE == 2 ? 0 : MODE)>(x[i], e, k, noise != nullptr, z);
        out[i] = ok ? r : qnan;
    }
}

// DPM-Solver++(2M) update, PRED 0/1: eps / v.  history[i] holds the previous step's x0 prediction and is replaced by this
// step's; x, out and history are each read and written by the same thread only.
template <int PRED>
__global__ void __launch_bounds__(256)
dpmpp_step_kernel(const float* x, const float* __restrict__ eu, const float* __restrict__ ec, float scale, float* hist,
                  int hist_valid, float* out, long long n, const float* __restrict__ table, int T,
                  const long long* __restrict__ t_dev, long long t_host, int vec_ok) {
    pdl_trigger();
    pdl_wait();
    Coef k;
    const bool ok = load_coef(table, T, t_dev, t_host, k);
    const bool second = ok && hist_valid && k.c[7] != 0.f;
    const float qnan = __int_as_float(0x7fc00000);
    const long long nvec = vec_ok ? (n >> 2) : 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        float4 xv = reinterpret_cast<const float4*>(x)[i];
        float4 uv = __ldg(reinterpret_cast<const float4*>(eu) + i);
        float ev[4] = {uv.x, uv.y, uv.z, uv.w};
        if (ec) {
            float4 cv = __ldg(reinterpret_cast<const float4*>(ec) + i);
            ev[0] = cfg_one(uv.x, cv.x, scale); ev[1] = cfg_one(uv.y, cv.y, scale);
            ev[2] = cfg_one(uv.z, cv.z, scale); ev[3] = cfg_one(uv.w, cv.w, scale);
        }
        float4 hv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (second) hv = reinterpret_cast<const float4*>(hist)[i];
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
        const float hs[4] = {hv.x, hv.y, hv.z, hv.w};
        float m[4], r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            m[j] = x0_one<PRED>(xs[j], ev[j], k);
            r[j] = dpmpp_one(xs[j], m[j], hs[j], k, second);
            if (!ok) { m[j] = qnan; r[j] = qnan; }
        }
        reinterpret_cast<float4*>(hist)[i] = make_float4(m[0], m[1], m[2], m[3]);
        reinterpret_cast<float4*>(out)[i] = make_float4(r[0], r[1], r[2], r[3]);
    }
    // scalar tail (n % 4, or everything when a pointer is not 16-byte aligned)
    for (long long i = (nvec << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float e = eu[i];
        if (ec) e = cfg_one(e, ec[i], scale);
        const float xi = x[i];
        const float m0 = x0_one<PRED>(xi, e, k);
        const float r = dpmpp_one(xi, m0, second ? hist[i] : 0.f, k, second);
        hist[i] = ok ? m0 : qnan;
        out[i] = ok ? r : qnan;
    }
}

// Inpainting step (models/diffusion.py:387-398), one pass, reference op order:
//   e      = s*(c - u) + c                      CFG in the inpaint loop's own form, model output ordered [cond ; uncond]
//   noised = sqrt(a_hat_t)*orig + sqrt(1 - a_hat_t)*e        forward_process(encoded_img, t, e)   (ddim.py:46-55)
//   xin    = mask ? x : noised                  torch.where(~mask, noised, latent); mask is per pixel, shared by batch and channels
//   x'     = DDIM(xin, e)  |  DDPM(xin, e, z)   reverse_process (MODE 0 / 1: DDIM eps / v; MODE 2: DDPM with the randn draw z of ddpm.py:80)
//          | DPM-Solver++(2M)(xin, e, hist)      MODE 3 / 4: eps / v, the update of dpmpp_step_kernel (history replaced by this step's x0)
template <int MODE>
__global__ void __launch_bounds__(256)
inpaint_step_kernel(const float* x, const float* __restrict__ ec, const float* __restrict__ eu, float scale,
                    const float* __restrict__ orig, long long orig_batch_stride, const unsigned char* __restrict__ mask,
                    const float* __restrict__ noise, float* out, long long n, long long chw, long long hw,
                    const float* __restrict__ table, int T, const long long* __restrict__ t_dev, long long t_host,
                    float* hist, int hist_valid) {
    pdl_trigger();
    pdl_wait();
    Coef k;
    const bool ok = load_coef(table, T, t_dev, t_host, k);
    const bool second = MODE >= 3 && ok && hist_valid && k.c[7] != 0.f;
    const float qnan = __int_as_float(0x7fc00000);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / chw, r = i - b * chw;
        float e = ec[i];
        if (eu) e = __fadd_rn(__fmul_rn(scale, __fsub_rn(e, eu[i])), e);
        const float noised = __fadd_rn(__fmul_rn(k.c[5], __ldg(orig + b * orig_batch_stride + r)), __fmul_rn(k.c[6], e));
        const float xin = mask[r % hw] ? x[i] : noised;
        float y;
        if (MODE >= 3) {
            const float m0 = x0_one<(MODE == 4 ? 1 : 0)>(xin, e, k);
            y = dpmpp_one(xin, m0, second ? hist[i] : 0.f, k, second);
            hist[i] = ok ? m0 : qnan;
        } else {
            y = MODE == 2 ? ddpm_one(xin, e, k, noise[i]) : ddim_one<(MODE == 2 ? 0 : MODE)>(xin, e, k, false, 0.f);
        }
        out[i] = ok ? y : qnan;
    }
}

__global__ void __launch_bounds__(256)
forward_process_kernel(const float* __restrict__ x0, const float* __restrict__ noise, float* __restrict__ out,
                       long long per_sample, const float* __restrict__ table, int T, const long long* __restrict__ t) {
    pdl_trigger();
    pdl_wait();
    const int b = blockIdx.y;
    long long tb = t[b];
    const bool ok = tb >= 0 && tb < T;
    const float sa = ok ? __ldg(table + tb * COEF_COLS + 5) : __int_as_float(0x7fc00000);
    const float sn = ok ? __ldg(table + tb * COEF_COLS + 6) : __int_as_float(0x7fc00000);
    const float* xs = x0 + (long long)b * per_sample;
    const float* ns = noise + (long long)b * per_sample;
    float* os = out + (long long)b * per_sample;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_sample; i += (long long)gridDim.x * blockDim.x)
        os[i] = __fadd_rn(__fmul_rn(sa, xs[i]), __fmul_rn(sn, ns[i]));
}

__global__ void __launch_bounds__(256)
x0_from_eps_kernel(const float* __restrict__ x, const float* __restrict__ e, float sigma, float alpha,
                   float* __restrict__ out, long long n) {
    pdl_trigger();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = __fdiv_rn(__fsub_rn(x[i], __fmul_rn(sigma, e[i])), alpha);
}

inline int grid_for(long long work_items, int threads) {
    long long blocks = (work_items + threads - 1) / threads;
    long long cap = (long long)sdk_num_sms() * 8;       // 8 resident 256-thread CTAs per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

extern "C" int sdk_ddim_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale,
                             const float* noise, float* out, int64_t n, const float* coef_table, int T,
                             const int64_t* t_dev, int64_t t_host, int prediction_type, void* stream) {
    SDK_CHECK_ARG(x && eps_u && out && coef_table, "sdk_ddim_step: null pointer");
    SDK_CHECK_ARG(n >= 0 && T > 0, "sdk_ddim_step: bad sizes n=%lld T=%d", (long long)n, T);
    SDK_CHECK_ARG(prediction_type == 0 || prediction_type == 1, "sdk_ddim_step: prediction_type %d", prediction_type);
    const int vec_ok = aligned16(x) && aligned16(eps_u) && aligned16(out) && (!eps_c || aligned16(eps_c)) && (!noise || aligned16(noise));
    if (n == 0) return SDK_OK;
    int grid = grid_for((n + 3) / 4, 256);
    cudaStream_t s = (cudaStream_t)stream;
    if (prediction_type == 0)
        SDK_CUDA(sdk_launch(step_kernel<0>, dim3(grid), dim3(256), (size_t)(0), s, x, eps_u, eps_c, cfg_scale, noise, out, n, coef_table, T, (const long long*)t_dev, t_host, vec_ok));
    else
        SDK_CUDA(sdk_launch(step_kernel<1>, dim3(grid), dim3(256), (size_t)(0), s, x, eps_u, eps_c, cfg_scale, noise, out, n, coef_table, T, (const long long*)t_dev, t_host, vec_ok));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

extern "C" int sdk_ddim_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                                     const float* orig, int64_t orig_batch, const uint8_t* mask, float* out,
                                     int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                                     const int64_t* t_dev, int64_t t_host, int prediction_type, void* stream) {
    SDK_CHECK_ARG(x && eps_c && orig && mask && out && coef_table, "sdk_ddim_inpaint_step: null pointer");
    SDK_CHECK_ARG(batch >= 0 && channels > 0 && hw > 0 && T > 0, "sdk_ddim_inpaint_step: bad sizes");
    SDK_CHECK_ARG(orig_batch == 1 || orig_batch == batch, "sdk_ddim_inpaint_step: orig batch %lld must be 1 or %lld", (long long)orig_batch, (long long)batch);
    SDK_CHECK_ARG(prediction_type == 0 || prediction_type == 1, "sdk_ddim_inpaint_step: prediction_type %d", prediction_type);
    const long long chw = channels * hw, n = batch * chw;
    if (n == 0) return SDK_OK;
    const long long ostride = orig_batch == 1 ? 0 : chw;
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = grid_for(n, 256);
    if (prediction_type == 0)
        SDK_CUDA(sdk_launch(inpaint_step_kernel<0>, dim3(grid), dim3(256), (size_t)0, s, x, eps_c, eps_u, cfg_scale, orig, ostride, mask, (const float*)nullptr, out, n, chw,
                            (long long)hw, coef_table, T, (const long long*)t_dev, (long long)t_host, (float*)nullptr, 0));
    else
        SDK_CUDA(sdk_launch(inpaint_step_kernel<1>, dim3(grid), dim3(256), (size_t)0, s, x, eps_c, eps_u, cfg_scale, orig, ostride, mask, (const float*)nullptr, out, n, chw,
                            (long long)hw, coef_table, T, (const long long*)t_dev, (long long)t_host, (float*)nullptr, 0));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

// the same loop body with the ancestral DDPM update (the reference's inpaint accepts sampler='ddpm', models/diffusion.py:314-316);
// noise = the randn draw of ddpm.py:80, caller-supplied
extern "C" int sdk_ddpm_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                                     const float* orig, int64_t orig_batch, const uint8_t* mask, const float* noise, float* out,
                                     int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                                     const int64_t* t_dev, int64_t t_host, void* stream) {
    SDK_CHECK_ARG(x && eps_c && orig && mask && noise && out && coef_table, "sdk_ddpm_inpaint_step: null pointer");
    SDK_CHECK_ARG(batch >= 0 && channels > 0 && hw > 0 && T > 0, "sdk_ddpm_inpaint_step: bad sizes");
    SDK_CHECK_ARG(orig_batch == 1 || orig_batch == batch, "sdk_ddpm_inpaint_step: orig batch %lld must be 1 or %lld", (long long)orig_batch, (long long)batch);
    const long long chw = channels * hw, n = batch * chw;
    if (n == 0) return SDK_OK;
    const long long ostride = orig_batch == 1 ? 0 : chw;
    SDK_CUDA(sdk_launch(inpaint_step_kernel<2>, dim3(grid_for(n, 256)), dim3(256), (size_t)0, (cudaStream_t)stream, x, eps_c, eps_u, cfg_scale, orig, ostride, mask,
                        noise, out, n, chw, (long long)hw, coef_table, T, (const long long*)t_dev, (long long)t_host, (float*)nullptr, 0));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

extern "C" int sdk_ddpm_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale,
                             const float* noise, float* out, int64_t n, const float* coef_table, int T,
                             const int64_t* t_dev, int64_t t_host, void* stream) {
    SDK_CHECK_ARG(x && eps_u && out && coef_table && noise, "sdk_ddpm_step: null pointer");
    SDK_CHECK_ARG(n >= 0 && T > 0, "sdk_ddpm_step: bad sizes");
    const int vec_ok = aligned16(x) && aligned16(eps_u) && aligned16(out) && aligned16(noise) && (!eps_c || aligned16(eps_c));
    if (n == 0) return SDK_OK;
    SDK_CUDA(sdk_launch(step_kernel<2>, dim3(grid_for((n + 3) / 4, 256)), dim3(256), (size_t)(0), (cudaStream_t)stream, 
        x, eps_u, eps_c, cfg_scale, noise, out, n, coef_table, T, (const long long*)t_dev, t_host, vec_ok));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

extern "C" int sdk_dpmpp_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale, float* history, int hist_valid,
                              float* out, int64_t n, const float* coef_table, int T, const int64_t* t_dev, int64_t t_host,
                              int prediction_type, void* stream) {
    SDK_CHECK_ARG(x && eps_u && history && out && coef_table, "sdk_dpmpp_step: null pointer");
    SDK_CHECK_ARG(n >= 0 && T > 0, "sdk_dpmpp_step: bad sizes n=%lld T=%d", (long long)n, T);
    SDK_CHECK_ARG(prediction_type == 0 || prediction_type == 1, "sdk_dpmpp_step: prediction_type %d", prediction_type);
    const int vec_ok = aligned16(x) && aligned16(eps_u) && aligned16(out) && aligned16(history) && (!eps_c || aligned16(eps_c));
    if (n == 0) return SDK_OK;
    const int grid = grid_for((n + 3) / 4, 256);
    cudaStream_t s = (cudaStream_t)stream;
    if (prediction_type == 0)
        SDK_CUDA(sdk_launch(dpmpp_step_kernel<0>, dim3(grid), dim3(256), (size_t)0, s, x, eps_u, eps_c, cfg_scale, history, hist_valid, out, n,
                            coef_table, T, (const long long*)t_dev, (long long)t_host, vec_ok));
    else
        SDK_CUDA(sdk_launch(dpmpp_step_kernel<1>, dim3(grid), dim3(256), (size_t)0, s, x, eps_u, eps_c, cfg_scale, history, hist_valid, out, n,
                            coef_table, T, (const long long*)t_dev, (long long)t_host, vec_ok));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

// the inpainting loop body with the DPM-Solver++(2M) update; history: [batch][channels][hw], the previous step's x0 prediction
extern "C" int sdk_dpmpp_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                                      const float* orig, int64_t orig_batch, const uint8_t* mask, float* out,
                                      int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                                      const int64_t* t_dev, int64_t t_host, int prediction_type, float* history, int hist_valid,
                                      void* stream) {
    SDK_CHECK_ARG(x && eps_c && orig && mask && out && coef_table && history, "sdk_dpmpp_inpaint_step: null pointer");
    SDK_CHECK_ARG(batch >= 0 && channels > 0 && hw > 0 && T > 0, "sdk_dpmpp_inpaint_step: bad sizes");
    SDK_CHECK_ARG(orig_batch == 1 || orig_batch == batch, "sdk_dpmpp_inpaint_step: orig batch %lld must be 1 or %lld", (long long)orig_batch, (long long)batch);
    SDK_CHECK_ARG(prediction_type == 0 || prediction_type == 1, "sdk_dpmpp_inpaint_step: prediction_type %d", prediction_type);
    const long long chw = channels * hw, n = batch * chw;
    if (n == 0) return SDK_OK;
    const long long ostride = orig_batch == 1 ? 0 : chw;
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = grid_for(n, 256);
    if (prediction_type == 0)
        SDK_CUDA(sdk_launch(inpaint_step_kernel<3>, dim3(grid), dim3(256), (size_t)0, s, x, eps_c, eps_u, cfg_scale, orig, ostride, mask, (const float*)nullptr, out, n, chw,
                            (long long)hw, coef_table, T, (const long long*)t_dev, (long long)t_host, history, hist_valid));
    else
        SDK_CUDA(sdk_launch(inpaint_step_kernel<4>, dim3(grid), dim3(256), (size_t)0, s, x, eps_c, eps_u, cfg_scale, orig, ostride, mask, (const float*)nullptr, out, n, chw,
                            (long long)hw, coef_table, T, (const long long*)t_dev, (long long)t_host, history, hist_valid));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

extern "C" int sdk_forward_process(const float* x0, const float* noise, float* out, int64_t batch, int64_t per_sample,
                                   const float* coef_table, int T, const int64_t* t_dev, void* stream) {
    SDK_CHECK_ARG(x0 && noise && out && coef_table && t_dev, "sdk_forward_process: null pointer");
    SDK_CHECK_ARG(batch >= 0 && batch < 65536 && per_sample >= 0, "sdk_forward_process: bad sizes");
    if (batch == 0 || per_sample == 0) return SDK_OK;
    dim3 grid(grid_for(per_sample, 256), (unsigned)batch);
    SDK_CUDA(sdk_launch(forward_process_kernel, dim3(grid), dim3(256), (size_t)(0), (cudaStream_t)stream, x0, noise, out, per_sample, coef_table, T, (const long long*)t_dev));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

extern "C" int sdk_x0_from_eps(const float* x, const float* eps, float sigma, float alpha, float* out, int64_t n, void* stream) {
    SDK_CHECK_ARG(x && eps && out, "sdk_x0_from_eps: null pointer");
    if (n <= 0) return SDK_OK;
    SDK_CUDA(sdk_launch(x0_from_eps_kernel, dim3(grid_for(n, 256)), dim3(256), (size_t)(0), (cudaStream_t)stream, x, eps, sigma, alpha, out, n));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}

// ---- loop bookkeeping on the device: t_out[0] = table[counter[0]]; counter[0]++ -------------------
// Lets a whole sampling step (UNet + CFG + scheduler update) be ONE CUDA-graph replay with no host
// work in between: the timestep sequence (host-built, bit-exact) is uploaded once and walked here.
namespace {
__global__ void next_timestep_kernel(const long long* __restrict__ table, int n, int* __restrict__ counter, long long* __restrict__ t_out) {
    pdl_trigger();
    pdl_wait();
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int i = counter[0];
        t_out[0] = (i >= 0 && i < n) ? table[i] : -1;     // -1 poisons the sampler update (NaN) instead of reading out of range
        counter[0] = i + 1;
    }
}
}  // namespace

extern "C" int sdk_next_timestep(const int64_t* table, int n, int* counter, int64_t* t_out, void* stream) {
    SDK_CHECK_ARG(table && counter && t_out && n > 0, "sdk_next_timestep: bad args");
    SDK_CUDA(sdk_launch(next_timestep_kernel, dim3(1), dim3(32), (size_t)(0), (cudaStream_t)stream, (const long long*)table, n, counter, (long long*)t_out));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}


// out[0:row_elems] = table[counter[0] + delta][:]  -- lets the step graph fetch per-step rows of a table that was
// precomputed for the whole timestep grid (the time-embedding projections depend only on the timestep: unet.py:209-220,182-183)
namespace {
__global__ void __launch_bounds__(256)
gather_row_kernel(const float* __restrict__ table, long long row_elems, int n_rows, const int* __restrict__ counter, int delta,
                  float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int row = counter[0] + delta;
    const bool ok = row >= 0 && row < n_rows;
    const float* src = table + (long long)(ok ? row : 0) * row_elems;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < row_elems; i += (long long)gridDim.x * blockDim.x)
        out[i] = ok ? __ldg(src + i) : __int_as_float(0x7fc00000);
}
}  // namespace

extern "C" int sdk_gather_row(const float* table, int64_t row_elems, int n_rows, const int* counter, int delta, float* out, void* stream) {
    SDK_CHECK_ARG(table && counter && out && row_elems > 0 && n_rows > 0, "sdk_gather_row: bad args");
    SDK_CUDA(sdk_launch(gather_row_kernel, dim3(grid_for(row_elems, 256)), dim3(256), (size_t)0, (cudaStream_t)stream, table, (long long)row_elems, n_rows,
                        counter, delta, out));
    SDK_LAUNCH_CHECK();
    return SDK_OK;
}
