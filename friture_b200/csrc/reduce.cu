// Widget-level reductions behind the spectrum widget (SURVEY 8f-1): exponential smoothing across
// the frames of a tick, weighting, dB, arg-max and harmonic product spectrum, fused in one pass
// over the power columns.  Stands behind friture/spectrum.py:158-181 (exp_smoothed_value_2d,
// friture/signal/exp_smoothing.py:59-107; log_spectrogram spectrum.py:95-101;
// harmonic_product_spectrum spectrum.py:103-123).
#include "frt_internal.cuh"

namespace {

__device__ __forceinline__ float lg2_fast(float v) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

__device__ __forceinline__ void argmax_merge(float &best, int &besti, float ob, int oi) {
    if (ob > best || (ob == best && oi < besti)) {
        best = ob;
        besti = oi;
    }
}

__device__ int block_argmax(float best, int besti, float *s_val, int *s_idx) {
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        argmax_merge(best, besti, ob, oi);
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) {
        s_val[w] = best;
        s_idx[w] = besti;
    }
    __syncthreads();
    if (w == 0) {
        const int nw = blockDim.x >> 5;
        best = l < nw ? s_val[l] : -INFINITY;
        besti = l < nw ? s_idx[l] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            argmax_merge(best, besti, ob, oi);
        }
        if (l == 0) s_idx[32] = besti;
    }
    __syncthreads();
    return s_idx[32];
}

__global__ void __launch_bounds__(256)
spectrum_reduce_kernel(const float *__restrict__ power, long long stride_c, long long stride_f,
                       int n_frames, int nbins, float alpha, float *__restrict__ disp,
                       const float *__restrict__ weight, float *__restrict__ db,
                       int *__restrict__ fmax_idx, int *__restrict__ pitch_idx) {
    extern __shared__ float s_sp[];   // [nbins] smoothed power of this channel
    __shared__ float s_val[32];
    __shared__ int s_idx[33];
    const int c = blockIdx.x;
    const float *p = power + (size_t)c * stride_c;
    float *d = disp + (size_t)c * nbins;
    float best = -INFINITY;
    int besti = 0x7fffffff;
    for (int k = threadIdx.x; k < nbins; k += blockDim.x) {
        float s = d[k];
        // s <- alpha x + (1-alpha) s  (exp_smoothing.py:59-107), in complement form s + alpha (x - s):
        // a float32-rounded 1-alpha would shift the time constant by up to 1e-3 at alpha ~ 3.5e-5
        // (N = 32, 5 s) and bias the steady state (tests/test_spectrum_host.py)
        for (int f = 0; f < n_frames; f++)
            s = fmaf(alpha, __ldg(p + (size_t)f * stride_f + k) - s, s);
        d[k] = s;
        s_sp[k] = s;
        float v = 3.01029995663981195f * lg2_fast(s + 1e-30f);   // spectrum.py:95-101
        if (weight) v += __ldg(weight + k);
        db[(size_t)c * nbins + k] = v;
        if (v > best) {
            best = v;
            besti = k;
        }
    }
    const int imax = block_argmax(best, besti, s_val, s_idx);      // spectrum.py:175
    // harmonic product spectrum, 3 harmonics (spectrum.py:103-123)
    const int h = nbins / 3;
    best = -INFINITY;
    besti = 0x7fffffff;
    for (int k = threadIdx.x; k < h; k += blockDim.x) {
        const float r = s_sp[k] * s_sp[2 * k] * s_sp[3 * k];
        if (r > best) {
            best = r;
            besti = k;
        }
    }
    const int ipitch = block_argmax(best, besti, s_val, s_idx);    // spectrum.py:180
    if (threadIdx.x == 0) {
        fmax_idx[c] = imax;
        pitch_idx[c] = ipitch;
    }
}

}   // namespace

extern "C" int frt_spectrum_reduce(frt_handle h, const float *power_dev, int64_t stride_c,
                                   int64_t stride_f, int n_channels, int n_frames, int nbins,
                                   float alpha, float *disp_dev, const float *weight_dev,
                                   float *db_dev, int *fmax_idx_dev, int *pitch_idx_dev,
                                   void *stream) {
    if (!h) return FRT_EINVAL;
    DeviceGuard g(h->device);
    FRT_CHECK_ARG(h, n_channels >= 0 && n_frames >= 0 && nbins >= 3, "bad shape");
    FRT_CHECK_ARG(h, n_frames <= 8192, "more frames than the reference's 8192-tap kernel");
    FRT_CHECK_ARG(h, alpha > 0.f && alpha <= 1.f, "alpha must be in (0, 1]");
    if (n_channels == 0) return FRT_OK;
    FRT_CHECK_ARG(h, (n_frames == 0 || power_dev) && disp_dev && db_dev && fmax_idx_dev &&
                         pitch_idx_dev, "NULL buffer");
    FRT_CHECK_ARG(h, sizeof(float) * (size_t)nbins <= 200 * 1024, "nbins too large");
    const size_t smem = sizeof(float) * (size_t)nbins;
    if (smem > 48 * 1024)
        FRT_CUDA(h, cudaFuncSetAttribute(spectrum_reduce_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    spectrum_reduce_kernel<<<n_channels, 256, smem, (cudaStream_t)stream>>>(
        power_dev, stride_c, stride_f, n_frames, nbins, alpha, disp_dev, weight_dev, db_dev,
        fmax_idx_dev, pitch_idx_dev);
    h->launches++;
    FRT_CUDA(h, cudaGetLastError());
    return FRT_OK;
}

// ---------------------------------------------------------------------------------------------
// Spectrogram display chain (SURVEY 8f-2): dB + weighting -> [0,1] scaling
// (friture/spectrogram.py:127-129,161-162) -> frequency-axis interpolation to the screen rows
// (np.interp on a Mel/Log/... grid, friture/signal/frequency_resampler.py:67-83) -> online linear
// resampling along time to the screen columns (friture/signal/online_linear_2D_resampler.py:61-97,
// friture/signal/linear_interp.py:11-62) -> clip + colour look-up lut[int(v*255)]
// (friture/signal/color_tranform.py:48-51, friture/signal/lookup_table.py:32-52), one kernel.
// The host works out which input column feeds which output column and with what weight (the
// resampler's scalar bookkeeping); the kernel is one thread per output pixel.
namespace {

__device__ __forceinline__ float screen_value(const float *__restrict__ col,
                                              const float *__restrict__ weight, int i0, float t,
                                              float spec_min, float inv_range) {
    // np.interp between bins i0 and i0+1 of (dB + w - spec_min) / (spec_max - spec_min)
    float a = __ldg(col + i0), b = __ldg(col + i0 + 1);
    if (weight) {
        a += __ldg(weight + i0);
        b += __ldg(weight + i0 + 1);
    }
    a = (a - spec_min) * inv_range;
    b = (b - spec_min) * inv_range;
    return fmaf(t, b - a, a);
}

__global__ void display_kernel(const float *__restrict__ db, long long stride_c, long long stride_f,
                               int n_frames, const float *__restrict__ weight, float spec_min,
                               float inv_range, const int *__restrict__ row_i0,
                               const float *__restrict__ row_t, int height,
                               const int *__restrict__ out_col, const float *__restrict__ out_a,
                               int n_out, float *__restrict__ old_data,
                               const unsigned *__restrict__ lut, unsigned *__restrict__ pixels) {
    const int c = blockIdx.y;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)height * (n_out > 0 ? n_out : 1);
    if (gid >= total) return;
    const int r = (int)(gid / (n_out > 0 ? n_out : 1));
    const int o = (int)(gid - (long long)r * (n_out > 0 ? n_out : 1));
    const float *base = db + (size_t)c * stride_c;
    const int i0 = __ldg(row_i0 + r);
    const float t = __ldg(row_t + r);
    if (n_out > 0) {
        const int j = __ldg(out_col + o);       // input column this output column is drawn from
        const float a = __ldg(out_a + o);       // weight of the previous input column
        const float cur = screen_value(base + (size_t)j * stride_f, weight, i0, t, spec_min, inv_range);
        const float old = (j > 0) ? screen_value(base + (size_t)(j - 1) * stride_f, weight, i0, t,
                                                 spec_min, inv_range)
                                  : old_data[(size_t)c * height + r];
        float v = cur * (1.0f - a) + old * a;   // linear_interp.py:56-59
        v = fminf(fmaxf(v, 0.f), 1.f);          // color_tranform.py:50
        pixels[((size_t)c * height + r) * n_out + o] = __ldg(lut + (int)(v * 255.0f));
    }
    // carry the last column of this tick (online_linear_2D_resampler.py "shift"); one writer per row
    // and only after every reader of the old value is done -> done by a second launch (n_out == 0)
    if (n_out == 0 && n_frames > 0)
        old_data[(size_t)c * height + r] =
            screen_value(base + (size_t)(n_frames - 1) * stride_f, weight, i0, t, spec_min, inv_range);
}

}   // namespace

extern "C" int frt_display_columns(frt_handle h, const float *db_dev, int64_t stride_c,
                                   int64_t stride_f, int n_channels, int n_frames, int nbins,
                                   const float *weight_dev, float spec_min, float spec_max,
                                   const int *row_i0_dev, const float *row_t_dev, int height,
                                   const int *out_col_dev, const float *out_a_dev, int n_out,
                                   float *old_data_dev, const uint32_t *lut_dev,
                                   uint32_t *pixels_dev, void *stream) {
    if (!h) return FRT_EINVAL;
    DeviceGuard g(h->device);
    FRT_CHECK_ARG(h, n_channels >= 0 && n_frames >= 0 && height >= 1 && n_out >= 0 && nbins >= 2,
                  "bad shape");
    FRT_CHECK_ARG(h, spec_max != spec_min, "empty dB range");
    if (n_channels == 0 || n_frames == 0) return FRT_OK;
    FRT_CHECK_ARG(h, db_dev && row_i0_dev && row_t_dev && old_data_dev && lut_dev, "NULL buffer");
    FRT_CHECK_ARG(h, n_out == 0 || (out_col_dev && out_a_dev && pixels_dev), "NULL output buffer");
    const float inv_range = 1.0f / (spec_max - spec_min);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_out > 0) {
        const long long total = (long long)height * n_out;
        dim3 grid((unsigned)((total + 255) / 256), (unsigned)n_channels);
        display_kernel<<<grid, 256, 0, st>>>(db_dev, stride_c, stride_f, n_frames, weight_dev,
                                             spec_min, inv_range, row_i0_dev, row_t_dev, height,
                                             out_col_dev, out_a_dev, n_out, old_data_dev,
                                             reinterpret_cast<const unsigned *>(lut_dev),
                                             reinterpret_cast<unsigned *>(pixels_dev));
        h->launches++;
    }
    dim3 grid2((unsigned)((height + 255) / 256), (unsigned)n_channels);
    display_kernel<<<grid2, 256, 0, st>>>(db_dev, stride_c, stride_f, n_frames, weight_dev, spec_min,
                                          inv_range, row_i0_dev, row_t_dev, height, nullptr, nullptr,
                                          0, old_data_dev, reinterpret_cast<const unsigned *>(lut_dev),
                                          nullptr);
    h->launches++;
    FRT_CUDA(h, cudaGetLastError());
    return FRT_OK;
}
