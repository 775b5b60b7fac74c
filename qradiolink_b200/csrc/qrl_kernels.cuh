// qrl_kernels.cuh -- sm_100a device code for the batched-channel IQ DSP hot path.
//
// Numerics contract (see DESIGN.md "Numerics"): compiled with -fmad=false; every fused multiply-add is
// an explicit fmaf(); FIR dot products follow ONE fixed order (polyphase branch r = j mod D accumulated
// oldest-sample-first into lane r mod 32, lanes combined by an xor-butterfly 16,8,4,2,1); sin/cos is
// qrl_sincosf below, never the CUDA libm one.  With that, integer outputs are bit-exact against the
// CPU oracle and float outputs are bit-identical in practice.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>
#include <stdint.h>

#include "qrl_tma.cuh"

namespace qrl {

// ------------------------------------------------------------------------------------------------
// device tables (uploaded once per process by qrl_upload_tables)
// ------------------------------------------------------------------------------------------------
__device__ float d_atan_tab[257];
__device__ float d_tanh_tab[256];
__device__ float d_mmse_tab[129 * 8];
__device__ float d_sine_tab[2048];
#ifdef QRL_SS_PROF
// -DQRL_SS_PROF (tools/ss_prof.py): where the symbol-sync loop warp of CTA 0 spends its cycles (clock64 deltas, summed per launch)
// [0] wait for the hand-off block  [1] wait for the window  [2] uniform rounds  [3] stragglers  [4] hand-off  [5] windows  [6] symbols  [7] rounds
// [8] ns entry -> loop warp starts  [9] ns entry -> first window there  [10] ns entry -> loop warp done  [11] launches (globaltimer)
__device__ long long d_ss_prof[16];
#define SSP(...) __VA_ARGS__
#else
#define SSP(...)
#endif

// ------------------------------------------------------------------------------------------------
// elementary functions shared by all loop kernels
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void qrl_sincosf(float x, float& s, float& c)
{
    // Cody-Waite reduction by pi/2 (3 constants) + Cephes single-precision minimax polynomials
    const float k = rintf(x * 0.636619772f);
    float r = fmaf(k, -1.5703125f, x);
    r = fmaf(k, -4.837512969970703125e-4f, r);
    r = fmaf(k, -7.54978995489188216e-8f, r);
    const int q = static_cast<int>(k) & 3;
    const float z = r * r;
    float ps = fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f);
    ps = fmaf(ps, z, -1.6666654611e-1f);
    ps = ps * z;
    const float sn = fmaf(ps, r, r);
    float pc = fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f);
    pc = fmaf(pc, z, 4.166664568298827e-2f);
    pc = pc * z;
    pc = pc * z;
    float cs = fmaf(z, -0.5f, 1.0f);
    cs = cs + pc;
    // quadrant fix-up without branches (lanes are different channels: a switch would diverge 4 ways):
    // q odd swaps sin/cos; sin is negated for q = 2,3, cos for q = 1,2 (sign-bit flips are exact)
    const bool swap = q & 1;
    const float s_ = swap ? cs : sn, c_ = swap ? sn : cs;
    s = __int_as_float(__float_as_int(s_) ^ ((q & 2) << 30));
    c = __int_as_float(__float_as_int(c_) ^ (((q + 1) & 2) << 30));
}

// gr::fast_atan2f restated (table + octant fix-up)
__device__ __forceinline__ float qrl_fast_atan2f(float y, float x)
{
    const float y_abs = fabsf(y), x_abs = fabsf(x);
    if (!((y_abs > 0.0f) || (x_abs > 0.0f))) return 0.0f;
    const float z = (y_abs < x_abs) ? (y_abs / x_abs) : (x_abs / y_abs);
    float base;
    if (static_cast<double>(z) < 0.003921569) base = z;
    else {
        float alpha = z * 255.0f;
        const int index = static_cast<int>(alpha) & 0xff;
        alpha -= static_cast<float>(index);
        base = d_atan_tab[index];
        base += (d_atan_tab[index + 1] - d_atan_tab[index]) * alpha;
    }
    float angle;
    if (x_abs > y_abs) {
        if (x >= 0.0f) angle = (y >= 0.0f) ? base : -base;
        else { angle = 3.14159265358979323846f; angle = (y >= 0.0f) ? (angle - base) : (base - angle); }
    } else {
        if (y >= 0.0f) { angle = 1.57079632679489661923f; angle = (x >= 0.0f) ? (angle - base) : (angle + base); }
        else { angle = -1.57079632679489661923f; angle = (x >= 0.0f) ? (angle + base) : (angle - base); }
    }
    return angle;
}

__device__ __forceinline__ float qrl_tanhf_lut(float x, const float* __restrict__ tab = d_tanh_tab)
{
    // x > 2 -> 1, x <= -2 -> -1, else table[(int)(128 + 64 x)] -- as selects, one table read
    int index = static_cast<int>(128.0f + 64.0f * fminf(fmaxf(x, -2.0f), 2.0f));
    index = index > 255 ? 255 : index;
    const float t = tab[index];
    return x > 2.0f ? 1.0f : (x <= -2.0f ? -1.0f : t);
}
__device__ __forceinline__ float qrl_clip(float x, float lim) { return x > lim ? lim : (x < -lim ? -lim : x); }

__device__ __forceinline__ unsigned char qrl_soft_u8(float v, float scale)
{
    float t = v * scale;
    t = t + 128.0f;
    float r = rintf(t);
    r = r < 0.0f ? 0.0f : (r > 255.0f ? 255.0f : r);
    return static_cast<unsigned char>(r);
}

// ------------------------------------------------------------------------------------------------
// Stage 1: batched polyphase decimating FIR  y[k] = sum_j h[j] x[D k - j]   (rational_resampler_ccf(1,D))
//   grid  = (strips, channels); one CTA = NOUT consecutive outputs of one channel.
//   lanes = polyphase branches: lane l owns branches r = l + 32*rho and keeps its Q taps per branch in
//   registers; each lane computes K consecutive outputs from (K+Q-1) strided shared-memory samples per
//   branch (register reuse 9K/(K+8) MAC per LDS.64); lane partials are combined with a transposed
//   butterfly (16 SHFL for 2K=16 values) whose association order equals the plain xor-butterfly.
//   Input samples are read once from HBM into shared memory (coalesced 8-byte loads); the previous
//   call's tail (history) comes from a small per-channel buffer.
// ------------------------------------------------------------------------------------------------
// front-end rotator state (gr_demod_base's rotator_cc): exact Q32 phase, phase = base + inc * (n_abs - n_base)
struct RotState { unsigned inc, base; long long n_base; };

// rot != nullptr: the carrier-offset rotator is applied to the window in shared memory right after the fill (same arithmetic as
// rotator_kernel, sample by sample), so a non-zero offset costs no extra pass over HBM (8.16 B per input sample instead of 24);
// the history tail then holds ALREADY ROTATED samples (frontend_hist_kernel), like the reference's resampler history.
template <int D, int Q, int K, int NOUT, int NWARPS>
__global__ void __launch_bounds__(NWARPS * 32)
fir_decim_poly_kernel(const float2* __restrict__ iq, long long iq_stride, long long T,
                      const float2* __restrict__ hist, int H,
                      const float* __restrict__ taps_padded,   // Q*D floats, zero padded
                      float2* __restrict__ out_ring, unsigned ring_mask, long long ring_stride,
                      long long n_in_before, long long k0, long long k1, const RotState* __restrict__ rot = nullptr)
{
    static_assert(K == 8, "transposed butterfly below is written for 2K = 16 values");
    constexpr int R = (D + 31) / 32;                 // branch rounds per lane
    constexpr int W = (NOUT + Q - 1) * D;            // samples in the strip window
    constexpr int WC = (W + 3) & ~1;                 // bulk-copy length: even (16-byte multiple), >= W + 1
    extern __shared__ __align__(128) float2 xs_raw[];   // WC samples
    __shared__ __align__(8) uint64_t fill_bar;

    const int c = blockIdx.y;
    const long long kbase = k0 + static_cast<long long>(blockIdx.x) * NOUT;
    if (kbase >= k1) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // per-lane taps: tap[rho][q] = h[D q + r], r = lane + 32 rho (zero beyond the filter / beyond D)
    float tap[R][Q];
#pragma unroll
    for (int rho = 0; rho < R; rho++) {
        const int r = lane + 32 * rho;
#pragma unroll
        for (int q = 0; q < Q; q++) tap[rho][q] = (r < D) ? taps_padded[D * q + r] : 0.0f;
    }

    // window covers absolute samples [A0, A0 + W); the copy starts one sample early when that makes the
    // global source 16-byte aligned (S0 even relative to the 16-byte aligned channel base)
    const long long A0 = D * kbase - (static_cast<long long>(Q) * D - 1);
    const float2* iqc = iq + static_cast<long long>(c) * iq_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    const long long i0 = A0 - n_in_before;                       // index of the window start in this call's input
    const int shift = static_cast<int>(i0 & 1);                  // 1 -> start the bulk copy at i0 - 1
    const float2* xs = xs_raw + shift;
    const bool bulk = (i0 - shift >= 0) && (i0 - shift + WC <= T) && ((iq_stride & 1) == 0) &&
                      ((reinterpret_cast<unsigned long long>(iq) & 15ull) == 0);
    if (bulk) {
        if (threadIdx.x == 0) { mbar_init(&fill_bar, 1); mbar_fence_init(); }
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(&fill_bar, WC * 8);
            bulk_g2s(xs_raw, iqc + (i0 - shift), WC * 8, &fill_bar);
        }
        mbar_wait(&fill_bar, 0);
    } else {
        float2* xw = xs_raw + shift;
        for (int idx = threadIdx.x; idx < W; idx += NWARPS * 32) {
            const long long i = i0 + idx;
            float2 v = make_float2(0.0f, 0.0f);
            if (i >= 0) { if (i < T) v = __ldg(iqc + i); }
            else if (H + i >= 0) v = hc[H + i];
            xw[idx] = v;
        }
        __syncthreads();
    }
    if (rot) {
        // rotate this call's samples of the window in place (history samples were rotated when they were new)
        const RotState r = rot[c];
        float2* xw = xs_raw + shift;
        for (int idx = threadIdx.x; idx < W; idx += NWARPS * 32) {
            const long long i = i0 + idx;
            if (i < 0 || i >= T) continue;
            const unsigned ph = r.base + r.inc * static_cast<unsigned>(n_in_before + i - r.n_base);
            const float ang = static_cast<float>(static_cast<double>(static_cast<int>(ph)) * (3.14159265358979323846 / 2147483648.0));
            float sn, cs;
            qrl_sincosf(ang, sn, cs);
            const float2 x = xw[idx];
            xw[idx] = make_float2(x.x * cs - x.y * sn, x.x * sn + x.y * cs);
        }
        __syncthreads();
    }

    float* outc = reinterpret_cast<float*>(out_ring + static_cast<long long>(c) * ring_stride);
    for (int b = warp; b < NOUT / K; b += NWARPS) {
        float2 acc[K];                                // (re, im) pairs: one FFMA2 per tap and output
#pragma unroll
        for (int i = 0; i < K; i++) acc[i] = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int rho = 0; rho < R; rho++) {
            int r = lane + 32 * rho;
            if (r > D - 1) r = D - 1;                 // idle lanes read a valid address, taps are zero
            const float2* p = xs + D * K * b + (D - 1 - r);
#pragma unroll
            for (int ip = 0; ip < K + Q - 1; ip++) {  // ip = i - q + (Q-1): ascending = oldest sample first
                const float2 x = p[D * ip];
#pragma unroll
                for (int i = 0; i < K; i++) {
                    const int q = i + (Q - 1) - ip;
                    if (q >= 0 && q < Q) ffma2(acc[i], tap[rho][q], x);
                }
            }
        }
        // transposed butterfly: value v = 2 i + comp; association order == xor-butterfly 16,8,4,2,1
        float a[16];
#pragma unroll
        for (int i = 0; i < K; i++) { a[2 * i] = acc[i].x; a[2 * i + 1] = acc[i].y; }
        {
            const bool hi = lane & 16;
#pragma unroll
            for (int v = 0; v < 8; v++) {
                const float send = hi ? a[v] : a[v + 8];
                const float keep = hi ? a[v + 8] : a[v];
                a[v] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
        }
        {
            const bool hi = lane & 8;
#pragma unroll
            for (int v = 0; v < 4; v++) {
                const float send = hi ? a[v] : a[v + 4];
                const float keep = hi ? a[v + 4] : a[v];
                a[v] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            }
        }
        {
            const bool hi = lane & 4;
#pragma unroll
            for (int v = 0; v < 2; v++) {
                const float send = hi ? a[v] : a[v + 2];
                const float keep = hi ? a[v + 2] : a[v];
                a[v] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
        }
        {
            const bool hi = lane & 2;
            const float send = hi ? a[0] : a[1];
            const float keep = hi ? a[1] : a[0];
            a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
        }
        a[0] = a[0] + __shfl_xor_sync(0xffffffffu, a[0], 1);
        // lane l (even) now holds value v = l >> 1  -> output i = v >> 1, component v & 1
        if ((lane & 1) == 0) {
            const int v = lane >> 1;
            const long long k = kbase + K * b + (v >> 1);
            if (k < k1) outc[2 * (k & ring_mask) + (v & 1)] = a[0];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Stage 1 for small decimations (QPSK-250k: D = 2): each thread owns K consecutive outputs and runs the
// D branch chains itself over a sliding register window; y = tree(S_0..S_{D-1}) with D <= 2 here.
// ------------------------------------------------------------------------------------------------
template <int NTP /*padded taps, even*/, int K, int NTHREADS>
__global__ void __launch_bounds__(NTHREADS)
fir_decim2_kernel(const float2* __restrict__ iq, long long iq_stride, long long T,
                  const float2* __restrict__ hist, int H,
                  const float* __restrict__ taps_padded,   // NTP floats
                  float2* __restrict__ out_ring, unsigned ring_mask, long long ring_stride,
                  long long n_in_before, long long k0, long long k1)
{
    constexpr int D = 2;
    constexpr int NOUT = NTHREADS * K;
    constexpr int W = D * (NOUT - 1) + NTP;              // samples needed by the strip
    constexpr int RUN = D * K;                           // samples per thread-run
    constexpr int PITCH = RUN + 1;                       // +1 float2 pad: lane stride odd -> conflict-free LDS.64
    extern __shared__ float2 xs[];
    __shared__ float hs[NTP];
    const int c = blockIdx.y;
    const long long kbase = k0 + static_cast<long long>(blockIdx.x) * NOUT;
    if (kbase >= k1) return;
    for (int i = threadIdx.x; i < NTP; i += NTHREADS) hs[i] = taps_padded[i];
    const long long A0 = D * kbase - (NTP - 1);
    const float2* iqc = iq + static_cast<long long>(c) * iq_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    for (int idx = threadIdx.x; idx < W; idx += NTHREADS) {
        const long long i = A0 + idx - n_in_before;
        float2 v = make_float2(0.0f, 0.0f);
        if (i >= 0) { if (i < T) v = __ldg(iqc + i); }
        else if (H + i >= 0) v = hc[H + i];
        xs[idx + idx / RUN] = v;                          // padded layout
    }
    __syncthreads();
    // thread t: outputs kbase + K t + i ; newest sample of output i at window index (NTP-1) + D (K t + i)
    float2 s0[K], s1[K];                                 // branch chains j even / j odd, (re, im) pairs: FFMA2
#pragma unroll
    for (int i = 0; i < K; i++) { s0[i] = make_float2(0.0f, 0.0f); s1[i] = make_float2(0.0f, 0.0f); }
    const int t = threadIdx.x;
    // walk window offsets w = 0 .. NTP-1 + D(K-1): sample index = D K t + w ; tap for output i: j = (NTP-1) + D i - w
#pragma unroll
    for (int w = 0; w < NTP + D * (K - 1); w++) {
        const int idx = D * K * t + w;
        const float2 x = xs[idx + idx / RUN];
#pragma unroll
        for (int i = 0; i < K; i++) {
            const int j = (NTP - 1) + D * i - w;
            if (j >= 0 && j < NTP) {
                const float h = hs[j];
                if ((j & 1) == 0) ffma2(s0[i], h, x);
                else ffma2(s1[i], h, x);
            }
        }
    }
    float2* outc = out_ring + static_cast<long long>(c) * ring_stride;
#pragma unroll
    for (int i = 0; i < K; i++) {
        const long long k = kbase + K * t + i;
        if (k < k1) outc[k & ring_mask] = make_float2(s0[i].x + s1[i].x, s0[i].y + s1[i].y);
    }
}

// ------------------------------------------------------------------------------------------------
// Stage 1 for the 10k modes: rational_resampler_ccf(L = 2, M = 25), 209 taps -> two arms of 105 taps.
// output i uses arm (i M) mod L at input position floor(i M / L); each arm is accumulated oldest-first.
// First version: one thread per output from a shared-memory window (cooperative fill).
// ------------------------------------------------------------------------------------------------
template <int L, int M, int NT /* taps per arm */, int NOUT>
__global__ void __launch_bounds__(256)
fir_resamp_ccf_kernel(const float2* __restrict__ iq, long long iq_stride, long long T,
                      const float2* __restrict__ hist, int H,
                      const float* __restrict__ arms /* [L][NT] */,
                      float2* __restrict__ out_ring, unsigned ring_mask, long long ring_stride,
                      long long n_in_before, long long k0, long long k1)
{
    constexpr int SPAN = (NOUT * M + L - 1) / L + NT + 1;      // input samples covering NOUT outputs
    extern __shared__ float2 xs_rs[];
    __shared__ float hs[L * NT];
    const int c = blockIdx.y;
    const long long kbase = k0 + static_cast<long long>(blockIdx.x) * NOUT;
    if (kbase >= k1) return;
    for (int i = threadIdx.x; i < L * NT; i += 256) hs[i] = arms[i];
    const long long pos0 = (kbase * M) / L;                    // input position of the first output
    const long long A0 = pos0 - (NT - 1);
    const float2* iqc = iq + static_cast<long long>(c) * iq_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    for (int idx = threadIdx.x; idx < SPAN; idx += 256) {
        const long long i = A0 + idx - n_in_before;
        float2 v = make_float2(0.0f, 0.0f);
        if (i >= 0) { if (i < T) v = __ldg(iqc + i); }
        else if (H + i >= 0) v = hc[H + i];
        xs_rs[idx] = v;
    }
    __syncthreads();
    float2* outc = out_ring + static_cast<long long>(c) * ring_stride;
    for (int o = threadIdx.x; o < NOUT; o += 256) {
        const long long k = kbase + o;
        if (k >= k1) break;
        const long long pos = (k * M) / L;
        const float* h = hs + static_cast<int>((k * M) % L) * NT;
        const float2* p = xs_rs + (pos - A0);                 // newest sample of this output
        float re = 0.0f, im = 0.0f;
#pragma unroll 5
        for (int j = NT - 1; j >= 0; j--) {
            const float2 v = p[-j];
            re = fmaf(h[j], v.x, re);
            im = fmaf(h[j], v.y, im);
        }
        outc[k & ring_mask] = make_float2(re, im);
    }
}

// ------------------------------------------------------------------------------------------------
// Low-rate stream stages (20 ksps .. 500 ksps): ring -> ring, one thread per output item, taps in smem,
// sequential oldest-first accumulation (the D = 1 case of the FIR order).
// ------------------------------------------------------------------------------------------------
constexpr int kMaxTapsSmem = 4096;

// complex stream, real taps (fft_filter_ccf restated in direct form); optional linear copy (port 0)
__global__ void fir_ccf_ring_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                                    float2* __restrict__ out, unsigned out_mask, long long out_stride,
                                    const float* __restrict__ taps, int ntaps, long long a0, long long a1,
                                    float2* __restrict__ lin, long long lin_stride, long long lin_base, int out_interleaved)
{
    extern __shared__ float hs_dyn[];
    for (int i = threadIdx.x; i < ntaps; i += blockDim.x) hs_dyn[i] = taps[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float2 y = make_float2(0.0f, 0.0f);
    for (int j = ntaps - 1; j >= 0; j--) ffma2(y, hs_dyn[j], x[(a - j) & in_mask]);
    if (out_interleaved) out[(static_cast<long long>(c >> 5) * out_stride + (a & out_mask)) * 32 + (c & 31)] = y;
    else out[static_cast<long long>(c) * out_stride + (a & out_mask)] = y;
    if (lin) lin[static_cast<long long>(c) * lin_stride + (a - lin_base)] = y;
}

// Register-tiled form of fir_ccf_ring_kernel (round 2): one CTA = NT * K consecutive outputs of one channel.  The tile's samples
// (+ ntaps - 1 of history) and the taps sit in shared memory; thread t owns K consecutive outputs and walks the samples oldest
// first, so every sample is loaded once (one LDS.64) and meets K taps that slide through a register window (one broadcast LDS.32
// per step): 2 LDS per K FFMA2 instead of 2 loads per FFMA2.  Per output the accumulation order is the ring kernel's (tap index
// descending = oldest sample first): results are bit-identical.  Sample index i lives at i + i / 16 (one pad slot per 16): the K-strided
// LDS.64 of a half-warp then hit distinct bank pairs.
template <int K, int NT>
__global__ void __launch_bounds__(NT)
fir_ccf_ring_tiled_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                          float2* __restrict__ out, unsigned out_mask, long long out_stride,
                          const float* __restrict__ taps, int ntaps, long long a0, long long a1,
                          float2* __restrict__ lin, long long lin_stride, long long lin_base, int out_interleaved)
{
    extern __shared__ __align__(16) float sm_tl[];
    constexpr int TILE = K * NT;
    float* hs = sm_tl;                                                    // ntaps floats (rounded up to even)
    float2* xs = reinterpret_cast<float2*>(sm_tl + ((ntaps + 1) & ~1));   // (TILE + ntaps - 1) samples, padded layout
    const int c = blockIdx.y;
    const long long tile0 = a0 + static_cast<long long>(blockIdx.x) * TILE;
    if (tile0 >= a1) return;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < ntaps; i += NT) hs[i] = taps[i];
    const int span = TILE + ntaps - 1;
    for (int i = threadIdx.x; i < span; i += NT) xs[i + (i >> 4)] = x[(tile0 - (ntaps - 1) + i) & in_mask];
    __syncthreads();
    float2 acc[K];
#pragma unroll
    for (int i = 0; i < K; i++) acc[i] = make_float2(0.0f, 0.0f);
    const int base = K * threadIdx.x;                  // xs index of the oldest sample of my output 0
    // step t meets sample base + t with tap j = i + (ntaps - 1) - t for output i; w[i] holds that tap (slides by one per step)
    float w[K];
#pragma unroll
    for (int i = 0; i < K; i++) w[i] = 0.0f;
    // head: t = 0 .. K-2, outputs i <= t are inside the filter
#pragma unroll
    for (int t = 0; t < K - 1; t++) {
#pragma unroll
        for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
        w[0] = hs[ntaps - 1 - t];
        const int idx = base + t;
        const float2 v = xs[idx + (idx >> 4)];
#pragma unroll
        for (int i = 0; i <= t; i++) ffma2(acc[i], w[i], v);
    }
    // main: t = K-1 .. ntaps-1, all K outputs.  Step K-1 and the last (ntaps mod K) steps shift the window register by register; the rest
    // runs K steps per iteration with the window ROTATING through the registers (step u of an iteration writes its tap to w[K-1-u] and
    // output i reads w[K-1 - ((u - i) mod K)]: all indices compile-time, so the K-1 moves per step are gone -- they were 7 of the 20
    // instructions per 8 FFMA).  After a whole iteration the window is in shifted order again.  Same taps meet the same samples in the
    // same order: bit-identical.
    auto shift_steps = [&](int ta, int tb) {
        for (int t = ta; t < tb; t++) {
#pragma unroll
            for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
            w[0] = hs[ntaps - 1 - t];
            const int idx = base + t;
            const float2 v = xs[idx + (idx >> 4)];
#pragma unroll
            for (int i = 0; i < K; i++) ffma2(acc[i], w[i], v);
        }
    };
    // rotating iterations start on a multiple of K (= 8): base + t0 is then a multiple of 8 as well, the 8 samples of an iteration sit
    // in one padding block and are addressed by immediates from one base
    static_assert(K == 8, "the rotating main phase assumes 8 outputs per thread (one padding block per iteration)");
    const int t_a = K, t_b = t_a + ((ntaps - t_a) / K) * K;
    shift_steps(K - 1, t_a < ntaps ? t_a : ntaps);
    for (int t0 = t_a; t0 < t_b; t0 += K) {
        const int idx0 = base + t0;
        const float2* xv = xs + idx0 + (idx0 >> 4);
        const float* hv = hs + (ntaps - 1 - t0);
#pragma unroll
        for (int u = 0; u < K; u++) {
            w[K - 1 - u] = hv[-u];
            const float2 v = xv[u];
#pragma unroll
            for (int i = 0; i < K; i++) ffma2(acc[i], w[K - 1 - ((u - i + K) % K)], v);
        }
    }
    shift_steps(t_b > t_a ? t_b : (t_a < ntaps ? t_a : ntaps), ntaps);
    // tail: t = ntaps .. ntaps+K-2, outputs i >= t - (ntaps - 1)
#pragma unroll
    for (int u = 1; u < K; u++) {
#pragma unroll
        for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
        const int idx = base + ntaps - 1 + u;
        const float2 v = xs[idx + (idx >> 4)];
#pragma unroll
        for (int i = u; i < K; i++) ffma2(acc[i], w[i], v);
    }
#pragma unroll
    for (int i = 0; i < K; i++) {
        const long long a = tile0 + base + i;
        if (a >= a1) break;
        if (out_interleaved) out[(static_cast<long long>(c >> 5) * out_stride + (a & out_mask)) * 32 + (c & 31)] = acc[i];
        else out[static_cast<long long>(c) * out_stride + (a & out_mask)] = acc[i];
        if (lin) lin[static_cast<long long>(c) * lin_stride + (a - lin_base)] = acc[i];
    }
}

// quadrature_demod_cf + real FIR, register-tiled like the kernel above (K outputs per thread, taps through a register window).
// The CTA first demodulates its tile + ntaps - 1 of history into shared memory, then filters from there.
template <int K, int NT>
__global__ void __launch_bounds__(NT)
qdemod_fir_fff_tiled_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                            float* __restrict__ out, unsigned out_mask, long long out_stride,
                            const float* __restrict__ taps, int ntaps, float gain, long long a0, long long a1)
{
    extern __shared__ __align__(16) float sm_tl[];
    constexpr int TILE = K * NT;
    float* hs = sm_tl;                         // ntaps
    float* ds = sm_tl + ntaps;                 // TILE + ntaps - 1 demodulated samples, index i at i + i / 32
    const int c = blockIdx.y;
    const long long tile0 = a0 + static_cast<long long>(blockIdx.x) * TILE;
    if (tile0 >= a1) return;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < ntaps; i += NT) hs[i] = taps[i];
    const int span = TILE + ntaps - 1;
    for (int i = threadIdx.x; i < span; i += NT) {
        const long long n = tile0 - (ntaps - 1) + i;       // absolute demod index
        float d = 0.0f;
        if (n >= 0 && n < a1) {
            const float2 cur = x[n & in_mask];
            float2 prev = make_float2(0.0f, 0.0f);
            if (n >= 1) prev = x[(n - 1) & in_mask];
            const float re = cur.x * prev.x + cur.y * prev.y;
            const float im = cur.y * prev.x - cur.x * prev.y;
            d = gain * qrl_fast_atan2f(im, re);
        }
        ds[i + (i >> 5)] = d;
    }
    __syncthreads();
    float acc[K], w[K];
#pragma unroll
    for (int i = 0; i < K; i++) { acc[i] = 0.0f; w[i] = 0.0f; }
    const int base = K * threadIdx.x;
#pragma unroll
    for (int t = 0; t < K - 1; t++) {
#pragma unroll
        for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
        w[0] = hs[ntaps - 1 - t];
        const int idx = base + t;
        const float v = ds[idx + (idx >> 5)];
#pragma unroll
        for (int i = 0; i <= t; i++) acc[i] = fmaf(w[i], v, acc[i]);
    }
    // (main phase: a few shifting steps, then K steps per iteration with the window rotating through the registers -- see
    // fir_ccf_ring_tiled_kernel)
    auto shift_steps = [&](int ta, int tb) {
        for (int t = ta; t < tb; t++) {
#pragma unroll
            for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
            w[0] = hs[ntaps - 1 - t];
            const int idx = base + t;
            const float v = ds[idx + (idx >> 5)];
#pragma unroll
            for (int i = 0; i < K; i++) acc[i] = fmaf(w[i], v, acc[i]);
        }
    };
    static_assert(K == 8, "the rotating main phase assumes 8 outputs per thread (one padding block per iteration)");
    const int t_a = K, t_b = t_a + ((ntaps - t_a) / K) * K;
    shift_steps(K - 1, t_a < ntaps ? t_a : ntaps);
    for (int t0 = t_a; t0 < t_b; t0 += K) {
        const int idx0 = base + t0;
        const float* dv = ds + idx0 + (idx0 >> 5);
        const float* hv = hs + (ntaps - 1 - t0);
#pragma unroll
        for (int u = 0; u < K; u++) {
            w[K - 1 - u] = hv[-u];
            const float v = dv[u];
#pragma unroll
            for (int i = 0; i < K; i++) acc[i] = fmaf(w[K - 1 - ((u - i + K) % K)], v, acc[i]);
        }
    }
    shift_steps(t_b > t_a ? t_b : (t_a < ntaps ? t_a : ntaps), ntaps);
#pragma unroll
    for (int u = 1; u < K; u++) {
#pragma unroll
        for (int i = K - 1; i > 0; i--) w[i] = w[i - 1];
        const int idx = base + ntaps - 1 + u;
        const float v = ds[idx + (idx >> 5)];
#pragma unroll
        for (int i = u; i < K; i++) acc[i] = fmaf(w[i], v, acc[i]);
    }
#pragma unroll
    for (int i = 0; i < K; i++) {
        const long long a = tile0 + base + i;
        if (a >= a1) break;
        out[(static_cast<long long>(c >> 5) * out_stride + (a & out_mask)) * 32 + (c & 31)] = acc[i];
    }
}

// quadrature_demod_cf fused in front of a real FIR (RRC shaping filter): in = complex ring, out = float ring.
// Each CTA demodulates its tile (+ntaps-1 halo) into shared memory, then filters from there.
__global__ void qdemod_fir_fff_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                                      float* __restrict__ out, unsigned out_mask, long long out_stride,
                                      const float* __restrict__ taps, int ntaps, float gain,
                                      long long a0, long long a1, float* __restrict__ demod_dbg, long long dbg_stride)
{
    extern __shared__ float sm_dyn[];
    float* hs = sm_dyn;                 // ntaps
    float* ds = sm_dyn + ntaps;         // blockDim.x + ntaps - 1 demodulated samples
    for (int i = threadIdx.x; i < ntaps; i += blockDim.x) hs[i] = taps[i];
    const int c = blockIdx.y;
    const long long tile0 = a0 + static_cast<long long>(blockIdx.x) * blockDim.x;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    const int span = blockDim.x + ntaps - 1;
    for (int i = threadIdx.x; i < span; i += blockDim.x) {
        const long long n = tile0 - (ntaps - 1) + i;       // absolute demod index
        float d = 0.0f;
        if (n >= 0 && n < a1) {
            const float2 cur = x[n & in_mask];
            float2 prev = make_float2(0.0f, 0.0f);
            if (n >= 1) prev = x[(n - 1) & in_mask];
            const float re = cur.x * prev.x + cur.y * prev.y;
            const float im = cur.y * prev.x - cur.x * prev.y;
            d = gain * qrl_fast_atan2f(im, re);
        }
        ds[i] = d;
        if (demod_dbg && n >= a0 && n < a1 && i >= ntaps - 1) demod_dbg[static_cast<long long>(c) * dbg_stride + (n - a0)] = d;
    }
    __syncthreads();
    const long long a = tile0 + threadIdx.x;
    if (a >= a1) return;
    float acc = 0.0f;
    const float* p = ds + threadIdx.x + (ntaps - 1);       // newest sample of this output
    for (int j = ntaps - 1; j >= 0; j--) acc = fmaf(hs[j], p[-j], acc);
    // channel-interleaved ring: [c / 32][slot][c % 32]  (one warp of the symbol-sync kernel = one 128-byte row per time step)
    out[(static_cast<long long>(c >> 5) * out_stride + (a & out_mask)) * 32 + (c & 31)] = acc;
}

// Channel-interleaved float ring [c / 32][slot][c % 32] -> linear per-channel port buffer [c][a - a0] (gr_demod_dmr's port 3:
// the symbol filter output, gr_demod_dmr.cpp:103).  grid = (tiles of blockDim.x samples, 32-channel groups), block = (32, ty):
// reads are whole 128-byte rows of the ring, writes go through a shared-memory transpose so each channel stores runs of 32 floats.
__global__ void ring_to_port_f32_kernel(const float* __restrict__ ring, unsigned mask, long long stride, int C,
                                        long long a0, long long a1, float* __restrict__ port, long long port_stride, long long port_off)
{
    __shared__ float tile[32][33];
    const int g = blockIdx.y, lane = threadIdx.x;
    const long long t0 = a0 + static_cast<long long>(blockIdx.x) * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long a = t0 + r;
        tile[r][lane] = (a < a1) ? ring[(static_cast<long long>(g) * stride + (a & mask)) * 32 + lane] : 0.0f;
    }
    __syncthreads();
    for (int ch = threadIdx.y; ch < 32; ch += blockDim.y) {
        const int c = g * 32 + ch;
        const long long a = t0 + lane;
        if (c < C && a < a1 && port_off + (a - a0) < port_stride)
            port[static_cast<long long>(c) * port_stride + port_off + (a - a0)] = tile[lane][ch];
    }
}

// THE FIR order for one output inside one thread: 32 partial sums (branch r = j mod D accumulated oldest sample first
// into slot r mod 32), combined 16, 8, 4, 2, 1 like the warp butterfly.  fetch(j) returns the sample that meets tap j.
template <class Fetch>
__device__ __forceinline__ float2 qrl_fir_dot_order_c(const float* __restrict__ taps, int ntaps, int D, Fetch fetch)
{
    float sr[32], si[32];
#pragma unroll
    for (int l = 0; l < 32; l++) { sr[l] = 0.0f; si[l] = 0.0f; }
    for (int r = 0; r < D && r < ntaps; r++) {
        float a = sr[r & 31], b = si[r & 31];
        for (int q = (ntaps - 1 - r) / D; q >= 0; q--) {
            const int j = D * q + r;
            const float2 v = fetch(j);
            a = fmaf(taps[j], v.x, a); b = fmaf(taps[j], v.y, b);
        }
        sr[r & 31] = a; si[r & 31] = b;
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1)
#pragma unroll
        for (int l = 0; l < off; l++) { sr[l] = sr[l] + sr[l + off]; si[l] = si[l] + si[l + off]; }
    return make_float2(sr[0], si[0]);
}

// Shape-generic stage 1 (any decimation / tap count) with the call-to-call history of the tiled instances: one thread per
// output.  Used for the stage-1 shapes that have no register-tiled instance (WBFM: /5, 41 taps).
__global__ void __launch_bounds__(128)
fir_decim_hist_generic_kernel(const float2* __restrict__ iq, long long iq_stride, long long T, const float2* __restrict__ hist, int H,
                              const float* __restrict__ taps, int ntaps, int D,
                              float2* __restrict__ out_ring, unsigned ring_mask, long long ring_stride,
                              long long n_in_before, long long k0, long long k1)
{
    const int c = blockIdx.y;
    const long long k = k0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k >= k1) return;
    const float2* x = iq + static_cast<long long>(c) * iq_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    const long long newest = static_cast<long long>(D) * k - n_in_before;          // index of x[D k] in this call's input
    const float2 y = qrl_fir_dot_order_c(taps, ntaps, D, [&](int j) {
        const long long i = newest - j;
        if (i >= 0) return i < T ? x[i] : make_float2(0.0f, 0.0f);
        return (H + i >= 0) ? hc[H + i] : make_float2(0.0f, 0.0f);
    });
    out_ring[static_cast<long long>(c) * ring_stride + (k & ring_mask)] = y;
}

// Shape-generic rational stage 1 (rational_resampler_ccf(L, M), L > 1): output i takes arm (i M) mod L at input position
// floor(i M / L); arms[p][k] = taps[p + k L]; plain oldest-first accumulation (the oracle's order for L > 1).  One thread per
// output; used for the shapes that have no tiled instance (M17: x3 / 125, 349 taps per arm).
__global__ void __launch_bounds__(128)
fir_resamp_hist_generic_kernel(const float2* __restrict__ iq, long long iq_stride, long long T, const float2* __restrict__ hist, int H,
                               const float* __restrict__ arms /* [L][nt] */, int nt, int L, int M,
                               float2* __restrict__ out_ring, unsigned ring_mask, long long ring_stride,
                               long long n_in_before, long long k0, long long k1)
{
    const int c = blockIdx.y;
    const long long i = k0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= k1) return;
    const float2* x = iq + static_cast<long long>(c) * iq_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    const long long im = i * M;
    const int p = static_cast<int>(im % L);
    const long long newest = im / L - n_in_before;                       // index of the newest sample in this call's input
    const float* h = arms + static_cast<long long>(p) * nt;
    float re = 0.0f, imv = 0.0f;
    for (int k = nt - 1; k >= 0; k--) {
        const long long a = newest - k;
        float2 v;
        if (a >= 0) v = a < T ? x[a] : make_float2(0.0f, 0.0f);
        else v = (H + a >= 0) ? hc[H + a] : make_float2(0.0f, 0.0f);
        re = fmaf(h[k], v.x, re); imv = fmaf(h[k], v.y, imv);
    }
    out_ring[static_cast<long long>(c) * ring_stride + (i & ring_mask)] = make_float2(re, imv);
}

// Stand-alone batched decimating FIR for any (ntaps, D), zero history: y[k] = sum_j h[j] x[D k - j] in THE FIR order
// (branch r = j mod D oldest-first into lane r mod 32, lanes combined 16, 8, 4, 2, 1).  One warp per output; this is the
// shape-generic entry point behind qrl_fir_decim_ccf_device (the chains use the register-tiled instances above).
__global__ void __launch_bounds__(256)
fir_decim_generic_kernel(const float* __restrict__ taps, int ntaps, int D, const float2* __restrict__ x, long long T, long long x_stride,
                         float2* __restrict__ y, long long y_stride, long long nout)
{
    const int lane = threadIdx.x & 31, c = blockIdx.y;
    const float2* xc = x + static_cast<long long>(c) * x_stride;
    float2* yc = y + static_cast<long long>(c) * y_stride;
    const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
    for (long long k = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); k < nout; k += warps) {
        float re = 0.0f, im = 0.0f;
        for (int r = lane; r < D && r < ntaps; r += 32) {
            for (int q = (ntaps - 1 - r) / D; q >= 0; q--) {
                const int j = D * q + r;
                const long long n = D * k - j;
                const float2 v = (n >= 0 && n < T) ? xc[n] : make_float2(0.0f, 0.0f);
                re = fmaf(taps[j], v.x, re); im = fmaf(taps[j], v.y, im);
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            re = re + __shfl_down_sync(0xffffffffu, re, off);
            im = im + __shfl_down_sync(0xffffffffu, im, off);
        }
        if (lane == 0) yc[k] = make_float2(re, im);
    }
}

// ------------------------------------------------------------------------------------------------
// Sequential loop stage: symbol_sync (PI clock loop, mod. Mueller&Muller TED, 8-tap MMSE interpolator)
// One lane per channel; a warp stages 32 channels x CH samples in shared memory with coalesced loads,
// then every lane runs its own loop from shared memory.  Epilogues:
//   EPI_4FSK_FM : float symbols -> phase_modulator_fc(pi/2) -> port1, soft bits (imag, real)
//   EPI_CPLX    : complex symbols -> port1, soft bits (real, imag)          (4FSK non-FM)
//   EPI_QPSK    : complex symbols -> costas(4, snr) -> diff_phasor -> rotate -> port1, soft bits
// ------------------------------------------------------------------------------------------------
enum { SL_RECT4 = 0, SL_DQPSK = 1, SL_BPSK = 2 };
//   EPI_EXT_4FSK_FM : as EPI_4FSK_FM, but the symbols leave the SM as they are (TMA bulk store of each hand-off
//                 block to a scratch buffer) and symsync_ext_epilogue_kernel does the phase modulator / soft bits
//                 on the wide SM partition: the scattered per-channel stores no longer share the MIO queue with the
//                 recurrence's shared-memory loads
enum { EPI_4FSK_FM = 0, EPI_CPLX = 1, EPI_QPSK = 2, EPI_BPSK = 3, EPI_REAL1 = 4, EPI_EXT_4FSK_FM = 5 };
enum { LOOP_SYMSYNC = 0, LOOP_CRMM = 1 };

struct LoopState {               // control_loop (costas)
    float phase, freq;
};
struct SymSyncState {
    long long ii;                // absolute index of the first unconsumed input sample
    long long n_sym;             // symbols produced so far (absolute)
    long long n_soft;            // soft bits produced so far (absolute, = write index of the soft ring)
    float avg_period, inst_period, mu;
    float xr[3], xi[3], dr[3], di[3];
    LoopState costas;            // second Costas loop (EPI_QPSK)
    float dp_r, dp_i;            // diff_phasor memory
};
__host__ __device__ inline int symsync_stride(int ch, int lookahead) { return ch - ((lookahead + 31) & ~31); }
constexpr int SYMSYNC_TAB_FLOATS = 132 * 8 + 129 * 12 + 4;   // tap-major bank + entry-major bank (16-byte pitch multiple)
struct SymSyncParams {
    float sps, alpha, beta, max_period, min_period;
    int lookahead;
    float pm_sens, soft_scale;
    float costas_alpha, costas_beta;
    float rot_r, rot_i;
    float fl0; int n0;           // n0 = floor(min_period - |alpha|) as float / int (fast floor window)
    int loop_kind;               // LOOP_SYMSYNC (symbol_sync_xx) or LOOP_CRMM (clock_recovery_mm_cc)
    float gain_omega, gain_mu, omega_mid, omega_lim;      // clock_recovery_mm_cc
    int costas_order;
    float sym_scale = 1.0f;      // gr_demod_dmr: multiply_const_ff(0.9) between the symbol sync and the phase modulator
    int reserved_[3] = { 0, 0, 0 };   // keeps the kernel parameters behind this struct on their 16-byte offsets (paired constant loads)
};

__device__ __forceinline__ void qrl_slice(int slicer, float re, float im, float& dr, float& di)
{
    if (slicer == SL_RECT4) {
        int sec = static_cast<int>(floorf(re + 2.0f));
        sec = sec < 0 ? 0 : (sec > 3 ? 3 : sec);
        dr = -1.5f + static_cast<float>(sec); di = 0.0f;
    } else if (slicer == SL_DQPSK) {
        dr = re > 0.0f ? 0.707107f : -0.707107f;
        di = im > 0.0f ? 0.707107f : -0.707107f;
    } else {
        dr = re > 0.0f ? 1.0f : -1.0f; di = 0.0f;
    }
}

__device__ __forceinline__ void qrl_costas_step(LoopState& st, float alpha, float beta, int order, bool use_snr,
                                                float xr, float xi, float& yr, float& yi,
                                                const float* __restrict__ tanh_tab = d_tanh_tab)
{
    float sn, cs;
    qrl_sincosf(-st.phase, sn, cs);
    const float orr = xr * cs - xi * sn;
    const float oi = xr * sn + xi * cs;
    float err;
    if (order == 2) {
        if (use_snr) { const float snr = orr * orr + oi * oi; err = qrl_tanhf_lut(snr * orr, tanh_tab) * oi; }
        else err = orr * oi;
    } else {
        if (use_snr) {
            const float snr = orr * orr + oi * oi;
            err = qrl_tanhf_lut(snr * orr, tanh_tab) * oi - qrl_tanhf_lut(snr * oi, tanh_tab) * orr;
        } else {
            err = (orr > 0.0f ? 1.0f : -1.0f) * oi - (oi > 0.0f ? 1.0f : -1.0f) * orr;
        }
    }
    err = qrl_clip(err, 1.0f);
    st.freq = st.freq + beta * err;
    st.phase = st.phase + st.freq + alpha * err;
    // (double)phase > 2*pi  <=>  phase >= 6.28318548f (the float just above 2*pi): float compare on the hot path,
    // the exact double subtraction only when a wrap really happens
    while (st.phase >= 6.2831854820251465f)
        st.phase = static_cast<float>(static_cast<double>(st.phase) - 2.0 * 3.14159265358979323846);
    while (st.phase <= -6.2831854820251465f)
        st.phase = static_cast<float>(static_cast<double>(st.phase) + 2.0 * 3.14159265358979323846);
    if (st.freq > 1.0f) st.freq = 1.0f;
    else if (st.freq < -1.0f) st.freq = -1.0f;
    yr = orr; yi = oi;
}

// ------------------------------------------------------------------------------------------------
// costas_loop_cc(order 4, use_snr) step for the per-sample recurrence of the QPSK chain, restated for a lone warp
// (same values as qrl_costas_step, bit for bit; no conversion instruction on the chain):
//   * |phase| < 2*pi + 2 here, so rintf(x * 2/pi) is the magic-number add (exact for |v| < 2^22) and its low
//     mantissa bits are the quadrant;
//   * the tanh table index floor(128 + 64 x) is an FADD with round-toward-minus-infinity onto 2^23;
//   * the 2*pi wrap (exact double subtraction) sits behind one unlikely branch.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void qrl_sincosf_small(float x, float& s, float& c)
{
    const float kb = (x * 0.636619772f) + 12582912.0f;       // == rintf(x * 0.636619772f) + 1.5 * 2^23: the product is rounded
                                                             // first (no fma), the add then rounds to nearest-even integer
    const float k = kb - 12582912.0f;
    const int q = __float_as_int(kb);
    float r = fmaf(k, -1.5703125f, x);
    r = fmaf(k, -4.837512969970703125e-4f, r);
    r = fmaf(k, -7.54978995489188216e-8f, r);
    const float z = r * r;
    float ps = fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f);
    ps = fmaf(ps, z, -1.6666654611e-1f);
    ps = ps * z;
    const float sn = fmaf(ps, r, r);
    float pc = fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f);
    pc = fmaf(pc, z, 4.166664568298827e-2f);
    pc = pc * z;
    pc = pc * z;
    float cs = fmaf(z, -0.5f, 1.0f);
    cs = cs + pc;
    const bool swap = q & 1;
    const float s_ = swap ? cs : sn, c_ = swap ? sn : cs;
    s = __int_as_float(__float_as_int(s_) ^ ((q & 2) << 30));
    c = __int_as_float(__float_as_int(c_) ^ (((q + 1) & 2) << 30));
}
__device__ __forceinline__ float qrl_tanhf_lut_rd(float x, const float* __restrict__ tab)
{
    const float v = 128.0f + 64.0f * fminf(fmaxf(x, -2.0f), 2.0f);          // in [0, 256]
    int index = __float_as_int(__fadd_rd(v, 8388608.0f)) & 0x1ff;           // floor(v): what static_cast<int>(v) gives
    index = index > 255 ? 255 : index;
    const float t = tab[index];
    return x > 2.0f ? 1.0f : (x <= -2.0f ? -1.0f : t);
}
__device__ __forceinline__ void qrl_costas4_snr_step(LoopState& st, float alpha, float beta, float xr, float xi,
                                                     float& yr, float& yi, const float* __restrict__ tanh_tab)
{
    float sn, cs;
    qrl_sincosf_small(-st.phase, sn, cs);
    const float orr = xr * cs - xi * sn;
    const float oi = xr * sn + xi * cs;
    const float snr = orr * orr + oi * oi;
    float err = qrl_tanhf_lut_rd(snr * orr, tanh_tab) * oi - qrl_tanhf_lut_rd(snr * oi, tanh_tab) * orr;
    err = qrl_clip(err, 1.0f);
    st.freq = st.freq + beta * err;
    st.phase = st.phase + st.freq + alpha * err;
    if (__builtin_expect(!(fabsf(st.phase) < 6.2831854820251465f), 0)) {
        while (st.phase >= 6.2831854820251465f)
            st.phase = static_cast<float>(static_cast<double>(st.phase) - 2.0 * 3.14159265358979323846);
        while (st.phase <= -6.2831854820251465f)
            st.phase = static_cast<float>(static_cast<double>(st.phase) + 2.0 * 3.14159265358979323846);
    }
    if (st.freq > 1.0f) st.freq = 1.0f;
    else if (st.freq < -1.0f) st.freq = -1.0f;
    yr = orr; yi = oi;
}

// Shared-memory copy of the tanh table as qrl_costas4_snr_chunk reads it: 256 entries, entry 256 = entry 255 (x = 2 exactly), entry
// 257 = 1.0f (x > 2), entry 258 = -1.0f (x <= -2, NaN).  Called by all threads of the block.
__device__ __forceinline__ void qrl_fill_tanh_s(float* tanh_s)
{
    for (int i = threadIdx.x; i < 259; i += blockDim.x)
        tanh_s[i] = i < 256 ? d_tanh_tab[i] : (i == 256 ? d_tanh_tab[255] : (i == 257 ? 1.0f : -1.0f));
}

// Rare path of the Costas phase wrap (exact double subtraction), kept out of line so the common path is one compare + branch.
__device__ __noinline__ float qrl_phase_wrap_slow(float ph)
{
    while (ph >= 6.2831854820251465f) ph = static_cast<float>(static_cast<double>(ph) - 2.0 * 3.14159265358979323846);
    while (ph <= -6.2831854820251465f) ph = static_cast<float>(static_cast<double>(ph) + 2.0 * 3.14159265358979323846);
    return ph;
}

// costas_loop_cc(order 4, use_snr) over `n` complex items that sit in shared memory `row_bytes` apart starting at shared address
// `addr` (one lane = one channel), IN PLACE.  Same values as qrl_costas_step bit for bit; written for a lone warp, where the
// loop-carried chain phase -> sincos -> rotate -> snr -> tanh table -> error -> phase is everything:
//   * items and table are addressed by 32-bit shared addresses (no generic-pointer / S2UR address arithmetic in the loop);
//   * the next item is loaded before the current one is worked on (the 30-cycle LDS leaves the chain);
//   * the table index floor(128 + 64 x) never passes through an integer register: the float rounded toward -inf onto 2^23 has
//     the index in its low mantissa bits, and (bits << 2) + (table - (0x4B000000 << 2)) is the entry's address; the table has a
//     257th entry (= entry 255) so that x = 2 needs no integer clamp, and entries 257 / 258 = +1 / -1 for the saturated ranges;
//   * the frequency limit is two FMNMX (exact for non-NaN), the 2*pi wrap one unlikely out-of-line call.
// tanh_addr_m = smem_u32(table of 259 floats: qrl_fill_tanh_s) - (0x4B000000u << 2) + (a zero read from shared memory: to the compiler the sum is then
// an ordinary register value; a visible constant gets re-derived (S2UR + ULEA) or split into two dependent adds inside the loop).
__device__ __forceinline__ void qrl_costas4_snr_chunk(LoopState& st, float k_a, float k_b, uint32_t addr, uint32_t row_bytes, int n,
                                                       uint32_t tanh_addr_m)
{
    float phase = st.phase, freq = st.freq;
    float2 x = lds_f32x2<0>(addr);
    for (int i = 0; i < n; i++) {
        const float2 xn = lds_f32x2<0>(addr + row_bytes);            // item i + 1 (the block has one row of padding behind it)
        float sn, cs;
        qrl_sincosf_small(-phase, sn, cs);
        const float orr = x.x * cs - x.y * sn;
        const float oi = x.x * sn + x.y * cs;
        const float snr = orr * orr + oi * oi;
        const float ar = snr * orr, ai = snr * oi;
        // tanhf_lut: x > 2 -> 1, x <= -2 -> -1, else table[(int)(128 + 64 x)]
        // 128 + 64 x == fma(64, x, 128): 64 x is exact, so the fused form rounds once like the separate add (one dependent operation less),
        // and for -2 < x <= 2 it lies in (0, 256] by itself.  The two saturated ranges are table entries too (257 = 1.0f, 258 = -1.0f),
        // picked by two selects IN FRONT of the load (they take the place of the two clamps), so nothing but the multiply stands
        // behind the 25-cycle LDS.  A NaN fails "x > -2" and reads entry 258: the load address is always inside the table.
        const float vr_ = fmaf(64.0f, ar, 128.0f), vi_ = fmaf(64.0f, ai, 128.0f);
        const float vr = ar > 2.0f ? 257.0f : (ar > -2.0f ? vr_ : 258.0f);
        const float vi = ai > 2.0f ? 257.0f : (ai > -2.0f ? vi_ : 258.0f);
        const float tr = lds_f32<0>((__float_as_uint(__fadd_rd(vr, 8388608.0f)) << 2) + tanh_addr_m);
        const float ti = lds_f32<0>((__float_as_uint(__fadd_rd(vi, 8388608.0f)) << 2) + tanh_addr_m);
        float err = tr * oi - ti * orr;
        err = qrl_clip(err, 1.0f);
        freq = freq + k_b * err;
        phase = phase + freq + k_a * err;
        sts_f32x2(addr, orr, oi);
        // The 2 pi wrap without a branch (a lone warp pays ~60 cycles per sample for an almost-never-taken one) and without double
        // precision: for every float a in [C, C + 1.6], C = 6.28318548f (the float just above 2 pi), (float)((double)a - 2 pi) ==
        // (a - C) + 1.74845553e-7f bit for bit (a - C is exact by Sterbenz, the constant is float(C - 2 pi); checked over ALL 3.4 M
        // floats of the range in tests/test_host_logic.py); one step moves the phase by at most 1 + alpha, so one wrap is enough.
        {
            const float a = fabsf(phase);
            const float w = (a - 6.2831854820251465f) + 1.7484555314695172e-07f;
            phase = a >= 6.2831854820251465f ? copysignf(w, phase) : phase;
        }
        freq = fminf(fmaxf(freq, -1.0f), 1.0f);
        addr += row_bytes;
        x = xn;
    }
    st.phase = phase; st.freq = freq;
}

// ------------------------------------------------------------------------------------------------
// fll_band_edge_cc (BPSK / 2FSK chains): per-sample NCO rotation + two N-tap complex band-edge filters on the
// rotated stream + second-order loop.  One lane per channel, channel-major rings, rotated-sample window in shared
// memory ([N][32] complex, bank = lane).  First correct version: the whole dot product sits in the sample loop
// (only its last tap really depends on the current NCO phase -- hoisting the rest is the next optimisation).
// ------------------------------------------------------------------------------------------------
struct FllState { float phase, freq; long long pos; };
struct FllParams { float alpha, beta, max_freq, min_freq; int N; };

template <int NMAX>
__global__ void __launch_bounds__(32)
fll_kernel(FllParams p, FllState* __restrict__ states, float2* __restrict__ hist_g /* [C][NMAX] rotated-sample window */,
           int C, const float* __restrict__ taps /* lower[2N] | upper[2N] */,
           const float2* __restrict__ in, unsigned in_mask, long long in_stride, long long avail_total,
           float2* __restrict__ out, unsigned out_mask, long long out_stride)
{
    __shared__ float2 win[NMAX][32];
    __shared__ float tl[2 * NMAX], tu[2 * NMAX];
    const int lane = threadIdx.x;
    const int c = blockIdx.x * 32 + lane;
    const int N = p.N;
    for (int i = lane; i < 2 * N; i += 32) { tl[i] = taps[i]; tu[i] = taps[2 * N + i]; }
    if (c < C) for (int k = 0; k < N; k++) win[k][lane] = hist_g[static_cast<long long>(c) * NMAX + k];
    __syncwarp();
    if (c >= C) return;
    FllState st = states[c];
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float2* y = out + static_cast<long long>(c) * out_stride;
    int head = static_cast<int>(st.pos & (N - 1));            // slot of the OLDEST sample (N is a power of two)
    for (long long a = st.pos; a < avail_total; a += 8) {
        float2 v[8];
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = (a + j < avail_total) ? x[(a + j) & in_mask] : make_float2(0.0f, 0.0f);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (a + j >= avail_total) break;
            float sn, cs;
            qrl_sincosf(st.phase, sn, cs);
            const float orr = v[j].x * cs - v[j].y * sn, oi = v[j].x * sn + v[j].y * cs;
            win[head][lane] = make_float2(orr, oi);            // overwrite the oldest: it becomes the newest
            head = (head + 1) & (N - 1);                       // head is the oldest again
            float ur = 0.0f, ui = 0.0f, lr = 0.0f, li = 0.0f;
            for (int k = 0; k < N; k++) {
                const float2 h = win[(head + k) & (N - 1)][lane];
                ur = fmaf(tu[2 * k], h.x, ur); ur = fmaf(-tu[2 * k + 1], h.y, ur);
                ui = fmaf(tu[2 * k], h.y, ui); ui = fmaf(tu[2 * k + 1], h.x, ui);
                lr = fmaf(tl[2 * k], h.x, lr); lr = fmaf(-tl[2 * k + 1], h.y, lr);
                li = fmaf(tl[2 * k], h.y, li); li = fmaf(tl[2 * k + 1], h.x, li);
            }
            const float err = (lr * lr + li * li) - (ur * ur + ui * ui);
            st.freq = st.freq + p.beta * err;
            st.phase = st.phase + st.freq + p.alpha * err;
            while (st.phase >= 6.2831854820251465f) st.phase = static_cast<float>(static_cast<double>(st.phase) - 2.0 * 3.14159265358979323846);
            while (st.phase <= -6.2831854820251465f) st.phase = static_cast<float>(static_cast<double>(st.phase) + 2.0 * 3.14159265358979323846);
            if (st.freq > p.max_freq) st.freq = p.max_freq;
            else if (st.freq < p.min_freq) st.freq = p.min_freq;
            y[(a + j) & out_mask] = make_float2(orr, oi);
        }
    }
    st.pos = avail_total;
    states[c] = st;
    // store the window oldest-first so that the next launch can start with head = pos & (N-1)
    // (slot of sample index i is i & (N-1): already true for the circular buffer as laid out)
    for (int k = 0; k < N; k++) hist_g[static_cast<long long>(c) * NMAX + k] = win[k][lane];
}

// ------------------------------------------------------------------------------------------------
// Sequential loop stage of the PSK chains: agc2_cc -> costas_loop_cc ("PLL" in gr_demod_qpsk.cpp:108-118), one
// lane per channel, per SAMPLE.  The two recurrences are independent of each other, so they run in two warps:
// warp 0 = AGC (gain recurrence), warp 2 = Costas (phase/frequency recurrence), connected by a shared-memory
// hand-off ring; warp 1 lane 0 = TMA producer.  Input and output rings are channel-interleaved.
// The hand-off ring is NHB = 3 blocks deep because a block has three owners in turn: the AGC warp fills it, the Costas
// warp works on it in place, the bulk store drains it -- and the Costas warp learns that block m-1 has been drained
// only while it closes block m.  With two blocks the AGC warp could not start block m+1 before the Costas warp had
// finished block m: the two recurrences ran one after the other (398 cycles per item for a 209-cycle Costas chain,
// tools/microbench/lone_warp.cu); with three they overlap.
// ------------------------------------------------------------------------------------------------
struct AgcCostasState {
    long long pos;            // absolute index of the next input sample
    float gain;               // agc2
    LoopState pll;            // costas
};
struct AgcCostasParams {
    float attack, decay, ref, max_gain;
    float alpha, beta;
    int order, use_snr;
};

constexpr int AC_NHB = 3;      // hand-off blocks between the AGC and the Costas warp (see above)
template <int CH, int NST, int ORDER = -1, int USE_SNR = -1>   // ORDER / USE_SNR >= 0: compile-time loop shape (else p.order / p.use_snr)
__global__ void __launch_bounds__(96)
agc_costas_kernel(AgcCostasParams p, AgcCostasState* __restrict__ states, int C,
                  const float2* __restrict__ in, unsigned in_mask, long long in_stride, long long avail_total,
                  float2* __restrict__ out, unsigned out_mask, long long out_stride)
{
    constexpr int NHB = AC_NHB;
    extern __shared__ __align__(128) float2 sm_ac[];          // [NST][CH][32] | hand-off [NHB][CH][32]
    __shared__ __align__(8) uint64_t bar_in[NST], bar_free[NST], bar_full[NHB], bar_empty[NHB];
    __shared__ float tanh_s[259];                             // entries 256 .. 258: see qrl_fill_tanh_s
    __shared__ volatile int opaque_zero;
    qrl_fill_tanh_s(tanh_s);
    if (threadIdx.x == 0) opaque_zero = 0;
    float2* stage0 = sm_ac;
    // [NHB][CH + 1][32]: every block carries its own padding row -- the Costas loop loads the item behind the one it works on, and behind
    // the last item of a block that must not be the first row of the next block, which the AGC warp may be filling (ThreadSanitizer
    // on the emulated library reported that read; the value was never used, the load is now inside the block's own storage)
    float2* hand = sm_ac + NST * CH * 32;
    constexpr int HB_ROWS = CH + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x;
    const int c = g * 32 + lane;
    const bool active = c < C;
    if (threadIdx.x == 0) {
        for (int b = 0; b < NST; b++) { mbar_init(&bar_in[b], 1); mbar_init(&bar_free[b], 1); }
        for (int b = 0; b < NHB; b++) { mbar_init(&bar_full[b], 1); mbar_init(&bar_empty[b], 1); }
        mbar_fence_init();
    }
    __syncthreads();
    // all channels of a handle advance in lock step (one output per input): the read position is uniform
    const long long base = states[g * 32 < C ? g * 32 : 0].pos;
    __syncthreads();      // all 96 threads hold `base` before the Costas warp stores the advanced position at its end
    if (base >= avail_total) return;
    const long long total = avail_total - base;
    const int nchunks = static_cast<int>((total + CH - 1) / CH);

    if (warp == 1) {
        if (lane == 0) {
            const float2* ring = in + static_cast<long long>(g) * in_stride * 32;
            const long long cap = static_cast<long long>(in_mask) + 1;
            for (int m = 0; m < nchunks; m++) {
                const int st = m % NST, u = m / NST;
                if (u > 0) mbar_wait(&bar_free[st], (u - 1) & 1);
                const long long w0 = base + static_cast<long long>(m) * CH;
                float2* dst = stage0 + st * CH * 32;
                const long long s0 = w0 & in_mask;
                const long long first = (s0 + CH <= cap) ? CH : (cap - s0);
                fence_proxy_async();
                mbar_expect_tx(&bar_in[st], CH * 256);
                bulk_g2s(dst, ring + s0 * 32, static_cast<uint32_t>(first * 256), &bar_in[st]);
                if (first < CH) bulk_g2s(dst + first * 32, ring, static_cast<uint32_t>((CH - first) * 256), &bar_in[st]);
            }
        }
    } else if (warp == 0) {
        // ---------------------------------------------------------------- AGC warp (agc2_cc::scale)
        float gain = active ? states[c].gain : 1.0f;
        const float k_att = p.attack, k_dec = p.decay, k_ref = p.ref, k_max = p.max_gain;
        for (int m = 0; m < nchunks; m++) {
            const int st = m % NST, b = m % NHB;
            if (m >= NHB) mbar_wait(&bar_empty[b], ((m / NHB) - 1) & 1);
            mbar_wait(&bar_in[st], (m / NST) & 1);
            const float2* buf = stage0 + st * CH * 32 + lane;
            float2* hb = hand + b * HB_ROWS * 32 + lane;
            const long long rem = total - static_cast<long long>(m) * CH;
            const int n = rem < CH ? static_cast<int>(rem) : CH;
            if (active) {
                for (int i = 0; i < n; i++) {
                    const float2 x = buf[i * 32];
                    const float orr = x.x * gain, oi = x.y * gain;
                    const float tmp = -k_ref + sqrtf(orr * orr + oi * oi);
                    const float rate = (tmp > gain) ? k_att : k_dec;           // agc2_cc: signed compare (agc2_ff takes fabsf), DESIGN.md section 2
                    gain = gain - tmp * rate;
                    if (gain < 0.0f) gain = 10e-5f;
                    if (k_max > 0.0f && gain > k_max) gain = k_max;
                    hb[i * 32] = make_float2(orr, oi);
                }
            }
            __syncwarp();
            if (lane == 0) { mbar_arrive(&bar_free[st]); mbar_arrive(&bar_full[b]); }
        }
        if (active) states[c].gain = gain;
    } else {
        // ---------------------------------------------------------------- Costas warp
        // works in place on the hand-off block and sends it to the output ring with one TMA bulk store per block
        LoopState pll{ 0.0f, 0.0f };
        if (active) pll = states[c].pll;
        float2* oring = out + static_cast<long long>(g) * out_stride * 32;
        const long long ocap = static_cast<long long>(out_mask) + 1;
        const float k_a = p.alpha, k_b = p.beta;
        const uint32_t tanh_m = smem_u32(tanh_s) - (0x4B000000u << 2) + static_cast<uint32_t>(opaque_zero);
        const int order = ORDER >= 0 ? ORDER : p.order;
        const bool use_snr = USE_SNR >= 0 ? (USE_SNR != 0) : (p.use_snr != 0);
        for (int m = 0; m < nchunks; m++) {
            const int b = m % NHB;
            mbar_wait(&bar_full[b], (m / NHB) & 1);
            float2* hb = hand + b * HB_ROWS * 32 + lane;
            const long long w0 = base + static_cast<long long>(m) * CH;
            const long long rem = total - static_cast<long long>(m) * CH;
            const int n = rem < CH ? static_cast<int>(rem) : CH;
            if (active && order != 0) {
                if (ORDER == 4 && USE_SNR == 1) {
                    qrl_costas4_snr_chunk(pll, k_a, k_b, smem_u32(hb), 256u, n, tanh_m);
                } else {
                    for (int i = 0; i < n; i++) {
                        const float2 x = hb[i * 32];
                        float yr, yi;
                        qrl_costas_step(pll, k_a, k_b, order, use_snr, x.x, x.y, yr, yi, tanh_s);
                        hb[i * 32] = make_float2(yr, yi);
                    }
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                const float2* src = hand + b * HB_ROWS * 32;
                const long long s0 = w0 & out_mask;
                const long long first = (s0 + n <= ocap) ? n : (ocap - s0);
                bulk_s2g(oring + s0 * 32, src, static_cast<uint32_t>(first * 256));
                if (first < n) bulk_s2g(oring, src + first * 32, static_cast<uint32_t>((n - first) * 256));
                bulk_commit();
                if (m >= 1) { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); mbar_arrive(&bar_empty[(m - 1) % NHB]); }
            }
        }
        if (lane == 0) { bulk_wait_all0(); mbar_arrive(&bar_empty[(nchunks - 1) % NHB]); }
        if (active) { states[c].pll = pll; states[c].pos = avail_total; }
    }
}

// exact threshold form of constellation_rect's floor(re + 2.0f) sector search (float addition rounds to nearest
// even, so fl(re+2) >= 1,2,3  <=>  re >= -1, -2^-24, 1-2^-23; checked in tests/test_host_logic.py)
__device__ __forceinline__ float qrl_ge1(float a, float b)     // (a >= b) ? 1.0f : 0.0f in one FSET, no predicate
{
    float r;
    asm("set.ge.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float qrl_slice_rect4(float re)
{
    // -1.5 + [re >= -1] + [re >= -2^-24] + [re >= 1 - 2^-23]  (all partial sums exact)
    return ((-1.5f + qrl_ge1(re, -1.0f)) + qrl_ge1(re, -5.9604644775390625e-8f)) + qrl_ge1(re, 0.99999988079071044921875f);
}
// clip for non-NaN arguments: two FMNMX instead of compare + select
__device__ __forceinline__ float qrl_clip1(float x) { return fminf(fmaxf(x, -1.0f), 1.0f); }

// out-of-lock step of the lean symbol-sync loop (never inlined: keeps FRND off the predicated common path)
__device__ __noinline__ float2 symsync_generic_step(float ph)
{
    const float fl = floorf(ph);
    return make_float2(ph - fl, fl);
}

// Input ring layout: [group = channel / 32][slot][32 lanes][NCOMP] -- a time step of one warp's 32 channels is one
// contiguous 128*NCOMP-byte row, so a CH-row window is ONE contiguous block fetched with cp.async.bulk (TMA 1-D).
// Warp-specialised CTA (one CTA per 32 channels):
//   warp 1 (lane 0) : TMA producer, NST-stage ring of CH-row windows (mbarrier full/free)
//   warp 0          : ONLY the loop-carried recurrence (interpolate -> TED -> PI loop -> next position); every lane
//                     reads column `lane` of the window (bank = lane: conflict-free)
//   warps 2..       : everything that does not feed back (phase modulator / 2nd Costas loop, soft bits, stores),
//                     fed through a double-buffered shared-memory symbol hand-off (mbarrier full/empty)
// VAR: 0 = generic recurrence (any NCOMP / slicer); 1 = lean real 4-level recurrence, interpolator bank as 12-float entries
// (two LDS.128 with bank conflicts); 2 = lean recurrence + 16-fold replicated bank (conflict-free, +66 KB of shared memory)
// 3 = generic recurrence with the PLAIN Mueller & Mueller detector (gr_demod_dmr.cpp:66; real symbols only) instead of the modified one
template <int NCOMP, int SLICER, int EPI, int CH, int NST, int NEPI, int LOOPK = LOOP_SYMSYNC, int VAR = 0>
__global__ void __launch_bounds__(64 + 32 * NEPI)
symsync_kernel(SymSyncParams p, SymSyncState* __restrict__ states, int C,
               const float* __restrict__ in, unsigned in_mask, long long in_stride /*slots per group*/, long long avail_total,
               float2* __restrict__ port1, long long port1_stride, int* __restrict__ port1_cnt, int port1_cap,
               unsigned char* __restrict__ soft_ring, unsigned soft_mask, long long soft_stride, int maxs,
               long long* __restrict__ n_soft_out /* [C] snapshot of the soft-bit write index after this launch */,
               float* __restrict__ ext_scratch = nullptr /* [groups][ext_chunk_cap][maxs + 2][32] (EPI_EXT_*) */,
               int ext_chunk_cap = 0 /* chunks this launch may emit */, int ext_chunk_stride = 0 /* chunks per group in the scratch */,
               int* __restrict__ ext_hdr = nullptr /* [groups][128] (EPI_EXT_*) */)
{
    static_assert(EPI != EPI_BPSK || NEPI == 1, "Costas epilogues carry loop state: one epilogue warp");
    static_assert(EPI != EPI_QPSK || NEPI == 1 || NEPI == 2, "QPSK: one epilogue warp, or a Costas warp + a feed-forward warp");
    // QPSK with NEPI == 2: warp 2 runs the second Costas loop in place, warp 3 everything behind it (diff_phasor, rotation, soft bits,
    // stores).  A symbol block then has three owners in turn (loop warp, Costas warp, feed-forward warp), so the ring is 3 deep (see
    // agc_costas_kernel) and a third barrier (bar_cdone) hands a block from the Costas warp to the feed-forward warp.
    constexpr bool SPLIT = (EPI == EPI_QPSK && NEPI == 2);
    constexpr int NB = SPLIT ? 3 : 2;
    constexpr bool EXT = (EPI == EPI_EXT_4FSK_FM);
    static_assert(!EXT || (NEPI == 1 && NCOMP == 1), "external epilogue: one drain warp, real symbols");
    constexpr int ROWF = 32 * NCOMP;                    // floats per row
    SSP(const unsigned long long pg0 = globaltimer_ns();)
    // window advance per chunk: a lane leaves a window once its position is within `lookahead` rows of the end, so
    // consecutive windows overlap by the lookahead rounded up to 32 rows (same formula on the host: symsync_stride)
    const int STRIDE = symsync_stride(CH, p.lookahead);
    extern __shared__ __align__(128) float sm_sync[];   // [NST][CH][ROWF] | mmse[129*8] | sym[2][maxs][ROWF] | cnt[2][32]
    __shared__ __align__(8) uint64_t bar_in[NST], bar_free[NST], bar_full[NB], bar_empty[NB], bar_cdone[NB];
    __shared__ volatile int lane_zero[32];
    __shared__ float tanh_s[EPI == EPI_QPSK ? 259 : 1];    // second Costas loop's table (entries 256 .. 258: see qrl_fill_tanh_s)
    __shared__ volatile int opaque_zero;
    if (EPI == EPI_QPSK) qrl_fill_tanh_s(tanh_s);
    if (threadIdx.x == 0) opaque_zero = 0;
    float* stage0 = sm_sync;
    float* mm = sm_sync + NST * CH * ROWF;
    float* mm2 = mm + 132 * 8;                          // entry-major copy (12-float pitch), taps reversed: two LDS.128
    float* symbuf = mm + SYMSYNC_TAB_FLOATS;
    const int blk_rows = EXT ? maxs + 2 : maxs;         // EXT: rows maxs / maxs+1 of a block hold the lane counts / lane bases
    int* cntbuf = reinterpret_cast<int*>(symbuf + NB * blk_rows * ROWF);
    // VAR == 2: 16-fold replicated bank [imu][half][lane & 15][4] (129 * 512 bytes) behind everything else: the 8 lanes
    // of an LDS.128 phase read 128 contiguous bytes, so the two tap loads of a symbol are conflict-free whatever imu is
    constexpr bool REP = (VAR == 2);
    float* mm3 = reinterpret_cast<float*>(cntbuf + 32 * (NB == 2 ? 2 : 4));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x;
    const int c = g * 32 + lane;
    const bool active = c < C;
    // tap-major copy of the MMSE bank: mm[k * 132 + imu] (a lane's 8 taps are 8 scalar loads in the order the
    // oldest-first FMA chain consumes them; random imu across lanes spreads over all 32 banks)
    // (all of a thread's table entries are loaded before the first store: one L2 latency per launch instead of one per entry -- the
    // fill used to be 6 us of every launch, profiles/r02_w_symsync_launch_phases.txt)
    constexpr int NT = 64 + 32 * NEPI, TPT = (129 * 8 + NT - 1) / NT;
    float tv[TPT];
#pragma unroll
    for (int k = 0; k < TPT; k++) { const int i = threadIdx.x + k * NT; tv[k] = i < 129 * 8 ? d_mmse_tab[i] : 0.0f; }
#pragma unroll
    for (int k = 0; k < TPT; k++) {
        const int i = threadIdx.x + k * NT;
        if (i >= 129 * 8) break;
        const float t = tv[k];
        mm[(i & 7) * 132 + (i >> 3)] = t;
        mm2[(i >> 3) * 12 + (7 - (i & 7))] = t;
        if (REP) {
            const int j = 7 - (i & 7);
            float* q = mm3 + (i >> 3) * 128 + (j >> 2) * 64 + (j & 3);
#pragma unroll
            for (int r = 0; r < 16; r++) q[r * 4] = t;
        }
    }
    if (threadIdx.x == 0) {
        for (int b = 0; b < NST; b++) { mbar_init(&bar_in[b], 1); mbar_init(&bar_free[b], 1); }
        for (int b = 0; b < NB; b++) { mbar_init(&bar_full[b], 1); mbar_init(&bar_empty[b], SPLIT ? 1 : NEPI); mbar_init(&bar_cdone[b], 1); }
        mbar_fence_init();
    }
    __syncthreads();

    // every warp derives the same chunk schedule from the (uniform) minimum read position
    long long my_ii = active ? states[c].ii : 0x7fffffffffffffffLL;
    long long base = my_ii;
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const long long o = __shfl_xor_sync(0xffffffffu, base, off);
        base = o < base ? o : base;
    }
    int nchunks = (base + p.lookahead > avail_total) ? 0 : static_cast<int>((avail_total - p.lookahead - base) / STRIDE) + 1;
    if (EXT) {
        // the launch's starting indices travel to the external epilogue in a header (this warp overwrites them at the end)
        nchunks = nchunks < ext_chunk_cap ? nchunks : ext_chunk_cap;     // a clipped launch catches up on the next one
        if (warp == 0) {
            const long long ns0 = active ? states[c].n_soft : 0;
            int* hdr = ext_hdr + g * 128;
            hdr[lane] = active ? port1_cnt[c] : 0;
            hdr[32 + lane] = static_cast<int>(ns0 & 0xffffffffLL);
            hdr[64 + lane] = static_cast<int>(ns0 >> 32);
            if (lane == 0) hdr[96] = nchunks;
            if (active) n_soft_out[c] = ns0;
        }
    } else if (warp == 2 && active) n_soft_out[c] = states[c].n_soft;
    // every warp has derived its schedule from states[].ii before the loop warp may store the advanced value at its end (with one
    // or two chunks nothing else orders the drain / epilogue warps' reads before that store)
    __syncthreads();
    if (nchunks == 0) return;

    if (warp == 1) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            const float* ring = in + static_cast<long long>(g) * in_stride * ROWF;
            const long long cap = static_cast<long long>(in_mask) + 1;
            for (int m = 0; m < nchunks; m++) {
                const int st = m % NST, u = m / NST;
                if (u > 0) mbar_wait(&bar_free[st], (u - 1) & 1);
                const long long w0 = base + static_cast<long long>(m) * STRIDE;
                float* dst = stage0 + st * CH * ROWF;
                const long long s0 = w0 & in_mask;
                const long long first = (s0 + CH <= cap) ? CH : (cap - s0);
                fence_proxy_async();
                mbar_expect_tx(&bar_in[st], CH * ROWF * 4);
                bulk_g2s(dst, ring + s0 * ROWF, static_cast<uint32_t>(first * ROWF * 4), &bar_in[st]);
                if (first < CH) bulk_g2s(dst + first * ROWF, ring, static_cast<uint32_t>((CH - first) * ROWF * 4), &bar_in[st]);
            }
        }
    } else if (warp == 0) {
        // ------------------------------------------------------------------ loop warp
        float avg_period = 0, inst_period = 0, mu = 0, x0 = 0, x1 = 0, x2 = 0, y0i = 0, y1i = 0, y2i = 0;
        float d0 = 0, d1 = 0, d2 = 0, e0 = 0, e1 = 0, e2 = 0;
        if (active) {
            const SymSyncState& st = states[c];
            avg_period = st.avg_period; inst_period = st.inst_period; mu = st.mu;
            x0 = st.xr[0]; x1 = st.xr[1]; x2 = st.xr[2]; y0i = st.xi[0]; y1i = st.xi[1]; y2i = st.xi[2];
            d0 = st.dr[0]; d1 = st.dr[1]; d2 = st.dr[2]; e0 = st.di[0]; e1 = st.di[1]; e2 = st.di[2];
        }
        int o = 0;                                         // my read position relative to the current window
        int nsym_run = 0;                                  // EXT: symbols this lane has emitted so far in this launch
        {
            const long long d = my_ii - base;
            o = d > 0x3fffffff ? 0x3fffffff : static_cast<int>(d);
        }
        const int la = p.lookahead;
        // a zero the compiler cannot see through (bounced through shared memory): pointers offset by it are
        // per-lane registers to the compiler, so the recurrence addresses shared memory as [R+imm], not [R+UR+imm]
        lane_zero[lane] = 0;
        __syncwarp();
        const int zoff = lane_zero[lane];
        const float* mmp = mm + zoff;
        const float* stp = stage0 + lane * NCOMP + zoff;
        // loop constants in registers (a constant-bank load inside the recurrence would sit on the critical path)
        const float k_alpha = p.alpha, k_beta = p.beta, k_maxp = p.max_period, k_minp = p.min_period;
        const float k_f0 = p.fl0, k_f1 = p.fl0 + 1.0f, k_f2 = p.fl0 + 2.0f, k_f3 = p.fl0 + 3.0f;
        const int k_n0 = p.n0;
        // constants of the lean loop, made opaque (+0.0f the compiler cannot see) so they stay in plain registers
        const float zf = __int_as_float(zoff);
        const float k_hb = 0.5f * p.beta + zf, k_ha = 0.5f * p.alpha + zf, k128 = 128.0f + zf;
        const float q_minp = p.min_period + zf, q_maxp = p.max_period + zf;
        const float q_f0 = p.fl0 + zf, q_f1 = (p.fl0 + 1.0f) + zf, q_f2 = (p.fl0 + 2.0f) + zf;
        // the tap-bank base minus the magic-number offset travels through shared memory: as a loaded value it is ONE register to the
        // compiler; as a visible sum its constant part is re-added behind the index multiply (an extra dependent op per tap load)
        lane_zero[lane] = static_cast<int>(REP ? smem_u32(mm3) + (lane & 15) * 16 - 0x4B400000u * 512u
                                               : smem_u32(mm2) - 0x4B400000u * 48u);
        __syncwarp();
        const uint32_t mm2_b = static_cast<uint32_t>(lane_zero[lane]);
        const bool lean_ok = p.min_period > fabsf(p.alpha) && p.fl0 >= 1.0f;
        const bool window_sure = lean_ok && (p.max_period + fabsf(p.alpha) + 1.0f < p.fl0 + 3.0f - 1e-3f) &&
                                 (p.min_period - fabsf(p.alpha) > p.fl0 + 1e-3f) && p.fl0 == static_cast<float>(p.n0);
        SSP(long long pf_we = 0; long long pf_wi = 0; long long pf_run = 0; long long pf_str = 0; long long pf_ho = 0; long long pf_rounds = 0; long long pf_sym = 0;)
        SSP(const unsigned long long pg1 = globaltimer_ns(); unsigned long long pg2 = pg1;)
        for (int m = 0; m < nchunks; m++) {
            const int st = m % NST, b = m % NB;
            SSP(const long long pt0 = clock64();)
            if (m >= NB) mbar_wait(&bar_empty[b], ((m / NB) - 1) & 1);   // epilogue released this hand-off buffer
            SSP(const long long pt1 = clock64();)
            mbar_wait(&bar_in[st], (m / NST) & 1);
            SSP(const long long pt2 = clock64(); pf_we += pt1 - pt0; pf_wi += pt2 - pt1; long long pt3 = pt2;)
            SSP(if (m == 0) pg2 = globaltimer_ns();)
            const float* buf = stp + st * CH * ROWF;
            float* sy = symbuf + b * blk_rows * ROWF + lane * NCOMP;
            const long long w0 = base + static_cast<long long>(m) * STRIDE;
            const long long rem = avail_total - w0;
            const int wlen = rem < CH ? static_cast<int>(rem) : CH;
            int cnt = 0;
            if (active && LOOPK == LOOP_CRMM) {
                // clock_recovery_mm_cc: avg_period holds omega, x*/y*i hold p_nT, d*/e* hold the 0/1 slicer outputs
                while (o + la <= wlen) {
                    const float* x = buf + o * ROWF;
                    const float* tp = mmp + (__float_as_int(fmaf(mu, 128.0f, 12582912.0f)) & 0x3ff);
                    float yr = 0.0f, yi = 0.0f;
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const float tt = tp[(7 - i) * 132];
                        yr = fmaf(tt, x[i * ROWF], yr);
                        if (NCOMP == 2) yi = fmaf(tt, x[i * ROWF + 1], yi);
                    }
                    x2 = x1; x1 = x0; x0 = yr;
                    y2i = y1i; y1i = y0i; y0i = yi;
                    d2 = d1; d1 = d0; e2 = e1; e1 = e0;
                    d0 = yr > 0.0f ? 1.0f : 0.0f; e0 = yi > 0.0f ? 1.0f : 0.0f;
                    const float ar = d0 - d2, ai = e0 - e2;
                    const float xr_ = ar * x1 + ai * y1i;
                    const float br = x0 - x2, bi = y0i - y2i;
                    const float yr_ = br * d1 + bi * e1;
                    const float mmv = qrl_clip1(yr_ - xr_);
                    avg_period = avg_period + p.gain_omega * mmv;
                    avg_period = p.omega_mid + fminf(fmaxf(avg_period - p.omega_mid, -p.omega_lim), p.omega_lim);
                    mu = mu + avg_period + p.gain_mu * mmv;
                    const float fl = floorf(mu);
                    o += static_cast<int>(fl);
                    mu = mu - fl;
                    sy[cnt * ROWF] = yr;
                    if (NCOMP == 2) sy[cnt * ROWF + 1] = yi;
                    cnt++;
                }
            } else if (active && LOOPK == LOOP_SYMSYNC && NCOMP == 1 && SLICER == SL_RECT4 && (VAR == 1 || VAR == 2) && lean_ok) {
                // Lean restatement of the real 4-level recurrence.  A lone warp pays ~1 cycle per issued instruction
                // plus ~4 per dependent one, so the loop is written for instruction count.  Every rewrite is exact:
                //  * err = clip(u/2, +-1) enters only as beta*err and alpha*err, formed as (beta/2)*clip(u, +-2)
                //    (scaling by 1/2 commutes with rounding);
                //  * the read position lives in a float as 2^23 + row (integer adds are exact, the row is the low
                //    mantissa bits), so the stride floor(ph) = n0 + [ph >= n0+1] + [ph >= n0+2] never leaves the
                //    float pipe and ph - floor(ph) is (ph - n0) minus the same two 0/1 terms (exact: integers
                //    subtracted from a float of at least their magnitude);
                //  * the TED history rotates through three registers (loop unrolled by 3) instead of being moved;
                //  * inst_period <= 0 cannot happen when min_period > |alpha| (checked by lean_ok).
                float ofm = 8388608.0f + static_cast<float>(o);
                const float lim = 8388608.0f + static_cast<float>(wlen - la);
                const uint32_t xb = smem_u32(buf) - (0x4B000000u << 7);
                uint32_t syp = smem_u32(sy);
                const uint32_t syp0 = syp;
                float A = x0, B = x1, Cc = x2, dA = d0, dB = d1, dC = d2;
                // The 8 input rows of a symbol are in registers BEFORE its position is known: the next position is ofn + s12 with
                // ofn = ofm + n0 known at the start of a symbol and s12 in {0, 1, 2} known at its end, so the ten rows ofn .. ofn + 9
                // are loaded in the shadow of the current symbol's chain and the eight that count are picked by two selects each.
                // Same values as loading at the final position (exact); what leaves the loop-carried chain is the shared-memory
                // latency of the sample loads (the tap load, which depends on mu, stays).
                float xs0 = 0.0f, xs1 = 0.0f, xs2 = 0.0f, xs3 = 0.0f, xs4 = 0.0f, xs5 = 0.0f, xs6 = 0.0f, xs7 = 0.0f;
                auto load_xs = [&]() {
                    const uint32_t xa = xb + (__float_as_uint(ofm) << 7);
                    xs0 = lds_f32<0>(xa); xs1 = lds_f32<ROWF * 4>(xa); xs2 = lds_f32<ROWF * 8>(xa); xs3 = lds_f32<ROWF * 12>(xa);
                    xs4 = lds_f32<ROWF * 16>(xa); xs5 = lds_f32<ROWF * 20>(xa); xs6 = lds_f32<ROWF * 24>(xa); xs7 = lds_f32<ROWF * 28>(xa);
                };
                if (ofm <= lim) load_xs();
                // one symbol; returns true when the lane fell out of the in-lock stride window (generic step taken).
                // ws_tag = true: the loop constants make that impossible (see window_sure), the check is compiled out.
                auto body_t = [&](auto ws_tag, float& n, const float h1, const float h2, float& dn, const float dh1, const float dh2) -> bool {
                    constexpr bool WS = decltype(ws_tag)::value;
                    const uint32_t ta = mm2_b + __float_as_uint(fmaf(mu, k128, 12582912.0f)) * (REP ? 512u : 48u);
                    const float ofn = ofm + q_f0;
                    const uint32_t xn = xb + (__float_as_uint(ofn) << 7);
                    const float r0 = lds_f32<0>(xn), r1 = lds_f32<ROWF * 4>(xn), r2 = lds_f32<ROWF * 8>(xn), r3 = lds_f32<ROWF * 12>(xn),
                                r4 = lds_f32<ROWF * 16>(xn), r5 = lds_f32<ROWF * 20>(xn), r6 = lds_f32<ROWF * 24>(xn), r7 = lds_f32<ROWF * 28>(xn),
                                r8 = lds_f32<ROWF * 32>(xn), r9 = lds_f32<ROWF * 36>(xn);
                    const float kd = -1.5f - dh2;
                    const float4 ta0 = lds_f32x4<0>(ta), ta1 = lds_f32x4<REP ? 256 : 16>(ta);   // taps[7..4], taps[3..0]
                    float yr = fmaf(ta0.x, xs0, 0.0f);                            // oldest sample first
                    yr = fmaf(ta0.y, xs1, yr);
                    yr = fmaf(ta0.z, xs2, yr);
                    yr = fmaf(ta0.w, xs3, yr);
                    yr = fmaf(ta1.x, xs4, yr);
                    yr = fmaf(ta1.y, xs5, yr);
                    yr = fmaf(ta1.z, xs6, yr);
                    yr = fmaf(ta1.w, xs7, yr);
                    n = yr;
                    // slicer levels are +-0.5, +-1.5: the sums below are exact in any order (two-level tree)
                    const float s1 = qrl_ge1(yr, -1.0f), s23 = qrl_ge1(yr, -5.9604644775390625e-8f) + qrl_ge1(yr, 0.99999988079071044921875f);
                    const float br = (s1 + kd) + s23;                             // dn - dh2
                    dn = (s1 - 1.5f) + s23;
                    const float u = (yr - h2) * dh1 - br * h1;
                    const float e2x = fminf(fmaxf(u, -2.0f), 2.0f);               // 2 * err
                    avg_period = avg_period + k_hb * e2x;
                    avg_period = fminf(fmaxf(avg_period, q_minp), q_maxp);
                    inst_period = avg_period + k_ha * e2x;
                    const float ph = mu + inst_period;
                    const float m0 = ph - q_f0;
                    sts_f32(syp, yr);
                    syp += ROWF * 4;
                    const float s12 = qrl_ge1(m0, 1.0f) + qrl_ge1(m0, 2.0f);     // == [ph >= n0+1] + [ph >= n0+2] (m0 exact)
                    const bool g1 = m0 >= 1.0f, g2 = m0 >= 2.0f;
                    mu = m0 - s12;
                    ofm = ofn + s12;
                    xs0 = g2 ? r2 : (g1 ? r1 : r0); xs1 = g2 ? r3 : (g1 ? r2 : r1); xs2 = g2 ? r4 : (g1 ? r3 : r2); xs3 = g2 ? r5 : (g1 ? r4 : r3);
                    xs4 = g2 ? r6 : (g1 ? r5 : r4); xs5 = g2 ? r7 : (g1 ? r6 : r5); xs6 = g2 ? r8 : (g1 ? r7 : r6); xs7 = g2 ? r9 : (g1 ? r8 : r7);
                    if (!WS) {
                        if (__builtin_expect(__float_as_uint(m0) >= 0x40400000u, 0)) {    // ph not in [n0, n0+3): generic floor
                            const float2 g = symsync_generic_step(ph);
                            mu = g.x;
                            ofm = (ofn - q_f0) + g.y;
                            if (ofm <= lim) load_xs();
                            return true;
                        }
                    }
                    return false;
                };
                // Trip counts are warp-uniform.  Positions telescope: o_j + mu_j = o_0 + mu_0 + sum of the instantaneous periods, each at
                // most max_period + |alpha| (the average is clamped to max_period, the proportional term is |alpha| |err| <= |alpha|),
                // so symbol j starts below o_0 + 1 + j pmax and every lane can take floor((rows left - 1) / pmax) + 1 symbols without
                // looking at the window end (the 0.9999 covers the float roundings of ph, ~5e-7 rows per symbol); recomputed until no
                // lane has a guaranteed symbol left, then each lane finishes under the exact per-lane check.  (The first version
                // divided by the largest possible stride n0 + 2 and needed ~3.9 rounds per window; this one needs 2.)
                const unsigned amask = __activemask();
                const float inv_s = 0.9999f / (p.max_period + fabsf(p.alpha));
                auto run = [&](auto ws_tag) {
                    auto body = [&](float& n, const float h1, const float h2, float& dn, const float dh1, const float dh2) -> bool {
                        return body_t(ws_tag, n, h1, h2, dn, dh1, dh2);
                    };
                    for (;;) {
                        SSP(pf_rounds++;)
                        const float left = lim - ofm;                      // exact (integers below 2^24)
                        int ksafe = left >= 0.0f ? static_cast<int>(fmaxf(left - 1.0f, 0.0f) * inv_s) + 1 : 0;
                        ksafe = __reduce_min_sync(amask, ksafe);
                        if (ksafe == 0) break;
                        bool fell = false;
                        for (; ksafe >= 3 && !fell; ksafe -= 3) {
                            if (body(Cc, A, B, dC, dA, dB)) { const float t = Cc, dt = dC; Cc = B; B = A; A = t; dC = dB; dB = dA; dA = dt; fell = true; }
                            else if (body(B, Cc, A, dB, dC, dA)) { const float t = B, dt = dB; B = Cc; Cc = A; A = t; dB = dC; dC = dA; dA = dt; fell = true; }
                            else if (body(A, B, Cc, dA, dB, dC)) fell = true;
                        }
                        for (; ksafe >= 1 && !fell; ksafe--) {
                            fell = body(Cc, A, B, dC, dA, dB);
                            const float t = Cc, dt = dC; Cc = B; B = A; A = t; dC = dB; dB = dA; dA = dt;
                        }
                        if (__any_sync(amask, fell)) break;
                    }
                    SSP(pt3 = clock64();)
                    while (ofm <= lim) {                                   // stragglers (and lanes that fell out of lock)
                        body(Cc, A, B, dC, dA, dB);
                        const float t = Cc, dt = dC; Cc = B; B = A; A = t; dC = dB; dB = dA; dA = dt;
                    }
                };
                // With mu in [0, 1) and the instantaneous period in [min_period - |alpha|, max_period + |alpha|], ph = mu + period
                // lies in [n0, n0 + 3) whenever max_period + |alpha| + 1 < n0 + 3 and min_period - |alpha| > n0 (margins far above
                // float rounding): the out-of-window test and its branch then leave the per-symbol path altogether.
                if (window_sure) run(std::true_type{}); else run(std::false_type{});
                x0 = A; x1 = B; x2 = Cc; d0 = dA; d1 = dB; d2 = dC;
                o = static_cast<int>(ofm - 8388608.0f);
                cnt = static_cast<int>((syp - syp0) / (ROWF * 4));
            } else if (active && LOOPK == LOOP_SYMSYNC && NCOMP == 2 && SLICER == SL_DQPSK && VAR == 2 && lean_ok && window_sure) {
                // Lean restatement of the COMPLEX recurrence (symbol_sync_cc with constellation_dqpsk: the QPSK chain), same construction as the
                // real one above: position in a float, fractional phase by two exact compares, TED history rotating through registers,
                // the ten candidate rows of the next symbol prefetched and picked by selects, tap bank replicated 16-fold.  The decision
                // terms (d0 - d2) x1 of the detector are formed for both signs off the chain and picked by the sign of the new sample.
                // Same operations in the same order per value as the generic loop below: bit-identical.
                float ofm = 8388608.0f + static_cast<float>(o);
                const float lim = 8388608.0f + static_cast<float>(wlen - la);
                const uint32_t xb = smem_u32(buf) - (0x4B000000u << 8);         // one row = 32 lanes x 8 bytes
                uint32_t syp = smem_u32(sy);
                const uint32_t syp0 = syp;
                float Ar = x0, Ai = y0i, Br = x1, Bi = y1i, Cr = x2, Ci = y2i;
                float dAr = d0, dAi = e0, dBr = d1, dBi = e1, dCr = d2, dCi = e2;
                const float k_b = p.beta + zf, k_a = p.alpha + zf, kp = 0.707107f + zf, kn = -0.707107f + zf;
                float2 xs0 = make_float2(0.0f, 0.0f), xs1 = make_float2(0.0f, 0.0f), xs2 = make_float2(0.0f, 0.0f), xs3 = make_float2(0.0f, 0.0f), xs4 = make_float2(0.0f, 0.0f), xs5 = make_float2(0.0f, 0.0f), xs6 = make_float2(0.0f, 0.0f), xs7 = make_float2(0.0f, 0.0f);
                auto load_xs = [&]() {
                    const uint32_t xa = xb + (__float_as_uint(ofm) << 8);
                    xs0 = lds_f32x2<ROWF * 0>(xa);
                    xs1 = lds_f32x2<ROWF * 4>(xa);
                    xs2 = lds_f32x2<ROWF * 8>(xa);
                    xs3 = lds_f32x2<ROWF * 12>(xa);
                    xs4 = lds_f32x2<ROWF * 16>(xa);
                    xs5 = lds_f32x2<ROWF * 20>(xa);
                    xs6 = lds_f32x2<ROWF * 24>(xa);
                    xs7 = lds_f32x2<ROWF * 28>(xa);
                };
                if (ofm <= lim) load_xs();
                auto body = [&](float& nr, float& ni, const float h1r, const float h1i, const float h2r, const float h2i,
                                float& dnr, float& dni, const float dh1r, const float dh1i, const float dh2r, const float dh2i) {
                    const uint32_t ta = mm2_b + __float_as_uint(fmaf(mu, k128, 12582912.0f)) * 512u;
                    const float ofn = ofm + q_f0;
                    const uint32_t xn = xb + (__float_as_uint(ofn) << 8);
                    const float2 r0 = lds_f32x2<ROWF * 0>(xn);
                    const float2 r1 = lds_f32x2<ROWF * 4>(xn);
                    const float2 r2 = lds_f32x2<ROWF * 8>(xn);
                    const float2 r3 = lds_f32x2<ROWF * 12>(xn);
                    const float2 r4 = lds_f32x2<ROWF * 16>(xn);
                    const float2 r5 = lds_f32x2<ROWF * 20>(xn);
                    const float2 r6 = lds_f32x2<ROWF * 24>(xn);
                    const float2 r7 = lds_f32x2<ROWF * 28>(xn);
                    const float2 r8 = lds_f32x2<ROWF * 32>(xn);
                    const float2 r9 = lds_f32x2<ROWF * 36>(xn);
                    const float4 ta0 = lds_f32x4<0>(ta), ta1 = lds_f32x4<256>(ta);   // taps[7..4], taps[3..0]
                    // (d0 - d2) x1 for both decisions of each component
                    const float prp = (kp - dh2r) * h1r, prn = (kn - dh2r) * h1r, pip = (kp - dh2i) * h1i, pin = (kn - dh2i) * h1i;
                    float yr = 0.0f, yi = 0.0f;                                   // oldest sample first
                    yr = fmaf(ta0.x, xs0.x, yr); yi = fmaf(ta0.x, xs0.y, yi);
                    yr = fmaf(ta0.y, xs1.x, yr); yi = fmaf(ta0.y, xs1.y, yi);
                    yr = fmaf(ta0.z, xs2.x, yr); yi = fmaf(ta0.z, xs2.y, yi);
                    yr = fmaf(ta0.w, xs3.x, yr); yi = fmaf(ta0.w, xs3.y, yi);
                    yr = fmaf(ta1.x, xs4.x, yr); yi = fmaf(ta1.x, xs4.y, yi);
                    yr = fmaf(ta1.y, xs5.x, yr); yi = fmaf(ta1.y, xs5.y, yi);
                    yr = fmaf(ta1.z, xs6.x, yr); yi = fmaf(ta1.z, xs6.y, yi);
                    yr = fmaf(ta1.w, xs7.x, yr); yi = fmaf(ta1.w, xs7.y, yi);
                    nr = yr; ni = yi;
                    const bool sr = yr > 0.0f, si = yi > 0.0f;
                    dnr = sr ? kp : kn; dni = si ? kp : kn;
                    const float t2 = (sr ? prp : prn) + (si ? pip : pin);         // br x1r + bi x1i
                    const float t1 = (yr - h2r) * dh1r + (yi - h2i) * dh1i;       // ar d1r + ai d1i
                    const float err = fminf(fmaxf(t1 - t2, -1.0f), 1.0f);
                    avg_period = avg_period + k_b * err;
                    avg_period = fminf(fmaxf(avg_period, q_minp), q_maxp);
                    inst_period = avg_period + k_a * err;
                    const float ph = mu + inst_period;
                    const float m0 = ph - q_f0;
                    sts_f32x2(syp, yr, yi);
                    syp += ROWF * 4;
                    const float s12 = qrl_ge1(m0, 1.0f) + qrl_ge1(m0, 2.0f);     // == [ph >= n0+1] + [ph >= n0+2] (m0 exact)
                    const bool g1 = m0 >= 1.0f, g2 = m0 >= 2.0f;
                    mu = m0 - s12;
                    ofm = ofn + s12;
                    xs0 = g2 ? r2 : (g1 ? r1 : r0);
                    xs1 = g2 ? r3 : (g1 ? r2 : r1);
                    xs2 = g2 ? r4 : (g1 ? r3 : r2);
                    xs3 = g2 ? r5 : (g1 ? r4 : r3);
                    xs4 = g2 ? r6 : (g1 ? r5 : r4);
                    xs5 = g2 ? r7 : (g1 ? r6 : r5);
                    xs6 = g2 ? r8 : (g1 ? r7 : r6);
                    xs7 = g2 ? r9 : (g1 ? r8 : r7);
                };
                auto rot = [&]() {
                    const float tr = Cr, ti = Ci, dtr = dCr, dti = dCi;
                    Cr = Br; Ci = Bi; Br = Ar; Bi = Ai; Ar = tr; Ai = ti;
                    dCr = dBr; dCi = dBi; dBr = dAr; dBi = dAi; dAr = dtr; dAi = dti;
                };
                const unsigned amask = __activemask();
                const float inv_s = 0.9999f / (p.max_period + fabsf(p.alpha));
                for (;;) {
                    const float left = lim - ofm;                              // exact (integers below 2^24)
                    int ksafe = left >= 0.0f ? static_cast<int>(fmaxf(left - 1.0f, 0.0f) * inv_s) + 1 : 0;
                    ksafe = __reduce_min_sync(amask, ksafe);
                    if (ksafe == 0) break;
                    for (; ksafe >= 3; ksafe -= 3) {
                        body(Cr, Ci, Ar, Ai, Br, Bi, dCr, dCi, dAr, dAi, dBr, dBi);
                        body(Br, Bi, Cr, Ci, Ar, Ai, dBr, dBi, dCr, dCi, dAr, dAi);
                        body(Ar, Ai, Br, Bi, Cr, Ci, dAr, dAi, dBr, dBi, dCr, dCi);
                    }
                    for (; ksafe >= 1; ksafe--) { body(Cr, Ci, Ar, Ai, Br, Bi, dCr, dCi, dAr, dAi, dBr, dBi); rot(); }
                }
                while (ofm <= lim) { body(Cr, Ci, Ar, Ai, Br, Bi, dCr, dCi, dAr, dAi, dBr, dBi); rot(); }     // stragglers
                x0 = Ar; y0i = Ai; x1 = Br; y1i = Bi; x2 = Cr; y2i = Ci;
                d0 = dAr; e0 = dAi; d1 = dBr; e1 = dBi; d2 = dCr; e2 = dCi;
                o = static_cast<int>(ofm - 8388608.0f);
                cnt = static_cast<int>((syp - syp0) / (ROWF * 4));
            } else if (active && LOOPK == LOOP_SYMSYNC) {
                while (o + la <= wlen) {
                    const float* x = buf + o * ROWF;
                    // rintf(mu*128) without a conversion unit: adding 1.5*2^23 rounds to nearest-even at integer
                    // granularity (mu*128 is exact, so the fused form rounds once); the integer sits in the low
                    // mantissa bits
                    const float* tp = mmp + (__float_as_int(fmaf(mu, 128.0f, 12582912.0f)) & 0x3ff);
                    // 8-tap MMSE interpolation, oldest sample first: taps[7], taps[6], ...
                    float yr = 0.0f, yi = 0.0f;
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const float tt = tp[(7 - i) * 132];
                        yr = fmaf(tt, x[i * ROWF], yr);
                        if (NCOMP == 2) yi = fmaf(tt, x[i * ROWF + 1], yi);
                    }
                    x2 = x1; x1 = x0; x0 = yr;
                    d2 = d1; d1 = d0;
                    if (NCOMP == 2) { y2i = y1i; y1i = y0i; y0i = yi; e2 = e1; e1 = e0; }
                    float err;
                    if (NCOMP == 2) {
                        if (SLICER == SL_RECT4) { d0 = qrl_slice_rect4(yr); e0 = 0.0f; }
                        else qrl_slice(SLICER, yr, yi, d0, e0);
                        const float ar = x0 - x2, ai = y0i - y2i;
                        const float br = d0 - d2, bi = e0 - e2;
                        const float u = (ar * d1 + ai * e1) - (br * x1 + bi * y1i);
                        err = qrl_clip1(u);
                    } else {
                        if (SLICER == SL_RECT4) d0 = qrl_slice_rect4(yr);
                        else { float ee; qrl_slice(SLICER, yr, yi, d0, ee); }
                        if (VAR == 3) {
                            // TED_MUELLER_AND_MULLER: e = d[n-1] x[n] - d[n] x[n-1], clipped to +-1
                            const float u = d1 * x0 - d0 * x1;
                            err = qrl_clip1(u);
                        } else {
                            const float u = (x0 - x2) * d1 - (d0 - d2) * x1;
                            err = qrl_clip1(u * 0.5f);
                        }
                    }
                    avg_period = avg_period + k_beta * err;
                    avg_period = fminf(fmaxf(avg_period, k_minp), k_maxp);   // == the two-sided clamp (no NaNs here)
                    inst_period = avg_period + k_alpha * err;
                    inst_period = inst_period <= 0.0f ? avg_period : inst_period;
                    const float ph = mu + inst_period;
                    // floorf(ph): in lock ph lies in [n0, n0+3) (n0 = floor(min_period - |alpha|)): two compares and
                    // selects replace FRND/F2I on the loop-carried path; anything else takes the generic route
                    const bool g1 = ph >= k_f1, g2 = ph >= k_f2;
                    float fl = g2 ? k_f2 : (g1 ? k_f1 : k_f0);
                    int step = k_n0 + (g1 ? 1 : 0) + (g2 ? 1 : 0);
                    if (__builtin_expect(!(ph >= k_f0 && ph < k_f3), 0)) { fl = floorf(ph); step = static_cast<int>(fl); }
                    mu = ph - fl;
                    o += step;
                    sy[cnt * ROWF] = yr;
                    if (NCOMP == 2) sy[cnt * ROWF + 1] = yi;
                    cnt++;
                }
            }
            SSP(const long long pt4 = clock64(); pf_run += pt3 - pt2; pf_str += pt4 - pt3; pf_sym += cnt;)
            o -= STRIDE;                                   // next window starts STRIDE rows later
            if (EXT) {
                float* blk = symbuf + b * blk_rows * ROWF;
                reinterpret_cast<int*>(blk)[maxs * 32 + lane] = cnt;
                reinterpret_cast<int*>(blk)[(maxs + 1) * 32 + lane] = nsym_run;
                nsym_run += cnt;
                fence_proxy_async();                       // the drain warp's bulk store reads this block through the async proxy
            } else cntbuf[b * 32 + lane] = cnt;
            __syncwarp();
            if (lane == 0) { mbar_arrive(&bar_free[st]); mbar_arrive(&bar_full[b]); }
            SSP(pf_ho += clock64() - pt4;)
        }
        SSP(const unsigned long long pg3 = globaltimer_ns();)
        SSP(if (g == 0 && lane == 0) { d_ss_prof[8] += pg1 - pg0; d_ss_prof[9] += pg2 - pg0; d_ss_prof[10] += pg3 - pg0; d_ss_prof[11] += 1; })
        SSP(if (g == 0 && lane == 0) { d_ss_prof[0] += pf_we; d_ss_prof[1] += pf_wi; d_ss_prof[2] += pf_run; d_ss_prof[3] += pf_str; d_ss_prof[4] += pf_ho;
                                       d_ss_prof[5] += nchunks; d_ss_prof[6] += pf_sym; d_ss_prof[7] += pf_rounds; })
        if (active) {
            SymSyncState& st = states[c];
            st.ii = base + static_cast<long long>(nchunks) * STRIDE + o;
            st.avg_period = avg_period; st.inst_period = inst_period; st.mu = mu;
            st.xr[0] = x0; st.xr[1] = x1; st.xr[2] = x2; st.xi[0] = y0i; st.xi[1] = y1i; st.xi[2] = y2i;
            st.dr[0] = d0; st.dr[1] = d1; st.dr[2] = d2; st.di[0] = e0; st.di[1] = e1; st.di[2] = e2;
            if (EXT) {
                st.n_sym += nsym_run; st.n_soft += 2LL * nsym_run;
                port1_cnt[c] += nsym_run;
                n_soft_out[c] = st.n_soft;
            }
        }
    } else if (EXT) {
        // ------------------------------------------------------------------ drain warp: hand-off block -> scratch (TMA)
        if (lane == 0) {
            const size_t blk_floats = static_cast<size_t>(blk_rows) * ROWF;
            float* dst0 = ext_scratch + static_cast<size_t>(g) * ext_chunk_stride * blk_floats;
            for (int m = 0; m < nchunks; m++) {
                const int b = m % NB;
                mbar_wait(&bar_full[b], (m / NB) & 1);
                bulk_s2g(dst0 + static_cast<size_t>(m) * blk_floats, symbuf + b * blk_floats, static_cast<uint32_t>(blk_floats * 4));
                bulk_commit();
                bulk_wait_read0();                         // the block may be refilled once its bytes have been read
                mbar_arrive(&bar_empty[b]);
            }
            bulk_wait_all0();
        }
    } else {
        // ------------------------------------------------------------------ epilogue warps
        const int e = SPLIT ? 0 : warp - 2;
        long long n_sym = 0, n_soft = 0; LoopState costas{ 0.0f, 0.0f }; float dp_r = 0, dp_i = 0;
        int p1cnt = 0;
        if (active) {
            const SymSyncState& st = states[c];
            n_sym = st.n_sym; n_soft = st.n_soft; costas = st.costas; dp_r = st.dp_r; dp_i = st.dp_i;
            p1cnt = port1_cnt[c];
        }
        unsigned char* sr = soft_ring + static_cast<long long>(c) * soft_stride;
        float2* p1 = port1 + static_cast<long long>(c) * port1_stride;
        for (int m = 0; m < nchunks; m++) {
            const int b = m % NB;
            if (SPLIT && warp == 3) mbar_wait(&bar_cdone[b], (m / NB) & 1);     // the Costas warp is through with this block
            else mbar_wait(&bar_full[b], (m / NB) & 1);
            const int n = cntbuf[b * 32 + lane];
            const float* sy = symbuf + b * blk_rows * ROWF + lane * NCOMP;
            if (EPI == EPI_QPSK && (!SPLIT || warp == 2)) {
                // pass 1: the second Costas loop (the only recurrence here) runs over this lane's symbols in place, lean;
                // pass 2 below is feed-forward (diff_phasor, rotation, soft bits, stores)
                qrl_costas4_snr_chunk(costas, p.costas_alpha, p.costas_beta, smem_u32(sy), ROWF * 4, active ? n : 0,
                                      smem_u32(tanh_s) - (0x4B000000u << 2) + static_cast<uint32_t>(opaque_zero));
            }
            if (SPLIT && warp == 2) {                      // hand the block on to the feed-forward warp
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_cdone[b]);
                continue;
            }
            for (int s = e; s < n; s += (SPLIT ? 1 : NEPI)) {
                const float yr = sy[s * ROWF];
                const float yi = (NCOMP == 2) ? sy[s * ROWF + 1] : 0.0f;
                float o_r, o_i;
                unsigned char sb0, sb1 = 0;
                if (EPI == EPI_BPSK) {
                    // costas_loop_cc(order 2) -> port 1; complex_to_real -> one soft bit per symbol
                    qrl_costas_step(costas, p.costas_alpha, p.costas_beta, 2, false, yr, yi, o_r, o_i);
                    sb0 = qrl_soft_u8(o_r, p.soft_scale);
                } else if (EPI == EPI_REAL1) {
                    o_r = yr; o_i = 0.0f;                      // float_to_complex(sym, 0)
                    sb0 = qrl_soft_u8(yr, p.soft_scale);
                } else if (EPI == EPI_4FSK_FM) {
                    const float phs = p.pm_sens * yr;
                    float sn, cs;
                    qrl_sincosf(phs, sn, cs);
                    o_r = cs; o_i = sn;
                    sb0 = qrl_soft_u8(sn, p.soft_scale);       // interleave: imag first, then real
                    sb1 = qrl_soft_u8(cs, p.soft_scale);
                } else if (EPI == EPI_CPLX) {
                    o_r = yr; o_i = yi;
                    sb0 = qrl_soft_u8(yr, p.soft_scale);
                    sb1 = qrl_soft_u8(yi, p.soft_scale);
                } else {
                    const float cr = yr, ci = yi;                  // already through the Costas loop (pass 1)
                    const float dr = cr * dp_r + ci * dp_i;
                    const float di = ci * dp_r - cr * dp_i;
                    dp_r = cr; dp_i = ci;
                    o_r = dr * p.rot_r - di * p.rot_i;
                    o_i = dr * p.rot_i + di * p.rot_r;
                    sb0 = qrl_soft_u8(o_r, p.soft_scale);
                    sb1 = qrl_soft_u8(o_i, p.soft_scale);
                }
                if (p1cnt + s < port1_cap) p1[p1cnt + s] = make_float2(o_r, o_i);
                if (EPI == EPI_BPSK || EPI == EPI_REAL1) sr[(n_soft + s) & soft_mask] = sb0;
                else { sr[(n_soft + 2 * s) & soft_mask] = sb0; sr[(n_soft + 2 * s + 1) & soft_mask] = sb1; }
            }
            p1cnt += n; n_soft += ((EPI == EPI_BPSK || EPI == EPI_REAL1) ? 1 : 2) * n; n_sym += n;
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_empty[b]);
        }
        if (active && SPLIT) {
            SymSyncState& st = states[c];
            if (warp == 2) st.costas = costas;
            else { st.n_sym = n_sym; st.n_soft = n_soft; st.dp_r = dp_r; st.dp_i = dp_i; port1_cnt[c] = p1cnt; n_soft_out[c] = n_soft; }
        } else if (active && e == 0) {
            SymSyncState& st = states[c];
            st.n_sym = n_sym; st.n_soft = n_soft; st.costas = costas; st.dp_r = dp_r; st.dp_i = dp_i;
            port1_cnt[c] = p1cnt;
            n_soft_out[c] = n_soft;
        }
    }
}

// External epilogue of symsync_kernel<.., EPI_EXT_4FSK_FM, ..>: phase_modulator_fc(pi/2) -> port 1, soft bits (imag, real)
// -> soft ring.  One block per (chunk, 32-channel group); x = channel lane (coalesced reads of the hand-off block),
// y strides over the symbols of the chunk.  Same arithmetic as the in-kernel EPI_4FSK_FM branch.  SCALE = 1 (gr_demod_dmr): the
// symbols pass multiply_const_ff(p.sym_scale) before the phase modulator.
template <int SCALE = 0>
__global__ void __launch_bounds__(256)
symsync_ext_epilogue_kernel(SymSyncParams p, int C, const float* __restrict__ scratch, int chunk_stride, int maxs,
                            const int* __restrict__ hdr_all,
                            float2* __restrict__ port1, long long port1_stride, int port1_cap,
                            unsigned char* __restrict__ soft_ring, unsigned soft_mask, long long soft_stride,
                            unsigned char* __restrict__ hard_port2 = nullptr /* M17: [C][hard_cap] bits */, long long hard_stride = 0,
                            int hard_cap = 0, int* __restrict__ hard_cnt = nullptr, const int* __restrict__ port1_cnt = nullptr)
{
    const int g = blockIdx.y, m = blockIdx.x, lane = threadIdx.x, c = g * 32 + lane;
    const int* hdr = hdr_all + g * 128;
    if (m >= hdr[96] || c >= C) return;
    const size_t blk_floats = static_cast<size_t>(maxs + 2) * 32;
    const float* blk = scratch + (static_cast<size_t>(g) * chunk_stride + m) * blk_floats;
    const int cnt = reinterpret_cast<const int*>(blk)[maxs * 32 + lane];
    const int sbase = reinterpret_cast<const int*>(blk)[(maxs + 1) * 32 + lane];
    const int p1cnt0 = hdr[lane];
    const long long n_soft0 = (static_cast<long long>(hdr[64 + lane]) << 32) | static_cast<unsigned>(hdr[32 + lane]);
    unsigned char* sr = soft_ring + static_cast<long long>(c) * soft_stride;
    float2* p1 = port1 + static_cast<long long>(c) * port1_stride;
    for (int k = threadIdx.y; k < cnt; k += blockDim.y) {
        const float yr = SCALE ? blk[k * 32 + lane] * p.sym_scale : blk[k * 32 + lane];
        float sn, cs;
        qrl_sincosf(p.pm_sens * yr, sn, cs);
        const int idx = sbase + k;
        if (p1cnt0 + idx < port1_cap) p1[p1cnt0 + idx] = make_float2(cs, sn);
        if (hard_port2) {
            // gr_demod_m17.cpp:98-107: (re, im) -> binary_slicer_fb -> pack_k_bits(2) -> map {3,1,2,0} -> unpack_k_bits(2)
            const int v = ((cs >= 0.0f) ? 2 : 0) | ((sn >= 0.0f) ? 1 : 0);
            const int mp = (0x27 >> (2 * v)) & 3;                     // {3,1,2,0} packed two bits per entry: 0b00'10'01'11
            const long long b = 2LL * (p1cnt0 + idx);
            unsigned char* hp = hard_port2 + static_cast<long long>(c) * hard_stride;
            if (b + 1 < hard_cap) { hp[b] = static_cast<unsigned char>((mp >> 1) & 1); hp[b + 1] = static_cast<unsigned char>(mp & 1); }
            continue;
        }
        const long long so = n_soft0 + 2LL * idx;
        sr[so & soft_mask] = qrl_soft_u8(sn, p.soft_scale);          // interleave: imag first, then real
        sr[(so + 1) & soft_mask] = qrl_soft_u8(cs, p.soft_scale);
    }
    if (hard_port2 && m == 0 && threadIdx.y == 0) hard_cnt[c] = 2 * port1_cnt[c];   // the symbol-sync launch has finished: final count
}

// ------------------------------------------------------------------------------------------------
// RSSI tap on port 0 (rssi_block.cpp:25-45 behind gr_demod_base.cpp:199-200): |x|^2 -> moving_average_ff(2000) ->
// single_pole_iir_filter_ff(0.04) -> 10 log10; only the latest value is observable (probe_signal_f).  The IIR forgets
// geometrically (0.96^1024 ~ 7e-19), so one CTA per channel evaluates the last min(new, 1024) moving sums directly from
// a 4096-deep ring of |x|^2 (window sums in a fixed order instead of the reference's drifting running sum: telemetry
// value, equal to the oracle within 1e-3 dB) and thread 0 runs the IIR over them.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rssi_kernel(const float2* __restrict__ port0, long long port0_stride, int n_new, long long n_before,
            float* __restrict__ ring /* [C][4096] */, float* __restrict__ y_state /* [C] */, float* __restrict__ out_db /* [C] */)
{
    constexpr int RING = 4096, LEN = 2000, KMAX = 1024;
    __shared__ float w[RING];
    __shared__ float m[KMAX];
    const int c = blockIdx.x;
    float* rg = ring + static_cast<long long>(c) * RING;
    const float2* x = port0 + static_cast<long long>(c) * port0_stride;
    for (int i = threadIdx.x; i < n_new; i += blockDim.x) {
        if (n_new - i > RING) continue;                          // only the last RING samples can matter
        const float2 v = x[i];
        rg[(n_before + i) & (RING - 1)] = v.x * v.x + v.y * v.y;
    }
    __syncthreads();
    const long long N = n_before + n_new;
    for (int k = threadIdx.x; k < RING; k += blockDim.x) {       // w[k] = |x|^2 at absolute index N - RING + k
        const long long a = N - RING + k;
        w[k] = a >= 0 ? rg[a & (RING - 1)] : 0.0f;
    }
    __syncthreads();
    const int K = n_new < KMAX ? n_new : KMAX;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {          // output n = N - K + 1 + k (1-based count) ends at w[RING - K + k]
        const int end = RING - K + k;
        float acc = 0.0f;
        for (int j = end - (LEN - 1); j <= end; j++) acc = acc + w[j];
        m[k] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0 && K > 0) {
        double y = (n_new >= KMAX) ? 0.0 : static_cast<double>(y_state[c]);
        float yf = static_cast<float>(y);
        for (int k = 0; k < K; k++) {
            y = 0.04 * static_cast<double>(m[k]) + (1.0 - 0.04) * y;
            yf = static_cast<float>(y);
            y = static_cast<double>(yf);
        }
        y_state[c] = yf;
        out_db[c] = 10.0f * log10f(yf > 1e-18f ? yf : 1e-18f);
    }
}

// ------------------------------------------------------------------------------------------------
// CCSDS K=7 r=1/2 soft Viterbi, fec::decoder(cc_decoder(80,7,2,{109,79}, CC_STREAMING)) stream semantics,
// + descrambler_bb(0x8A,0x7F,7).  One warp per channel: lane i = butterfly i (states 2i, 2i+1).
// 32-bit path metrics without renormalisation are decision-equivalent to VOLK's 8-bit generic kernel
// (which renormalises every step and never wraps: spread <= 6*31+31 < 256).
// ------------------------------------------------------------------------------------------------
struct ViterbiState {
    long long rd;            // absolute soft-bit index of the next frame's first NEW symbol (frame start - 12 = rd - 12)
    int start_state;
    unsigned descr_reg;
};

// Two warps per channel: warp 0 runs the add-compare-select recursion (lane i = butterfly i), finds the best end
// state and walks back the 6 tail steps that fix the next frame's start state, then immediately starts the next
// frame; warp 1 does the 80-step traceback, descrambling and the stores for the previous frame.  Decisions are
// double buffered in shared memory (mbarrier full/empty); the next frame's soft symbols are prefetched into
// registers during the current ACS.
//
// The ACS step is written for a warp whose only business is the loop-carried metric exchange (round 2; 157 -> ~45 cycles):
//   * the two path metrics of a lane travel as ONE register (two 16-bit halves: a frame adds at most 86 * 31 to the
//     start value 63, far below 2^16, so the comparisons are those of the 32-bit form): 2 SHFL per step instead of 4,
//     the half a lane needs comes out with one PRMT whose selector is a per-lane constant;
//   * the branch metrics do not depend on the path: at the start of a frame the warp turns its 172 soft symbols into 86
//     words holding the metric of each of the four branch-label classes (b0, b1) in {0, 255}^2; in the loop a lane takes its
//     class byte with one PRMT from a word that was loaded four steps earlier (LDS.128 per four steps, off the chain);
//   * new metric = min(x + m, x' + m') is one VIADDMNMX per state; the two ballots of a step leave with one predicated
//     STS.64; the last six steps' ballots stay in registers for the tail walk; the best end state is one REDUX.MIN.
template <int CPB /* channels per CTA */>
__global__ void __launch_bounds__(64 * CPB)
viterbi_k7_kernel(ViterbiState* __restrict__ vstates, const long long* __restrict__ n_soft_avail, int C,
                  const unsigned char* __restrict__ soft_ring, unsigned soft_mask, long long soft_stride,
                  unsigned char* __restrict__ port2, long long port2_stride, int* __restrict__ port2_cnt, int port2_cap,
                  int delay /* blocks::delay(1) in front of the second decoder: stream index shifted by `delay` */)
{
    __shared__ unsigned char syms_all[CPB][176];
    __shared__ __align__(16) unsigned mw_all[CPB][88];        // per step: metric of label class (b0 ? 2 : 0) | (b1 ? 1 : 0) in byte `class`
    __shared__ __align__(8) uint2 dec_all[CPB][2][86];        // per step: ballots of d0 (new state 2 lane) and d1 (new state 2 lane + 1)
    __shared__ unsigned endst_all[CPB][2];
    __shared__ unsigned char obits_all[CPB][80];
    __shared__ __align__(8) uint64_t bar_full_all[CPB][2], bar_empty_all[CPB][2];
    const int slot = threadIdx.x >> 6;                       // channel slot inside the CTA (2 warps each)
    const int c = blockIdx.x * CPB + slot;
    const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & 1;
    unsigned char* syms = syms_all[slot];
    unsigned* mw = mw_all[slot];
    uint2 (*dec)[86] = dec_all[slot];
    unsigned* endst = endst_all[slot];
    unsigned char* obits = obits_all[slot];
    uint64_t* bar_full = bar_full_all[slot];
    uint64_t* bar_empty = bar_empty_all[slot];
    if ((threadIdx.x & 63) == 0) {
        for (int b = 0; b < 2; b++) { mbar_init(&bar_full[b], 1); mbar_init(&bar_empty[b], 1); }
        mbar_fence_init();
    }
    __syncthreads();
    if (c >= C) return;
    const ViterbiState vs0 = vstates[c];
    const long long avail = n_soft_avail[c] + delay;
    const int nframes = (avail - vs0.rd) >= 160 ? static_cast<int>((avail - vs0.rd) / 160) : 0;
    if (nframes == 0) return;
    const unsigned char* sr = soft_ring + static_cast<long long>(c) * soft_stride;

    if (warp == 0) {
        // ---------------------------------------------------------------- ACS warp
        // branch labels of butterfly `lane`: parity((2*lane) & poly) -> label class and the PRMT selectors of this lane
        const unsigned l0 = __popc((2u * lane) & 109u) & 1u, l1 = __popc((2u * lane) & 79u) & 1u;
        const unsigned sel_m = 0x4440u | (l0 * 2u + l1);                 // byte `class` of the metric word, zero extended
        const unsigned sel_x = (lane & 1) ? 0x4432u : 0x4410u;           // high / low 16-bit half, zero extended
        const int src0 = lane >> 1, src1 = (lane >> 1) + 16;
        int start_state = vs0.start_state;
        // soft symbols of a frame: absolute indices [rd - 12, rd + 160); each lane carries bytes i = lane + 32 k
        unsigned char pre[6];
        auto fetch = [&](long long rd) {
#pragma unroll
            for (int k = 0; k < 6; k++) {
                const int i = lane + 32 * k;
                const long long a = rd - 12 + i - delay;
                pre[k] = (i < 172 && a >= 0) ? sr[a & soft_mask] : 0;
            }
        };
        fetch(vs0.rd);
        for (int f = 0; f < nframes; f++) {
            const int b = f & 1;
#pragma unroll
            for (int k = 0; k < 6; k++) { const int i = lane + 32 * k; if (i < 172) syms[i] = pre[k]; }
            if (f + 1 < nframes) fetch(vs0.rd + 160LL * (f + 1));      // latency hidden behind this frame's ACS
            __syncwarp();
            // branch metrics of the frame: (((b0 ^ s0) >> 2) + ((b1 ^ s1) >> 2)) >> 2 for the four label classes
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const int st = lane + 32 * k;
                if (st < 86) {
                    const unsigned s0 = syms[2 * st], s1 = syms[2 * st + 1];
                    const unsigned a0 = s0 >> 2, a1 = (255u ^ s0) >> 2, c0 = s1 >> 2, c1 = (255u ^ s1) >> 2;
                    mw[st] = ((a0 + c0) >> 2) | (((a0 + c1) >> 2) << 8) | (((a1 + c0) >> 2) << 16) | (((a1 + c1) >> 2) << 24);
                }
            }
            if (f >= 2) mbar_wait(&bar_empty[b], ((f >> 1) - 1) & 1);  // traceback warp released dec[b]
            __syncwarp();
            unsigned ya = 63, yb = 63;                                  // Y[2 lane], Y[2 lane + 1]
            if ((start_state & 63) == 2 * lane) ya = 0;
            if ((start_state & 63) == 2 * lane + 1) yb = 0;
            unsigned P = ya | (yb << 16);
            unsigned t0[6], t1[6];                                      // ballots of steps 80..85 (tail walk)
            auto step = [&](const unsigned W, const int s, unsigned& B0, unsigned& B1) {
                const unsigned v0 = __shfl_sync(0xffffffffu, P, src0);
                const unsigned v1 = __shfl_sync(0xffffffffu, P, src1);
                const unsigned xi = __byte_perm(v0, 0u, sel_x);         // X[lane]
                const unsigned xj = __byte_perm(v1, 0u, sel_x);         // X[lane + 32]
                const unsigned m = __byte_perm(W, 0u, sel_m), nm = 31u - m;
                const unsigned m0 = xi + m, m1 = xj + nm, m2 = xi + nm, m3 = xj + m;
                const unsigned na = __viaddmin_u32(xi, m, m1);          // min(m0, m1)
                const unsigned nb = __viaddmin_u32(xi, nm, m3);         // min(m2, m3)
                B0 = __ballot_sync(0xffffffffu, m0 > m1);
                B1 = __ballot_sync(0xffffffffu, m2 > m3);
                P = __byte_perm(na, nb, 0x5410u);                       // na | nb << 16
                if (lane == 0) dec[b][s] = make_uint2(B0, B1);
            };
            const uint4* mw4 = reinterpret_cast<const uint4*>(mw);
#pragma unroll 1
            for (int s4 = 0; s4 < 20; s4++) {                           // steps 0..79, four per metric-word load
                const uint4 W = mw4[s4];
                unsigned B0, B1;
                step(W.x, 4 * s4 + 0, B0, B1);
                step(W.y, 4 * s4 + 1, B0, B1);
                step(W.z, 4 * s4 + 2, B0, B1);
                step(W.w, 4 * s4 + 3, B0, B1);
            }
            {
                const uint4 Wa = mw4[20]; const uint2 Wb = reinterpret_cast<const uint2*>(mw)[42];
                step(Wa.x, 80, t0[0], t1[0]); step(Wa.y, 81, t0[1], t1[1]); step(Wa.z, 82, t0[2], t1[2]); step(Wa.w, 83, t0[3], t1[3]);
                step(Wb.x, 84, t0[4], t1[4]); step(Wb.y, 85, t0[5], t1[5]);
            }
            // best end state: minimum metric, lowest index on ties
            ya = P & 0xffffu; yb = P >> 16;
            const unsigned key_l = (ya <= yb) ? ((ya << 6) | (2u * lane)) : ((yb << 6) | (2u * lane + 1u));
            const unsigned key = __reduce_min_sync(0xffffffffu, key_l);
            // the first 6 traceback steps (bits 79..74, trellis steps 85..80) give the state the next frame starts from
            unsigned st = key & 63u;
#pragma unroll
            for (int j = 5; j >= 0; j--) {
                const unsigned k = (((st & 1u) ? t1[j] : t0[j]) >> (st >> 1)) & 1u;
                st = (st >> 1) | (k << 5);
            }
            start_state = static_cast<int>(st);
            __syncwarp();                                               // lane 0's dec[b][*] stores are ordered before its arrive
            if (lane == 0) { endst[b] = key & 63u; mbar_arrive(&bar_full[b]); }
        }
        if (lane == 0) { vstates[c].start_state = start_state; vstates[c].rd = vs0.rd + 160LL * nframes; }
    } else {
        // ---------------------------------------------------------------- traceback / output warp
        unsigned descr_reg = vs0.descr_reg;
        int cnt = port2_cnt[c];
        unsigned char* outp = port2 + static_cast<long long>(c) * port2_stride;
        for (int f = 0; f < nframes; f++) {
            const int b = f & 1;
            mbar_wait(&bar_full[b], (f >> 1) & 1);
            if (lane == 0) {
                unsigned st = endst[b];
                // the decision words do not depend on the state: loaded eight steps ahead of the walk
#pragma unroll 1
                for (int nb8 = 72; nb8 >= 0; nb8 -= 8) {
                    uint2 d[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) d[j] = dec[b][nb8 + j + 6];
#pragma unroll
                    for (int j = 7; j >= 0; j--) {
                        const unsigned k = (((st & 1u) ? d[j].y : d[j].x) >> (st >> 1)) & 1u;
                        st = (st >> 1) | (k << 5);
                        obits[nb8 + j] = static_cast<unsigned char>(k);
                    }
                }
                mbar_arrive(&bar_empty[b]);
            }
            __syncwarp();
            // descrambler: out[n] = in[n] ^ in[n-1] ^ in[n-5] ^ in[n-7]; reg bit (8-d) holds in[n-d]
            for (int i = lane; i < 80; i += 32) {
                auto bit = [&](int n) -> unsigned { return n >= 0 ? obits[n] : ((descr_reg >> (8 + n)) & 1u); };
                const unsigned o = bit(i) ^ bit(i - 1) ^ bit(i - 5) ^ bit(i - 7);
                if (cnt + i < port2_cap) outp[cnt + i] = static_cast<unsigned char>(o);
            }
            unsigned reg = 0;
#pragma unroll
            for (int d = 1; d <= 8; d++) reg |= static_cast<unsigned>(obits[80 - d]) << (8 - d);
            descr_reg = reg;
            cnt += 80;
            __syncwarp();
        }
        if (lane == 0) { vstates[c].descr_reg = descr_reg; port2_cnt[c] = cnt; }
    }
}

// ------------------------------------------------------------------------------------------------
// NBFM audio chain after the channel filter (gr_demod_nbfm.cpp:68-76): pwr_squelch_cc(gate) -> quadrature_demod_cf
// -> rational_resampler_fff(2,5) -> fft_filter_fff (audio LPF, direct form) -> iir_filter_ffd (de-emphasis) -> x2.
// 20 ksps per channel: one CTA per channel; the two recurrences (squelch state machine with its double-precision
// power IIR, de-emphasis IIR) run on thread 0, the FIR-type stages are spread over the CTA.  All streams are
// small per-channel rings addressed by absolute item index, so chunking is invisible.
// ------------------------------------------------------------------------------------------------
struct NbfmState {
    double pwr, iir_x1, iir_y1;
    long long n_in;           // channel-filter items consumed
    long long n_gate;         // items passed by the squelch (= demod stream length)
    long long n_res;          // resampler outputs produced
    long long n_aud;          // audio-filter / de-emphasis outputs produced
    int sq_state, ramped;
    float envelope;
    float prev_r, prev_i;     // quadrature demod memory
    float agc_gain;           // AM: agc2_ff gain
    // NBFM tone squelch (ctcss_squelch_ff): gated audio items written so far, three Goertzel filters, squelch_base_ff state
    long long n_q;
    float gl1, gl2, gc1, gc2, gr1, gr2;
    int g_processed, c_mute, c_state, c_ramped;
    double c_env;
};
struct NbfmCtcss { int on, len, ramp, gate; float level, wr_l, wi_l, wr_c, wi_c, wr_r, wi_r; };
struct NbfmParams {
    double sq_alpha, sq_threshold;
    int sq_ramp, sq_gate;
    float qd_gain;
    int nt_arm;               // taps per resampler arm (L = 2, M = 5)
    int nt_audio;
    double b0, b1, a1;
    float out_gain;
    // mode 2 = WBFM (gr_demod_wbfm.cpp:56-64): squelch -> quadrature demod -> x am_gain -> de-emphasis iir (b0, b1, a1) on the
    // 200 ksps stream, then rational_resampler_fff(1, 25) (nt_audio taps, THE FIR order with D = 25) straight to port 1
    // mode 1 = AM detector (gr_demod_am.cpp:57-71): squelch -> complex_to_mag -> agc2_ff -> iir_filter_ffd (b0, b1, a1) -> x am_gain
    // on the 20 ksps stream, then resampler 2/5 and audio low-pass straight to port 1 (no de-emphasis behind them)
    int mode;
    float agc_attack, agc_decay, agc_ref, agc_max, am_gain;
};
enum { SQ_MUTED = 0, SQ_ATTACK = 1, SQ_UNMUTED = 2, SQ_DECAY = 3 };

__global__ void __launch_bounds__(128)
nbfm_audio_kernel(NbfmParams p, NbfmState* __restrict__ states,
                  const float2* __restrict__ in, unsigned in_mask, long long in_stride, long long avail_in,
                  const float* __restrict__ env_tab,            // sq_ramp + 1 envelope values
                  float2* __restrict__ gate_ring, unsigned gate_mask, long long gate_stride,
                  float* __restrict__ dem_ring, unsigned dem_mask, long long dem_stride,
                  float* __restrict__ res_ring, unsigned res_mask, long long res_stride,
                  const float* __restrict__ arm_taps,           // [2][nt_arm]
                  const float* __restrict__ audio_taps,
                  float* __restrict__ port1, long long port1_stride, int* __restrict__ port1_cnt, int port1_cap,
                  // NBFM (mode 0) only: when given, the audio filter's output goes to this ring and the de-emphasis runs in
                  // nbfm_deemph_kernel on another stream (its recurrence then overlaps the next slice's squelch recurrence);
                  // aud_snap[c] = audio items produced so far
                  float* __restrict__ aud_ring = nullptr, unsigned aud_mask = 0, long long aud_stride = 0, long long* __restrict__ aud_snap = nullptr,
                  // NBFM only: the stream between the 2/5 resampler and the audio filter goes through this ring: a plain copy, or
                  // ctcss_squelch_ff (gate: the stream shrinks while the tone is absent) when ct.on (gr_demod_nbfm::set_ctcss)
                  float* __restrict__ q_ring = nullptr, unsigned q_mask = 0, long long q_stride = 0, NbfmCtcss ct = NbfmCtcss{},
                  const double* __restrict__ c_env_tab = nullptr)
{
    const int c = blockIdx.x;
    __shared__ NbfmState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float2* gr_ = gate_ring + static_cast<long long>(c) * gate_stride;
    float* dr = dem_ring + static_cast<long long>(c) * dem_stride;
    float* rr = res_ring + static_cast<long long>(c) * res_stride;
    const long long gate0 = st.n_gate;

    // ---- 1. squelch (sequential on thread 0; input tiles staged in shared memory by the whole CTA so the
    //         recurrence never waits on a global load)
    // Fast path (round 2): while the squelch sits in a stable state (open, or closed) the only recurrence is the power estimate
    // pwr = alpha |x|^2 + (1 - alpha) pwr (double, two dependent operations per sample).  Thread 0 runs just that over the
    // tile's |x|^2 (computed by the whole CTA) until the first sample that would change the state; the samples before it
    // are passed (or dropped) in bulk by all threads, the rest of the tile goes through the full state machine below.
    __shared__ float2 xin[2048];
    __shared__ double t1s[2048];          // alpha * |x|^2 in double, computed by the whole CTA: an FP64 instruction occupies the SM's FP64
                                          // pipe for ~64 cycles whatever its lane count, so the recurrence thread keeps only the two
                                          // operations that are on the chain
    __shared__ float aud[2048];           // staging of the audio-rate (WBFM: 200 ksps) recurrences
    __shared__ int fast_n, fast_state;
    __shared__ long long fast_ng0;
    __shared__ float fast_env;
    for (long long tile0 = st.n_in; tile0 < avail_in; tile0 += 2048) {
        const int nt = (avail_in - tile0) < 2048 ? static_cast<int>(avail_in - tile0) : 2048;
        for (int j = threadIdx.x; j < nt; j += blockDim.x) {
            const float2 v = x[(tile0 + j) & in_mask];
            xin[j] = v;
            t1s[j] = p.sq_alpha * static_cast<double>(v.x * v.x + v.y * v.y);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double pwr = st.pwr; int state = st.sq_state, ramped = st.ramped; float env = st.envelope;
            float agc = st.agc_gain; double ix1 = st.iir_x1, iy1 = st.iir_y1;
            long long ng = st.n_gate;
            const double one_m_alpha = 1.0 - p.sq_alpha;
            int j0 = 0;
            fast_n = 0;
            if (p.mode != 1 && (state == SQ_UNMUTED || state == SQ_MUTED)) {
                const bool want = (state == SQ_MUTED);           // the state holds while every sample's mute flag equals `want`
                // pn and the threshold are non-negative doubles: pn < thr is the same comparison on their bit patterns (an integer
                // compare instead of a third FP64-pipe instruction per sample)
                const long long thr_bits = __double_as_longlong(p.sq_threshold);
                int j = 0;
                for (; j < nt; j++) {
                    const double pn = t1s[j] + one_m_alpha * pwr;
                    if ((__double_as_longlong(pn) < thr_bits) != want) break;
                    pwr = pn;
                }
                fast_n = j; fast_state = state; fast_ng0 = ng; fast_env = env;
                if (state == SQ_UNMUTED || !p.sq_gate) ng += j;
                j0 = j;
            }
            for (int j = j0; j < nt; j++) {
                const float2 v = xin[j];
                const float mag2 = v.x * v.x + v.y * v.y;
                pwr = p.sq_alpha * static_cast<double>(mag2) + one_m_alpha * pwr;
                const bool mute = pwr < p.sq_threshold;
                switch (state) {
                case SQ_MUTED: if (!mute) state = p.sq_ramp ? SQ_ATTACK : SQ_UNMUTED; break;
                case SQ_UNMUTED: if (mute) state = p.sq_ramp ? SQ_DECAY : SQ_MUTED; break;
                case SQ_ATTACK:
                    env = env_tab[++ramped];
                    if (ramped >= p.sq_ramp) { state = SQ_UNMUTED; env = 1.0f; }
                    break;
                case SQ_DECAY:
                    env = env_tab[--ramped];
                    if (ramped == 0) state = SQ_MUTED;
                    break;
                }
                if (p.mode == 1) {
                    if (state != SQ_MUTED) {
                        const float vr = v.x * env, vi = v.y * env;
                        const float mag = sqrtf(vr * vr + vi * vi);                    // complex_to_mag
                        const float outv = mag * agc;                                   // agc2_ff::scale
                        const float tmp = fabsf(outv) - p.agc_ref;
                        const float rate = (fabsf(tmp) > agc) ? p.agc_attack : p.agc_decay;
                        agc = agc - tmp * rate;
                        if (agc < 0.0f) agc = 10e-5f;
                        if (p.agc_max > 0.0f && agc > p.agc_max) agc = p.agc_max;
                        const double xin = static_cast<double>(outv);                   // iir_filter_ffd
                        double acc = p.b0 * xin;
                        acc = acc + p.b1 * ix1;
                        acc = acc - p.a1 * iy1;
                        ix1 = xin; iy1 = acc;
                        dr[ng & dem_mask] = static_cast<float>(acc) * p.am_gain;
                        ng++;
                    }
                } else if (state != SQ_MUTED) { gr_[ng & gate_mask] = make_float2(v.x * env, v.y * env); ng++; }
                else if (!p.sq_gate) { gr_[ng & gate_mask] = make_float2(0.0f, 0.0f); ng++; }
            }
            st.pwr = pwr; st.sq_state = state; st.ramped = ramped; st.envelope = env; st.n_gate = ng;
            if (p.mode == 1) { st.agc_gain = agc; st.iir_x1 = ix1; st.iir_y1 = iy1; }
        }
        __syncthreads();
        {   // bulk part of the tile: open squelch -> items x envelope, closed and not gating -> zeros, closed and gating -> nothing
            const int n = fast_n;
            const long long g0 = fast_ng0;
            if (fast_state == SQ_UNMUTED) {
                const float env = fast_env;
                for (int j = threadIdx.x; j < n; j += blockDim.x) { const float2 v = xin[j]; gr_[(g0 + j) & gate_mask] = make_float2(v.x * env, v.y * env); }
            } else if (!p.sq_gate) {
                for (int j = threadIdx.x; j < n; j += blockDim.x) gr_[(g0 + j) & gate_mask] = make_float2(0.0f, 0.0f);
            }
        }
        __syncthreads();
    }
    __syncthreads();      // (empty input: no tile barrier above) every thread has read st.n_in for its loop bounds
    if (threadIdx.x == 0) st.n_in = avail_in;
    __syncthreads();
    const long long gate1 = st.n_gate;
    // ---- 2. quadrature demod over the gated stream (AM: the detector already wrote the 20 ksps stream)
    for (long long n = gate0 + threadIdx.x; n < gate1 && p.mode != 1; n += blockDim.x) {
        const float2 cur = gr_[n & gate_mask];
        float2 prev;
        if (n == gate0) prev = make_float2(st.prev_r, st.prev_i);
        else prev = gr_[(n - 1) & gate_mask];
        const float re = cur.x * prev.x + cur.y * prev.y;
        const float im = cur.y * prev.x - cur.x * prev.y;
        dr[n & dem_mask] = p.qd_gain * qrl_fast_atan2f(im, re);
    }
    __syncthreads();
    if (threadIdx.x == 0 && gate1 > gate0 && p.mode != 1) { const float2 l = gr_[(gate1 - 1) & gate_mask]; st.prev_r = l.x; st.prev_i = l.y; }
    if (p.mode == 2) {
        // ---- WBFM: x am_gain and de-emphasis IIR over the new demodulated samples (sequential), into the res ring at 200 ksps
        // (tiles through shared memory; b0 x[n] + b1 x[n-1] by all threads, thread 0 keeps the two FP64 operations on the chain)
        {
            float* wx = aud;
            double* u = t1s;
            for (long long base = gate0; base < gate1; base += 2048) {
                const int nb = (gate1 - base) < 2048 ? static_cast<int>(gate1 - base) : 2048;
                for (int j = threadIdx.x; j < nb; j += blockDim.x) wx[j] = dr[(base + j) & dem_mask] * p.am_gain;
                __syncthreads();
                const double x1c = st.iir_x1;
                for (int j = threadIdx.x; j < nb; j += blockDim.x) {
                    const double xin = static_cast<double>(wx[j]);
                    const double x1 = j > 0 ? static_cast<double>(wx[j - 1]) : x1c;
                    double acc = p.b0 * xin;
                    acc = acc + p.b1 * x1;
                    u[j] = acc;
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    double y1 = st.iir_y1;
                    for (int j = 0; j < nb; j++) { const double acc = u[j] - p.a1 * y1; y1 = acc; u[j] = acc; }
                    st.iir_y1 = y1; st.iir_x1 = static_cast<double>(wx[nb - 1]);
                }
                __syncthreads();
                for (int j = threadIdx.x; j < nb; j += blockDim.x) rr[(base + j) & res_mask] = static_cast<float>(u[j]);
                __syncthreads();
            }
        }
        __syncthreads();
        // ---- rational_resampler_fff(1, 25): output i = sum_j h[j] z[25 i - j], outputs with 25 i <= gate1 - 1
        const long long o0 = st.n_res, o1 = (gate1 + 24) / 25;
        const int cnt0 = port1_cnt[c];
        float* o = port1 + static_cast<long long>(c) * port1_stride;
        for (long long i = o0 + threadIdx.x; i < o1; i += blockDim.x) {
            const long long newest = 25 * i;
            const float2 y = qrl_fir_dot_order_c(audio_taps, p.nt_audio, 25, [&](int j) {
                const long long n = newest - j;
                return make_float2(n >= 0 ? rr[n & res_mask] : 0.0f, 0.0f);
            });
            const long long slot = cnt0 + (i - o0);
            if (slot < port1_cap) o[slot] = y.x;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            if (o1 > o0) port1_cnt[c] = cnt0 + static_cast<int>(o1 - o0);
            st.n_res = o1 > o0 ? o1 : o0; st.n_aud = st.n_res; states[c] = st;
        }
        return;
    }
    // ---- 3. rational resampler 2/5: output i uses arm (5 i) mod 2 at input position floor(5 i / 2)
    const long long res0 = st.n_res;
    long long res1 = res0;
    res1 = (2 * gate1 + 4) / 5;                                  // ceil(2 G / 5): outputs i with floor(5 i / 2) <= G - 1
    if (res1 < res0) res1 = res0;
    for (long long i = res0 + threadIdx.x; i < res1; i += blockDim.x) {
        const long long pos = (5 * i) >> 1;
        const float* h = arm_taps + ((5 * i) & 1) * p.nt_arm;
        float acc = 0.0f;
        for (int k = p.nt_arm - 1; k >= 0; k--) {
            const long long n = pos - k;
            const float v = n >= 0 ? dr[n & dem_mask] : 0.0f;
            acc = fmaf(h[k], v, acc);
        }
        rr[i & res_mask] = acc;
    }
    __syncthreads();
    // ---- 3b. NBFM: copy, or tone squelch, into the audio filter's input ring
    float* qr = q_ring ? q_ring + static_cast<long long>(c) * q_stride : nullptr;
    if (qr) {
        const long long q0 = st.n_q;
        if (!ct.on) {
            for (long long i = res0 + threadIdx.x; i < res1; i += blockDim.x) qr[(q0 + (i - res0)) & q_mask] = rr[i & res_mask];
            __syncthreads();
            if (threadIdx.x == 0) st.n_q = q0 + (res1 - res0);
        } else {
            for (long long base = res0; base < res1; base += 2048) {
                const int nb = (res1 - base) < 2048 ? static_cast<int>(res1 - base) : 2048;
                for (int j = threadIdx.x; j < nb; j += blockDim.x) aud[j] = rr[(base + j) & res_mask];
                __syncthreads();
                if (threadIdx.x == 0) {
                    float gl1 = st.gl1, gl2 = st.gl2, gc1 = st.gc1, gc2 = st.gc2, gr1 = st.gr1, gr2 = st.gr2;
                    int proc = st.g_processed, mute = st.c_mute, state = st.c_state, ramped = st.c_ramped;
                    double env = st.c_env;
                    long long nq = st.n_q;
                    for (int j = 0; j < nb; j++) {
                        const float xv = aud[j];
                        float y = xv + ct.wr_l * gl1; y = y - gl2; gl2 = gl1; gl1 = y;              // fft::goertzel::input
                        y = xv + ct.wr_c * gc1; y = y - gc2; gc2 = gc1; gc1 = y;
                        y = xv + ct.wr_r * gr1; y = y - gr2; gr2 = gr1; gr1 = y;
                        proc++;
                        if (proc == ct.len) {
                            auto mag = [&](float wr, float wi, float d1, float d2) -> float {
                                const float re = static_cast<float>((0.5 * wr * d1 - d2) / ct.len), im = (wi * d1) / ct.len;
                                const float m = static_cast<float>(sqrt(static_cast<double>(re) * re + static_cast<double>(im) * im));
                                return floorf(100000.0f * m) / 100000.0f;
                            };
                            const float ml = mag(ct.wr_l, ct.wi_l, gl1, gl2), mc = mag(ct.wr_c, ct.wi_c, gc1, gc2), mr = mag(ct.wr_r, ct.wi_r, gr1, gr2);
                            gl1 = gl2 = gc1 = gc2 = gr1 = gr2 = 0.0f; proc = 0;
                            mute = (mc < ct.level || mc < ml || mc < mr) ? 1 : 0;
                        }
                        switch (state) {                                                                // squelch_base_ff
                        case SQ_MUTED: if (!mute) state = ct.ramp ? SQ_ATTACK : SQ_UNMUTED; break;
                        case SQ_UNMUTED: if (mute) state = ct.ramp ? SQ_DECAY : SQ_MUTED; break;
                        case SQ_ATTACK: env = c_env_tab[++ramped]; if (ramped >= ct.ramp) { state = SQ_UNMUTED; env = 1.0; } break;
                        case SQ_DECAY: env = c_env_tab[--ramped]; if (ramped == 0) state = SQ_MUTED; break;
                        }
                        if (state != SQ_MUTED) { qr[nq & q_mask] = static_cast<float>(static_cast<double>(xv) * env); nq++; }
                        else if (!ct.gate) { qr[nq & q_mask] = 0.0f; nq++; }
                    }
                    st.gl1 = gl1; st.gl2 = gl2; st.gc1 = gc1; st.gc2 = gc2; st.gr1 = gr1; st.gr2 = gr2;
                    st.g_processed = proc; st.c_mute = mute; st.c_state = state; st.c_ramped = ramped; st.c_env = env; st.n_q = nq;
                }
                __syncthreads();
            }
        }
        __syncthreads();
    }
    // ---- 4. audio low-pass (direct form), into shared staging for the IIR
    const float* fsrc = qr ? qr : rr;                               // the filter's input stream and its length so far
    const unsigned fmask = qr ? q_mask : res_mask;
    const long long fend = qr ? st.n_q : res1;
    const long long aud0 = st.n_aud;
    const int n_aud = static_cast<int>(fend - aud0);                // one output per input item
    for (int base = 0; base < n_aud; base += 2048) {
        const int nb = (n_aud - base) < 2048 ? (n_aud - base) : 2048;
        for (int j = threadIdx.x; j < nb; j += blockDim.x) {
            const long long a = aud0 + base + j;
            float acc = 0.0f;
            for (int k = p.nt_audio - 1; k >= 0; k--) {
                const long long n = a - k;
                const float v = n >= 0 ? fsrc[n & fmask] : 0.0f;
                acc = fmaf(audio_taps[k], v, acc);
            }
            aud[j] = acc;
            if (aud_ring && p.mode == 0) aud_ring[static_cast<long long>(c) * aud_stride + (a & aud_mask)] = acc;
        }
        __syncthreads();
        // ---- 5. de-emphasis IIR (double) + output gain (sequential)
        if (aud_ring && p.mode == 0) {
            // split form: nbfm_deemph_kernel does it
        } else if (p.mode == 1) {
            const int cnt0 = port1_cnt[c];
            float* o = port1 + static_cast<long long>(c) * port1_stride;
            for (int j = threadIdx.x; j < nb; j += blockDim.x) if (cnt0 + j < port1_cap) o[cnt0 + j] = aud[j];
            __syncthreads();
            if (threadIdx.x == 0) port1_cnt[c] = cnt0 + nb;
        } else {
            // b0 x[n] + b1 x[n-1] does not depend on the recurrence: all threads (t1s is free by now); thread 0 keeps y[n] = u[n] - a1 y[n-1]
            double* u = t1s;
            const double x1c = st.iir_x1;
            for (int j = threadIdx.x; j < nb; j += blockDim.x) {
                const double xin = static_cast<double>(aud[j]);
                const double x1 = j > 0 ? static_cast<double>(aud[j - 1]) : x1c;
                double acc = p.b0 * xin;
                acc = acc + p.b1 * x1;
                u[j] = acc;
            }
            __syncthreads();
            const int cnt0 = port1_cnt[c];
            if (threadIdx.x == 0) {
                double y1 = st.iir_y1;
                for (int j = 0; j < nb; j++) { const double acc = u[j] - p.a1 * y1; y1 = acc; u[j] = acc; }
                st.iir_y1 = y1; st.iir_x1 = static_cast<double>(aud[nb - 1]);
            }
            __syncthreads();
            float* o = port1 + static_cast<long long>(c) * port1_stride;
            for (int j = threadIdx.x; j < nb; j += blockDim.x) if (cnt0 + j < port1_cap) o[cnt0 + j] = static_cast<float>(u[j]) * p.out_gain;
            __syncthreads();
            if (threadIdx.x == 0) port1_cnt[c] = cnt0 + nb;
        }
        __syncthreads();
    }
    __syncthreads();      // (nothing new: no barrier above) every thread has read st.n_aud
    if (threadIdx.x == 0) { st.n_res = res1; st.n_aud = fend; states[c] = st; if (aud_snap) aud_snap[c] = fend; }
}

// The de-emphasis recurrence of the NBFM chain (iir_filter_ffd, double: two dependent FP64 operations per audio item) in a kernel of
// its own: launched on a second stream behind the slice's nbfm_audio_kernel, it runs while the NEXT slice's squelch recurrence does.
// One CTA per channel; the audio items are staged through shared memory so the recurrence never waits on a global load.
struct NbfmDeemphState { double iir_x1, iir_y1; long long n_done; };
__global__ void __launch_bounds__(128)
nbfm_deemph_kernel(double b0, double b1, double a1, float out_gain, NbfmDeemphState* __restrict__ states,
                   const float* __restrict__ aud_ring, unsigned aud_mask, long long aud_stride, const long long* __restrict__ aud_snap,
                   float* __restrict__ port1, long long port1_stride, int* __restrict__ port1_cnt, int port1_cap)
{
    const int c = blockIdx.x;
    __shared__ float aud[2048];
    __shared__ double u[2048];            // b0 x[n] + b1 x[n-1] from all threads (does not depend on the recurrence), then y[n] in place
    __shared__ NbfmDeemphState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    const long long a0 = st.n_done, a1n = aud_snap[c];
    const float* ar = aud_ring + static_cast<long long>(c) * aud_stride;
    float* o = port1 + static_cast<long long>(c) * port1_stride;
    for (long long base = a0; base < a1n; base += 2048) {
        const int nb = (a1n - base) < 2048 ? static_cast<int>(a1n - base) : 2048;
        for (int j = threadIdx.x; j < nb; j += blockDim.x) aud[j] = ar[(base + j) & aud_mask];
        __syncthreads();
        const double x1c = st.iir_x1;
        for (int j = threadIdx.x; j < nb; j += blockDim.x) {
            const double xin = static_cast<double>(aud[j]);
            const double x1 = j > 0 ? static_cast<double>(aud[j - 1]) : x1c;
            double acc = b0 * xin;
            acc = acc + b1 * x1;
            u[j] = acc;
        }
        __syncthreads();
        const int cnt0 = port1_cnt[c];
        if (threadIdx.x == 0) {
            double y1 = st.iir_y1;
            for (int j = 0; j < nb; j++) { const double acc = u[j] - a1 * y1; y1 = acc; u[j] = acc; }      // the two operations on the chain
            st.iir_y1 = y1; st.iir_x1 = static_cast<double>(aud[nb - 1]);
        }
        __syncthreads();
        for (int j = threadIdx.x; j < nb; j += blockDim.x) if (cnt0 + j < port1_cap) o[cnt0 + j] = static_cast<float>(u[j]) * out_gain;
        __syncthreads();
        if (threadIdx.x == 0) port1_cnt[c] = cnt0 + nb;
        __syncthreads();
    }
    if (threadIdx.x == 0) { st.n_done = a1n > a0 ? a1n : a0; states[c] = st; }
}

// complex stream, COMPLEX taps (fft_filter_ccc restated in direct form), optional input gain (multiply_const_cc in front)
__global__ void fir_ccc_ring_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                                    float2* __restrict__ out, unsigned out_mask, long long out_stride,
                                    const float* __restrict__ taps_c /* interleaved */, int ntaps, float in_gain,
                                    long long a0, long long a1, float2* __restrict__ lin, long long lin_stride, long long lin_base)
{
    extern __shared__ float hs_dyn[];
    for (int i = threadIdx.x; i < 2 * ntaps; i += blockDim.x) hs_dyn[i] = taps_c[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float re = 0.0f, im = 0.0f;
    for (int j = ntaps - 1; j >= 0; j--) {
        float2 v = x[(a - j) & in_mask];
        v.x = v.x * in_gain; v.y = v.y * in_gain;
        const float hr = hs_dyn[2 * j], hi = hs_dyn[2 * j + 1];
        re = fmaf(hr, v.x, re); re = fmaf(-hi, v.y, re);
        im = fmaf(hr, v.y, im); im = fmaf(hi, v.x, im);
    }
    const float2 y = make_float2(re, im);
    out[static_cast<long long>(c) * out_stride + (a & out_mask)] = y;
    if (lin) lin[static_cast<long long>(c) * lin_stride + (a - lin_base)] = y;
}

// ------------------------------------------------------------------------------------------------
// SSB audio chain after the side-band filter (gr_demod_ssb.cpp:62-84): pwr_squelch_cc(gate, no ramp) -> agc2_cc ->
// cessb::clipper_cc(0.95) -> cessb::stretcher_cc -> complex_to_real -> x1.333 -> audio band-pass (direct form).
// 8 ksps per channel: one CTA per channel; squelch + AGC recurrences on thread 0, the rest spread over the CTA.
// ------------------------------------------------------------------------------------------------
struct SsbState {
    double pwr;
    long long n_in, n_gate, n_str, n_aud;
    int sq_state; float gain;
};
struct SsbParams {
    double sq_alpha, sq_threshold;
    float attack, decay, ref, max_gain, clip, emax, out_gain;
    int nt_audio;
};

__global__ void __launch_bounds__(128)
ssb_audio_kernel(SsbParams p, SsbState* __restrict__ states,
                 const float2* __restrict__ in, unsigned in_mask, long long in_stride, long long avail_in,
                 float2* __restrict__ clip_ring, unsigned clip_mask, long long clip_stride,
                 float* __restrict__ str_ring, unsigned str_mask, long long str_stride,
                 const float* __restrict__ audio_taps,
                 float* __restrict__ port1, long long port1_stride, int* __restrict__ port1_cnt, int port1_cap)
{
    const int c = blockIdx.x;
    __shared__ SsbState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float2* cr = clip_ring + static_cast<long long>(c) * clip_stride;
    float* sr = str_ring + static_cast<long long>(c) * str_stride;
    const long long gate0 = st.n_gate;
    __syncthreads();      // every thread holds its copy of gate0 before thread 0 advances st.n_gate at the end of step 1
    // ---- 1. squelch + AGC (sequential); the AGC output is parked in the clip ring, clipped in place in step 2
    if (threadIdx.x == 0) {
        double pwr = st.pwr; int state = st.sq_state; float gain = st.gain; long long ng = st.n_gate;
        for (long long a = st.n_in; a < avail_in; a++) {
            const float2 v = x[a & in_mask];
            const float mag2 = v.x * v.x + v.y * v.y;
            pwr = p.sq_alpha * static_cast<double>(mag2) + (1.0 - p.sq_alpha) * pwr;
            const bool mute = pwr < p.sq_threshold;
            if (state == SQ_MUTED) { if (!mute) state = SQ_UNMUTED; }
            else if (mute) state = SQ_MUTED;
            if (state != SQ_MUTED) {
                const float orr = v.x * gain, oi = v.y * gain;          // envelope is 1.0 without a ramp
                const float tmp = -p.ref + sqrtf(orr * orr + oi * oi);
                const float rate = (tmp > gain) ? p.attack : p.decay;      // agc2_cc: signed compare
                gain = gain - tmp * rate;
                if (gain < 0.0f) gain = 10e-5f;
                if (p.max_gain > 0.0f && gain > p.max_gain) gain = p.max_gain;
                cr[ng & clip_mask] = make_float2(orr, oi);
                ng++;
            }
        }
        st.pwr = pwr; st.sq_state = state; st.gain = gain; st.n_in = avail_in; st.n_gate = ng;
    }
    __syncthreads();
    const long long gate1 = st.n_gate;
    // ---- 2. clipper: magnitude limited to `clip`, phase kept (fast_atan2f + sincos)
    for (long long n = gate0 + threadIdx.x; n < gate1; n += blockDim.x) {
        const float2 v = cr[n & clip_mask];
        const float mag = sqrtf(v.x * v.x + v.y * v.y);
        const float ph = qrl_fast_atan2f(v.y, v.x);
        const float cl = mag < p.clip ? mag : p.clip;
        float sn, cs;
        qrl_sincosf(ph, sn, cs);
        cr[n & clip_mask] = make_float2(cs * cl, sn * cl);
    }
    __syncthreads();
    // ---- 3. stretcher: gain from the 5-point envelope maximum around n (needs n+2), real part x out_gain
    const long long str0 = st.n_str;
    const long long str1 = gate1 >= 2 ? gate1 - 2 : 0;
    for (long long n = str0 + threadIdx.x; n < str1; n += blockDim.x) {
        auto env = [&](long long k) -> float {
            if (k < 0) return 0.0f;
            const float2 v = cr[k & clip_mask];
            return sqrtf(v.x * v.x + v.y * v.y);
        };
        float h = env(n);
        h = fmaxf(h, env(n - 2)); h = fmaxf(h, env(n - 1)); h = fmaxf(h, env(n + 1)); h = fmaxf(h, env(n + 2));
        h = h * p.emax; h = fmaxf(h, 1.0f); h = h - 1.0f; h = h * 2.0f; h = h + 1.0f;
        const float re = cr[n & clip_mask].x / h;
        sr[n & str_mask] = re * p.out_gain;
    }
    __syncthreads();
    // ---- 4. audio band-pass (direct form), one output per stretcher output
    const long long aud0 = st.n_aud;
    int cnt0 = port1_cnt[c];
    float* o = port1 + static_cast<long long>(c) * port1_stride;
    const long long str1c = str1 > str0 ? str1 : str0;
    for (long long a = aud0 + threadIdx.x; a < str1c; a += blockDim.x) {
        float acc = 0.0f;
        for (int k = p.nt_audio - 1; k >= 0; k--) {
            const long long n = a - k;
            const float v = n >= 0 ? sr[n & str_mask] : 0.0f;
            acc = fmaf(audio_taps[k], v, acc);
        }
        const long long idx = cnt0 + (a - aud0);
        if (idx < port1_cap) o[idx] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        port1_cnt[c] = cnt0 + static_cast<int>(str1c - aud0);
        st.n_str = str1c; st.n_aud = str1c;
        states[c] = st;
    }
}

// ------------------------------------------------------------------------------------------------
// Non-FM FSK detectors: a bank of NB complex band-pass filters (fft_filter_ccc, direct form) on the channel-filter
// output, complex_to_mag, then
//   NB = 4: gr_4fsk_discriminator (strict-greater argmax -> +-0.707107 +-0.707107j, or 0)   gr_4fsk_discriminator.cpp:17-44
//   NB = 2: divide_ff(upper / lower) -> rail_ff(0, 2) -> add_const_ff(-1)                     gr_demod_2fsk.cpp:137-148
// one thread per sample, channel-major rings.
// ------------------------------------------------------------------------------------------------
template <int NB>
__global__ void fsk_bank_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                                const float* __restrict__ taps_c /* [NB][2*ntaps] */, int ntaps, long long a0, long long a1,
                                float* __restrict__ out /* float2 ring (NB=4) or float ring (NB=2) */, unsigned out_mask, long long out_stride)
{
    extern __shared__ float hs_dyn[];
    for (int i = threadIdx.x; i < NB * 2 * ntaps; i += blockDim.x) hs_dyn[i] = taps_c[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    const float2* x = in + static_cast<long long>(c) * in_stride;
    float m[NB];
#pragma unroll
    for (int b = 0; b < NB; b++) {
        const float* h = hs_dyn + b * 2 * ntaps;
        float re = 0.0f, im = 0.0f;
        for (int j = ntaps - 1; j >= 0; j--) {
            const float2 v = x[(a - j) & in_mask];
            re = fmaf(h[2 * j], v.x, re); re = fmaf(-h[2 * j + 1], v.y, re);
            im = fmaf(h[2 * j], v.y, im); im = fmaf(h[2 * j + 1], v.x, im);
        }
        m[b] = sqrtf(re * re + im * im);
    }
    if (NB == 4) {
        float orr = 0.0f, oi = 0.0f;
        const float P = static_cast<float>(0.707107), N = static_cast<float>(-0.707107);
        if ((m[0] > m[1]) && (m[0] > m[2]) && (m[0] > m[3])) { orr = N; oi = N; }
        else if ((m[1] > m[0]) && (m[1] > m[2]) && (m[1] > m[3])) { orr = N; oi = P; }
        else if ((m[2] > m[1]) && (m[2] > m[0]) && (m[2] > m[3])) { orr = P; oi = P; }
        else if ((m[3] > m[1]) && (m[3] > m[0]) && (m[3] > m[2])) { orr = P; oi = N; }
        reinterpret_cast<float2*>(out)[static_cast<long long>(c) * out_stride + (a & out_mask)] = make_float2(orr, oi);
    } else {
        const float q = m[0] / m[1];
        const float t = fmaxf(fminf(q, 2.0f), 0.0f);          // NaN (0/0 at start-up) -> the rail, like the oracle
        out[static_cast<long long>(c) * out_stride + (a & out_mask)] = t + -1.0f;
    }
}

// float stream, real taps (fft_filter_fff direct form): channel-major ring in, channel-interleaved ring out
__global__ void fir_fff_ring_kernel(const float* __restrict__ in, unsigned in_mask, long long in_stride,
                                    float* __restrict__ out, unsigned out_mask, long long out_stride,
                                    const float* __restrict__ taps, int ntaps, long long a0, long long a1)
{
    extern __shared__ float hs_dyn[];
    for (int i = threadIdx.x; i < ntaps; i += blockDim.x) hs_dyn[i] = taps[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    const float* x = in + static_cast<long long>(c) * in_stride;
    float acc = 0.0f;
    for (int j = ntaps - 1; j >= 0; j--) acc = fmaf(hs_dyn[j], x[(a - j) & in_mask], acc);
    out[(static_cast<long long>(c >> 5) * out_stride + (a & out_mask)) * 32 + (c & 31)] = acc;
}

// Front-end rotator (gr_demod_base's rotator_cc, carrier offset): out[c][n] = in[c][n] * exp(j theta), exact Q32 phase
// phase = base[c] + inc[c] * (n_abs - n_base[c]).  Only launched when some channel has a non-zero offset (the
// reference default is 0); it costs one extra pass over the slab -- fusing it needs complex stage-1 taps (next).
__global__ void rotator_kernel(const RotState* __restrict__ rs, const float2* __restrict__ in, long long in_stride,
                               float2* __restrict__ out, long long out_stride, long long T, long long n_abs0)
{
    const int c = blockIdx.y;
    const RotState r = rs[c];
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < T; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned ph = r.base + r.inc * static_cast<unsigned>(n_abs0 + i - r.n_base);
        const float ang = static_cast<float>(static_cast<double>(static_cast<int>(ph)) * (3.14159265358979323846 / 2147483648.0));
        float sn, cs;
        qrl_sincosf(ang, sn, cs);
        const float2 x = in[static_cast<long long>(c) * in_stride + i];
        out[static_cast<long long>(c) * out_stride + i] = make_float2(x.x * cs - x.y * sn, x.x * sn + x.y * cs);
    }
}

// Front end at device rates >= 2 Msps (gr_demod_base.cpp:1303-1362): rotator_cc at the device rate fused into the /D decimating FIR
// (83 taps at 2 Msps).  One CTA = 128 outputs of one channel: the window is rotated while it is loaded into shared memory (same Q32
// phase arithmetic as rotator_kernel), the previous calls' tail comes ALREADY ROTATED from `hist` (a retune must not touch samples that
// are already inside the filter, like the reference's resampler history); each thread then runs THE FIR order over its window.
__global__ void __launch_bounds__(128)
frontend_fir_kernel(const RotState* __restrict__ rs /* nullptr: no rotation */, const float2* __restrict__ in, long long in_stride, long long T,
                    long long n_abs0 /* absolute index of in[c][0] */, const float2* __restrict__ hist /* [C][H] rotated */, int H,
                    const float* __restrict__ taps, int ntaps, int D, float2* __restrict__ out, long long out_stride,
                    long long k0, long long k1 /* absolute output range of this call */)
{
    extern __shared__ __align__(16) float sm_fe[];
    float* hs = sm_fe;                                                  // ntaps (rounded up to even)
    float2* xs = reinterpret_cast<float2*>(sm_fe + ((ntaps + 1) & ~1));
    const int c = blockIdx.y;
    const long long kb = k0 + static_cast<long long>(blockIdx.x) * 128;
    if (kb >= k1) return;
    const int nout = (k1 - kb) < 128 ? static_cast<int>(k1 - kb) : 128;
    const long long a_first = D * kb - (ntaps - 1);                    // absolute index of the oldest sample of the window
    const int W = (nout - 1) * D + ntaps;
    for (int i = threadIdx.x; i < ntaps; i += 128) hs[i] = taps[i];
    const float2* x = in + static_cast<long long>(c) * in_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    RotState r{ 0u, 0u, 0 };
    if (rs) r = rs[c];
    for (int i = threadIdx.x; i < W; i += 128) {
        const long long a = a_first + i, li = a - n_abs0;               // li: index into this call's input
        float2 v = make_float2(0.0f, 0.0f);
        if (li >= 0) {
            if (li < T) {
                v = x[li];
                if (rs) {
                    const unsigned ph = r.base + r.inc * static_cast<unsigned>(a - r.n_base);
                    const float ang = static_cast<float>(static_cast<double>(static_cast<int>(ph)) * (3.14159265358979323846 / 2147483648.0));
                    float sn, cs;
                    qrl_sincosf(ang, sn, cs);
                    v = make_float2(v.x * cs - v.y * sn, v.x * sn + v.y * cs);
                }
            }
        } else if (H + li >= 0) v = hc[H + li];
        xs[i] = v;
    }
    __syncthreads();
    if (threadIdx.x >= nout) return;
    const float2* newest = xs + threadIdx.x * D + (ntaps - 1);
    const float2 y = qrl_fir_dot_order_c(hs, ntaps, D, [&](int j) { return newest[-j]; });
    out[static_cast<long long>(c) * out_stride + (kb + threadIdx.x - k0)] = y;
}
// rotated tail for the next call: new_hist = last H samples of (old_hist ++ rotate(in[0..T)))
__global__ void frontend_hist_kernel(const RotState* __restrict__ rs, const float2* __restrict__ in, long long in_stride, long long T, long long n_abs0,
                                     const float2* __restrict__ old_hist, float2* __restrict__ new_hist, int H)
{
    const int c = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= H) return;
    const long long li = T - H + i;
    float2 v;
    if (li >= 0) {
        v = in[static_cast<long long>(c) * in_stride + li];
        if (rs) {
            const RotState r = rs[c];
            const unsigned ph = r.base + r.inc * static_cast<unsigned>(n_abs0 + li - r.n_base);
            const float ang = static_cast<float>(static_cast<double>(static_cast<int>(ph)) * (3.14159265358979323846 / 2147483648.0));
            float sn, cs;
            qrl_sincosf(ang, sn, cs);
            v = make_float2(v.x * cs - v.y * sn, v.x * sn + v.y * cs);
        }
    } else v = old_hist[static_cast<long long>(c) * H + (H + li)];
    new_hist[static_cast<long long>(c) * H + i] = v;
}

// ------------------------------------------------------------------------------------------------
// TX front end (gr_mod_base.cpp:38,211-290): rotator_cc at 1 Msps, then rational_resampler_ccf(N, 1) up to the device rate
//   y[N m + p] = sum_k arm[p][k] x[m - k],  arm[p][k] = h[p + k N],  one fmaf chain per output, oldest sample first.
// grid = (tiles, channels); one CTA = P passes of G*R consecutive inputs of one channel, all N phases; thread (p = tid % N,
// q = tid / N) owns phase p and R consecutive inputs per pass.  The taps sit in shared memory in chain order, row i = the taps of
// step i ([NTP][N]: lanes on consecutive phases read consecutive words), the window holds the rotated samples (rotator fused into
// the load, the previous calls' tail comes ALREADY ROTATED from `hist`, so a retune never reaches samples already in the filter).
// Per step: one LDS (tap), one LDS.64 (the sample that slides into the R-slot register window), R FFMA2.  The arm is padded at
// its oldest end to NTP = a multiple of R with zero taps: the chain starts at +0 and stays there through them, as the oracle's
// own zero padding does, so the sums are the oracle's bit for bit.
// Bound: 2 NTP lane-FMAs per output (NTP ~ 216 at every rate), FP32-pipe bound -- 148 SMs x 128 lanes / 432 per output; the
// stores (8 B, or 4 B with SC16, per output) are an order of magnitude below the HBM write rate.
// SC16: per component (short) clamp(rintf(v * scale), -32768, 32767), interleaved I/Q (a definition chosen here: the SIMD
// fc32 -> sc16 converter's arithmetic, one multiply and round-half-even).
__device__ __forceinline__ float2 txfront_rotate(const RotState& r, long long a, float2 v)
{
    const unsigned ph = r.base + r.inc * static_cast<unsigned>(a - r.n_base);
    const float ang = static_cast<float>(static_cast<double>(static_cast<int>(ph)) * (3.14159265358979323846 / 2147483648.0));
    float sn, cs;
    qrl_sincosf(ang, sn, cs);
    return make_float2(v.x * cs - v.y * sn, v.x * sn + v.y * cs);
}
__device__ __forceinline__ short txfront_sc16(float v, float scale)
{
    const float t = rintf(v * scale);
    return static_cast<short>(t < -32768.0f ? -32768.0f : (t > 32767.0f ? 32767.0f : t));
}
template <bool SC16>
__device__ __forceinline__ void txfront_store(void* out, long long i, float2 v, float scale)
{
    if (SC16) {
        short2 s; s.x = txfront_sc16(v.x, scale); s.y = txfront_sc16(v.y, scale);
        static_cast<short2*>(out)[i] = s;
    } else static_cast<float2*>(out)[i] = v;
}

template <int R, bool SC16>
__global__ void __launch_bounds__(256)
txfront_interp_kernel(const RotState* __restrict__ rs /* nullptr: no rotation */, const float2* __restrict__ in, long long in_stride, long long T,
                      long long n_abs0 /* absolute index of in[c][0] */, const float2* __restrict__ hist /* [C][H] rotated, H = NTP - 1 */,
                      const float* __restrict__ taps /* [NTP][N] chain order */, int N, int NTP, int G, int P,
                      void* __restrict__ out, long long out_stride /* items */, float scale)
{
    extern __shared__ __align__(16) float sm_txf[];
    const int TM = G * R * P, H = NTP - 1;
    float* hs = sm_txf;                                                 // NTP * N (rounded up to even)
    float2* xs = reinterpret_cast<float2*>(sm_txf + ((NTP * N + 1) & ~1)); // TM + NTP - 1 rotated samples
    const int c = blockIdx.y;
    const long long t0 = static_cast<long long>(blockIdx.x) * TM;      // first input of the tile, relative to this call
    const int nin = (T - t0) < TM ? static_cast<int>(T - t0) : TM;
    const int nthr = N * G;
    for (int i = threadIdx.x; i < NTP * N; i += nthr) hs[i] = taps[i];
    const float2* x = in + static_cast<long long>(c) * in_stride;
    const float2* hc = hist + static_cast<long long>(c) * H;
    RotState r{ 0u, 0u, 0 };
    if (rs) r = rs[c];
    for (int i = threadIdx.x; i < TM + NTP - 1; i += nthr) {
        const long long li = t0 - H + i;                               // index into this call's input
        float2 v = make_float2(0.0f, 0.0f);
        if (li >= 0) {
            if (li < T) {
                v = x[li];
                if (rs) v = txfront_rotate(r, n_abs0 + li, v);
            }
        } else v = hc[H + li];
        xs[i] = v;
    }
    __syncthreads();
    const int p = threadIdx.x % N, q = threadIdx.x / N;
    for (int ps = 0; ps < P; ps++) {
        const int mi = (ps * G + q) * R;                                // tile-relative first input of this thread's R outputs
        if (mi >= nin) break;
        const float2* s = xs + mi;                                      // s[t] = x[t0 + mi - H + t]
        float2 acc[R], w[R];
#pragma unroll
        for (int u = 0; u < R; u++) acc[u] = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int u = 0; u < R - 1; u++) w[u] = s[u];
        for (int i0 = 0; i0 < NTP; i0 += R) {
#pragma unroll
            for (int u = 0; u < R; u++) {
                // step i = i0 + u: output j takes x[m_j - (NTP - 1 - i)] = s[i + j], which sits in slot (u + j) % R
                w[(u + R - 1) % R] = s[i0 + u + R - 1];
                const float h = hs[(i0 + u) * N + p];
#pragma unroll
                for (int j = 0; j < R; j++) ffma2(acc[j], h, w[(u + j) % R]);
            }
        }
        const long long ob = static_cast<long long>(c) * out_stride + (t0 + mi) * N + p;
#pragma unroll
        for (int j = 0; j < R; j++)
            if (mi + j < nin) txfront_store<SC16>(out, ob + static_cast<long long>(j) * N, acc[j], scale);
    }
}

// N = 1 (device rate 1 Msps: the reference's rotator feeds the sink directly): rotation and the output format only
template <bool SC16>
__global__ void __launch_bounds__(256)
txfront_rot_kernel(const RotState* __restrict__ rs, const float2* __restrict__ in, long long in_stride, long long T, long long n_abs0,
                   void* __restrict__ out, long long out_stride, float scale)
{
    const int c = blockIdx.y;
    RotState r{ 0u, 0u, 0 };
    if (rs) r = rs[c];
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < T; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float2 v = in[static_cast<long long>(c) * in_stride + i];
        if (rs) v = txfront_rotate(r, n_abs0 + i, v);
        txfront_store<SC16>(out, static_cast<long long>(c) * out_stride + i, v, scale);
    }
}

// roll the stage-1 history: new_hist = last H samples of (old_hist ++ iq[0..T))
__global__ void hist_update_kernel(const float2* __restrict__ iq, long long iq_stride, long long T,
                                   const float2* __restrict__ old_hist, float2* __restrict__ new_hist, int H)
{
    const int c = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= H) return;
    const long long src = T - H + i;     // index into iq; negative -> old history
    float2 v;
    if (src >= 0) v = iq[static_cast<long long>(c) * iq_stride + src];
    else v = old_hist[static_cast<long long>(c) * H + (H + src)];
    new_hist[static_cast<long long>(c) * H + i] = v;
}

// ================================================================================================
// TX chains (gr_mod_4fsk.cpp:95-115, gr_mod_qpsk.cpp:76-86)
// ================================================================================================
struct TxBitState {
    unsigned scr_reg;      // scrambler_bb(0x8A, 0x7F, 7) register
    unsigned enc_state;    // cc_encoder(80,7,2,{109,79}) CC_STREAMING shift register
    unsigned diff_prev;    // diff_encoder_bb(4)
    unsigned phase_q;      // Q32 phase accumulator of the frequency modulator
};

// bytes -> packed_to_unpacked(MSB) -> scrambler -> CC encoder -> pack_k_bits(2) -> map {0,1,3,2}
//       -> chunks_to_symbols (4FSK: float level, QPSK: diff_encoder(4) + complex point)
// one thread per channel (the scrambler is a feedback LFSR); 16 symbols per input byte... 8 per byte.
enum { TXM_4FSK = 0, TXM_QPSK = 1, TXM_BPSK = 2, TXM_2FSK = 3, TXM_M17 = 4, TXM_DSSS = 5 };
// TXM_DSSS (gr_mod_dsss.cpp:77-82, dsss_encoder_bb_impl.cc:86-97): per coded bit 13 chips, Barker-13 for a 0 and its complement for a 1, chips -> {-1, +1}
// TXM_M17 (gr_mod_m17.cpp:52-58,79-82): no scrambler / encoder in the block: bytes -> packed_to_unpacked(MSB) -> pack_k_bits(2) ->
// map {2,3,1,0} -> chunks_to_symbols {-1.5 .. 1.5}: 4 symbols per input byte
template <int MODE>
__global__ void tx_bits_kernel(TxBitState* __restrict__ states, int C, const unsigned char* __restrict__ bytes, long long n, long long stride,
                               float* __restrict__ sym_ring /* float or float2 */, unsigned sym_mask, long long sym_stride, long long sym0)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    TxBitState st = states[c];
    const unsigned char* b = bytes + static_cast<long long>(c) * stride;
    long long si = sym0;
    for (long long i = 0; i < n; i++) {
        const unsigned byte = b[i];
        if (MODE == TXM_M17) {
#pragma unroll
            for (int k = 3; k >= 0; k--) {
                const unsigned dibit = (byte >> (2 * k)) & 3u;
                const unsigned chunk = (0x1Eu >> (2 * dibit)) & 3u;           // map {2,3,1,0}, two bits per entry
                sym_ring[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = -1.5f + static_cast<float>(chunk);
                si++;
            }
            continue;
        }
        unsigned coded = 0;                       // 16 coded bits, first emitted = MSB
#pragma unroll
        for (int k = 7; k >= 0; k--) {
            const unsigned in = (byte >> k) & 1u;
            const unsigned out = st.scr_reg & 1u;
            const unsigned nb = (__popc(st.scr_reg & 0x8Au) & 1u) ^ in;
            st.scr_reg = ((st.scr_reg >> 1) | (nb << 7)) & 0xffu;
            st.enc_state = ((st.enc_state << 1) | out) & 0x7fu;
            coded = (coded << 2) | ((__popc(st.enc_state & 109u) & 1u) << 1) | (__popc(st.enc_state & 79u) & 1u);
        }
        if (MODE == TXM_DSSS) {
            for (int k = 15; k >= 0; k--) {
                const unsigned bit = (coded >> k) & 1u;
#pragma unroll
                for (int q = 0; q < 13; q++) {
                    const unsigned chip = ((0x1F35u >> (12 - q)) & 1u) ^ bit;      // {1,1,1,1,1,0,0,1,1,0,1,0,1}, first chip = MSB
                    reinterpret_cast<float2*>(sym_ring)[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = make_float2(chip ? 1.0f : -1.0f, 0.0f);
                    si++;
                }
            }
            continue;
        }
        if (MODE == TXM_BPSK || MODE == TXM_2FSK) {
            // one symbol per coded bit: chunks_to_symbols {-1, +1} (complex for BPSK, float for 2FSK)
#pragma unroll
            for (int k = 15; k >= 0; k--) {
                const float lv = ((coded >> k) & 1u) ? 1.0f : -1.0f;
                if (MODE == TXM_BPSK) reinterpret_cast<float2*>(sym_ring)[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = make_float2(lv, 0.0f);
                else sym_ring[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = lv;
                si++;
            }
            continue;
        }
#pragma unroll
        for (int k = 7; k >= 0; k--) {
            const unsigned dibit = (coded >> (2 * k)) & 3u;
            const unsigned chunk = dibit ^ (dibit >> 1);                  // map {0,1,3,2}
            if (MODE == TXM_QPSK) {
                st.diff_prev = (chunk + st.diff_prev) & 3u;
                const float qr = (st.diff_prev >= 2u) ? 0.707f : -0.707f;
                const float qi = (st.diff_prev == 1u || st.diff_prev == 2u) ? 0.707f : -0.707f;
                reinterpret_cast<float2*>(sym_ring)[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = make_float2(qr, qi);
            } else {
                sym_ring[static_cast<long long>(c) * sym_stride + (si & sym_mask)] = -1.5f + static_cast<float>(chunk);
            }
            si++;
        }
    }
    // field by field: phase_q belongs to tx_shape_fm_kernel, which may be running on another stream
    states[c].scr_reg = st.scr_reg; states[c].enc_state = st.enc_state; states[c].diff_prev = st.diff_prev;
}

// 4FSK-FM: rational_resampler_fff(L,1,RRC) -> x0.66666666 -> frequency_modulator_fc -> x amplif -> x bb_gain.
// The phase accumulator is a Q32 integer (increment quantised once per sample, summed exactly mod 2^32), so the
// per-channel phase is a prefix sum: one CTA per channel scans its samples block by block.
template <int NTHREADS, int ITEMS>
__global__ void __launch_bounds__(NTHREADS)
tx_shape_fm_kernel(TxBitState* __restrict__ states, const float* __restrict__ sym_ring, unsigned sym_mask, long long sym_stride,
                   long long sym0, long long nsym, int L, int nt_arm, const float* __restrict__ arms /* [L][nt_arm] */, int repeat_only,
                   float pulse_scale, float fm_sens, float amplif, float bb_gain,
                   float2* __restrict__ if_ring, unsigned if_mask, long long if_stride)
{
    const int c = blockIdx.x;
    const float* sy = sym_ring + static_cast<long long>(c) * sym_stride;
    float2* o = if_ring + static_cast<long long>(c) * if_stride;
    __shared__ unsigned warp_sums[NTHREADS / 32];
    __shared__ unsigned carry;
    if (threadIdx.x == 0) carry = states[c].phase_q;
    __syncthreads();
    const long long n0 = sym0 * L, n1 = (sym0 + nsym) * L;              // absolute IF sample range
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (long long blk = n0; blk < n1; blk += NTHREADS * ITEMS) {
        unsigned inc[ITEMS];
        unsigned local = 0;
#pragma unroll
        for (int it = 0; it < ITEMS; it++) {
            const long long a = blk + static_cast<long long>(threadIdx.x) * ITEMS + it;
            unsigned q = 0;
            if (a < n1) {
                const long long m = a / L; const int ph = static_cast<int>(a - m * L);
                float x;
                if (repeat_only) x = sy[m & sym_mask];
                else {
                    const float* h = arms + ph * nt_arm;
                    float acc = 0.0f;
                    for (int k = nt_arm - 1; k >= 0; k--) acc = fmaf(h[k], sy[(m - k) & sym_mask], acc);
                    x = acc * pulse_scale;
                }
                const float finc = fm_sens * x;
                const double dq = rint(static_cast<double>(finc) * (2147483648.0 / 3.14159265358979323846));
                q = static_cast<unsigned>(static_cast<int>(static_cast<long long>(dq)));
            }
            local += q;
            inc[it] = local;                                             // inclusive prefix inside the thread
        }
        // block-wide exclusive scan of the per-thread totals
        unsigned v = local;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, v, off); if (lane >= off) v += t; }
        if (lane == 31) warp_sums[warp] = v;
        __syncthreads();
        unsigned wbase = 0;
        for (int w = 0; w < warp; w++) wbase += warp_sums[w];
        const unsigned excl = carry + wbase + (v - local);
        unsigned total = 0;
        for (int w = 0; w < NTHREADS / 32; w++) total += warp_sums[w];
#pragma unroll
        for (int it = 0; it < ITEMS; it++) {
            const long long a = blk + static_cast<long long>(threadIdx.x) * ITEMS + it;
            if (a < n1) {
                const unsigned ux = excl + inc[it];
                const int si = ux >> 22;
                const float sn = d_sine_tab[2 * si] * static_cast<float>(ux >> 1) + d_sine_tab[2 * si + 1];
                const unsigned uc = ux + 0x40000000u;
                const int ci = uc >> 22;
                const float cs = d_sine_tab[2 * ci] * static_cast<float>(uc >> 1) + d_sine_tab[2 * ci + 1];
                float re = cs * amplif, im = sn * amplif;
                re = re * bb_gain; im = im * bb_gain;
                o[a & if_mask] = make_float2(re, im);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) states[c].phase_q = carry;
}

// Interpolating FIR  y[L m + p] = sum_k arm[p][k] x[m - k]  (rational_resampler_ccf(L,1)), complex stream.
// Thread = (m-block, phase p): its NT arm taps live in registers, its input window slides through registers
// (one shared-memory load per m), 2 NT FFMA per output sample; L*MB threads keep every lane busy.
template <int L, int NT, int MB, int MLEN>
__global__ void __launch_bounds__(L * MB)
interp_fir_ccf_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride, long long m0, long long m1,
                      const float* __restrict__ arms /* [L][NT] */, float post_gain1, float post_gain2, int apply_gain,
                      float2* __restrict__ out, long long out_stride, long long out_base /* absolute output index of out[c][0] */)
{
    static_assert(MLEN % NT == 0, "m-loop is unrolled in groups of NT");
    __shared__ float2 xs[MB * MLEN + NT];
    const int c = blockIdx.y;
    const long long tile0 = m0 + static_cast<long long>(blockIdx.x) * (MB * MLEN);
    if (tile0 >= m1) return;
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < MB * MLEN + NT - 1; i += L * MB) {
        const long long m = tile0 - (NT - 1) + i;
        xs[i] = (m < m1) ? x[m & in_mask] : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    const int p = threadIdx.x % L, mb = threadIdx.x / L;
    float h[NT];
#pragma unroll
    for (int k = 0; k < NT; k++) h[k] = arms[p * NT + k];
    float2 w[NT];
#pragma unroll
    for (int j = 0; j < NT - 1; j++) w[j] = xs[mb * MLEN + j];
    float2* oc = out + static_cast<long long>(c) * out_stride;
    for (int g = 0; g < MLEN / NT; g++) {
#pragma unroll
        for (int i = 0; i < NT; i++) {
            // window slot (NT-1+i) % NT receives the newest sample; sample m-k sits in slot (NT-1+i-k) % NT
            w[(NT - 1 + i) % NT] = xs[mb * MLEN + g * NT + i + (NT - 1)];
            float2 acc2 = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int k = NT - 1; k >= 0; k--) ffma2(acc2, h[k], w[(NT - 1 + i - k + NT) % NT]);
            float re = acc2.x, im = acc2.y;
            if (apply_gain) { re = re * post_gain1; im = im * post_gain1; re = re * post_gain2; im = im * post_gain2; }
            const long long m = tile0 + mb * MLEN + g * NT + i;
            if (m < m1) oc[(m * L + p) - out_base] = make_float2(re, im);
        }
    }
}

// Register-tiled variant: thread (phase p = tid % L, group q = tid / L) produces R consecutive outputs of its phase
// at once.  Each input sample is loaded once (a broadcast LDS: the lanes of a group read the same address) and feeds
// R accumulators, so consecutive FFMAs share an operand (register reuse) instead of streaming 2 new operands each:
// 2 NT FFMA per output as before, about twice the FP32 issue rate.  Same accumulation order (oldest sample first).
// (round 2 experiment, profiles/README.md: several tiles per CTA with a double-buffered window measured 8 % SLOWER on B200 -- 131.6 vs
// 121.9 us per launch, the window fill competes with the FFMA stream for the LSU -- and keeping the taps resident across tiles costs
// an occupancy step (64 registers); the one-tile form below stays)
template <int L, int NT, int R, int G>
__global__ void __launch_bounds__(L * G)
interp_fir_ccf_rt_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride, long long m0, long long m1,
                         const float* __restrict__ arms /* [L][NT] */, float post_gain1, float post_gain2, int apply_gain,
                         float2* __restrict__ out, long long out_stride, long long out_base)
{
    constexpr int TM = G * R;
    __shared__ float2 xs[TM + NT];
    const int c = blockIdx.y;
    const long long tile0 = m0 + static_cast<long long>(blockIdx.x) * TM;
    if (tile0 >= m1) return;
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < TM + NT - 1; i += L * G) {
        const long long m = tile0 - (NT - 1) + i;
        xs[i] = (m < m1) ? x[m & in_mask] : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    const int p = threadIdx.x % L, q = threadIdx.x / L;
    float h[NT];
#pragma unroll
    for (int k = 0; k < NT; k++) h[k] = arms[p * NT + k];
    float2 acc[R];                                              // (re, im) pairs: one FFMA2 per tap and output
#pragma unroll
    for (int r = 0; r < R; r++) acc[r] = make_float2(0.0f, 0.0f);
    const float2* s = xs + q * R;                               // s[j] = x[tile0 + qR - (NT-1) + j]
#pragma unroll
    for (int j = 0; j < R + NT - 1; j++) {
        const float2 v = s[j];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int k = r + NT - 1 - j;                       // output m = tile0 + qR + r uses x[m - k]
            if (k >= 0 && k < NT) ffma2(acc[r], h[k], v);
        }
    }
    float2* oc = out + static_cast<long long>(c) * out_stride;
#pragma unroll
    for (int r = 0; r < R; r++) {
        float re = acc[r].x, im = acc[r].y;
        if (apply_gain) { re = re * post_gain1; im = im * post_gain1; re = re * post_gain2; im = im * post_gain2; }
        const long long m = tile0 + q * R + r;
        if (m < m1) oc[(m * L + p) - out_base] = make_float2(re, im);
    }
}

// Shape-generic interpolating FIR (any L, NT): one thread per output sample, arm taps and the input window in shared
// memory.  Used for the TX shapes that have no register-tiled instance (QPSK x100/x500, BPSK x250/x500, 2FSK x10 ...).
__global__ void __launch_bounds__(256)
interp_fir_ccf_generic_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride, long long m0, long long m1,
                              const float* __restrict__ arms /* [L][NT] */, int L, int NT, int MT /* m per CTA */,
                              float post_gain1, float post_gain2, int apply_gain,
                              float2* __restrict__ out, long long out_stride, long long out_base)
{
    extern __shared__ float sm_gi[];
    float* hs = sm_gi;                                           // L*NT
    float2* xs = reinterpret_cast<float2*>(sm_gi + ((L * NT + 1) & ~1));   // MT + NT - 1
    const int c = blockIdx.y;
    const long long tile0 = m0 + static_cast<long long>(blockIdx.x) * MT;
    if (tile0 >= m1) return;
    for (int i = threadIdx.x; i < L * NT; i += 256) hs[i] = arms[i];
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < MT + NT - 1; i += 256) {
        const long long m = tile0 - (NT - 1) + i;
        xs[i] = (m < m1) ? x[m & in_mask] : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    float2* oc = out + static_cast<long long>(c) * out_stride;
    const long long nout = static_cast<long long>(MT) * L;
    for (long long o = threadIdx.x; o < nout; o += 256) {
        const int ml = static_cast<int>(o / L), p = static_cast<int>(o - static_cast<long long>(ml) * L);
        const long long m = tile0 + ml;
        if (m >= m1) break;
        const float* h = hs + p * NT;
        const float2* w = xs + ml + (NT - 1);                    // newest sample of this output
        float re = 0.0f, im = 0.0f;
        for (int k = NT - 1; k >= 0; k--) { const float2 v = w[-k]; re = fmaf(h[k], v.x, re); im = fmaf(h[k], v.y, im); }
        if (apply_gain) { re = re * post_gain1; im = im * post_gain1; re = re * post_gain2; im = im * post_gain2; }
        oc[(m * L + p) - out_base] = make_float2(re, im);
    }
}

// Shape-generic rational interpolator from a complex ring (rational_resampler_ccf(L, M) with L > M; gr_mod_m17.cpp:70-73: x125 / 3):
// output i takes arm (i M) mod L at ring position floor(i M / L), arms[p][k] = taps[p + k L], plain oldest-first accumulation (the
// oracle's order for L > 1).  One thread per output sample, the arm table in shared memory; consecutive outputs share their inputs.
__global__ void __launch_bounds__(256)
resamp_ring_ccf_generic_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride,
                               const float* __restrict__ arms /* [L][NT] */, int L, int M, int NT, long long o0, long long o1,
                               float2* __restrict__ out, long long out_stride)
{
    extern __shared__ float sm_rr[];
    for (int i = threadIdx.x; i < L * NT; i += 256) sm_rr[i] = arms[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long i = o0 + static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    if (i >= o1) return;
    const long long im = i * M;
    const long long newest = im / L;                                      // absolute index of the newest input sample
    const float* h = sm_rr + static_cast<int>(im - newest * L) * NT;
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    float re = 0.0f, imv = 0.0f;
    for (int k = NT - 1; k >= 0; k--) {
        const float2 v = x[(newest - k) & in_mask];                       // before the first sample: the zero-initialised top of the ring
        re = fmaf(h[k], v.x, re); imv = fmaf(h[k], v.y, imv);
    }
    out[static_cast<long long>(c) * out_stride + (i - o0)] = make_float2(re, imv);
}

// the same resampler writing a ring (a later stage needs the history across calls), with the two multiply_const_cc gains behind it
// when apply_gain is set (gr_mod_dsss.cpp:83-86: x25 pulse shaping -> x0.65 -> x bb_gain -> x50 / 13)
__global__ void __launch_bounds__(256)
resamp_ring_to_ring_ccf_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride,
                               const float* __restrict__ arms /* [L][NT] */, int L, int M, int NT, long long o0, long long o1,
                               float g1, float g2, int apply_gain, float2* __restrict__ out_ring, unsigned out_mask, long long out_stride)
{
    extern __shared__ float sm_r2r[];
    for (int i = threadIdx.x; i < L * NT; i += 256) sm_r2r[i] = arms[i];
    __syncthreads();
    const int c = blockIdx.y;
    const long long i = o0 + static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    if (i >= o1) return;
    const long long im = i * M;
    const long long newest = im / L;
    const float* h = sm_r2r + static_cast<int>(im - newest * L) * NT;
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    float re = 0.0f, imv = 0.0f;
    for (int k = NT - 1; k >= 0; k--) {
        const long long a = newest - k;
        const float2 v = a >= 0 ? x[a & in_mask] : make_float2(0.0f, 0.0f);
        re = fmaf(h[k], v.x, re); imv = fmaf(h[k], v.y, imv);
    }
    if (apply_gain) { re = re * g1; imv = imv * g1; re = re * g2; imv = imv * g2; }
    out_ring[static_cast<long long>(c) * out_stride + (i & out_mask)] = make_float2(re, imv);
}

// Tiled form of resamp_ring_to_ring_ccf_kernel for M >= L (a decimating rational resampler, gr_demod_mmdvm_multi2's 24 / 25): a CTA takes
// 256 consecutive outputs, stages the input span they touch (256 M / L + NT items) and the arm table in shared memory once, and every
// thread walks its NT taps over shared memory with the loop fully unrolled (independent loads in flight instead of one L1 round trip
// per tap).  Same taps, same order (oldest first) as the generic kernel: bit-identical.
template <int NT>
__global__ void __launch_bounds__(256)
resamp_ring_to_ring_tiled_kernel(const float2* __restrict__ in_ring, unsigned in_mask, long long in_stride,
                                 const float* __restrict__ arms /* [L][NT] */, int L, int M, long long o0, long long o1,
                                 float2* __restrict__ out_ring, unsigned out_mask, long long out_stride, int span_cap)
{
    extern __shared__ float sm_rt[];
    float* hs = sm_rt;                                               // L * NT
    float2* xs = reinterpret_cast<float2*>(sm_rt + ((L * NT + 1) & ~1));
    const int c = blockIdx.y;
    const long long ob = o0 + static_cast<long long>(blockIdx.x) * 256;
    if (ob >= o1) return;
    const long long oe = ob + 256 < o1 ? ob + 256 : o1;
    const long long first = (ob * M) / L - (NT - 1), last = ((oe - 1) * M) / L;      // input span of this CTA
    const int span = static_cast<int>(last - first + 1);
    for (int i = threadIdx.x; i < L * NT; i += 256) hs[i] = arms[i];
    const float2* x = in_ring + static_cast<long long>(c) * in_stride;
    for (int i = threadIdx.x; i < span && i < span_cap; i += 256) {
        const long long a = first + i;
        xs[i] = a >= 0 ? x[a & in_mask] : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    const long long o = ob + threadIdx.x;
    if (o >= oe) return;
    const long long im = o * M, newest = im / L;
    const float* h = hs + static_cast<int>(im - newest * L) * NT;
    const float2* w = xs + static_cast<int>(newest - first);          // newest item of this output
    float re = 0.0f, imv = 0.0f;
#pragma unroll
    for (int k = NT - 1; k >= 0; k--) { const float2 v = w[-k]; re = fmaf(h[k], v.x, re); imv = fmaf(h[k], v.y, imv); }
    out_ring[static_cast<long long>(c) * out_stride + (o & out_mask)] = make_float2(re, imv);
}

// ================================================================================================
// Analog modulators (gr_mod_nbfm.cpp:26-75, gr_mod_ssb.cpp:28-82): 8 ksps float audio in.  One CTA per channel runs
// the low-rate front part; the FM scan / IF filters / final interpolator reuse the digital TX kernels.
// ================================================================================================
struct TxAnalogState { long long n_in, n_rs, n_str; double iir_x1, iir_y1; float agc; int pad_; };     // agc: gr_mod_am's agc2_ff gain

// NBFM: audio LPF -> x0.99 -> pre-emphasis IIR (double) -> rational_resampler_fff(25,4) -> float ring (FM input)
__global__ void __launch_bounds__(128)
tx_nbfm_front_kernel(TxAnalogState* __restrict__ states, const float* __restrict__ audio, long long n, long long a_stride,
                     float* __restrict__ ra, unsigned ra_mask, long long ra_stride,      // audio ring
                     float* __restrict__ rb, unsigned rb_mask, long long rb_stride,      // filtered + pre-emphasised
                     const float* __restrict__ lpf, int nt_lpf, double b0, double b1, double a1,
                     const float* __restrict__ arms /* [25][nt_arm] */, int nt_arm,
                     float* __restrict__ rs_out, unsigned rs_mask, long long rs_stride,
                     float audio_gain, int tone_on, unsigned tone_phase0, unsigned tone_inc)      // gr_mod_nbfm::set_ctcss: gain + CTCSS tone
{
    const int c = blockIdx.x;
    __shared__ TxAnalogState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    float* A = ra + static_cast<long long>(c) * ra_stride;
    float* B = rb + static_cast<long long>(c) * rb_stride;
    float* R = rs_out + static_cast<long long>(c) * rs_stride;
    const long long a0 = st.n_in, a1n = st.n_in + n;
    for (long long a = a0 + threadIdx.x; a < a1n; a += blockDim.x) A[a & ra_mask] = audio[static_cast<long long>(c) * a_stride + (a - a0)];
    __syncthreads();
    for (long long a = a0 + threadIdx.x; a < a1n; a += blockDim.x) {
        float acc = 0.0f;
        for (int k = nt_lpf - 1; k >= 0; k--) { const long long m = a - k; acc = fmaf(lpf[k], m >= 0 ? A[m & ra_mask] : 0.0f, acc); }
        float v = acc * audio_gain;                                   // multiply_const_ff(0.99 / 0.98 / 0.85)
        if (tone_on) {
            // add_ff with sig_source_f(8000, cos, f, 0.15) = fxpt_nco: (float)(fxpt::cos(phase) * 0.15); phase of this call's sample j
            // is tone_phase0 + j * inc (mod 2^32)
            const unsigned uc = tone_phase0 + tone_inc * static_cast<unsigned>(a - a0) + 0x40000000u;
            const int ci = static_cast<int>(uc >> 22);
            const float cs = d_sine_tab[2 * ci] * static_cast<float>(uc >> 1) + d_sine_tab[2 * ci + 1];
            v = v + static_cast<float>(static_cast<double>(cs) * 0.15);
        }
        B[a & rb_mask] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double x1 = st.iir_x1, y1 = st.iir_y1;
        for (long long a = a0; a < a1n; a++) {
            const double xin = static_cast<double>(B[a & rb_mask]);
            double acc = b0 * xin;
            acc = acc + b1 * x1;
            acc = acc - a1 * y1;
            x1 = xin; y1 = acc;
            B[a & rb_mask] = static_cast<float>(acc);
        }
        st.iir_x1 = x1; st.iir_y1 = y1;
    }
    __syncthreads();
    // resampler 25/4: output i uses arm (4 i) mod 25 at input position floor(4 i / 25); available while pos <= a1n - 1
    const long long r0 = st.n_rs, r1 = (a1n * 25 + 3) / 4;
    for (long long i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
        const long long pos = (4 * i) / 25;
        const float* h = arms + static_cast<int>((4 * i) % 25) * nt_arm;
        float acc = 0.0f;
        for (int k = nt_arm - 1; k >= 0; k--) { const long long m = pos - k; acc = fmaf(h[k], m >= 0 ? B[m & rb_mask] : 0.0f, acc); }
        R[i & rs_mask] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) { st.n_in = a1n; st.n_rs = r1; states[c] = st; }
}

// SSB: audio band-pass -> float_to_complex -> cessb::clipper_cc(0.95) -> cessb::stretcher_cc -> complex ring
__global__ void __launch_bounds__(128)
tx_ssb_front_kernel(TxAnalogState* __restrict__ states, const float* __restrict__ audio, long long n, long long a_stride,
                    float* __restrict__ ra, unsigned ra_mask, long long ra_stride,
                    float2* __restrict__ rclip, unsigned rc_mask, long long rc_stride,
                    const float* __restrict__ bpf, int nt_bpf, float clip, float emax,
                    float2* __restrict__ rstr, unsigned rs_mask, long long rs_stride)
{
    const int c = blockIdx.x;
    __shared__ TxAnalogState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    float* A = ra + static_cast<long long>(c) * ra_stride;
    float2* Cc = rclip + static_cast<long long>(c) * rc_stride;
    float2* S = rstr + static_cast<long long>(c) * rs_stride;
    const long long a0 = st.n_in, a1n = st.n_in + n;
    for (long long a = a0 + threadIdx.x; a < a1n; a += blockDim.x) A[a & ra_mask] = audio[static_cast<long long>(c) * a_stride + (a - a0)];
    __syncthreads();
    for (long long a = a0 + threadIdx.x; a < a1n; a += blockDim.x) {
        float acc = 0.0f;
        for (int k = nt_bpf - 1; k >= 0; k--) { const long long m = a - k; acc = fmaf(bpf[k], m >= 0 ? A[m & ra_mask] : 0.0f, acc); }
        const float mag = sqrtf(acc * acc + 0.0f * 0.0f);
        const float ph = qrl_fast_atan2f(0.0f, acc);
        const float cl = mag < clip ? mag : clip;
        float sn, cs;
        qrl_sincosf(ph, sn, cs);
        Cc[a & rc_mask] = make_float2(cs * cl, sn * cl);
    }
    __syncthreads();
    const long long s0 = st.n_str, s1 = a1n >= 2 ? a1n - 2 : 0;
    for (long long k = s0 + threadIdx.x; k < s1; k += blockDim.x) {
        auto env = [&](long long j) -> float { if (j < 0) return 0.0f; const float2 v = Cc[j & rc_mask]; return sqrtf(v.x * v.x + v.y * v.y); };
        float h = env(k);
        h = fmaxf(h, env(k - 2)); h = fmaxf(h, env(k - 1)); h = fmaxf(h, env(k + 1)); h = fmaxf(h, env(k + 2));
        h = h * emax; h = fmaxf(h, 1.0f); h = h - 1.0f; h = h * 2.0f; h = h + 1.0f;
        const float2 v = Cc[k & rc_mask];
        S[k & rs_mask] = make_float2(v.x / h, v.y / h);
    }
    __syncthreads();
    if (threadIdx.x == 0) { st.n_in = a1n; st.n_str = s1 > s0 ? s1 : s0; states[c] = st; }
}

// AM (gr_mod_am.cpp:41-62): agc2_ff(1e-2, 1e-4, 1, 1; max gain 1) -> rail_ff(+-0.98) -> x0.95 (thread 0, per-sample recurrence) -> audio ring;
// band-pass FIR -> + carrier term -> float_to_complex -> complex ring at 8 ksps (all threads)
__global__ void __launch_bounds__(128)
tx_am_front_kernel(TxAnalogState* __restrict__ states, const float* __restrict__ audio, long long n, long long a_stride,
                   float attack, float decay, float ref, float max_gain,
                   float* __restrict__ ra, unsigned ra_mask, long long ra_stride, const float* __restrict__ bpf, int nt_bpf, float dc,
                   float2* __restrict__ rsym, unsigned rs_mask, long long rs_stride)
{
    const int c = blockIdx.x;
    __shared__ TxAnalogState st;
    if (threadIdx.x == 0) st = states[c];
    __syncthreads();
    float* A = ra + static_cast<long long>(c) * ra_stride;
    float2* S = rsym + static_cast<long long>(c) * rs_stride;
    const long long a0 = st.n_in, a1n = st.n_in + n;
    if (threadIdx.x == 0) {
        float gain = st.agc;
        const float* au = audio + static_cast<long long>(c) * a_stride;
        for (long long i = 0; i < n; i++) {
            const float out = au[i] * gain;                         // analog::kernel::agc2_ff::scale
            const float tmp = fabsf(out) - ref;
            const float rate = (fabsf(tmp) > gain) ? attack : decay;
            gain = gain - tmp * rate;
            if (gain < 0.0f) gain = 10e-5f;
            if (max_gain > 0.0f && gain > max_gain) gain = max_gain;
            float v = out < -0.98f ? -0.98f : (out > 0.98f ? 0.98f : out);
            v = v * 0.95f;
            A[(a0 + i) & ra_mask] = v;
        }
        st.agc = gain;
    }
    __syncthreads();
    for (long long a = a0 + threadIdx.x; a < a1n; a += blockDim.x) {
        float acc = 0.0f;
        for (int k = nt_bpf - 1; k >= 0; k--) { const long long m = a - k; acc = fmaf(bpf[k], m >= 0 ? A[m & ra_mask] : 0.0f, acc); }
        S[a & rs_mask] = make_float2(acc + dc, 0.0f);
    }
    __syncthreads();
    if (threadIdx.x == 0) { st.n_in = a1n; states[c] = st; }
}

// in-place x g1 x g2 on a channel-major complex ring segment (multiply_const_cc twice)
__global__ void scale2_ring_kernel(float2* __restrict__ ring, unsigned mask, long long stride, long long a0, long long a1, float g1, float g2)
{
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    float2 v = ring[static_cast<long long>(c) * stride + (a & mask)];
    v.x = v.x * g1; v.y = v.y * g1; v.x = v.x * g2; v.y = v.y * g2;
    ring[static_cast<long long>(c) * stride + (a & mask)] = v;
}

// ================================================================================================
// gr_demod_dsss behind stage 1 (gr_demod_dsss.cpp:89-112): a 16 symbol/s mode -- everything after the /50 FIR runs at 5200 items/s and
// below, so one CTA per channel walks the whole chain for a call, phase by phase (parallel phases on all threads, the three feedback
// loops on thread 0 over shared-memory chunks):
//   A  rational_resampler_ccf(13, 50)  r1 (20 ksps) -> ra          B  costas_loop_cc(pi/200, 2, snr) in place on ra
//   C  low_pass FIR ra -> rc + port 0                               D  agc2_cc(.1, .1, 1, 10) in place on rc
//   E  dsss_decoder_cc: per symbol m the N correlations of the N + 11 sps tap matched filter over rc[m N - 2 N + 1 + j ...], first
//      strict maximum of |y| (|y| = (float)sqrt((double)re re + (double)im im), glibc's hypotf) times 2 / N -> rd
//   F  clock_recovery_mm_cc(1, 2.5e-5, .5, .05, .005) on rd -> costas_loop_cc(2 pi/100, 2) -> port 1, soft bits (real x64 + 128) -> r5
// Arithmetic and orders as oracle/qrl_oracle.c (qo_rx_work, QO_DEMOD_DSSS).  Counters are absolute and live in the state.
// ================================================================================================
struct DsssState {
    long long o_n;            // 5200 sps items produced so far (phases A-D)
    long long m_n;            // despread symbols produced so far
    long long cr_ii;          // clock recovery: absolute index in rd of the next interpolation window
    long long n_sym, n_soft;
    LoopState pll, costas;
    float agc;
    float omega, mu, p0r, p0i, p1r, p1i, p2r, p2i, c0r, c0i, c1r, c1i, c2r, c2i;
};
struct DsssParams {
    int nt_arm;               // taps per arm of the 13 / 50 resampler
    int nt2;                  // low-pass in front of the AGC
    int N, ntaps;             // despreader: N = sps * 13 correlations per symbol, ntaps = N + 11 sps
    float pll_alpha, pll_beta, costas_alpha, costas_beta;
    float agc_attack, agc_decay, agc_ref, agc_max;
    float gain_omega, gain_mu, omega_mid, omega_lim, soft_scale;
};
constexpr int kDsssChunk = 1024;

__global__ void __launch_bounds__(256)
dsss_chain_kernel(DsssParams p, DsssState* __restrict__ states,
                  const float2* __restrict__ r1, unsigned r1_mask, long long r1_stride, long long k1,
                  const float* __restrict__ arms /* [13][nt_arm] */, const float* __restrict__ taps2, const float2* __restrict__ dtaps_rev,
                  float2* __restrict__ ra, float2* __restrict__ rc, unsigned ring_mask, long long ring_stride,
                  float2* __restrict__ rd, unsigned rd_mask, long long rd_stride,
                  float2* __restrict__ port0, long long port0_stride, long long o_call0,
                  float2* __restrict__ port1, long long port1_stride, int* __restrict__ port1_cnt, int port1_cap,
                  unsigned char* __restrict__ soft_ring, unsigned soft_mask, long long soft_stride, long long* __restrict__ n_soft_out)
{
    __shared__ DsssState st;
    __shared__ float s_arms[13 * 8], s_t2[64];
    __shared__ float2 s_dt[640];
    __shared__ float2 s_buf[kDsssChunk];
    __shared__ float s_mag[256]; __shared__ int s_idx[256]; __shared__ float2 s_val[256];
    const int c = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) st = states[c];
    for (int i = tid; i < 13 * p.nt_arm; i += 256) s_arms[i] = arms[i];
    for (int i = tid; i < p.nt2; i += 256) s_t2[i] = taps2[i];
    for (int i = tid; i < p.ntaps; i += 256) s_dt[i] = dtaps_rev[i];
    __syncthreads();
    const float2* x1 = r1 + static_cast<long long>(c) * r1_stride;
    float2* xa = ra + static_cast<long long>(c) * ring_stride;
    float2* xc = rc + static_cast<long long>(c) * ring_stride;
    float2* xd = rd + static_cast<long long>(c) * rd_stride;
    const long long o0 = st.o_n;
    const long long o1 = (k1 * 13 + 49) / 50;                    // outputs o whose newest input floor(50 o / 13) has arrived
    // ---- A: rational resampler 13 / 50 (arm (50 o) mod 13 at input floor(50 o / 13), oldest tap first)
    for (long long o = o0 + tid; o < o1; o += 256) {
        const long long im = o * 50, newest = im / 13;
        const float* hh = s_arms + static_cast<int>(im - newest * 13) * p.nt_arm;
        float re = 0.0f, imv = 0.0f;
        for (int k = p.nt_arm - 1; k >= 0; k--) {
            const long long a = newest - k;
            const float2 v = a >= 0 ? x1[a & r1_mask] : make_float2(0.0f, 0.0f);
            re = fmaf(hh[k], v.x, re); imv = fmaf(hh[k], v.y, imv);
        }
        xa[o & ring_mask] = make_float2(re, imv);
    }
    __syncthreads();
    // ---- B: frequency / phase lock (per-item recurrence) over shared-memory chunks
    for (long long b0 = o0; b0 < o1; b0 += kDsssChunk) {
        const int n = static_cast<int>(o1 - b0 < kDsssChunk ? o1 - b0 : kDsssChunk);
        for (int i = tid; i < n; i += 256) s_buf[i] = xa[(b0 + i) & ring_mask];
        __syncthreads();
        if (tid == 0) {
            LoopState pll = st.pll;
            for (int i = 0; i < n; i++) {
                float yr, yi;
                qrl_costas_step(pll, p.pll_alpha, p.pll_beta, 2, true, s_buf[i].x, s_buf[i].y, yr, yi);
                s_buf[i] = make_float2(yr, yi);
            }
            st.pll = pll;
        }
        __syncthreads();
        for (int i = tid; i < n; i += 256) xa[(b0 + i) & ring_mask] = s_buf[i];
        __syncthreads();
    }
    // ---- C: low-pass -> port 0 and the AGC's input
    for (long long o = o0 + tid; o < o1; o += 256) {
        float re = 0.0f, imv = 0.0f;
        for (int k = p.nt2 - 1; k >= 0; k--) {
            const long long a = o - k;
            const float2 v = a >= 0 ? xa[a & ring_mask] : make_float2(0.0f, 0.0f);
            re = fmaf(s_t2[k], v.x, re); imv = fmaf(s_t2[k], v.y, imv);
        }
        xc[o & ring_mask] = make_float2(re, imv);
        if (o - o_call0 < port0_stride) port0[static_cast<long long>(c) * port0_stride + (o - o_call0)] = make_float2(re, imv);
    }
    __syncthreads();
    // ---- D: agc2_cc::scale (signed rate compare, see agc_costas_kernel)
    for (long long b0 = o0; b0 < o1; b0 += kDsssChunk) {
        const int n = static_cast<int>(o1 - b0 < kDsssChunk ? o1 - b0 : kDsssChunk);
        for (int i = tid; i < n; i += 256) s_buf[i] = xc[(b0 + i) & ring_mask];
        __syncthreads();
        if (tid == 0) {
            float gain = st.agc;
            for (int i = 0; i < n; i++) {
                const float orr = s_buf[i].x * gain, oi = s_buf[i].y * gain;
                const float tmp = -p.agc_ref + sqrtf(orr * orr + oi * oi);
                const float rate = (tmp > gain) ? p.agc_attack : p.agc_decay;
                gain = gain - tmp * rate;
                if (gain < 0.0f) gain = 10e-5f;
                if (p.agc_max > 0.0f && gain > p.agc_max) gain = p.agc_max;
                s_buf[i] = make_float2(orr, oi);
            }
            st.agc = gain;
        }
        __syncthreads();
        for (int i = tid; i < n; i += 256) xc[(b0 + i) & ring_mask] = s_buf[i];
        __syncthreads();
    }
    // ---- E: despreader.  Symbol m needs items up to m N + (ntaps - N) - 1.
    const long long m0 = st.m_n;
    const long long m1 = o1 >= (p.ntaps - p.N) ? (o1 - (p.ntaps - p.N)) / p.N + 1 : 0;
    const int wlen = p.N + p.ntaps - 1;                           // items one symbol's correlations touch (<= kDsssChunk, checked at create)
    for (long long m = m0; m < m1; m++) {
        const long long w0 = m * p.N - 2LL * p.N + 1;
        for (int i = tid; i < wlen; i += 256) {
            const long long a = w0 + i;
            s_buf[i] = a >= 0 ? xc[a & ring_mask] : make_float2(0.0f, 0.0f);
        }
        __syncthreads();
        float best = 0.0f; int bj = 0x7fffffff; float2 bv = make_float2(0.0f, 0.0f);
        for (int j = tid; j < p.N; j += 256) {
            float ar = 0.0f, ai = 0.0f;
            for (int k = 0; k < p.ntaps; k++) {
                const float2 v = s_buf[j + k], t = s_dt[k];
                const float pr = v.x * t.x - v.y * t.y, pi = v.x * t.y + v.y * t.x;
                ar = ar + pr; ai = ai + pi;
            }
            const float mag = static_cast<float>(sqrt(static_cast<double>(ar) * static_cast<double>(ar) + static_cast<double>(ai) * static_cast<double>(ai)));
            if (mag > best) { best = mag; bj = j; bv = make_float2(ar, ai); }       // ascending j per thread: first strict maximum
        }
        s_mag[tid] = best; s_idx[tid] = bj; s_val[tid] = bv;
        __syncthreads();
        for (int off = 128; off >= 1; off >>= 1) {
            if (tid < off) {
                const float om = s_mag[tid + off]; const int oj = s_idx[tid + off];
                if (om > s_mag[tid] || (om == s_mag[tid] && oj < s_idx[tid])) { s_mag[tid] = om; s_idx[tid] = oj; s_val[tid] = s_val[tid + off]; }
            }
            __syncthreads();
        }
        if (tid == 0) {
            const float sc = 2.0f / static_cast<float>(p.N);
            xd[m & rd_mask] = s_mag[0] > 0.0f ? make_float2(s_val[0].x * sc, s_val[0].y * sc) : make_float2(0.0f * sc, 0.0f * sc);
        }
        __syncthreads();
    }
    // ---- F: symbol clock, carrier phase, soft bits
    if (tid == 0) {
        st.o_n = o1; st.m_n = m1 > m0 ? m1 : m0;
        const long long avail = st.m_n;
        int cnt = port1_cnt[c];
        // (each step advances mu by at least omega_min - gain_mu > 0.9, so two steps consume an item; the guard only stops a NaN stream)
        long long guard = 2 * (avail - st.cr_ii) + 16;
        while (st.cr_ii + 24 <= avail && guard-- > 0) {                // 8 interpolator taps + the block's 16-item margin (oracle crmm_work)
            const int imu = static_cast<int>(rintf(st.mu * 128.0f));
            const float* tt = d_mmse_tab + imu * 8;
            float yr = 0.0f, yi = 0.0f;
            for (int i = 0; i < 8; i++) {
                const float2 v = xd[(st.cr_ii + i) & rd_mask];
                yr = fmaf(tt[7 - i], v.x, yr); yi = fmaf(tt[7 - i], v.y, yi);
            }
            st.p2r = st.p1r; st.p2i = st.p1i; st.p1r = st.p0r; st.p1i = st.p0i; st.p0r = yr; st.p0i = yi;
            st.c2r = st.c1r; st.c2i = st.c1i; st.c1r = st.c0r; st.c1i = st.c0i;
            st.c0r = yr > 0.0f ? 1.0f : 0.0f; st.c0i = yi > 0.0f ? 1.0f : 0.0f;
            const float ar = st.c0r - st.c2r, ai = st.c0i - st.c2i;
            const float xr_ = ar * st.p1r + ai * st.p1i;
            const float br = st.p0r - st.p2r, bi = st.p0i - st.p2i;
            const float yr_ = br * st.c1r + bi * st.c1i;
            const float mm = qrl_clip(yr_ - xr_, 1.0f);
            st.omega = st.omega + p.gain_omega * mm;
            st.omega = p.omega_mid + qrl_clip(st.omega - p.omega_mid, p.omega_lim);
            st.mu = st.mu + st.omega + p.gain_mu * mm;
            const float fl = floorf(st.mu);
            st.cr_ii += static_cast<long long>(static_cast<int>(fl));
            st.mu = st.mu - fl;
            float cr, ci;
            qrl_costas_step(st.costas, p.costas_alpha, p.costas_beta, 2, false, yr, yi, cr, ci);
            if (cnt < port1_cap) port1[static_cast<long long>(c) * port1_stride + cnt] = make_float2(cr, ci);
            cnt++;
            soft_ring[static_cast<long long>(c) * soft_stride + (st.n_soft & soft_mask)] = qrl_soft_u8(cr, p.soft_scale);
            st.n_soft++; st.n_sym++;
        }
        port1_cnt[c] = cnt < port1_cap ? cnt : port1_cap;
        n_soft_out[c] = st.n_soft;
        states[c] = st;
    }
}

// ================================================================================================
// gr_demod_mmdvm_multi2 / gr_mod_mmdvm_multi2 per channel, either side of the polyphase filter bank (gr_demod_mmdvm_multi2.cpp:56-126,
// gr_mod_mmdvm_multi2.cpp:47-126).  No feedback anywhere: every stage is one thread per output item.
// ================================================================================================
// rows of a [n_rows][in_stride] slab (the channelizer's output) -> per-channel input ring (the resampler's history lives there)
__global__ void mmdvm_gather_kernel(const float2* __restrict__ in, long long in_stride, const int* __restrict__ rows, long long n,
                                    float2* __restrict__ ring, unsigned mask, long long stride, long long a0)
{
    const int c = blockIdx.y;
    const float2* src = in + static_cast<long long>(rows[c]) * in_stride;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
        ring[static_cast<long long>(c) * stride + ((a0 + i) & mask)] = src[i];
}
// quadrature_demod_cf(gain) -> x level (multiply_const_ff) -> float_to_short(1, 32767) = volk_32f_s32f_convert_16i: x scale, clip, rintf
__global__ void mmdvm_demod_short_kernel(const float2* __restrict__ ring, unsigned mask, long long stride, long long o0, long long o1,
                                         float gain, float level, short* __restrict__ out, long long out_stride)
{
    const int c = blockIdx.y;
    const long long o = o0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (o >= o1) return;
    const float2* x = ring + static_cast<long long>(c) * stride;
    const float2 a = x[o & mask];
    const float2 p = o > 0 ? x[(o - 1) & mask] : make_float2(0.0f, 0.0f);
    const float re = a.x * p.x + a.y * p.y;                              // x[n] * conj(x[n-1])
    const float im = a.y * p.x - a.x * p.y;
    float v = gain * qrl_fast_atan2f(im, re);
    v = v * level;
    v = v * 32767.0f;
    v = v > 32767.0f ? 32767.0f : (v < -32768.0f ? -32768.0f : v);
    out[static_cast<long long>(c) * out_stride + (o - o0)] = static_cast<short>(rintf(v));
}
// rssi_tag_block (rssi_tag_block.cpp:42-63): one value per 300 items, the block's own sequential float sum of (|x|^2)^2
__global__ void mmdvm_rssi_kernel(const float2* __restrict__ ring, unsigned mask, long long stride, long long b0, int nblocks, float cal,
                                  float* __restrict__ db, long long db_stride)
{
    const int c = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nblocks) return;
    const float2* x = ring + static_cast<long long>(c) * stride;
    const long long base = (b0 + j) * 300;
    float sum = 0.0f;
    for (int i = 0; i < 300; i++) {
        const float2 v = x[(base + i) & mask];
        const float pwr = v.x * v.x + v.y * v.y;
        sum = sum + pwr * pwr;
    }
    const float lv = sqrtf(sum / 300.0f);
    db[static_cast<long long>(c) * db_stride + j] = 10.0f * log10f(static_cast<float>(static_cast<double>(lv) + 1.0e-20)) + cal;
}
// short_to_float(1, 32767) = volk_16i_s32f_convert_32f (SIMD form: x (float)(1 / 32767)) -> x level -> the FM modulator's input ring
__global__ void mmdvm_short_float_kernel(const short* __restrict__ in, long long in_stride, long long n, float level,
                                         float* __restrict__ ring, unsigned mask, long long stride, long long a0)
{
    const int c = blockIdx.y;
    const float inv = static_cast<float>(1.0 / 32767.0);
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float v = static_cast<float>(in[static_cast<long long>(c) * in_stride + i]) * inv;
        v = v * level;
        ring[static_cast<long long>(c) * stride + ((a0 + i) & mask)] = v;
    }
}
// per-channel linear rows -> rows of the synthesizer's [n_rows][stride] input slab
__global__ void mmdvm_scatter_kernel(const float2* __restrict__ in, long long in_stride, const int* __restrict__ rows, long long n,
                                     float2* __restrict__ out, long long out_stride)
{
    const int c = blockIdx.y;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
        out[static_cast<long long>(rows[c]) * out_stride + i] = in[static_cast<long long>(c) * in_stride + i];
}
// multiply_const_cc twice on a linear buffer (behind the synthesizer: x 1 / num_channels, x bb_gain)
__global__ void scale2_linear_kernel(float2* __restrict__ x, long long n, float g1, float g2)
{
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float2 v = x[i];
        v.x = v.x * g1; v.y = v.y * g1; v.x = v.x * g2; v.y = v.y * g2;
        x[i] = v;
    }
}

// interleaved int16 I/Q (the SDR's wire format) -> gr_complex: float(v) * scale, as the host-side converter in front of the reference's
// source block does.  4 samples per thread: one 16-byte load, two 16-byte stores.
__global__ void sc16_to_fc32_kernel(const short2* __restrict__ in, long long in_stride, float2* __restrict__ out, long long out_stride,
                                    long T, float scale)
{
    const int c = blockIdx.y;
    const short2* src = in + static_cast<long long>(c) * in_stride;
    float2* dst = out + static_cast<long long>(c) * out_stride;
    const bool al = ((reinterpret_cast<unsigned long long>(src) & 15) == 0) && ((reinterpret_cast<unsigned long long>(dst) & 15) == 0);
    for (long q = (static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; q < T; q += static_cast<long>(gridDim.x) * blockDim.x * 4) {
        if (al && q + 4 <= T) {
            const uint4 v = *reinterpret_cast<const uint4*>(src + q);
            const unsigned w[4] = { v.x, v.y, v.z, v.w };
            float4 o[2];
            float* of = reinterpret_cast<float*>(o);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                of[2 * k] = static_cast<float>(static_cast<short>(w[k] & 0xFFFFu)) * scale;
                of[2 * k + 1] = static_cast<float>(static_cast<short>(w[k] >> 16)) * scale;
            }
            *reinterpret_cast<float4*>(dst + q) = o[0];
            *reinterpret_cast<float4*>(dst + q + 2) = o[1];
        } else {
            for (long t = q; t < T && t < q + 4; t++) dst[t] = make_float2(static_cast<float>(src[t].x) * scale, static_cast<float>(src[t].y) * scale);
        }
    }
}

// interleaved int8 I/Q (HackRF / 8-bit front ends through gr-osmosdr: 2 bytes per sample) -> gr_complex: float(v) * scale.  8 samples per
// thread: one 16-byte load, four 16-byte stores.
__global__ void sc8_to_fc32_kernel(const char2* __restrict__ in, long long in_stride, float2* __restrict__ out, long long out_stride,
                                   long T, float scale)
{
    const int c = blockIdx.y;
    const char2* src = in + static_cast<long long>(c) * in_stride;
    float2* dst = out + static_cast<long long>(c) * out_stride;
    const bool al = ((reinterpret_cast<unsigned long long>(src) & 15) == 0) && ((reinterpret_cast<unsigned long long>(dst) & 15) == 0);
    for (long q = (static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x) * 8; q < T; q += static_cast<long>(gridDim.x) * blockDim.x * 8) {
        if (al && q + 8 <= T) {
            const uint4 v = *reinterpret_cast<const uint4*>(src + q);
            const unsigned w[4] = { v.x, v.y, v.z, v.w };
            float4 o[4];
            float* of = reinterpret_cast<float*>(o);
#pragma unroll
            for (int k = 0; k < 4; k++)
#pragma unroll
                for (int b = 0; b < 4; b++) of[4 * k + b] = static_cast<float>(static_cast<signed char>((w[k] >> (8 * b)) & 0xFFu)) * scale;
#pragma unroll
            for (int k = 0; k < 4; k++) *reinterpret_cast<float4*>(dst + q + 2 * k) = o[k];
        } else {
            for (long t = q; t < T && t < q + 8; t++) dst[t] = make_float2(static_cast<float>(src[t].x) * scale, static_cast<float>(src[t].y) * scale);
        }
    }
}

// gr_zero_idle_bursts (gr_zero_idle_bursts.cpp:45-82) as two ring passes.  (1) the sync block's history: out[a] = in[a - delay_items]
// (zero before the stream began); (2) the "zero_samples" counter: the host has turned the tags of this call into [begin, end) item
// ranges per channel (qrl_tx_work), one CTA per range clears them.
__global__ void tx_delay_ring_kernel(const float2* __restrict__ in, unsigned in_mask, long long in_stride,
                                     float2* __restrict__ out, unsigned out_mask, long long out_stride,
                                     long long a0, long long a1, long long delay_items)
{
    const int c = blockIdx.y;
    const long long a = a0 + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (a >= a1) return;
    const long long s = a - delay_items;
    float2 v = make_float2(0.0f, 0.0f);
    if (s >= 0) v = in[static_cast<long long>(c) * in_stride + (s & in_mask)];
    out[static_cast<long long>(c) * out_stride + (a & out_mask)] = v;
}
__global__ void tx_zero_ranges_kernel(float2* __restrict__ ring, unsigned mask, long long stride, const long long* __restrict__ ranges)
{
    const long long c = ranges[3 * blockIdx.x], a0 = ranges[3 * blockIdx.x + 1], a1 = ranges[3 * blockIdx.x + 2];
    for (long long a = a0 + threadIdx.x; a < a1; a += blockDim.x) ring[c * stride + (a & mask)] = make_float2(0.0f, 0.0f);
}

}  // namespace qrl
