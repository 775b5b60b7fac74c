/* txfront_ref.c -- the TX front end's definition (tests/txfront_ref.py builds and drives it; test infrastructure only).
 *
 * gr_mod_base (gr_mod_base.cpp:38,211-290,799-805): mod -> rotator_cc(2 pi offset / 1e6) -> (samp_rate >= 2 Msps)
 * rational_resampler_ccf(N, 1, low_pass(N, samp_rate, 480000, 20000, BLACKMAN_HARRIS)).  The two loops that need exact float
 * arithmetic live here (built with -ffp-contract=off: a fused multiply-add exists only where fmaf() is written); the stream state
 * (phase bookkeeping, history) is kept by the Python side. */
#include <math.h>
#include <stdint.h>

void qo_sincosf(float x, float* s, float* c);      /* the oracle's sin / cos (oracle/libqrl_oracle.so) */

/* y[i] = x[i] * exp(j theta_i): the oracle's exact Q32 NCO, phase_i = base + inc * (k0 + i), theta = phase (as int32) * pi / 2^31 */
void txref_rotate(const float* x, long n, uint32_t base, uint32_t inc, uint32_t k0, float* y)
{
    for (long i = 0; i < n; i++) {
        uint32_t ph = base + inc * (uint32_t)(k0 + (uint32_t)i);
        float ang = (float)((double)(int32_t)ph * (M_PI / 2147483648.0));
        float sn, cs;
        qo_sincosf(ang, &sn, &cs);
        float xr = x[2 * i], xi = x[2 * i + 1];
        y[2 * i] = xr * cs - xi * sn;
        y[2 * i + 1] = xr * sn + xi * cs;
    }
}

/* xN interpolator: x = nt - 1 history items followed by n new ones (complex); arms[p][k] = taps[p + k N];
 * y[N m + p] = sum_k arms[p][k] x_new[m - k], one fmaf chain per component, oldest sample (k = nt - 1) first */
void txref_interp(const float* arms, int N, int nt, const float* x, long n, float* y)
{
    for (long m = 0; m < n; m++) {
        const float* newest = x + 2 * (m + nt - 1);
        for (int p = 0; p < N; p++) {
            const float* h = arms + (long)p * nt;
            float re = 0.0f, im = 0.0f;
            for (int k = nt - 1; k >= 0; k--) {
                re = fmaf(h[k], newest[-2L * k], re);
                im = fmaf(h[k], newest[-2L * k + 1], im);
            }
            y[2 * (m * N + p)] = re;
            y[2 * (m * N + p) + 1] = im;
        }
    }
}
