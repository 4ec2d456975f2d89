/*
 * mse_oracle.c -- CPU restatement of the MSE observer's clipping-range search (vsiquantization_b200/csrc/mse_search.cu,
 * observers/mse.py).  TEST INFRASTRUCTURE ONLY: the checker the GPU tests and tools/mse_bench.py compare against.
 * Kept beside oracle/ rather than in it so the pinned oracle stays byte-identical to what its golden vectors were
 * checked against; the fake-quant arithmetic below is oracle/vsiq_oracle.c's (every fp32 operation individually rounded,
 * IEEE division, round-half-even, torch.clamp semantics; compile with -ffp-contract=off).
 *
 * Layout: [outer, C, inner], channel c of flat index i is (i / inner) % C; a channels_last [rows, C] tensor is
 * {rows, C, 1}.  Every sum runs in index order.
 */
#include <math.h>
#include <stdint.h>

static inline float clamp_torch(float r, float lo, float hi) {
    if (r != r) return r;
    if (r < lo) return lo;
    if (r > hi) return hi;
    return r;
}

/* observers/minmax.py:67-74 in Python doubles (oracle/vsiq_oracle.c: vsiq_oracle_qparams) */
static void qparams(double mn, double mx, int bits, int symmetric, double eps, double *scale, double *zp) {
    if (symmetric) {
        double a = fabs(mn), b = fabs(mx);
        double max_abs = (b > a) ? b : a;
        *scale = max_abs / ((double)((1 << (bits - 1)) - 1) + eps);
        *zp = 0.0;
    } else {
        double s = (mx - mn) / ((double)((1 << bits) - 1) + eps);
        *scale = s;
        *zp = rint(-mn / (s + eps));
    }
}

/* sum over channel c of ((double)fq(x) - (double)x)^2 with fp32 qparams (s, z) and integer range [qmin, qmax] */
static double channel_error(const float *x, int64_t outer, int64_t C, int64_t inner, int64_t c, float s, float z,
                            int qmin, int qmax) {
    const float lo = (float)qmin, hi = (float)qmax;
    double e = 0.0;
    for (int64_t o = 0; o < outer; ++o) {
        const float *p = x + (o * C + c) * inner;
        for (int64_t i = 0; i < inner; ++i) {
            float v = p[i] / s;
            float t = v + z;
            float q = clamp_torch(rintf(t), lo, hi);
            float y = (q - z) * s;
            double d = (double)y - (double)p[i];
            e += d * d;
        }
    }
    return e;
}

/*
 * One MSEObserver.observe(x) call.  state: [C][10] fp64 (run_min, run_max, scale, zero_point, n_calls, sum mean|x|,
 * sum mean x, sum std, mean clipped min, mean clipped max), updated in place.  err [C][K] and alpha [C] may be NULL.
 */
void mse_oracle_search(const float *x, int64_t outer, int64_t C, int64_t inner, double *state, int bits, int symmetric,
                       double eps, int K, double *err, double *alpha) {
    const int qmin = symmetric ? -(1 << (bits - 1)) : 0;
    const int qmax = symmetric ? (1 << (bits - 1)) - 1 : (1 << bits) - 1;
    const double count = (double)outer * (double)inner;
    for (int64_t c = 0; c < C; ++c) {
        double *st = state + c * 10;
        /* 1. running range and call statistics: observers/minmax.py:42-47, quantization_manager.py:66-68 */
        float mn = INFINITY, mx = -INFINITY;
        int has_nan = 0;
        double sa = 0.0, s1 = 0.0, s2 = 0.0;
        for (int64_t o = 0; o < outer; ++o) {
            const float *p = x + (o * C + c) * inner;
            for (int64_t i = 0; i < inner; ++i) {
                float v = p[i];
                if (v != v) has_nan = 1;
                if (v < mn) mn = v;
                if (v > mx) mx = v;
                sa += fabs((double)v);
                s1 += (double)v;
                s2 += (double)v * (double)v;
            }
        }
        if (!has_nan) {
            if ((double)mn < st[0]) st[0] = (double)mn;
            if ((double)mx > st[1]) st[1] = (double)mx;
        }
        const double mean = s1 / count;
        const double var = (s2 - count * mean * mean) / (count - 1.0);
        st[4] += 1.0;
        st[5] += sa / count;
        st[6] += mean;
        st[7] += sqrt(var > 0.0 ? var : 0.0);
        const double lo = st[0], hi = st[1];
        /* 2-4. candidates, errors, choice */
        int best = 0, bad = !(isfinite(lo) && isfinite(hi));
        double best_e = 0.0;
        for (int k = 1; k <= K; ++k) {
            const double a = (double)k / (double)K;
            double s, z;
            qparams(a * lo, a * hi, bits, symmetric, eps, &s, &z);
            const double e = channel_error(x, outer, C, inner, c, (float)s, (float)z, qmin, qmax);
            if (err) err[c * K + (k - 1)] = e;
            if (!isfinite(e)) bad = 1;
            else if (best == 0 || e <= best_e) {
                best = k;
                best_e = e;
            }
        }
        const double a = (bad || best == 0) ? 1.0 : (double)best / (double)K;
        if (alpha) alpha[c] = a;
        /* 5-6. running means of the clipped extrema, qparams from them */
        st[8] += (a * lo - st[8]) / st[4];
        st[9] += (a * hi - st[9]) / st[4];
        qparams(st[8], st[9], bits, symmetric, eps, &st[2], &st[3]);
    }
}

/* scale / zero-point of (mn, mx) by the same formula, for the checks */
void mse_oracle_qparams(double mn, double mx, int bits, int symmetric, double eps, double *scale, double *zp) {
    qparams(mn, mx, bits, symmetric, eps, scale, zp);
}
