// =====================================================================================
// tests/bpr_strict_reference.cpp  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The StrictMath restatement of one BPR epoch (recommender/cf/ranking/BPRRecommender.java:48-93) that defines the device's
// reference-order BPR mode (LRK_UPDATE_REFERENCE_ORDER with LRK_MODEL_BPR): the same loop as lro_bpr_epoch in
// oracle/lrk_oracle.cpp, with fdlibm's exp in Maths.logistic and fdlibm's log in the loss, on a java.util.Random state of its own
// that the caller sets and reads back.  Self-contained, so that the oracle the other tests pin stays as it is; the fdlibm log
// below is the oracle's restatement, repeated.  Built by tests/bpr_strict.py (g++ -O2 -ffp-contract=off: Java never contracts
// a*b+c into an FMA).
// =====================================================================================
#include <algorithm>
#include <cstdint>
#include <cstring>

#define LRO_API extern "C" __attribute__((visibility("default")))

// fdlibm __ieee754_log  ==  java.lang.StrictMath.log, restated from the published fdlibm 5.3 e_log.c algorithm
// (Sun Microsystems, freely distributable)
static inline int32_t hi_word(double x) { uint64_t b; memcpy(&b, &x, 8); return (int32_t)(b >> 32); }
static inline uint32_t lo_word(double x) { uint64_t b; memcpy(&b, &x, 8); return (uint32_t)b; }
static inline double with_hi(double x, int32_t hi) {
    uint64_t b; memcpy(&b, &x, 8);
    b = (b & 0xffffffffULL) | ((uint64_t)(uint32_t)hi << 32);
    memcpy(&x, &b, 8); return x;
}

static double fdlibm_log(double x) {
    static const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10,
                        two54 = 1.80143985094819840000e+16,
                        Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01,
                        Lg3 = 2.857142874366239149e-01, Lg4 = 2.222219843214978396e-01,
                        Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                        Lg7 = 1.479819860511658591e-01;
    const double zero = 0.0;
    double hfsq, f, s, z, R, w, t1, t2, dk;
    int32_t k, hx, i, j;
    uint32_t lx;
    hx = hi_word(x); lx = lo_word(x);
    k = 0;
    if (hx < 0x00100000) {
        if (((hx & 0x7fffffff) | lx) == 0) return -two54 / zero;
        if (hx < 0) return (x - x) / zero;
        k -= 54; x *= two54; hx = hi_word(x);
    }
    if (hx >= 0x7ff00000) return x + x;
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    i = (hx + 0x95f64) & 0x100000;
    x = with_hi(x, hx | (i ^ 0x3ff00000));
    k += (i >> 20);
    f = x - 1.0;
    if ((0x000fffff & (2 + hx)) < 3) {
        if (f == zero) { if (k == 0) return zero; dk = (double)k; return dk * ln2_hi + dk * ln2_lo; }
        R = f * f * (0.5 - 0.33333333333333333 * f);
        if (k == 0) return f - R;
        dk = (double)k; return dk * ln2_hi - ((R - dk * ln2_lo) - f);
    }
    s = f / (2.0 + f);
    dk = (double)k;
    z = s * s;
    i = hx - 0x6147a;
    w = z * z;
    j = 0x6b851 - hx;
    t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    i |= j;
    R = t2 + t1;
    if (i > 0) {
        hfsq = 0.5 * f * f;
        if (k == 0) return f - (hfsq - s * (hfsq + R));
        return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
    } else {
        if (k == 0) return f - s * (f - R);
        return dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f);
    }
}

// -------------------------------------------------------------------------------------
// fdlibm __ieee754_exp  ==  java.lang.StrictMath.exp.  Restated from the published fdlibm 5.3 e_exp.c algorithm (Sun
// Microsystems, freely distributable).  Maths.logistic calls Math.exp, whose JIT intrinsic may differ from StrictMath.exp in
// the last bit on some JVMs; the reference-order BPR mode is defined with this one, as the oracle pins nextGaussian's log to fdlibm's.
// -------------------------------------------------------------------------------------
static double fdlibm_exp(double x) {
    static const double one = 1.0, halF[2] = {0.5, -0.5}, huge = 1.0e+300, twom1000 = 9.33263618503218878990e-302,
                        o_threshold = 7.09782712893383973096e+02, u_threshold = -7.45133219101941108420e+02,
                        ln2HI[2] = {6.93147180369123816490e-01, -6.93147180369123816490e-01},
                        ln2LO[2] = {1.90821492927058770002e-10, -1.90821492927058770002e-10},
                        invln2 = 1.44269504088896338700e+00, P1 = 1.66666666666666019037e-01,
                        P2 = -2.77777777770155933842e-03, P3 = 6.61375632143793436117e-05,
                        P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    double y, hi = 0.0, lo = 0.0, c, t;
    int32_t k = 0;
    uint32_t hx = (uint32_t)hi_word(x);
    const int xsb = (int)((hx >> 31) & 1);
    hx &= 0x7fffffff;
    if (hx >= 0x40862E42) {                                   // |x| >= 709.78...
        if (hx >= 0x7ff00000) {
            if (((hx & 0xfffff) | lo_word(x)) != 0) return x + x;   // NaN
            return xsb == 0 ? x : 0.0;                        // exp(+-inf) = {inf, 0}
        }
        if (x > o_threshold) return huge * huge;
        if (x < u_threshold) return twom1000 * twom1000;
    }
    if (hx > 0x3fd62e42) {                                    // |x| > 0.5 ln2
        if (hx < 0x3FF0A2B2) {                                // and |x| < 1.5 ln2
            hi = x - ln2HI[xsb]; lo = ln2LO[xsb]; k = 1 - xsb - xsb;
        } else {
            k = (int32_t)(invln2 * x + halF[xsb]);
            t = k;
            hi = x - t * ln2HI[0];                            // t * ln2HI is exact here
            lo = t * ln2LO[0];
        }
        x = hi - lo;
    } else if (hx < 0x3e300000) {                             // |x| < 2^-28
        if (huge + x > one) return one + x;
    } else {
        k = 0;
    }
    t = x * x;
    c = x - t * (P1 + t * (P2 + t * (P3 + t * (P4 + t * P5))));
    if (k == 0) return one - ((x * c) / (c - 2.0) - x);
    y = one - ((lo - (x * c) / (2.0 - c)) - hi);
    if (k >= -1021) return with_hi(y, (int32_t)((uint32_t)hi_word(y) + ((uint32_t)k << 20)));
    return with_hi(y, (int32_t)((uint32_t)hi_word(y) + ((uint32_t)(k + 1000) << 20))) * twom1000;
}
LRO_API double lro_fdlibm_exp(double x) { return fdlibm_exp(x); }

// the 48-bit state of the generator (Randoms.r's Random.seed; BPR draws only nextInt, so there is no cached Gaussian)
static uint64_t g_seed = 0;
LRO_API uint64_t lro_jrandom_state() { return g_seed; }
LRO_API void lro_set_jrandom_state(uint64_t s) { g_seed = s & ((1ULL << 48) - 1); }

// java.util.Random.next(31) / nextInt(bound) (JDK 8), Randoms.uniform(int) (math/algorithm/Randoms.java:41-43)
static inline int32_t jr_next31() {
    g_seed = (g_seed * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
    return (int32_t)(uint32_t)(g_seed >> 17);
}
static inline int32_t lro_uniform_int(int32_t bound) {
    int32_t v = jr_next31();
    const int32_t m = bound - 1;
    if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)v) >> 31);
    for (int32_t u = v;; u = jr_next31()) {
        v = u % bound;
        if ((int32_t)((uint32_t)u - (uint32_t)v + (uint32_t)m) >= 0) return v;   // Java int arithmetic wraps: "u - r + m < 0"
    }
}

// DenseVector.dot: math/structure/DenseVector.java:104-111 -- left to right from 0.0
static inline double dot_lr(const double* a, const double* b, int k) {
    double r = 0.0;
    for (int f = 0; f < k; ++f) r += b[f] * a[f];
    return r;
}

// oracle/lrk_oracle.cpp's lro_bpr_epoch with StrictMath semantics: fdlibm exp in Maths.logistic and fdlibm log in the loss.  This is the definition of
// the device's reference-order BPR mode (LRK_UPDATE_REFERENCE_ORDER with LRK_MODEL_BPR), whose factors and generator state
// equal this function's bit for bit.  Same trip / trip_out arguments as lro_bpr_epoch.
static inline double logistic_strict(double x) { return 1.0 / (1.0 + fdlibm_exp(-x)); }
LRO_API double lro_bpr_epoch_strict(int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, int32_t k,
                                    double* P, double* Q, float lr_f, float regU_f, float regI_f,
                                    int64_t n_samples, const int32_t* trip, int32_t* trip_out) {
    const double learnRate = (double)lr_f, regUser = (double)regU_f, regItem = (double)regI_f;
    double loss = 0.0;
    for (int64_t s = 0; s < n_samples; ++s) {
        int32_t u, pi, nj;
        if (trip) { u = trip[3 * s]; pi = trip[3 * s + 1]; nj = trip[3 * s + 2]; }
        else {
            for (;;) {
                u = lro_uniform_int(U);
                const int64_t b = rowptr[u], e = rowptr[u + 1];
                const int64_t len = e - b;
                if (len == 0 || len == I) continue;
                pi = col[b + lro_uniform_int((int32_t)len)];
                do { nj = lro_uniform_int(I); } while (std::binary_search(col + b, col + e, nj));
                break;
            }
        }
        if (trip_out) { trip_out[3 * s] = u; trip_out[3 * s + 1] = pi; trip_out[3 * s + 2] = nj; }
        double* pu = P + (int64_t)u * k;
        double* qi = Q + (int64_t)pi * k;
        double* qj = Q + (int64_t)nj * k;
        const double diff = dot_lr(pu, qi, k) - dot_lr(pu, qj, k);
        loss += -fdlibm_log(logistic_strict(diff));
        const double deri = logistic_strict(-diff);
        for (int f = 0; f < k; ++f) {
            const double uf = pu[f], pf = qi[f], nf = qj[f];
            pu[f] += learnRate * (deri * (pf - nf) - regUser * uf);
            qi[f] += learnRate * (deri * uf - regItem * pf);
            qj[f] += learnRate * (deri * (-uf) - regItem * nf);
            loss += regUser * uf * uf + regItem * pf * pf + regItem * nf * nf;
        }
    }
    return loss;  // no *0.5 for BPR
}

