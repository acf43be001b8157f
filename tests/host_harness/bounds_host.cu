// Test infrastructure (not part of the product library): the two fp32 bounds of K3a's exact search - the candidate
// filter threshold and the slack of a tracked match, generalized-icp_b200/csrc/objective.cuh - compiled for the HOST
// together with a restatement of the device arithmetic around them (fp32 candidate distance, roundings), so that
// tests/test_host.py can check their soundness against __float128 distances on millions of adversarial cases.
#include "../../generalized-icp_b200/csrc/objective.cuh"

typedef __float128 f128;

static float f_ru(double x) {   // __double2float_ru
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
}
static float f_rd(double x) {   // __double2float_rd
    float f = (float)x;
    if ((double)f > x) f = nextafterf(f, -INFINITY);
    return f;
}
static float ulps(float x, int n) {
    for (; n > 0; --n) x = nextafterf(x, INFINITY);
    for (; n < 0; ++n) x = nextafterf(x, -INFINITY);
    return x;
}
static f128 sqrt128(f128 v) {   // one Newton step from the 64-bit square root: ~113 bits
    if (!(v > 0)) return 0;
    f128 x = (f128)sqrtl((long double)v);
    return 0.5 * (x + v / x);
}
// the oracle's key (dx*dx + dy*dy) + dz*dz, every operation rounded separately (exact_d2 of common.cuh)
static double key_d2(const double* c, const double* p) {
    const double dx = c[0] - p[0], dy = c[1] - p[1], dz = c[2] - p[2];
    volatile double xx = dx * dx, yy = dy * dy, zz = dz * dz;
    volatile double s = xx + yy;
    return s + zz;
}
static f128 true_d2(const double* c, const double* p) {
    f128 s = 0;
    for (int i = 0; i < 3; ++i) { const f128 d = (f128)c[i] - (f128)p[i]; s += d * d; }
    return s;
}
struct Query { float fx, fy, fz, Pf, c1; };
static Query query(const double* p) {
    Query q;
    q.fx = (float)p[0]; q.fy = (float)p[1]; q.fz = (float)p[2];
    q.Pf = fmaxf(fabsf(q.fx), fmaxf(fabsf(q.fy), fabsf(q.fz))) * 1.0000002f;
    q.c1 = gicp::filter_c1(q.Pf);
    return q;
}
// the fp32 squared distance K3a filters with (f32 storage: candidate coordinates are fp32)
static float d32_of(const double* c, const Query& q) {
    const float dx = (float)c[0] - q.fx, dy = (float)c[1] - q.fy, dz = (float)c[2] - q.fz;
    return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

// Filter soundness.  Case i: query p[i] (fp64), candidate c[i] (fp32 values), best distance so far bd[i].  The
// threshold is evaluated with the reciprocal square root perturbed by every offset in [-rs_ulps, rs_ulps] (the
// device's rsqrtf is approximate); out[i] = 1 when the candidate must pass (its key or its exact squared distance
// is <= bd) and fails for some perturbation, 0 otherwise.  Returns the number of such failures.
extern "C" long long gicp_test_filter(long long n, const double* p, const double* c, const double* bd, int rs_ulps,
                                      int* out) {
    long long bad = 0;
    for (long long i = 0; i < n; ++i) {
        const double* pi = p + 3 * i;
        const double* ci = c + 3 * i;
        const Query q = query(pi);
        const bool must = key_d2(ci, pi) <= bd[i] || true_d2(ci, pi) <= (f128)bd[i];
        const float d32 = d32_of(ci, q);
        const float b = f_ru(bd[i]);
        const float rs = (float)(1.0 / sqrt((double)fmaxf(b, 1e-30f)));
        bool fail = false;
        for (int u = -rs_ulps; u <= rs_ulps; ++u) fail |= !(d32 <= gicp::filter_thr_of(b, ulps(rs, u), q.c1));
        out[i] = must && fail;
        bad += out[i];
    }
    return bad;
}

// Slack soundness.  Case i: query p[i], two target points a[i], b[i] (the nearest and the runner-up, in either
// order).  f32 != 0: fp32 storage (the fp32 distances K3a keeps for the slack are the filter's d2_32); otherwise
// fp64 storage (the key rounded down).  The device's slack for the match is computed with rad32 = +inf (every other
// target point is farther than both) and compared with half the exact gap.  slack[i] / gap[i] receive both (as
// doubles); returns the number of cases with slack > gap / 2.
extern "C" long long gicp_test_slack(long long n, const double* p, const double* a, const double* b, int f32,
                                     double* slack, double* half_gap) {
    long long bad = 0;
    for (long long i = 0; i < n; ++i) {
        const double* pi = p + 3 * i;
        const Query q = query(pi);
        const double ka = key_d2(a + 3 * i, pi), kb = key_d2(b + 3 * i, pi);
        const f128 ta = true_d2(a + 3 * i, pi), tb = true_d2(b + 3 * i, pi);
        float da, db;
        if (f32) { da = d32_of(a + 3 * i, q); db = d32_of(b + 3 * i, q); }
        else { da = f_rd(ka); db = f_rd(kb); }
        const float m2 = fmaxf(da, db);            // second smallest of the two
        const double bestd = ka <= kb ? ka : kb;   // the match: smaller key (equal keys: either one, same distance)
        const float sl = gicp::match_slack(f_ru(sqrt(bestd)), m2, INFINITY, q.c1, q.Pf);
        const f128 g = sqrt128(ta) - sqrt128(tb);
        const f128 hg = 0.5 * (g < 0 ? -g : g);
        slack[i] = sl;
        half_gap[i] = (double)hg;
        bad += ((f128)sl > hg) ? 1 : 0;
    }
    return bad;
}
