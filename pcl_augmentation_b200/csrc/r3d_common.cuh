// Shared device math for the Real3D-Aug hot path (sm_100a).  Everything that decides a bin, a mask or a choice is
// evaluated in fp64 with the reference's expression order and WITHOUT fused multiply-add (the library is compiled with
// --fmad=false; the helpers below also spell the roundings out), so results are bit-identical to numpy wherever the
// reference uses +,-,*,/,sqrt.  The only ops that can differ from numpy by an ulp are the transcendentals
// (atan2/acos), see DESIGN.md "numerics".
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define R3D_EMPTY_U64 0xFFFFFFFFFFFFFFFFull
#define R3D_MAX_CLASSES 16
#define R3D_MAX_SURFACE 8
#define R3D_NUM_RADII 50

namespace r3d {

constexpr double kPi = 3.141592653589793;        // numpy.pi
constexpr double kTwoPi = 6.283185307179586;     // 2 * math.pi
constexpr double kEmptyRange = 500.0;            // od/ins:100 "train = ones * 500"

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }

// od/ins:75  r = sqrt(x**2 + y**2 + z**2)
__device__ __forceinline__ double range3(double x, double y, double z) {
    return sqrt(add(add(mul(x, x), mul(y, y)), mul(z, z)));
}
// od/ins:76  azimuth = arctan2(y, x) + pi
__device__ __forceinline__ double azimuth(double x, double y) { return add(atan2(y, x), kPi); }
// od/ins:77  elevation = arccos(z / r)
__device__ __forceinline__ double elevation(double z, double r) { return acos(__ddiv_rn(z, r)); }

// od/ins:106  int((az % (2*pi)) / d_azimuth) ; az is in [0, 2*pi] so the Python float modulo is a conditional subtract
__device__ __forceinline__ double az_mod(double az) { return az >= kTwoPi ? sub(az, kTwoPi) : az; }

struct ImageGeom {
    int rows, cols;
    int pix_stride;       // the reference's module-global NUMCOLUMN used in pix_id (od/ins:117)
    double min_el, max_el;
    double d_el, d_az;
};

__host__ __device__ __forceinline__ ImageGeom make_geom(int rows, int cols, int pix_stride, double max_el, double min_el) {
    ImageGeom g;
    g.rows = rows; g.cols = cols; g.pix_stride = pix_stride;
    g.min_el = min_el; g.max_el = max_el;
    g.d_el = (max_el - min_el) / (double)rows;          // od/ins:97
    g.d_az = kTwoPi / (double)cols;                     // od/ins:98
    return g;
}

// truncation toward zero like Python int(); values that do not fit are reported as INT_MIN
__device__ __forceinline__ int trunc_to_int(double v) {
    if (!(v > -2147483000.0 && v < 2147483000.0)) return INT_MIN;
    return (int)v;                                       // cvt.rzi
}
// od/ins:105  int((el - min_el - 0.00001) / d_elevation)
__device__ __forceinline__ int bin_row(const ImageGeom& g, double el) {
    return trunc_to_int(__ddiv_rn(sub(sub(el, g.min_el), 0.00001), g.d_el));
}
__device__ __forceinline__ int bin_col(const ImageGeom& g, double az) {
    return trunc_to_int(__ddiv_rn(az_mod(az), g.d_az));
}

// ---- mean of n = 1 .. 15 ranges (the close / fill neighbour mean, cl:57), correctly rounded like sum / n but without
// the fp64 division: y = RN(1/n) from a table, q = RN(sum * y) is within an ulp of the quotient, the remainder
// sum - q * n is exact in one fma, and by Markstein's theorem q + r * y rounded once is RN(sum / n).
// (tests/test_mean_div_host.py checks it against sum / n in exact rational arithmetic.)  The table is read through the
// L1 (__ldg) rather than the constant cache, whose reads serialise when the lanes of a warp index different entries.
static __device__ const double kRecipSmall[16] = {0.0, 1.0, 1.0 / 2, 1.0 / 3, 1.0 / 4, 1.0 / 5, 1.0 / 6, 1.0 / 7, 1.0 / 8,
                                                  1.0 / 9, 1.0 / 10, 1.0 / 11, 1.0 / 12, 1.0 / 13, 1.0 / 14, 1.0 / 15};
__device__ __forceinline__ double mean_div(double sum, int n) {
#ifdef R3D_MEAN_DDIV                                     // A/B builds only: the plain division
    return __ddiv_rn(sum, (double)n);
#else
    const double y = __ldg(&kRecipSmall[n]);
    const double q = __dmul_rn(sum, y);
    const double r = __fma_rn(-q, (double)n, sum);
    return __fma_rn(r, y, q);
#endif
}

// ---- fast binning.  A bin index only needs the transcendental to ~1e-6 rad unless the point sits next to a bin edge:
// float atan2f / acosf (CUDA: <= 3 / 2 ulp) give the position in bin units with a known error bound; if that position
// is at least the bound away from both edges of its bin (and from both ends of the image), floor() of it IS the index
// the fp64 expression of the reference yields; otherwise the caller evaluates the exact fp64 path.  Error budget in
// radians: arguments rounded to float 2e-7, function 7e-7 (azimuth near 2 pi) resp. 2.4e-7 / sqrt(1 - t^2) (elevation,
// |t| <= 0.9 only), offsets 2.4e-7 -> < 1.5e-6 rad, taken as 6e-6; the product with the float reciprocal of the bin
// width adds 2.4e-7 relative to the position (<= nbins).
struct FastGeom { float inv_d_az, inv_d_el, el0, err_az, err_el; };
__device__ __forceinline__ FastGeom make_fast_geom(const ImageGeom& g) {
    FastGeom f;
    f.inv_d_az = (float)(1.0 / g.d_az); f.inv_d_el = (float)(1.0 / g.d_el);
    f.el0 = (float)(g.min_el + 0.00001);
    f.err_az = 6e-6f * f.inv_d_az + 5e-7f * (float)g.cols + 1e-5f;
    f.err_el = 6e-6f * f.inv_d_el + 5e-7f * (float)g.rows + 1e-5f;
    if (!(f.err_az < 0.25f)) f.err_az = 2.0f;            // hopeless geometry: the test below never passes
    if (!(f.err_el < 0.25f)) f.err_el = 2.0f;
    return f;
}
__device__ __forceinline__ bool fast_bin(float t, float err, int nbins, int& bin) {
    const float f = floorf(t), fr = t - f;
    if (!(fr > err && fr < 1.0f - err && t > err && t < (float)nbins - err)) return false;      // also NaN
    bin = (int)f;
    return true;
}
// od/ins:106 without the fp64 arctan2 where the azimuth is clear of the bin edges
__device__ __forceinline__ bool fast_col(float inv_d_az, float err_az, int cols, float x, float y, int& col) {
    return fast_bin((atan2f(y, x) + 3.14159274f) * inv_d_az, err_az, cols, col);
}
// od/ins:105 without the fp64 arccos where the elevation is clear of the bin edges
__device__ __forceinline__ bool fast_row(const FastGeom& f, int rows, float z, float r, int& row) {
    const float t = z / r;
    if (!(fabsf(t) <= 0.9f)) return false;
    return fast_bin((acosf(t) - f.el0) * f.inv_d_el, f.err_el, rows, row);
}

// ---------------------------------------------------------------------------------------------- boxes
// Host-prepared oriented box: centre (z = box BOTTOM, cb:56-66), rotation matrix (row-major) and extents.
struct Box {
    double cx, cy, cz;
    double m[9];
    double length, width, height;
    double reach;          // horizontal bounding radius used only for conservative pruning
};

// The six thresholds of cut_bounding_box (cb:30-66) in the reference's expression order.
struct BoxTest {
    double c0x, c0y, c0z, hi0, lo0;      // column 0 of m, length
    double c1x, c1y, c1z, hi1, lo1;      // column 1 of m, width
    double c2x, c2y, c2z, hi2, lo2;      // column 2 of m, height (from the bottom)
};

__device__ __forceinline__ BoxTest make_box_test(const Box& b) {
    BoxTest t;
    const double* m = b.m;
    t.c0x = m[0]; t.c0y = m[3]; t.c0z = m[6];
    t.c1x = m[1]; t.c1y = m[4]; t.c1z = m[7];
    t.c2x = m[2]; t.c2y = m[5]; t.c2z = m[8];
    const double L = b.length, W = b.width, H = b.height;
    // m00*(xc + m00*L/2) + m10*(yc + m10*L/2) + m20*(zc + m20*L/2)      ("m00*L/2" is (m00*L)/2)
    t.hi0 = add(add(mul(t.c0x, add(b.cx, __ddiv_rn(mul(t.c0x, L), 2.0))), mul(t.c0y, add(b.cy, __ddiv_rn(mul(t.c0y, L), 2.0)))),
                mul(t.c0z, add(b.cz, __ddiv_rn(mul(t.c0z, L), 2.0))));
    t.lo0 = add(add(mul(t.c0x, sub(b.cx, __ddiv_rn(mul(t.c0x, L), 2.0))), mul(t.c0y, sub(b.cy, __ddiv_rn(mul(t.c0y, L), 2.0)))),
                mul(t.c0z, sub(b.cz, __ddiv_rn(mul(t.c0z, L), 2.0))));
    t.hi1 = add(add(mul(t.c1x, add(b.cx, __ddiv_rn(mul(t.c1x, W), 2.0))), mul(t.c1y, add(b.cy, __ddiv_rn(mul(t.c1y, W), 2.0)))),
                mul(t.c1z, add(b.cz, __ddiv_rn(mul(t.c1z, W), 2.0))));
    t.lo1 = add(add(mul(t.c1x, sub(b.cx, __ddiv_rn(mul(t.c1x, W), 2.0))), mul(t.c1y, sub(b.cy, __ddiv_rn(mul(t.c1y, W), 2.0)))),
                mul(t.c1z, sub(b.cz, __ddiv_rn(mul(t.c1z, W), 2.0))));
    t.hi2 = add(add(mul(t.c2x, add(b.cx, mul(t.c2x, H))), mul(t.c2y, add(b.cy, mul(t.c2y, H)))),
                mul(t.c2z, add(b.cz, mul(t.c2z, H))));
    t.lo2 = add(add(mul(t.c2x, sub(b.cx, mul(t.c2x, 0.0))), mul(t.c2y, sub(b.cy, mul(t.c2y, 0.0)))),
                mul(t.c2z, sub(b.cz, mul(t.c2z, 0.0))));
    return t;
}

// cb:30-66 — strict inequalities, (a*x + b*y) + c*z evaluation order
__device__ __forceinline__ bool inside_box(const BoxTest& t, double x, double y, double z) {
    const double a0 = add(add(mul(t.c0x, x), mul(t.c0y, y)), mul(t.c0z, z));
    if (!(a0 < t.hi0) || !(a0 > t.lo0)) return false;
    const double a1 = add(add(mul(t.c1x, x), mul(t.c1y, y)), mul(t.c1z, z));
    if (!(a1 < t.hi1) || !(a1 > t.lo1)) return false;
    const double a2 = add(add(mul(t.c2x, x), mul(t.c2y, y)), mul(t.c2z, z));
    return (a2 < t.hi2) && (a2 > t.lo2);
}

// Candidate k of a cut object: one rotation by k*step about the SENSOR z-axis (closed form of the reference's k
// cumulative +1 degree rotations od/fs:263-265; identical feasible sets, xyz within ~1e-12 m — SURVEY.md §8).
struct YawBox {            // yaw-only box of candidate k
    double cx, cy;         // centre after rotation about the sensor
    double m00, m10;       // R_k = R0 . Rz(theta_k): [[m00, -m10', 0], [m10, m00, 0], [0, 0, 1]]
    double m01;            // = -(a*s + b*c)
};

__device__ __forceinline__ YawBox make_yaw_box(double c0x, double c0y, double a, double b, double c, double s) {
    YawBox y;
    y.cx = sub(mul(c, c0x), mul(s, c0y));
    y.cy = add(mul(s, c0x), mul(c, c0y));
    y.m00 = sub(mul(a, c), mul(b, s));
    y.m10 = add(mul(b, c), mul(a, s));
    y.m01 = -add(mul(a, s), mul(b, c));
    return y;
}

__device__ __forceinline__ Box yaw_box_to_box(const YawBox& y, double cz, double L, double W, double H) {
    Box b;
    b.cx = y.cx; b.cy = y.cy; b.cz = cz;
    b.m[0] = y.m00; b.m[1] = y.m01; b.m[2] = 0.0;
    b.m[3] = y.m10; b.m[4] = y.m00; b.m[5] = 0.0;
    b.m[6] = 0.0;   b.m[7] = 0.0;   b.m[8] = 1.0;
    b.length = L; b.width = W; b.height = H; b.reach = 0.0;
    return b;
}

// ------------------------------------------------------------------------------------------- utilities
__device__ __forceinline__ unsigned long long dbl_bits(double v) { return (unsigned long long)__double_as_longlong(v); }
__device__ __forceinline__ double bits_dbl(unsigned long long b) { return __longlong_as_double((long long)b); }

__device__ __forceinline__ float4 ldg_f4(const float4* p) { return __ldg(p); }

}  // namespace r3d
