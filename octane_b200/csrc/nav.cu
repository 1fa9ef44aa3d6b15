// nav.cu -- pixel displacement -> navigated u/v (m/s), packed to shorts.
// Replaces octnavcalcuda / oct_navpixel_uv_cuda / oct_haversine_cuda and the host loops of
// oct_pix2uv_cuda, src/oct_pix2uv_cuda.cu:13-221,265-370 (reference tree).
//
// Parity here is a rounding-reproduction problem: latitude / longitude are narrowed to float at the
// haversine call (:13,151,160), so the fp64 values feeding that narrowing have to be the reference's
// to the last bit.  The kernel therefore computes every fp64 quantity with the same CUDA math-library
// call on the same argument, and every piece of glue arithmetic with an explicitly rounded intrinsic
// (__dmul_rn / __dadd_rn / __fma_rn ...) in the association and with the fused multiply-adds the
// reference's own sm_100 build uses (read off its PTX), so that the compiler has no contraction
// choice left.  What is NOT reproduced is the reference's amount of work:
//
//   * the unmoved pixel (iv = 0, :99-100) sits on the fixed grid: sin / cos / pow(.,2) of its scan
//     angles depend on the column or on the row only.  A small setup kernel tabulates them per
//     column and per row (same calls, same arguments, same bits); the per-pixel kernel starts from the
//     tables.  In the Mercator grid the unmoved pixel's latitude depends on the row and its
//     longitude on the column only, so they are tabulated outright;
//   * the two haversines (:151,160) are called with one pair of equal arguments each, so one
//     squared sine is exactly +0 and drops out with the cosines it multiplies: 2 sin + 1 cos instead of
//     4 sin + 4 cos, 2 pow instead of 4;
//   * constants (pow(req,2) / pow(rpol,2), pow(H,2) - pow(req,2), sin / cos of the polar reference
//     latitude) are evaluated once, on the device, by the setup kernel.
//
// Per pixel that leaves 7 sin / cos, 12 pow, 8 sqrt, 4 atan, 2 atan2 of the reference's 16, 20, 8, 4, 2.
// Data movement: the reference fills int index arrays and double copies of u, v on the host
// (:308-321, 24 B/px over PCIe / managed memory); here (i, j) come from the thread index, the
// float flow is read directly and the four short planes are written (8 B in, 8 B out per pixel).
#include "kernels.cuh"

namespace octane {

namespace {

// The reference packs U_raw / V_raw (and U / V with -pd, and CTP) on the HOST: (short)(float) on
// x86-64 is cvttss2si to int32 followed by truncation to 16 bits, which wraps for |x| >= 32768
// (e.g. the -9999 fill value times 100) where the GPU's cvt.s16.f32 would saturate.
__device__ __forceinline__ short host_short(float x) { return (short)(int)x; }

constexpr double PI_NAV = 3.14159265359;             // :28
constexpr double PI_K = 3.14159265;                  // octnavcalcuda's caller: DTOR = pi / 180 with this pi
constexpr double DTOR = PI_K / 180.;
constexpr double DTOR2 = DTOR / 2.;
constexpr double EARTH_R = 6371000.00;               // :15
constexpr double FILL = -999.;

struct LatLon { double lat, lon; };                  // degrees; lat = FILL marks "not on the earth"

// ---- layout of the table buffer (doubles) ------------------------------------------------------
// [0, NT_HEAD) constants, then per-column arrays of nx, then per-row arrays of nrows
enum { K_H, K_HM2, K_RATIO, K_CTERM, K_LAM0, K_SINL, K_COSL, K_LON0R, K_LAT1R, NT_HEAD = 16 };
enum { CX_ANG, CX_SIN, CX_COS, CX_SIN2, CX_COS2, NT_COL };      // GOES; Mercator uses CX_ANG (x) and CX_SIN (lon0)
enum { RY_ANG, RY_SIN, RY_COS, RY_T, NT_ROW };                  // GOES; Mercator uses RY_ANG (y) and RY_SIN (lat0)

// scan angle of grid index k: evaluated in FLOAT with one fused multiply-add, then widened (:99-100)
__device__ __forceinline__ double grid_angle(int k, float scale, float offset)
{
    return (double)fmaf(scale, (float)k, offset);
}
// ... of the displaced position: (d * dt + k) * scale + offset in double, two fused multiply-adds (:102-103)
__device__ __forceinline__ double moved_angle(double d, double dt, int k, float scale, float offset)
{
    return __fma_rn(__fma_rn(d, dt, (double)k), (double)scale, (double)offset);
}

// GOES-R ABI fixed grid -> geodetic latitude / longitude (:108-139), from the sines and cosines of the two
// scan angles.  s2x = pow(sin x, 2), c2x = pow(cos x, 2), ty = pow(cos y, 2) + ratio * pow(sin y, 2).
__device__ __forceinline__ LatLon fixed_grid_inverse(double sinx, double cosx, double s2x, double c2x, double siny,
                                                     double cosy, double ty, const double* __restrict__ K)
{
    LatLon o = { FILL, FILL };
    const double H = K[K_H], ratio = K[K_RATIO];
    const double a = __fma_rn(c2x, ty, s2x);
    const double b = __dmul_rn(__dmul_rn(K[K_HM2], cosx), cosy);
    const double d = __fma_rn(__dmul_rn(a, -4.), K[K_CTERM], pow(b, 2));
    if (!(d >= 0)) return o;
    const double rs = __ddiv_rn(__dsub_rn(-b, __dsqrt_rn(d)), __dadd_rn(a, a));
    const double t = __dmul_rn(cosx, rs);
    const double sx = __dmul_rn(cosy, t);
    const double sy = __dmul_rn(sinx, -rs);
    const double sz = __dmul_rn(siny, t);
    const double hx = __dsub_rn(H, sx);
    const double e = __dadd_rn(pow(hx, 2), pow(sy, 2));
    if (sz == 0 || e <= 0 || hx == 0) return o;
    o.lat = __ddiv_rn(atan(__dmul_rn(__ddiv_rn(sz, __dsqrt_rn(e)), ratio)), DTOR);
    o.lon = __ddiv_rn(__dsub_rn(K[K_LAM0], atan(__ddiv_rn(sy, hx))), DTOR);
    return o;
}

// orthographic polar grid (metres) -> latitude / longitude (:34-67)
__device__ __forceinline__ LatLon polar_inverse(double x, double y, double R, bool pole, const double* __restrict__ K)
{
    LatLon o;
    const double rho = __dsqrt_rn(__fma_rn(x, x, __dmul_rn(y, y)));
    const double c = asin(__ddiv_rn(rho, R));
    const double sc = sin(c), cc = cos(c);
    if (pole) {
        o.lon = __dadd_rn(K[K_LON0R], atan2(x, -y));
    } else {
        const double den = __dsub_rn(__dmul_rn(__dmul_rn(rho, K[K_COSL]), cc), __dmul_rn(sc, __dmul_rn(K[K_SINL], y)));
        o.lon = __dadd_rn(K[K_LON0R], atan2(__dmul_rn(sc, x), den));
    }
    if (rho > 0.0000001)
        o.lat = asin(__dadd_rn(__dmul_rn(cc, K[K_SINL]), __ddiv_rn(__dmul_rn(__dmul_rn(sc, y), K[K_COSL]), rho)));
    else
        o.lat = K[K_LAT1R];
    o.lat = __ddiv_rn(o.lat, DTOR);
    o.lon = __ddiv_rn(o.lon, DTOR);
    return o;
}

// spherical Mercator (metres): the two coordinates separate (:70-87)
__device__ __forceinline__ double mercator_lat(double y, double R)
{
    const double t = atan(exp(__ddiv_rn(-y, R)));
    return __ddiv_rn(__dsub_rn(PI_NAV / 2., __dadd_rn(t, t)), DTOR);
}
__device__ __forceinline__ double mercator_lon(double x, double R, double lon1)
{
    return __ddiv_rn(__dadd_rn(__ddiv_rn(x, R), lon1), DTOR);
}

// great-circle distance along a parallel: both latitudes equal, so the squared sine of the latitude
// difference is exactly +0 (:13-25 with lat1 == lat2)
__device__ __forceinline__ double arc_zonal(float lat, float lon_a, float lon_b)
{
    const double dlon = lon_b - lon_a;                       // float subtraction, widened (the arguments are floats)
    const double cl = cos(__dmul_rn((double)lat, DTOR));
    const double a = __dmul_rn(__dmul_rn(cl, cl), pow(sin(__dmul_rn(DTOR2, dlon)), 2));
    const double c = atan2(__dsqrt_rn(a), __dsqrt_rn(__dsub_rn(1., a)));
    return __dmul_rn(__dadd_rn(c, c), EARTH_R);
}
// ... along a meridian: both longitudes equal, the cosine product multiplies an exact +0
__device__ __forceinline__ double arc_meridional(float lat_a, float lat_b)
{
    const double dlat = lat_b - lat_a;
    const double a = pow(sin(__dmul_rn(DTOR2, dlat)), 2);
    const double c = atan2(__dsqrt_rn(a), __dsqrt_rn(__dsub_rn(1., a)));
    return __dmul_rn(__dadd_rn(c, c), EARTH_R);
}

// ---- setup: constants and the per-column / per-row tables of the unmoved pixel -------------------
// BATCH: pair blockIdx.z, with navs[blockIdx.z] and its own table tstride doubles further on
template <bool BATCH>
__global__ void __launch_bounds__(128) k_nav_tables(NavParams nav0, int nx, int row0, int nrows, double* __restrict__ tab,
                                                    const NavParams* __restrict__ navs, size_t tstride)
{
    const NavParams nav = BATCH ? navs[blockIdx.z] : nav0;
    if (BATCH) tab += blockIdx.z * tstride;
    const int t = blockIdx.x * 128 + threadIdx.x;
    double* col = tab + NT_HEAD;
    double* row = col + (size_t)NT_COL * nx;
    const bool goes = !nav.dp && !nav.dm;
    // every thread needs the axial ratio for its own entry; thread 0 also publishes the constants
    const double H = __dadd_rn(nav.pph, nav.req);
    const double req2 = pow(nav.req, 2);
    const double ratio = __ddiv_rn(req2, pow(nav.rpol, 2));
    if (t == 0) {
        tab[K_H] = H;
        tab[K_HM2] = __dmul_rn(H, -2.);
        tab[K_RATIO] = ratio;
        tab[K_CTERM] = __dsub_rn(pow(H, 2), req2);
        tab[K_LAM0] = nav.lam0;
        const double lat1r = __dmul_rn((double)nav.lat1, DTOR);
        tab[K_LAT1R] = lat1r;
        tab[K_SINL] = sin(lat1r);
        tab[K_COSL] = cos(lat1r);
        tab[K_LON0R] = __dmul_rn((double)nav.lon0, DTOR);
    }
    if (t < nx) {
        const double x = grid_angle(t + nav.minX, nav.xScale, nav.xOffset);
        col[(size_t)CX_ANG * nx + t] = x;
        if (goes) {
            const double s = sin(x), c = cos(x);
            col[(size_t)CX_SIN * nx + t] = s;
            col[(size_t)CX_COS * nx + t] = c;
            col[(size_t)CX_SIN2 * nx + t] = pow(s, 2);
            col[(size_t)CX_COS2 * nx + t] = pow(c, 2);
        } else if (nav.dm) {
            col[(size_t)CX_SIN * nx + t] = mercator_lon(x, (double)nav.R, (double)nav.lon1);
        }
    } else if (t - nx < nrows) {
        const int j = t - nx;
        const double y = grid_angle(j + row0 + nav.minY, nav.yScale, nav.yOffset);
        row[(size_t)RY_ANG * nrows + j] = y;
        if (goes) {
            const double s = sin(y), c = cos(y);
            row[(size_t)RY_SIN * nrows + j] = s;
            row[(size_t)RY_COS * nrows + j] = c;
            row[(size_t)RY_T * nrows + j] = __fma_rn(ratio, pow(s, 2), pow(c, 2));
        } else if (nav.dm) {
            row[(size_t)RY_SIN * nrows + j] = mercator_lat(y, (double)nav.R);
        }
    }
}

// ---- per pixel: a block owns 128 columns x NAV_ROWS rows; a thread walks one column down --------
constexpr int NAV_ROWS = 8;

// BATCH: pair blockIdx.z, with navs[blockIdx.z], its table tstride doubles and its planes n values further on
template <int GRID, bool BATCH>     // GRID: 0 GOES fixed grid, 1 polar, 2 Mercator
__global__ void __launch_bounds__(128)
k_pix2uv(NavParams nav0, const float* __restrict__ u, const float* __restrict__ v, int nx, int row0, int nrows,
         const double* __restrict__ tab, short* __restrict__ ur, short* __restrict__ vr, short* __restrict__ ur2,
         short* __restrict__ vr2, const NavParams* __restrict__ navs, size_t tstride, size_t n)
{
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= nx) return;
    const NavParams nav = BATCH ? navs[blockIdx.z] : nav0;
    if (BATCH) {
        const size_t po = blockIdx.z * n;
        tab += blockIdx.z * tstride;
        u += po; v += po; ur += po; vr += po; ur2 += po; vr2 += po;
    }
    const double* col = tab + NT_HEAD;
    const double* row = col + (size_t)NT_COL * nx;
    const double dt = nav.t2 - nav.t1;
    const int xi = i + nav.minX;
    // this column's share of the unmoved pixel
    const double x0 = col[(size_t)CX_ANG * nx + i];
    double sx0 = 0., cx0 = 0., s2x0 = 0., c2x0 = 0., lon0m = 0.;
    if (GRID == 0) {
        sx0 = col[(size_t)CX_SIN * nx + i]; cx0 = col[(size_t)CX_COS * nx + i];
        s2x0 = col[(size_t)CX_SIN2 * nx + i]; c2x0 = col[(size_t)CX_COS2 * nx + i];
    } else if (GRID == 2) {
        lon0m = col[(size_t)CX_SIN * nx + i];
    }
    const bool pole = nav.lat1 > 89.9999;
    const int j_end = min(nrows, (int)(blockIdx.y + 1) * NAV_ROWS);
    for (int j = blockIdx.y * NAV_ROWS; j < j_end; j++) {
        const size_t l = (size_t)j * nx + i;
        const float uf = u[l], vf = v[l];
        const short u100 = host_short(100 * uf), v100 = host_short(100 * vf);       // :335-336
        ur2[l] = u100;
        vr2[l] = v100;
        if (nav.pixuv) {                                                             // :348-356
            ur[l] = u100;
            vr[l] = v100;
            continue;
        }
        if (!((double)uf > -9998.)) {                                                // fill value, :213-218
            ur[l] = (short)(-32768);
            vr[l] = (short)(-32768);
            continue;
        }
        const int yi = j + row0 + nav.minY;
        const double du = __ddiv_rn((double)uf, dt), dv = __ddiv_rn((double)vf, dt);   // pixels per second, :187-188
        const double y0 = row[(size_t)RY_ANG * nrows + j];
        LatLon p0, p1;
        bool limb = false;
        if (GRID == 0) {
            limb = __fma_rn(x0, x0, __dmul_rn(y0, y0)) > 0.021;                      // :105,144
            p0 = fixed_grid_inverse(sx0, cx0, s2x0, c2x0, row[(size_t)RY_SIN * nrows + j], row[(size_t)RY_COS * nrows + j],
                                    row[(size_t)RY_T * nrows + j], tab);
            const double x1 = moved_angle(du, dt, xi, nav.xScale, nav.xOffset);
            const double y1 = moved_angle(dv, dt, yi, nav.yScale, nav.yOffset);
            const double s1 = sin(x1), c1 = cos(x1), sy1 = sin(y1), cy1 = cos(y1);
            p1 = fixed_grid_inverse(s1, c1, pow(s1, 2), pow(c1, 2), sy1, cy1,
                                    __fma_rn(tab[K_RATIO], pow(sy1, 2), pow(cy1, 2)), tab);
        } else if (GRID == 1) {
            p0 = polar_inverse(x0, y0, (double)nav.R, pole, tab);
            p1 = polar_inverse(moved_angle(du, dt, xi, nav.xScale, nav.xOffset),
                               moved_angle(dv, dt, yi, nav.yScale, nav.yOffset), (double)nav.R, pole, tab);
        } else {
            p0.lat = row[(size_t)RY_SIN * nrows + j];
            p0.lon = lon0m;
            p1.lat = mercator_lat(moved_angle(dv, dt, yi, nav.yScale, nav.yOffset), (double)nav.R);
            p1.lon = mercator_lon(moved_angle(du, dt, xi, nav.xScale, nav.xOffset), (double)nav.R, (double)nav.lon1);
        }
        double ums = 0., vms = 0.;
        if (!(p0.lat < -998 || p1.lat < -998 || limb)) {                            // :144-148
            const float lat0 = (float)p0.lat, lon0 = (float)p0.lon;                 // the haversine's float parameters
            const double east = arc_zonal(lat0, lon0, (float)p1.lon);
            ums = __ddiv_rn(p1.lon >= p0.lon ? east : -east, dt);                    // :152-158
            const double north = arc_meridional(lat0, (float)p1.lat);
            vms = __ddiv_rn(p1.lat >= p0.lat ? north : -north, dt);                  // :161-167
        }
        ur[l] = (short)(100 * ums);                                                   // :196-197
        vr[l] = (short)(100 * vms);
    }
}

// CTP pack of oct_optical_flow.cc:71-88
__global__ void __launch_bounds__(256) k_ctp_pack(const float* __restrict__ cth, short* __restrict__ ctp, size_t n, int ir)
{
    for (size_t k = (size_t)blockIdx.x * 256 + threadIdx.x; k < n; k += (size_t)gridDim.x * 256)
        ctp[k] = ir ? host_short((cth[k] - 300) * 100) : host_short(cth[k]);
}

}  // namespace

size_t pix2uv_table_doubles(int nx, int nrows)
{
    return (size_t)NT_HEAD + (size_t)NT_COL * nx + (size_t)NT_ROW * nrows;
}

int launch_pix2uv(const NavParams& np, const float* u, const float* v, int nx, int row0, int nrows, double* tab,
                  short* U, short* V, short* Uraw, short* Vraw, cudaStream_t st)
{
    if (nx <= 0 || nrows <= 0) return 0;
    k_nav_tables<false><<<(nx + nrows + 127) / 128, 128, 0, st>>>(np, nx, row0, nrows, tab, nullptr, 0);
    const dim3 grid((nx + 127) / 128, (nrows + NAV_ROWS - 1) / NAV_ROWS);
    if (np.dp)      k_pix2uv<1, false><<<grid, 128, 0, st>>>(np, u, v, nx, row0, nrows, tab, U, V, Uraw, Vraw, nullptr, 0, 0);
    else if (np.dm) k_pix2uv<2, false><<<grid, 128, 0, st>>>(np, u, v, nx, row0, nrows, tab, U, V, Uraw, Vraw, nullptr, 0, 0);
    else            k_pix2uv<0, false><<<grid, 128, 0, st>>>(np, u, v, nx, row0, nrows, tab, U, V, Uraw, Vraw, nullptr, 0, 0);
    return 2;
}

int launch_pix2uv_batch(const NavParams& np0, const NavParams* d_navs, int npairs, const float* u, const float* v, int nx,
                        int ny, double* tab, short* U, short* V, short* Uraw, short* Vraw, cudaStream_t st)
{
    if (nx <= 0 || ny <= 0 || npairs <= 0) return 0;
    const size_t ts = pix2uv_table_doubles(nx, ny), n = (size_t)nx * ny;
    k_nav_tables<true><<<dim3((nx + ny + 127) / 128, 1, npairs), 128, 0, st>>>(np0, nx, 0, ny, tab, d_navs, ts);
    const dim3 grid((nx + 127) / 128, (ny + NAV_ROWS - 1) / NAV_ROWS, npairs);
    if (np0.dp)      k_pix2uv<1, true><<<grid, 128, 0, st>>>(np0, u, v, nx, 0, ny, tab, U, V, Uraw, Vraw, d_navs, ts, n);
    else if (np0.dm) k_pix2uv<2, true><<<grid, 128, 0, st>>>(np0, u, v, nx, 0, ny, tab, U, V, Uraw, Vraw, d_navs, ts, n);
    else             k_pix2uv<0, true><<<grid, 128, 0, st>>>(np0, u, v, nx, 0, ny, tab, U, V, Uraw, Vraw, d_navs, ts, n);
    return 2;
}

void launch_ctp_pack(const float* cth, short* ctp, size_t n, int ir, cudaStream_t st)
{
    if (!n) return;
    size_t grid = (n + 255) / 256;
    if (grid > 148 * 32) grid = 148 * 32;
    k_ctp_pack<<<(unsigned)grid, 256, 0, st>>>(cth, ctp, n, ir);
}

}  // namespace octane
