// build.cu -- linearised data term + robust smoothness weights -> the 2x2-block
// 5-point system of one inner iteration, matrix-free.
// Replaces the body of the inner loop of octConjugateGradient,
// src/oct_variational_optical_flow.cu:611-1097 (reference tree): same
// neighbourhoods, same warp/clamp rules, same float/double promotion points.
// Instead of CSR arrays (12 nnz x 12 B per pixel) it stores 5 coefficients per
// pixel (the 2x2 diagonal block and the couplings to i+1 and j+1; the other two
// couplings are their neighbours' by symmetry), the right-hand side, and seeds
// the PCG scalars (r0 = b because x0 = 0).
#include <stdlib.h>

#include "kernels.cuh"

namespace octane {

#define BUILD_ROWS 64
#ifndef OCTANE_BUILD_OCC
#define OCTANE_BUILD_OCC 4      // resident blocks of 256 threads per SM the register allocation aims at (64 registers,
                                // no spills; measured 2 / 3 / 4: profiles/r02_build_occ_ab.txt)
#endif

__device__ __forceinline__ float jsq(float x) { return x * x; }

// ---- exact shortcuts for the reference's mixed-precision expressions ----------------------
// The reference's promotion rules force fp64 divisions where the operands are floats; each
// helper below returns the SAME float, bit for bit, with less work (CPU proof by enumeration:
// tests/test_abi_host.py::test_exact_division_shortcuts).

// float(1. / double(s)) for a float s.  1/s cannot fall within 2^-49 (relative) of a float
// rounding boundary unless it is exactly on one (s times a 25-bit midpoint would have to be
// within 1 of a power of two), so rounding to double first never changes the float result:
// it is the correctly rounded single-precision reciprocal.
__device__ __forceinline__ float recip_f(float s) { return __frcp_rn(s); }

// double(x) / a for a float x and a double constant a with y = RN(1/a): one Markstein
// correction step after the multiply gives the correctly rounded quotient.
__device__ __forceinline__ double div_const(float x, double a, double y)
{
    const double xd = (double)x;
    const double q = xd * y;
    const double r = fma(-q, a, xd);
    return fma(r, y, q);
}

// oct_PSI_smooth_cu, :72-88: float(1. / double(sqrtf(float(double(x) + 1E-6))))
__device__ __forceinline__ float psi_smooth(float x)
{
    const float s = (float)(x + 1E-6);
    return recip_f(sqrtf(s));
}
// oct_PSI_data_cu, :90-108: float(1. / sqrt(double(x) + 1E-6))
__device__ __forceinline__ float psi_data(float x)
{
    float answer;
    answer = 1. / (sqrt(x + 1E-6));
    return answer;
}
// :57-71
__device__ __forceinline__ float binterp(float p1, float p2, float p3, float p4, float f11, float f21, float f12,
                                         float f22)
{
    return p3 * ((p1)*f11 + (p2)*f21) + p4 * ((p1)*f12 + (p2)*f22);
}
__device__ __forceinline__ float gather(const float* __restrict__ q, int pitch, float p1, float p2, float p3, float p4)
{
    return binterp(p1, p2, p3, p4, __ldg(q), __ldg(q + 1), __ldg(q + pitch), __ldg(q + pitch + 1));
}

// GNC stage of a launch (:604-606): al1 = 1 - 0.5*gnc.  Every coefficient is
// al1*(quadratic term) + (1-al1)*(robust term) evaluated in double and cast to float; with
// al1 == 1 the robust term is multiplied by zero and with al1 == 0 the quadratic one is, so
// those launches skip it (x*1 + y*0 == x exactly for finite y; the robust weights are finite
// because psi(x) = 1/sqrt(x + 1e-6) with x >= 0).
enum { GNC_QUADRATIC = 0, GNC_BLEND = 1, GNC_ROBUST = 2 };

// SPLIT: the batched instance, whose six image fields (g1, g1x, g1y, g2, g2x, g2y) of pair blockIdx.z lie `is` floats
// after pair 0's, every other plane ps floats; the single-pair instance ignores `is`.
template <int MODE, int OCC, bool SPLIT>
__global__ void __launch_bounds__(256, OCC)
k_build(LevelFields f, PcgBuffers b, Geom g, int ja, int jb, int da, int db, BuildParams bp, int halo_check, size_t ps,
        size_t is)
{
    constexpr bool ROBUST = (MODE != GNC_QUADRATIC);   // robust terms needed
    constexpr bool QUAD = (MODE != GNC_ROBUST);        // quadratic terms needed
    __shared__ double red[2 * 32];
    const int ii = blockIdx.x * 32 + threadIdx.x;
    const int xi = g.nx, yi = g.ny, pitch = g.pitch;
    const double alpha = bp.alpha, ralpha = bp.ralpha, lambdadalpha = bp.lambdadalpha, al1 = bp.al1;
    const float lambdac = bp.lambdac;
    double acc[2] = { 0.0, 0.0 };
    const size_t po = (size_t)blockIdx.z * ps;         // pair blockIdx.z: every plane is ps floats further on
    const size_t pi = SPLIT ? (size_t)blockIdx.z * is : po;   // ... every image field pi floats

    // a block covers 32 columns x BUILD_ROWS rows, 8 rows at a time
    for (int jt = 0; jt < BUILD_ROWS; jt += 8) {
    const int jj = ja + blockIdx.y * BUILD_ROWS + jt + threadIdx.y;
    if (ii < xi && jj < jb) {
        // mirror-without-repeat neighbours (:629-652)
        const int im = (ii == 0) ? ii + 1 : ii - 1;
        const int ip = (ii == xi - 1) ? ii - 1 : ii + 1;
        const int jm = (jj == 0) ? jj + 1 : jj - 1;
        const int jp = (jj == yi - 1) ? jj - 1 : jj + 1;
        const size_t r0 = g.at(0, jj) + po;
        const float* u0 = f.u + r0;
        const float* v0 = f.v + r0;
        const int dm = (jm - jj) * pitch, dp = (jp - jj) * pitch;     // +-pitch
        const float up0p0 = u0[ii], up1p0 = u0[ip], um1p0 = u0[im], up0p1 = u0[dp + ii], up0m1 = u0[dm + ii];
        const float vp0p0 = v0[ii], vp1p0 = v0[ip], vm1p0 = v0[im], vp0p1 = v0[dp + ii], vp0m1 = v0[dm + ii];

        float psis3 = 0.f, psis4 = 0.f, psistot = 0.f, psisnmiu = 0.f, psisnmiv = 0.f;
        if (ROBUST) {
            const float up1p1 = u0[dp + ip], up1m1 = u0[dm + ip], um1p1 = u0[dp + im], um1m1 = u0[dm + im];
            const float vp1p1 = v0[dp + ip], vp1m1 = v0[dm + ip], vm1p1 = v0[dp + im], vm1m1 = v0[dm + im];
            // :680-683 (0.25 * x is exact in either precision, so the reference's detour through double is dropped)
            float Uip1 = jsq(up1p0 - up0p0) + jsq(0.25f * ((up1p1 - up1m1) + (up0p1 - up0m1))) + jsq(vp1p0 - vp0p0) + jsq(0.25f * ((vp1p1 - vp1m1) + (vp0p1 - vp0m1)));
            float Uim1 = jsq(up0p0 - um1p0) + jsq(0.25f * ((um1p1 - um1m1) + (up0p1 - up0m1))) + jsq(vp0p0 - vm1p0) + jsq(0.25f * ((vm1p1 - vm1m1) + (vp0p1 - vp0m1)));
            float Ujp1 = jsq(up0p1 - up0p0) + jsq(0.25f * ((up1p1 - um1p1) + (up1p0 - um1p0))) + jsq(vp0p1 - vp0p0) + jsq(0.25f * ((vp1p1 - vm1p1) + (vp1p0 - vm1p0)));
            float Ujm1 = jsq(up0p0 - up0m1) + jsq(0.25f * ((up1m1 - um1m1) + (up1p0 - um1p0))) + jsq(vp0p0 - vp0m1) + jsq(0.25f * ((vp1m1 - vm1m1) + (vp1p0 - vm1p0)));
            // :714-724
            float psis1 = psi_smooth(Uim1);
            float psis2 = psi_smooth(Ujm1);
            psis3 = psi_smooth(Uip1);
            psis4 = psi_smooth(Ujp1);
            psistot = psis1 + psis2 + psis3 + psis4;
            psisnmiu = psis1 * (um1p0) + psis2 * (up0m1) + psis3 * (up1p0) + psis4 * (up0p1);
            psisnmiv = psis1 * (vm1p0) + psis2 * (vp0m1) + psis3 * (vp1p0) + psis4 * (vp0p1);
        }
        const float psistotq = 4.;
        const float psisnmiuq = um1p0 + up0m1 + up1p0 + up0p1;
        const float psisnmivq = vm1p0 + vp0m1 + vp1p0 + vp0p1;

        float vr1 = 0, vr2 = 0, vr4 = 0, vr5 = 0, vr6 = 0, intcomp = 0;
        float vr12 = 0, vr22 = 0, vr42 = 0, vr52 = 0, vr62 = 0, intcomp2 = 0;
        // warped position with clamp, :732-745
        bool bc2 = false, bc3 = false;
        float iv = (float)(ii + up0p0);
        if (iv < 0) { iv = 0; bc2 = true; }
        if (iv >= xi) { iv = xi - 1; bc2 = true; }
        float jv = (float)(jj + vp0p0);
        if (jv < 0) { jv = 0; bc3 = true; }
        if (jv >= yi) { jv = yi - 1; bc3 = true; }
        int iv1 = int(iv);
        int jv1 = int(jv);
        if (iv1 == xi - 1) iv1 = xi - 2;
        if (jv1 == yi - 1) jv1 = yi - 2;
        if (halo_check) {     // banded run: rows jv1, jv1+1 must carry valid second derivatives
            const int vlo = (g.jlo() == 0) ? 0 : g.jlo() + 4, vhi = (g.jhi() == yi) ? yi : g.jhi() - 4;
            if (jv1 < vlo || jv1 + 1 >= vhi) {
                atomicOr(&b.scal->halo_err, 1);
                jv1 = min(max(jv1, g.jlo()), g.jhi() - 2);
            }
        }
        const size_t c1 = g.at(iv1, jv1) + po;
        const size_t c1i = SPLIT ? g.at(iv1, jv1) + pi : c1;
        const size_t l = r0 + ii;
        const size_t li = SPLIT ? g.at(0, jj) + pi + ii : l;
        // bilinear weights, :57-65; x2-x1 == y2-y1 == 1.0f exactly, so the divisions are dropped
        const float x1 = iv1, x2 = iv1 + 1, y1 = jv1, y2 = jv1 + 1;
        const float p1 = x2 - iv;
        const float p2 = iv - x1;
        const float p3 = y2 - jv;
        const float p4 = jv - y1;
        for (int c = 0; c < bp.nchan; c++) {
            const size_t off = (size_t)c * g.plane;
            const size_t oc = off + c1, oci = off + c1i;
            float g2 = gather(f.g2 + oci, pitch, p1, p2, p3, p4);
            float Ix = gather(f.g2x + oci, pitch, p1, p2, p3, p4);
            float Iy = gather(f.g2y + oci, pitch, p1, p2, p3, p4);
            float Ixx = gather(f.g2xx + oc, pitch, p1, p2, p3, p4);
            float Ixy = gather(f.g2xy + oc, pitch, p1, p2, p3, p4);
            float Iyy = gather(f.g2yy + oc, pitch, p1, p2, p3, p4);
            // derivative zeroing where the warp was clamped, :768-779
            if (bc2) { Ix = 0.; Ixx = 0.; Ixy = 0.; }
            if (bc3) { Iy = 0.; Ixy = 0.; Iyy = 0.; }
            // :782-828
            float It = g2 - __ldg(f.g1 + off + li);
            float Ixt = Ix - __ldg(f.g1x + off + li);
            float Iyt = Iy - __ldg(f.g1y + off + li);
            float IxIx = Ix * Ix;
            float IyIy = Iy * Iy;
            float IxxIxx = Ixx * Ixx;
            float IxyIxy = Ixy * Ixy;
            float IyyIyy = Iyy * Iyy;
            float na, nb, nc;
            if (bp.dozim) {
                na = 1. / (IxIx + IyIy + 1.);
                nb = 1. / (IxxIxx + IxyIxy + 1.);
                nc = 1. / (IxyIxy + IyyIyy + 1.);
            } else {
                na = 1.; nb = 1.; nc = 1.;
            }
            if (ROBUST) {
                intcomp += na * It * It;
                intcomp2 += (nb * Ixt * Ixt + nc * Iyt * Iyt);
            }
            vr1 += (na * IxIx);
            vr12 += (nb * IxxIxx + nc * IxyIxy);
            vr2 += na * Ix * Iy;
            vr22 += (nb * Ixx * Ixy + nc * Iyy * Ixy);
            vr4 += (na * IyIy);
            vr42 += ((nb * IxyIxy + nc * IyyIyy));
            float natIt = -na * It;
            float nbtIxt = nb * Ixt;
            float nctIyt = nc * Iyt;
            vr5 += natIt * Ix;
            vr52 += -(nbtIxt * Ixx + nctIyt * Ixy);
            vr6 += natIt * Iy;
            vr62 += -(nbtIxt * Ixy + nctIyt * Iyy);
        }
        // right-hand-side hint term, :1087-1092
        const float uvt = f.uh ? __ldg(f.uh + l) : 0.f;
        const float vvt = f.vh ? __ldg(f.vh + l) : 0.f;
        const float val2u = lambdac * (up0p0 - uvt);
        const float val2v = lambdac * (vp0p0 - vvt);
        // :831-864.  Quadratic (q*) and robust (r*) halves of every entry, then the GNC blend.
        double q1 = 0., q2 = 0., q4 = 0., qbu = 0., qbv = 0.;
        float r1 = 0.f, r2 = 0.f, r4 = 0.f, rbu = 0.f, rbv = 0.f;
        if (QUAD) {
            q1 = div_const(vr1, alpha, ralpha) + lambdadalpha * (vr12) + lambdac + psistotq;
            q2 = div_const(vr2, alpha, ralpha) + lambdadalpha * vr22;
            q4 = div_const(vr4, alpha, ralpha) + lambdadalpha * vr42 + lambdac + psistotq;
            qbu = div_const(vr5, alpha, ralpha) + lambdadalpha * vr52 - val2u + psisnmiuq - psistotq * up0p0;
            qbv = div_const(vr6, alpha, ralpha) + lambdadalpha * vr62 - val2v + psisnmivq - psistotq * vp0p0;
        }
        if (ROBUST) {
            float psid = div_const(psi_data(intcomp), alpha, ralpha);
            float psid2 = lambdadalpha * psi_data(intcomp2);
            r1 = psid * (vr1) + psid2 * vr12 + lambdac + psistot;
            r2 = psid * (vr2) + psid2 * vr22;
            r4 = psid * (vr4) + psid2 * vr42 + lambdac + psistot;
            rbu = psid * (vr5) + psid2 * vr52 - val2u + psisnmiu - psistot * up0p0;
            rbv = psid * (vr6) + psid2 * vr62 - val2v + psisnmiv - psistot * vp0p0;
        }
        float a1, a2, a4, a7, a8, bu, bv;
        if (MODE == GNC_QUADRATIC) {
            a1 = (float)q1; a2 = (float)q2; a4 = (float)q4; bu = (float)qbu; bv = (float)qbv;
            a7 = -1.f; a8 = -1.f;
        } else if (MODE == GNC_ROBUST) {
            a1 = r1; a2 = r2; a4 = r4; bu = rbu; bv = rbv;
            a7 = -psis3; a8 = -psis4;
        } else {
            a1 = (float)((al1) * (q1) + (1 - al1) * (r1));
            a2 = (float)((al1) * (q2) + (1 - al1) * (r2));
            a4 = (float)((al1) * (q4) + (1 - al1) * (r4));
            a7 = (float)(-1 * (al1 + (1 - al1) * (psis3)));
            a8 = (float)(-1 * (al1 + (1 - al1) * (psis4)));
            bu = (float)(al1 * (qbu) + (1. - al1) * (rbu));
            bv = (float)(al1 * (qbv) + (1 - al1) * (rbv));
        }
        // Only the couplings to i+1 and j+1 are stored: a5(i,j) == a7(i-1,j) and
        // a6(i,j) == a8(i,j-1) bit for bit (same expression, two commuted additions), and at a
        // mirrored edge a5 == a7 (a6 == a8), so the boundary merging of :929-1077 -- the weight
        // of an absent neighbour is added to the opposite one -- is a doubling that the PCG
        // kernels apply on the fly (kernels.cuh, PcgBuffers).
        b.coef[C_A1][l] = a1;
        b.coef[C_A2][l] = a2;
        b.coef[C_A4][l] = a4;
        b.coef[C_W][l] = a7;
        b.coef[C_N][l] = a8;
        b.ru[l] = bu;
        b.rv[l] = bv;
        if (jj >= da && jj < db) {
            // residc = b.b (:1126); rkTzk = b.z with z = (1/M) b (:1115-1117,1157)
            const float mu = recip_f(a1), mv = recip_f(a4);
            const float zu = mu * bu, zv = mv * bv;
            acc[0] += (double)(bu * bu) + (double)(bv * bv);
            acc[1] += (double)(bu * zu) + (double)(bv * zv);
        }
    }
    }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        const unsigned nblocks = gridDim.x * gridDim.y, bid = blockIdx.y * gridDim.x + blockIdx.x;
        double* part = b.partials + (size_t)blockIdx.z * 2 * nblocks;   // one region per pair
        part[bid] = acc[0];
        part[(size_t)nblocks + bid] = acc[1];
    }
}

// second stage of the build's dot products (fixed order) + PCG scalar seeding:
// residc = b.b, rkTzk = b.z; stop rule already true -> no iterations (:1131).  Pair blockIdx.z: its partials and
// its scalars b.scal[blockIdx.z].
__global__ void __launch_bounds__(1024) k_build_finish(PcgBuffers b, unsigned nblocks, float tol)
{
    __shared__ double red[2 * 32];
    double acc[2] = { 0.0, 0.0 };
    const double* part = b.partials + (size_t)blockIdx.z * 2 * nblocks;
    for (unsigned i = threadIdx.x; i < nblocks; i += 1024) {
        acc[0] += part[i];
        acc[1] += part[(size_t)nblocks + i];
    }
    block_sum<2>(acc, red);
    if (b.p2p.world > 1) p2p_allreduce<2>(b.p2p, P2P_BUILD, acc, &b.scal->comm_err);
    if (threadIdx.x == 0 && b.defer) {
        b.pending[0] = acc[0];
        b.pending[1] = acc[1];
    } else if (threadIdx.x == 0) {
        PcgScalars* s = b.scal + blockIdx.z;
        s->rr = (float)acc[0];
        s->rz = (float)acc[1];
        s->rz_old = 0.f;
        s->pAp = 0.f;
        s->alpha = 0.f;
        s->tol = tol;
        s->its = 0;
        s->done = !((float)acc[0] > tol);
    }
}

void launch_build(const LevelFields& f, const PcgBuffers& b, const Geom& g, int ja, int jb, int da, int db,
                  const BuildParams& bp, int halo_check, cudaStream_t st, int npairs, size_t ps, size_t is)
{
    dim3 grid((g.nx + 31) / 32, (jb - ja + BUILD_ROWS - 1) / BUILD_ROWS, npairs), block(32, 8);
#define LAUNCH_BUILD(MODE)                                                                                               \
    do {                                                                                                                 \
        if (npairs > 1) k_build<MODE, OCTANE_BUILD_OCC, true><<<grid, block, 0, st>>>(f, b, g, ja, jb, da, db, bp, halo_check, ps, is); \
        else k_build<MODE, OCTANE_BUILD_OCC, false><<<grid, block, 0, st>>>(f, b, g, ja, jb, da, db, bp, halo_check, ps, is); \
    } while (0)
    if (bp.al1 == 1.0)      LAUNCH_BUILD(GNC_QUADRATIC);
    else if (bp.al1 == 0.0) LAUNCH_BUILD(GNC_ROBUST);
    else                    LAUNCH_BUILD(GNC_BLEND);
#undef LAUNCH_BUILD
    k_build_finish<<<dim3(1, 1, npairs), 1024, 0, st>>>(b, grid.x * grid.y, bp.tol);
}

int build_partial_blocks(const Geom& g, int nrows)
{
    return ((g.nx + 31) / 32) * ((nrows + BUILD_ROWS - 1) / BUILD_ROWS);
}

}  // namespace octane
