// pyramid.cu -- Gaussian pyramid (blur + decimate), 4th-order gradients and
// bicubic flow prolongation.  Replaces the device functions fill_GK, convh,
// convv, zoom_out, oct_compgrad_cu, zoom_in, oct_bicubic_cu of
// src/oct_variational_optical_flow.cu:208-466 (reference tree).
#include <stdint.h>

#include "kernels.cuh"

namespace octane {

// ---- Gaussian taps, :208-228 (one thread, same expression order) -----------
__global__ void k_fill_gk(float* GK, float factor, int R)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    float sigma, r, s;
    sigma = 0.6 * sqrt(1.0 / (factor * factor) - 1.0);
    s = 2.0 * sigma * sigma;
    float sum = 0.0;
    for (int x = -R; x <= R; x++) {
        r = x;
        GK[x + R] = (exp(-(r * r) / s)) / (3.14159265358979323846 * s);
        sum += GK[x + R];
    }
    for (int i = 0; i < 2 * R + 1; ++i) GK[i] /= sum;
}

// ---- fused convh + convv + zoom_out, :312-408 --------------------------------
// The reference blurs the whole full-resolution plane (taps kk in [-R,R): the +R
// tap is dropped, :322,344) and then samples it with a bicubic at integer
// coordinates, which is an exact decimation (oct_cell_cu(v,0) == v[1], :236).
// Here each output pixel evaluates the separable blur only where it is sampled,
// with the same tap order (horizontal sums first, then the vertical sum), so
// the result is bit-identical while the full-res blurred planes never exist.
// A block computes a (TX x TY) output tile: the horizontal sums for the
// TY-tile's (TY-1)*step + 2R source rows are staged in shared memory.
template <int TX, int TY>
__global__ void __launch_bounds__(TX* TY)
k_blur_decimate(const float* __restrict__ src, Geom gs, float* __restrict__ dst, Geom gd,
                int ja, int jb, float factor, const float* __restrict__ GK, int R, float scale, int nc, size_t ps)
{
    extern __shared__ float sm[];
    float* gk = sm;                  // 2R+1 taps
    float* hs = sm + 2 * R + 1;      // [nrow_h][TX] horizontal sums
    const int tid = threadIdx.y * TX + threadIdx.x;
    for (int t = tid; t < 2 * R + 1; t += TX * TY) gk[t] = GK[t];
    const int ii = blockIdx.x * TX + threadIdx.x;
    const int jj0 = ja + blockIdx.y * TY;
    // Reference quirk kept for parity: zoom_out reads the blurred plane without a channel
    // offset (:406), so every coarse-level channel is channel 0's blurred, decimated image.
    // blockIdx.z = pair * nc + channel; pairs are ps floats apart in both planes.
    const unsigned pair = blockIdx.z / nc;
    src += pair * ps;
    dst += (size_t)(blockIdx.z - pair * nc) * gd.plane + pair * ps;
    const int i2 = (int)(ii / factor);                          // :369
    const int jj_last = min(jj0 + TY, jb) - 1;
    const int jsrc0 = (int)(jj0 / factor) - R;                  // first source row of the tile
    const int jsrc1 = (int)(jj_last / factor) + R;              // one past the last
    const int nrow_h = jsrc1 - jsrc0;
    __syncthreads();
    if (ii < gd.nx) {
        for (int rr = threadIdx.y; rr < nrow_h; rr += TY) {
            int js = clampi(jsrc0 + rr, gs.ny);                 // global clamp-to-edge
            js = min(max(js, gs.jlo()), gs.jhi() - 1);          // stay inside the local band
            const float* row = src + gs.at(0, js);
            float wsum = 0;
            for (int kk = -R; kk < R; ++kk)
                wsum = fmaf(gk[kk + R], __ldg(row + clampi(i2 + kk, gs.nx)), wsum);
            hs[rr * TX + threadIdx.x] = wsum;
        }
    }
    __syncthreads();
    const int jj = jj0 + threadIdx.y;
    if (ii < gd.nx && jj < jb) {
        const int j2 = (int)(jj / factor);
        // rows j2-R .. j2+R-1; a clamped source row repeats the clamped row's sum,
        // exactly as convv reading the clamped row of the convh output (:346-347)
        float wsum = 0;
        for (int kk = -R; kk < R; ++kk) {
            int rr = (j2 + kk) - jsrc0;
            wsum = fmaf(gk[kk + R], hs[rr * TX + threadIdx.x], wsum);
        }
        dst[gd.at(ii, jj)] = wsum * scale;
    }
}

// ---- 4th-order central differences, :411-449 ---------------------------------
// numerator in double (the literal 8. promotes it), divided by 12.0, stored float.
__device__ __forceinline__ double grad_num(float p2, float p1, float m1, float m2) { return (-p2 + 8. * p1 - 8. * m1 + m2); }

// x / 12.0, correctly rounded, without the division: y = RN(1/12) has a relative error of 2^-54, so q = RN(x*y) is
// within one ulp of the quotient, the residual r = x - 12 q is exact in one FMA, and one Markstein correction step
// returns RN(x / 12) -- the same double the reference's division produces
// (tests/test_abi_host.py::test_exact_division_shortcuts checks the identity on the CPU).
__device__ __forceinline__ double div12(double x)
{
    const double y = 1.0 / 12.0;
    const double q = x * y;
    const double r = fma(-q, 12.0, x);
    return fma(r, y, q);
}

// A thread owns 4 consecutive columns and walks GRAD_ROWS rows with the five rows of the y-stencil rolling through
// registers (every input row is loaded once per 8 output rows, as one 16-byte vector); the two columns either side
// that the x-stencil needs come from the neighbouring lanes.  Columns at and beyond nx carry the value of column
// nx - 1, rows are clamped to the image and to the rows the band holds -- the reference's clamp-to-edge taps.
// gy may be null (the reference's third call: its y-output is overwritten by the fourth).
#define GRAD_ROWS 8
template <bool VEC>
__device__ __forceinline__ float4 grad_row(const float* __restrict__ f, const Geom& g, int i0, int j)
{
    const int lo = g.jlo(), hi = g.jhi() - 1;
    const float* r = f + g.at(0, min(max(clampi(j, g.ny), lo), hi));
    float4 c;
    if (i0 + 3 < g.nx) {
        if (VEC) c = __ldg(reinterpret_cast<const float4*>(r + i0));
        else { c.x = __ldg(r + i0); c.y = __ldg(r + i0 + 1); c.z = __ldg(r + i0 + 2); c.w = __ldg(r + i0 + 3); }
    } else {
        const float e = __ldg(r + g.nx - 1);
        c.x = i0 < g.nx ? __ldg(r + i0) : e;
        c.y = i0 + 1 < g.nx ? __ldg(r + i0 + 1) : e;
        c.z = i0 + 2 < g.nx ? __ldg(r + i0 + 2) : e;
        c.w = e;
    }
    return c;
}

// VEC: rows start on 16-byte boundaries (every plane of a plan does; the dense arrays of the stage entry point need not).
// SPLIT: the batched instance, whose input planes of pair p lie p * ps_in floats after pair 0's and its outputs p * ps
// (a sequence's second derivatives read image slots and write per-pair planes); the single-pair instance ignores ps_in.
template <bool VEC, bool SPLIT>
__global__ void __launch_bounds__(256)
k_gradient(const float* __restrict__ f, float* __restrict__ gx, float* __restrict__ gy, Geom g,
           int ja, int jb, int nc, size_t ps, size_t ps_in)
{
    const int lane = threadIdx.x;
    const int i0 = (blockIdx.x * 32 + lane) * 4;
    const int js = ja + (blockIdx.y * 8 + threadIdx.y) * GRAD_ROWS;
    if (js >= jb) return;                                  // whole warp: js depends on threadIdx.y only
    const unsigned pair = blockIdx.z / nc;            // blockIdx.z = pair * nc + channel
    const size_t coff = (size_t)(blockIdx.z - pair * nc) * g.plane + pair * ps;
    f += SPLIT ? (size_t)(blockIdx.z - pair * nc) * g.plane + pair * ps_in : coff;
    gx += coff;
    if (gy) gy += coff;
    const int lo = g.jlo(), hi = g.jhi() - 1;
    float4 w0 = grad_row<VEC>(f, g, i0, js - 2), w1 = grad_row<VEC>(f, g, i0, js - 1), w2 = grad_row<VEC>(f, g, i0, js),
           w3 = grad_row<VEC>(f, g, i0, js + 1), w4 = grad_row<VEC>(f, g, i0, js + 2);
    const int je = min(js + GRAD_ROWS, jb);
    for (int j = js; j < je; j++) {
        // columns i0-2, i0-1 and i0+4, i0+5 of row j
        float l2 = __shfl_up_sync(0xffffffffu, w2.z, 1), l1 = __shfl_up_sync(0xffffffffu, w2.w, 1);
        float r1 = __shfl_down_sync(0xffffffffu, w2.x, 1), r2 = __shfl_down_sync(0xffffffffu, w2.y, 1);
        if (lane == 0 || lane == 31) {
            const float* r = f + g.at(0, min(max(clampi(j, g.ny), lo), hi));
            if (lane == 0) { l2 = __ldg(r + clampi(i0 - 2, g.nx)); l1 = __ldg(r + clampi(i0 - 1, g.nx)); }
            else { r1 = __ldg(r + clampi(i0 + 4, g.nx)); r2 = __ldg(r + clampi(i0 + 5, g.nx)); }
        }
        if (i0 < g.nx) {
            float4 ox, oy;
            ox.x = div12(grad_num(w2.z, w2.y, l1, l2));
            ox.y = div12(grad_num(w2.w, w2.z, w2.x, l1));
            ox.z = div12(grad_num(r1, w2.w, w2.y, w2.x));
            ox.w = div12(grad_num(r2, r1, w2.z, w2.y));
            oy.x = div12(grad_num(w4.x, w3.x, w1.x, w0.x));
            oy.y = div12(grad_num(w4.y, w3.y, w1.y, w0.y));
            oy.z = div12(grad_num(w4.z, w3.z, w1.z, w0.z));
            oy.w = div12(grad_num(w4.w, w3.w, w1.w, w0.w));
            const size_t o = g.at(i0, j);
            if (VEC && i0 + 3 < g.nx) {
                *reinterpret_cast<float4*>(gx + o) = ox;
                if (gy) *reinterpret_cast<float4*>(gy + o) = oy;
            } else if (i0 + 3 < g.nx) {
                gx[o] = ox.x; gx[o + 1] = ox.y; gx[o + 2] = ox.z; gx[o + 3] = ox.w;
                if (gy) { gy[o] = oy.x; gy[o + 1] = oy.y; gy[o + 2] = oy.z; gy[o + 3] = oy.w; }
            } else {                                        // last, partial vector of a row: padding is not written
                gx[o] = ox.x;
                if (i0 + 1 < g.nx) gx[o + 1] = ox.y;
                if (i0 + 2 < g.nx) gx[o + 2] = ox.z;
                if (gy) {
                    gy[o] = oy.x;
                    if (i0 + 1 < g.nx) gy[o + 1] = oy.y;
                    if (i0 + 2 < g.nx) gy[o + 2] = oy.z;
                }
            }
        }
        w0 = w1; w1 = w2; w2 = w3; w3 = w4;
        if (j + 1 < je) w4 = grad_row<VEC>(f, g, i0, j + 3);
    }
}

// ---- bicubic, :231-309 ---------------------------------------------------------
__device__ __forceinline__ float oct_cell(const float v[4], float x)
{
    return v[1] + 0.5 * x * (v[2] - v[0] +
           x * (2.0 * v[0] - 5.0 * v[1] + 4.0 * v[2] - v[3] +
           x * (3.0 * (v[1] - v[2]) + v[3] - v[0])));
}

__device__ __forceinline__ float bicubic(const float* __restrict__ in, const Geom& g, float uu, float vv)
{
    // tap indices: (int)-truncation of the float coordinate, then clamp (:266-273)
    const int x = clampi((int)uu, g.nx), y = clampi((int)vv, g.ny);
    const int mx = clampi((int)(uu - 1), g.nx), my = clampi((int)(vv - 1), g.ny);
    const int dx = clampi((int)(uu + 1), g.nx), dy = clampi((int)(vv + 1), g.ny);
    const int ddx = clampi((int)(uu + 2), g.nx), ddy = clampi((int)(vv + 2), g.ny);
    const int xs[4] = { mx, x, dx, ddx };
    const int ys[4] = { my, y, dy, ddy };
    float v[4];
#pragma unroll
    for (int a = 0; a < 4; a++) {
        float p[4];
#pragma unroll
        for (int b = 0; b < 4; b++) {
            int jr = min(max(ys[b], g.jlo()), g.jhi() - 1);
            p[b] = __ldg(in + g.at(xs[a], jr));
        }
        v[a] = oct_cell(p, vv - y);
    }
    return oct_cell(v, uu - x);
}

// ---- flow prolongation, :453-466 -------------------------------------------------
// The bicubic of :231-309 interpolates four columns along y and the four results along x.  The y-part of a column
// depends on the coarse column and the fine row only, so a warp (one fine row, 128 fine columns) evaluates it once
// per coarse column it touches (about 68 for a factor of 2, into shared memory) instead of four times per pixel:
// 1.5 instead of 5 cell evaluations and 2 instead of 16 loads per pixel, same operands and same operations per value.
#define ZOOM_COLS 128          // fine columns per warp
#define ZOOM_VMAX 144          // coarse columns a warp can hold (ZOOM_COLS / factor + 4, factor >= 1 up to rounding)
__device__ __forceinline__ float zoom_u(int ii, float factorx) { return (float)((ii / factorx) - (0.5 - 0.5 / factorx)); }

__global__ void __launch_bounds__(256)
k_zoom_in(const float* __restrict__ flow, Geom gc, float* __restrict__ out, Geom gf, int ja, int jb, float sf, size_t ps)
{
    __shared__ float V[8][ZOOM_VMAX];
    const int lane = threadIdx.x, wy = threadIdx.y;
    const int ibase = blockIdx.x * ZOOM_COLS;
    const int jj = ja + blockIdx.y * 8 + wy;
    if (jj >= jb || ibase >= gf.nx) return;                // whole warp
    flow += blockIdx.z * ps;                               // pair blockIdx.z
    out += blockIdx.z * ps;
    const float factorx = ((float)gf.nx / gc.nx);
    const float factory = ((float)gf.ny / gc.ny);
    const float vv = (float)((jj / factory) - (0.5 - 0.5 / factory));
    // the warp's coarse columns: the taps (int)(u - 1) .. (int)(u + 2), clamped, are monotone in the fine column
    const int ilast = min(ibase + ZOOM_COLS, gf.nx) - 1;
    const int cmin = clampi((int)(zoom_u(ibase, factorx) - 1), gc.nx);
    const int cmax = clampi((int)(zoom_u(ilast, factorx) + 2), gc.nx);
    const int ncol = cmax - cmin + 1;
    if (ncol > ZOOM_VMAX) {                                 // a factor below 1: the direct form
        for (int ii = ibase + lane; ii <= ilast; ii += 32)
            out[gf.at(ii, jj)] = bicubic(flow, gc, zoom_u(ii, factorx), vv) / sf;
        return;
    }
    const int y = clampi((int)vv, gc.ny), my = clampi((int)(vv - 1), gc.ny);
    const int dy = clampi((int)(vv + 1), gc.ny), ddy = clampi((int)(vv + 2), gc.ny);
    const int ys[4] = { my, y, dy, ddy };
    const float* rows[4];
#pragma unroll
    for (int b = 0; b < 4; b++) rows[b] = flow + gc.at(0, min(max(ys[b], gc.jlo()), gc.jhi() - 1));
    for (int c = lane; c < ncol; c += 32) {
        float p[4];
#pragma unroll
        for (int b = 0; b < 4; b++) p[b] = __ldg(rows[b] + cmin + c);
        V[wy][c] = oct_cell(p, vv - y);
    }
    __syncwarp();
    for (int ii = ibase + lane; ii <= ilast; ii += 32) {
        const float uu = zoom_u(ii, factorx);
        const int x = clampi((int)uu, gc.nx), mx = clampi((int)(uu - 1), gc.nx);
        const int dx = clampi((int)(uu + 1), gc.nx), ddx = clampi((int)(uu + 2), gc.nx);
        const float v[4] = { V[wy][mx - cmin], V[wy][x - cmin], V[wy][dx - cmin], V[wy][ddx - cmin] };
        out[gf.at(ii, jj)] = oct_cell(v, uu - x) / sf;
    }
}

// ---- dense <-> pitched copies, u += x ---------------------------------------------
__global__ void __launch_bounds__(256)
k_zero_rows(float* __restrict__ a, Geom g, int ja, int jb)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    const int j = ja + blockIdx.y;
    if (i < g.pitch && j < jb) a[g.at(i, j)] = 0.f;
}

// ---- host launchers ------------------------------------------------------------------
void launch_fill_gk(float* GK, float factor, int R, cudaStream_t st)
{
    k_fill_gk<<<1, 32, 0, st>>>(GK, factor, R);
}

size_t blur_decimate_smem_bytes(float factor, int R)
{
    constexpr int TX = 32, TY = 8;
    const int step = (int)(1.0f / factor) + 1;
    const int nrow_h = (TY - 1) * step + 2 * R + 2;
    return sizeof(float) * ((size_t)nrow_h * TX + 2 * R + 1);
}

void launch_blur_decimate(const float* src, const Geom& gs, float* dst, const Geom& gd, int ja, int jb,
                          float factor, const float* GK, int R, float scale, int nc, cudaStream_t st, int npairs, size_t ps)
{
    if (jb <= ja) return;
    constexpr int TX = 32, TY = 8;
    const size_t smem = blur_decimate_smem_bytes(factor, R);
    dim3 grid((gd.nx + TX - 1) / TX, (jb - ja + TY - 1) / TY, nc * npairs), block(TX, TY);
    static unsigned long long configured = 0;
    if (first_launch_on_device(&configured))
        cudaFuncSetAttribute(k_blur_decimate<TX, TY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BLUR_DECIMATE_SMEM_LIMIT);
    k_blur_decimate<TX, TY><<<grid, block, smem, st>>>(src, gs, dst, gd, ja, jb, factor, GK, R, scale, nc, ps);
}

void launch_gradient(const float* f, float* gx, float* gy, const Geom& g, int ja, int jb, int nc, cudaStream_t st,
                     int npairs, size_t ps, size_t ps_in)
{
    if (jb <= ja) return;
    dim3 grid((g.nx + 127) / 128, (jb - ja + 8 * GRAD_ROWS - 1) / (8 * GRAD_ROWS), nc * npairs), block(32, 8);
    const bool vec = (g.pitch & 3) == 0 && (g.plane & 3) == 0 &&
                     (((uintptr_t)f | (uintptr_t)gx | (uintptr_t)gy) & 15) == 0;
    if (npairs > 1) {
        if (vec) k_gradient<true, true><<<grid, block, 0, st>>>(f, gx, gy, g, ja, jb, nc, ps, ps_in);
        else k_gradient<false, true><<<grid, block, 0, st>>>(f, gx, gy, g, ja, jb, nc, ps, ps_in);
    } else {
        if (vec) k_gradient<true, false><<<grid, block, 0, st>>>(f, gx, gy, g, ja, jb, nc, ps, ps_in);
        else k_gradient<false, false><<<grid, block, 0, st>>>(f, gx, gy, g, ja, jb, nc, ps, ps_in);
    }
}

void launch_zoom_in(const float* flow, const Geom& gc, float* out, const Geom& gf, int ja, int jb, float sf,
                    cudaStream_t st, int npairs, size_t ps)
{
    if (jb <= ja) return;
    dim3 grid((gf.nx + ZOOM_COLS - 1) / ZOOM_COLS, (jb - ja + 7) / 8, npairs), block(32, 8);
    k_zoom_in<<<grid, block, 0, st>>>(flow, gc, out, gf, ja, jb, sf, ps);
}

}  // namespace octane
