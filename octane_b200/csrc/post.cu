// post.cu -- the optional post-smoother of the pixel displacements (-srsal): a 37 x 37 bilateral
// filter whose range weight comes from the cloud-top heights (Apke et al. 2018).
// Replaces octsrsalcuda + the host loops of oct_srsal_cu, src/oct_srsal_cuda.cu:16-71,73-147
// (reference tree).
//
// The reference widens u, v and CTH to double planes in managed memory on the host, fills per-pixel
// index arrays, and lets every thread gather its 1369 neighbours from global memory.  Here a CTA of
// 32 x 8 threads stages the (32+36) x (8+36) float neighbourhood of its tile (CTH, u, v: 36 KB) in
// shared memory once, the reflecting index rule applied while staging, and each thread runs the
// 37 x 37 window out of shared memory.  The pass is bound by the fp64 exp() of every tap (1369 per
// pixel), not by memory: 12 B read + 8 B written per pixel.
//
// Arithmetic kept from the reference: double accumulators, kc (x offset) outer / lc (y offset) inner,
// a1 = GK[kc]*GK[lc]*exp(d*d*sigpix2) with d the FLOAT difference of the two heights widened to
// double (:52,56-57), default FMA contraction of `au += u * a1`, result narrowed to float by the
// host copy-back (:139-143).  The taps are computed on the host like the reference's (glibc exp).
//
// Row window (banded runs): the input planes hold global rows [e0, ...), the output planes global rows
// [o0, o1).  The reflecting index stays in global coordinates (the scene edges are the edges of the whole
// scene, not of a band); e0 is subtracted only when addressing.  One GPU: e0 = o0 = 0, o1 = ny.
//
// Batches (octane_optical_flow_batch_ex_dev): pair blockIdx.z reads and writes planes ps floats further on, each pair
// filtered with its own heights; one launch covers every pair.  The offset enters the staging loads and the two
// stores only, so the 37 x 37 loop, which reads shared memory only, is the single-pair loop instruction for
// instruction.
#include "kernels.cuh"

namespace octane {

namespace {
constexpr int SR = 18;                 // filtsize = 2 * filtsigma, :78-79
constexpr int TX = 32, TY = 8;
constexpr int SW = TX + 2 * SR, SH = TY + 2 * SR;

// oct_bc_cuda, :16-28: -x below zero, 2 nx - x - 1 at or above nx
__device__ __forceinline__ int reflect(int x, int nx)
{
    if (x < 0) x = 0 - x;
    if (x >= nx) x = nx - (x - nx + 1);
    return x;
}

__global__ void __launch_bounds__(TX * TY)
k_srsal(const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ cth, int nx, int ny,
        int e0, int o0, int o1, SrsalTaps t, float* __restrict__ u_out, float* __restrict__ v_out, size_t ps)
{
    __shared__ float s_c[SH][SW], s_u[SH][SW], s_v[SH][SW];
    const size_t po = (size_t)blockIdx.z * ps;
    u += po; v += po; cth += po;
    const int i0 = blockIdx.x * TX, j0 = o0 + blockIdx.y * TY;
    for (int k = threadIdx.y * TX + threadIdx.x; k < SW * SH; k += TX * TY) {
        const int sy = k / SW, sx = k - sy * SW;
        // pixels beyond the scene (the window) in a partial tile are never read by a thread that stores
        const int gi = reflect(min(i0 + sx - SR, nx - 1 + SR), nx), gj = reflect(min(j0 + sy - SR, o1 - 1 + SR), ny);
        const size_t at = (size_t)gi + (size_t)(gj - e0) * nx;
        s_c[sy][sx] = cth[at];
        s_u[sy][sx] = u[at];
        s_v[sy][sx] = v[at];
    }
    __syncthreads();
    const int ic = i0 + threadIdx.x, jc = j0 + threadIdx.y;
    if (ic >= nx || jc >= o1) return;
    const float pixc = s_c[threadIdx.y + SR][threadIdx.x + SR];
    double au = 0, av = 0, a2 = 0;
    for (int kc = 0; kc < 2 * SR + 1; kc++) {
        for (int lc = 0; lc < 2 * SR + 1; lc++) {
            const float pixl = s_c[threadIdx.y + lc][threadIdx.x + kc];
            const double pixm = pixl - pixc;
            const double a1 = t.gk[kc] * t.gk[lc] * exp((pixm) * (pixm)*t.sigpix2);
            a2 += a1;
            au += (double)s_u[threadIdx.y + lc][threadIdx.x + kc] * a1;
            av += (double)s_v[threadIdx.y + lc][threadIdx.x + kc] * a1;
        }
    }
    // the pair index is read again rather than kept from the staging loop: a value live across the filter loop moves
    // the loop's uniform registers and its schedule
    unsigned z;
    asm volatile("mov.u32 %0, %%ctaid.z;" : "=r"(z));
    const size_t at = (size_t)z * ps + (size_t)ic + (size_t)(jc - o0) * nx;
    u_out[at] = (au / a2);
    v_out[at] = (av / a2);
}
}  // namespace

void launch_srsal(const float* u, const float* v, const float* cth, int nx, int ny, int e0, int o0, int o1,
                  const SrsalTaps& t, float* u_out, float* v_out, cudaStream_t st, int npairs, size_t ps)
{
    dim3 grid((nx + TX - 1) / TX, (o1 - o0 + TY - 1) / TY, npairs), block(TX, TY);
    k_srsal<<<grid, block, 0, st>>>(u, v, cth, nx, ny, e0, o0, o1, t, u_out, v_out, ps);
}

}  // namespace octane
