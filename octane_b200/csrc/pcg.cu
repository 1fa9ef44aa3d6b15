// pcg.cu -- matrix-free Jacobi-preconditioned conjugate gradient on the 2x2-block
// 5-point system.  Replaces jMatXVec / jVecXVec / jVecPVec / jDiagInv and the
// PCG driver of src/oct_variational_optical_flow.cu:112-205,1105-1195
// (reference tree).  The reference spends ~12 grid-wide barriers and ~520 B/px
// per iteration on explicit CSR; here one iteration is two streaming kernels:
//
//   pass 1  x += alpha' p   (the PREVIOUS iteration's update: p is being read anyway)
//           p = z + beta p   (z = M^-1 r, recomputed, never stored)
//           q = A p          (stencil, rolling three rows of p in registers)
//           partial p.q                                   68 B/px
//   pass 2  r -= alpha q ; partial r.r and z.r
//           stop rule + scalar roll in the last block      32 B/px
//
// Same recurrence, same fp32 scalar arithmetic (alpha = rz/pAp, beta =
// rz_new/rz_old, stop on !(r.r > tol) or the launch cap), same FMA order inside
// each matrix row as multiply_row (:112-121) over the entry order the build
// writes.  Dot products are reduced in a fixed order in double, so a solve is
// bit-reproducible run to run (the reference's float atomics are not).
// Every launch re-reads the device-side `done` flag and returns at once when
// the stop rule has fired, so the host can enqueue the cap's worth of launches
// (or replay a CUDA graph of them) without synchronising.
#include <cooperative_groups.h>

#include "kernels.cuh"

namespace octane {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4_stream(const float* p)
{
    return __ldcs(reinterpret_cast<const float4*>(p));   // read-once coefficient planes: evict-first
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float& el(float4& v, int k) { return reinterpret_cast<float*>(&v)[k]; }
__device__ __forceinline__ const float& el(const float4& v, int k) { return reinterpret_cast<const float*>(&v)[k]; }

// x-update mode of a pass-1 launch: iteration 0 has no previous term; iteration 1 starts x
// (x = alpha_0 p_0, no read of x); later iterations accumulate.
enum { XM_NONE = 0, XM_INIT = 1, XM_ACC = 2 };

struct P1Args {
    PcgBuffers b;
    Geom g;
    int ja, jb;        // rows whose q = A p this rank computes
    int cur;           // p[cur] = p_old, p[cur^1] = p_new
    int store_halo;    // banded: also store p_new of rows ja-1 and jb
    int rs;            // rows per warp task
    int nstrips, nsegs;
};

struct PRow {
    float4 pu, pv;     // p_new of the lane's 4 pixels
    float4 a1, a4;     // diagonal entries of the same pixels
    float eu, ev;      // p_new of the pixel just outside the warp's strip (lanes 0 and 31)
};

// p_new = (1/M) r + beta p_old for one row segment of the warp's strip; when `own`, also the
// pending x += alpha_prev p_old of the previous iteration (:1172) for the same pixels.
// (1/M) as jDiagInv (:142-149): 1./M rounded to float; z = Minv*r (:1117,1138);
// p = Bk*p + z (:1146, one FMA).
template <int XM>
__device__ __forceinline__ PRow compute_p(const P1Args& a, int cur, int j, int i0, int lane, float beta, float alpha_prev,
                                          bool own)
{
    constexpr bool FIRST = (XM == XM_NONE);
    PRow o;
    o.pu = o.pv = o.a1 = o.a4 = make_float4(0.f, 0.f, 0.f, 0.f);
    o.eu = o.ev = 0.f;
    const Geom& g = a.g;
    if (j < 0 || j >= g.ny) return o;
    const float* pu_old = a.b.pu[cur];
    const float* pv_old = a.b.pv[cur];
    if (i0 < g.nx) {
        const size_t off = g.at(i0, j);
        const float4 ru = ld4(a.b.ru + off), rv = ld4(a.b.rv + off);
        o.a1 = ld4(a.b.coef[C_A1] + off);
        o.a4 = ld4(a.b.coef[C_A4] + off);
        float4 po_u = make_float4(0.f, 0.f, 0.f, 0.f), po_v = po_u;
        if (!FIRST) { po_u = ld4(pu_old + off); po_v = ld4(pv_old + off); }
        if (!FIRST && own) {
            float4 x_u = make_float4(0.f, 0.f, 0.f, 0.f), x_v = x_u;
            if (XM == XM_ACC) { x_u = ld4(a.b.xu + off); x_v = ld4(a.b.xv + off); }
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (i0 + k < g.nx) {
                    el(x_u, k) = fmaf(alpha_prev, el(po_u, k), el(x_u, k));      // :1172
                    el(x_v, k) = fmaf(alpha_prev, el(po_v, k), el(x_v, k));
                } else {
                    el(x_u, k) = 0.f; el(x_v, k) = 0.f;
                }
            }
            st4(a.b.xu + off, x_u);
            st4(a.b.xv + off, x_v);
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (i0 + k < g.nx) {
                const float mu = 1.0f / el(o.a1, k), mv = 1.0f / el(o.a4, k);
                const float zu = mu * el(ru, k), zv = mv * el(rv, k);
                el(o.pu, k) = FIRST ? zu : fmaf(beta, el(po_u, k), zu);
                el(o.pv, k) = FIRST ? zv : fmaf(beta, el(po_v, k), zv);
            }
        }
    }
    if (lane == 0 || lane == 31) {
        const int ie = (lane == 0) ? i0 - 1 : i0 + 4;
        if (ie >= 0 && ie < g.nx) {
            const size_t off = g.at(ie, j);
            const float mu = 1.0f / a.b.coef[C_A1][off], mv = 1.0f / a.b.coef[C_A4][off];
            const float zu = mu * a.b.ru[off], zv = mv * a.b.rv[off];
            o.eu = FIRST ? zu : fmaf(beta, pu_old[off], zu);
            o.ev = FIRST ? zv : fmaf(beta, pv_old[off], zv);
        }
    }
    return o;
}

// boundary merging of the stored couplings (:929-1077): multiplier of W(i-1) / W(i) as the
// entry towards i-1 / i+1 of pixel i (and the same in j for N)
__device__ __forceinline__ float mul_lo(int i, int n) { return i == 0 ? 0.f : (i == n - 1 ? 2.f : 1.f); }
__device__ __forceinline__ float mul_hi(int i, int n) { return i == n - 1 ? 0.f : (i == 0 ? 2.f : 1.f); }

// q = A p of block `bid`'s share (of `nblk` blocks) of the (strip x row segment) tasks, p and x updated on the way;
// returns the thread's partial p.q.  Shared by the per-iteration kernel and the whole-solve cooperative kernels.
template <int XM>
__device__ __forceinline__ double pass1_tasks(const P1Args& a, int cur, float beta, float alpha_prev, int bid, int nblk)
{
    constexpr bool FIRST = (XM == XM_NONE);
    const Geom& g = a.g;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ntasks = a.nstrips * a.nsegs;
    float* pu_new = a.b.pu[cur ^ 1];
    float* pv_new = a.b.pv[cur ^ 1];
    const float* W = a.b.coef[C_W];
    const float* N = a.b.coef[C_N];
    double dot[1] = { 0.0 };

    for (int t = bid * 8 + wib; t < ntasks; t += nblk * 8) {
        const int seg = t / a.nstrips, strip = t - seg * a.nstrips;
        const int i0 = strip * 128 + lane * 4;
        const int j_a = a.ja + seg * a.rs, j_b = min(a.jb, j_a + a.rs);
        const bool active = i0 < g.nx;
        PRow up = compute_p<XM>(a, cur, j_a - 1, i0, lane, beta, alpha_prev, false);
        PRow ce = compute_p<XM>(a, cur, j_a, i0, lane, beta, alpha_prev, true);
        float4 n_up = make_float4(0.f, 0.f, 0.f, 0.f);                 // N of the row above the centre
        if (active && j_a > 0) n_up = ld4(N + g.at(i0, j_a - 1));
        if (a.store_halo && j_a == a.ja && j_a - 1 >= 0 && active) {
            st4(pu_new + g.at(i0, j_a - 1), up.pu);
            st4(pv_new + g.at(i0, j_a - 1), up.pv);
        }
        for (int j = j_a; j < j_b; j++) {
            PRow dn = compute_p<XM>(a, cur, j + 1, i0, lane, beta, alpha_prev, j + 1 < j_b);
            // horizontal neighbours of the centre row: lanes exchange their edge pixels
            float lu = __shfl_up_sync(0xffffffffu, ce.pu.w, 1), lv = __shfl_up_sync(0xffffffffu, ce.pv.w, 1);
            float ru_ = __shfl_down_sync(0xffffffffu, ce.pu.x, 1), rv_ = __shfl_down_sync(0xffffffffu, ce.pv.x, 1);
            if (lane == 0) { lu = ce.eu; lv = ce.ev; }
            if (lane == 31) { ru_ = ce.eu; rv_ = ce.ev; }
            float4 a2 = make_float4(0.f, 0.f, 0.f, 0.f), w = a2, nn = a2;
            size_t off = 0;
            if (active) {
                off = g.at(i0, j);
                a2 = ld4_stream(a.b.coef[C_A2] + off);
                w = ld4_stream(W + off);
                nn = ld4_stream(N + off);
            }
            float wl = __shfl_up_sync(0xffffffffu, w.w, 1);            // W of the pixel left of the lane's first
            if (lane == 0) wl = (active && i0 > 0) ? W[off - 1] : 0.f;
            if (active) {
                const float m6 = mul_lo(j, g.ny), m8 = mul_hi(j, g.ny);
                float4 qu, qv;
                float part = 0.f;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const float pl_u = (k == 0) ? lu : el(ce.pu, k - 1), pl_v = (k == 0) ? lv : el(ce.pv, k - 1);
                    const float pr_u = (k == 3) ? ru_ : el(ce.pu, k + 1), pr_v = (k == 3) ? rv_ : el(ce.pv, k + 1);
                    const float a5 = mul_lo(i0 + k, g.nx) * ((k == 0) ? wl : el(w, k - 1));
                    const float a7 = mul_hi(i0 + k, g.nx) * el(w, k);
                    const float a6 = m6 * el(n_up, k), a8 = m8 * el(nn, k);
                    // row of u: [j-1] [i-1] a1 a2 [i+1] [j+1]   (multiply_row order)
                    float su = 0.f;
                    su = fmaf(a6, el(up.pu, k), su);
                    su = fmaf(a5, pl_u, su);
                    su = fmaf(el(ce.a1, k), el(ce.pu, k), su);
                    su = fmaf(el(a2, k), el(ce.pv, k), su);
                    su = fmaf(a7, pr_u, su);
                    su = fmaf(a8, el(dn.pu, k), su);
                    // row of v: [j-1] [i-1] a2 a4 [i+1] [j+1]
                    float sv = 0.f;
                    sv = fmaf(a6, el(up.pv, k), sv);
                    sv = fmaf(a5, pl_v, sv);
                    sv = fmaf(el(a2, k), el(ce.pu, k), sv);
                    sv = fmaf(el(ce.a4, k), el(ce.pv, k), sv);
                    sv = fmaf(a7, pr_v, sv);
                    sv = fmaf(a8, el(dn.pv, k), sv);
                    const bool in = i0 + k < g.nx;
                    el(qu, k) = in ? su : 0.f;
                    el(qv, k) = in ? sv : 0.f;
                    if (in) part += el(ce.pu, k) * su + el(ce.pv, k) * sv;
                }
                st4(pu_new + off, ce.pu);
                st4(pv_new + off, ce.pv);
                st4(a.b.qu + off, qu);
                st4(a.b.qv + off, qv);
                dot[0] += (double)part;
            }
            n_up = nn;
            up = ce;
            ce = dn;
        }
        if (a.store_halo && j_b == a.jb && j_b < g.ny && active) {     // ce now holds row j_b
            st4(pu_new + g.at(i0, j_b), ce.pu);
            st4(pv_new + g.at(i0, j_b), ce.pv);
        }
    }
    return dot[0];
}

template <int XM>
__global__ void __launch_bounds__(256, 2) k_pcg_pass1(P1Args a)
{
    constexpr bool FIRST = (XM == XM_NONE);
    __shared__ double red[32];
    const PcgScalars* s = a.b.scal;
    if (s->done) return;
    const float beta = FIRST ? 0.f : s->rz / s->rz_old;      // Bk, :1144
    const float alpha_prev = FIRST ? 0.f : s->alpha;
    double dot[1] = { pass1_tasks<XM>(a, a.cur, beta, alpha_prev, blockIdx.x, gridDim.x) };
    block_sum<1>(dot, red);
    double tot[1];
    if (grid_sum_finish<1>(dot, a.b.partials, a.b.ticket, tot, red)) {
        if (a.b.p2p.world > 1) p2p_allreduce<1>(a.b.p2p, P2P_PASS1, tot, &a.b.scal->comm_err);
        if (threadIdx.x == 0) {
            if (a.b.defer) a.b.pending[0] = tot[0];
            else a.b.scal->pAp = (float)tot[0];                        // pkTApk, :1165
        }
    }
}

typedef P1Args P2Args;       // pass 2 reads b, g, ja, jb of the same argument block

// r -= alpha q over block `bid`'s share (of `nblk` blocks) of the rows; acc += partial r.r and z.r.  Shared by the
// per-iteration kernel and the whole-solve cooperative kernels.
__device__ __forceinline__ void pass2_units(const P1Args& a, float alphak, bool p2p, double (&acc)[2], int bid, int nblk)
{
    const float nalpha = -1. * alphak;                        // :1174
    const Geom& g = a.g;
    const int upr = g.pitch >> 2;                             // float4 units per row
    const long long nunits = (long long)(a.jb - a.ja) * upr;
    for (long long t = (long long)bid * 256 + threadIdx.x; t < nunits; t += (long long)nblk * 256) {
        const int jr = (int)(t / upr), i0 = (int)(t - (long long)jr * upr) * 4;
        if (i0 >= g.nx) continue;
        const size_t off = g.at(i0, a.ja + jr);
        const float4 q_u = ld4_stream(a.b.qu + off), q_v = ld4_stream(a.b.qv + off);
        float4 r_u = ld4(a.b.ru + off), r_v = ld4(a.b.rv + off);
        const float4 a1 = ld4(a.b.coef[C_A1] + off), a4 = ld4(a.b.coef[C_A4] + off);
        float prr = 0.f, prz = 0.f;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (i0 + k < g.nx) {
                const float ru = fmaf(nalpha, el(q_u, k), el(r_u, k));   // :1174
                const float rv = fmaf(nalpha, el(q_v, k), el(r_v, k));
                el(r_u, k) = ru;
                el(r_v, k) = rv;
                const float zu = (1.0f / el(a1, k)) * ru, zv = (1.0f / el(a4, k)) * rv;
                prr += ru * ru + rv * rv;                                // residc, :1178
                prz += zu * ru + zv * rv;                                // zktrk of the next iteration, :1142
            } else {
                el(r_u, k) = 0.f; el(r_v, k) = 0.f;
            }
        }
        st4(a.b.ru + off, r_u);
        st4(a.b.rv + off, r_v);
        if (p2p) {
            // the band's first / last owned row is the neighbour's halo row: store it there as well
            // (peer memory over NVLink), so the next pass 1 rebuilds p on the halo without an exchange step
            const int j = a.ja + jr;
            if (j == a.ja && a.b.up_ru) { st4(a.b.up_ru + off, r_u); st4(a.b.up_rv + off, r_v); }
            if (j == a.jb - 1 && a.b.dn_ru) { st4(a.b.dn_ru + off, r_u); st4(a.b.dn_rv + off, r_v); }
        }
        acc[0] += (double)prr;
        acc[1] += (double)prz;
    }
}

// r -= alpha q; partial r.r and z.r; the last block rolls the scalars and applies the stop rule.
__global__ void __launch_bounds__(256) k_pcg_pass2(P2Args a)
{
    __shared__ double red[2 * 32];
    PcgScalars* s = a.b.scal;
    if (s->done) return;
    const float alphak = s->rz / s->pAp;                      // :1169
    const bool p2p = a.b.p2p.world > 1;
    double acc[2] = { 0.0, 0.0 };
    pass2_units(a, alphak, p2p, acc, blockIdx.x, gridDim.x);
    block_sum<2>(acc, red);
    double tot[2];
    if (grid_sum_finish<2>(acc, a.b.partials, a.b.ticket, tot, red, p2p)) {
        if (p2p) p2p_allreduce<2>(a.b.p2p, P2P_PASS2, tot, &a.b.scal->comm_err);
        if (threadIdx.x == 0 && a.b.defer) {
            a.b.pending[0] = tot[0];
            a.b.pending[1] = tot[1];
        } else if (threadIdx.x == 0) {
            const float rr = (float)tot[0];
            s->alpha = alphak;                 // x += alpha p rides on the next pass 1 / the final update
            s->rz_old = s->rz;                 // z0tr0 of the next iteration, :1135
            s->rz = (float)tot[1];
            s->rr = rr;
            s->its = s->its + 1;
            s->done = !(rr > s->tol);          // while((*residc) > tol ...), :1131
        }
    }
}

// ---- a whole solve in ONE cooperative launch (small levels, one GPU) ------------------------------------------
// A 500 x 500 level is a few microseconds of work per pass: 60 launches per solve spend their time in launch
// latency and in the GPU's front end (64 pairs in flight on 8 to 32 streams all run at the same 1.6 us per kernel,
// profiles/r02_bench_batch64_streams*.json).  Here the same two passes of the same recurrence run inside one kernel,
// separated by grid-wide barriers; every block sums the per-block partials itself, in the same fixed order, so all
// blocks take the same alpha, beta and stop decision without a ticket or a scalar round trip through memory.
template <int NV>
__device__ __forceinline__ void coop_sum(double (&v)[NV], double* partials, double* red, cooperative_groups::grid_group& grid)
{
    const int tid = threadIdx.x;
    block_sum<NV>(v, red);
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NV; k++) partials[(size_t)k * gridDim.x + blockIdx.x] = v[k];
    }
    grid.sync();
#pragma unroll
    for (int k = 0; k < NV; k++) {
        double t = 0.0;
        for (unsigned b = tid; b < gridDim.x; b += 256) t += __ldcg(&partials[(size_t)k * gridDim.x + b]);
        v[k] = t;
    }
    __syncthreads();                       // red is reused
    block_sum<NV>(v, red);
    // broadcast thread 0's totals to the block
    __shared__ double bc[NV];
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NV; k++) bc[k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; k++) v[k] = bc[k];
}

__global__ void __launch_bounds__(256, 2) k_pcg_coop(P1Args a, int iters)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[2 * 32];
    PcgScalars* s = a.b.scal;
    // the scalars of the solve live in registers, identically in every thread of the grid
    float rz = s->rz, rr = s->rr, rz_old = 0.f, alpha = 0.f;
    const float tol = s->tol;
    int its = 0;
    bool done = s->done != 0;
    double* part1 = a.b.partials;                       // p.q
    double* part2 = a.b.partials + gridDim.x;           // r.r, z.r (two more regions: a block may still read one while
                                                        // a faster block already writes the other)
    for (int ki = 0; ki < iters && !done; ki++) {
        const int cur = ki & 1;
        double d1[1];
        if (ki == 0)      d1[0] = pass1_tasks<XM_NONE>(a, cur, 0.f, 0.f, blockIdx.x, gridDim.x);
        else if (ki == 1) d1[0] = pass1_tasks<XM_INIT>(a, cur, rz / rz_old, alpha, blockIdx.x, gridDim.x);       // Bk, :1144
        else              d1[0] = pass1_tasks<XM_ACC>(a, cur, rz / rz_old, alpha, blockIdx.x, gridDim.x);
        coop_sum<1>(d1, part1, red, grid);
        const float pAp = (float)d1[0];                                              // pkTApk, :1165
        const float alphak = rz / pAp;                                               // :1169
        double d2[2] = { 0.0, 0.0 };
        pass2_units(a, alphak, false, d2, blockIdx.x, gridDim.x);
        coop_sum<2>(d2, part2, red, grid);
        alpha = alphak;
        rz_old = rz;
        rz = (float)d2[1];
        rr = (float)d2[0];
        its++;
        done = !(rr > tol);                                                          // :1131
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        s->alpha = alpha; s->rz_old = rz_old; s->rz = rz; s->rr = rr; s->its = its; s->done = done ? 1 : 0;
    }
}

// ---- a whole solve of MANY pairs in one cooperative launch (small levels, batched calls) ------------------------
// Pair `pair0 + k` of the launch is solved by the k-th group of G consecutive blocks, with its own partial sums, its
// own barrier and its own scalars: a pair that meets its stop rule leaves without waiting for the others.  G and
// the task partition depend only on the level geometry (coop_batch_blocks), so a pair's bits do not depend on how
// many other pairs share the launch or where in the batch it sits.
struct CoopBatch {
    int G;                 // blocks per pair
    int pair0;             // first pair of this launch (index into the batch)
    size_t ps;             // pair stride of the workspace planes (floats)
    double* partials;      // [launch pairs][3 G]: p.q, then r.r and z.r
    unsigned* bar;         // [launch pairs][2]: arrive counter, generation -- zero before the launch
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned* p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned atom_add_acq_rel_gpu(unsigned* p, unsigned v)
{
    unsigned old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}

// Barrier of one group of G blocks (all co-resident: the launch is cooperative).  Thread 0 reads the generation
// (acquire) BEFORE it arrives, so the last arrival cannot advance it unseen; the last arrival resets the counter and
// then releases the next generation, so a block that has seen the new generation also sees the counter at zero.
// The fences make the writes of all the block's threads (ordered before thread 0 by __syncthreads) visible to the
// group, as grid.sync() does for a whole grid.
__device__ __forceinline__ void group_barrier(unsigned* bar, unsigned G)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned gen = ld_acquire_gpu(bar + 1);
        __threadfence();
        if (atom_add_acq_rel_gpu(bar, 1u) == G - 1) {
            bar[0] = 0u;
            st_release_gpu(bar + 1, gen + 1u);
        } else {
            while (ld_acquire_gpu(bar + 1) == gen) __nanosleep(20);
        }
        __threadfence();
    }
    __syncthreads();
}

// coop_sum over the blocks of one group: block lb of G writes its partials, then every block sums all G in the same
// fixed order
template <int NV>
__device__ __forceinline__ void group_sum(double (&v)[NV], double* partials, double* red, unsigned* bar, int G, int lb)
{
    const int tid = threadIdx.x;
    block_sum<NV>(v, red);
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NV; k++) partials[(size_t)k * G + lb] = v[k];
    }
    group_barrier(bar, (unsigned)G);
#pragma unroll
    for (int k = 0; k < NV; k++) {
        double t = 0.0;
        for (int b = tid; b < G; b += 256) t += __ldcg(&partials[(size_t)k * G + b]);
        v[k] = t;
    }
    __syncthreads();
    block_sum<NV>(v, red);
    __shared__ double bc[NV];
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NV; k++) bc[k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; k++) v[k] = bc[k];
}

__global__ void __launch_bounds__(256, 2) k_pcg_coop_batch(P1Args a, CoopBatch cb, int iters)
{
    __shared__ double red[2 * 32];
    const int grp = blockIdx.x / cb.G, lb = blockIdx.x - grp * cb.G, G = cb.G;
    const int pair = cb.pair0 + grp;
    const size_t po = (size_t)pair * cb.ps;
    for (int i = 0; i < NCOEF; i++) a.b.coef[i] += po;
    a.b.ru += po; a.b.rv += po; a.b.xu += po; a.b.xv += po;
    a.b.pu[0] += po; a.b.pu[1] += po; a.b.pv[0] += po; a.b.pv[1] += po;
    a.b.qu += po; a.b.qv += po;
    PcgScalars* s = a.b.scal + pair;
    double* part1 = cb.partials + (size_t)grp * 3 * G;       // p.q
    double* part2 = part1 + G;                               // r.r, z.r
    unsigned* bar = cb.bar + 2 * grp;
    float rz = s->rz, rr = s->rr, rz_old = 0.f, alpha = 0.f;
    const float tol = s->tol;
    int its = 0;
    bool done = s->done != 0;
    for (int ki = 0; ki < iters && !done; ki++) {
        const int cur = ki & 1;
        double d1[1];
        if (ki == 0)      d1[0] = pass1_tasks<XM_NONE>(a, cur, 0.f, 0.f, lb, G);
        else if (ki == 1) d1[0] = pass1_tasks<XM_INIT>(a, cur, rz / rz_old, alpha, lb, G);       // Bk, :1144
        else              d1[0] = pass1_tasks<XM_ACC>(a, cur, rz / rz_old, alpha, lb, G);
        group_sum<1>(d1, part1, red, bar, G, lb);
        const float pAp = (float)d1[0];                                              // pkTApk, :1165
        const float alphak = rz / pAp;                                               // :1169
        double d2[2] = { 0.0, 0.0 };
        pass2_units(a, alphak, false, d2, lb, G);
        group_sum<2>(d2, part2, red, bar, G, lb);
        alpha = alphak;
        rz_old = rz;
        rz = (float)d2[1];
        rr = (float)d2[0];
        its++;
        done = !(rr > tol);                                                          // :1131
    }
    if (lb == 0 && threadIdx.x == 0) {
        s->alpha = alpha; s->rz_old = rz_old; s->rz = rz; s->rr = rr; s->its = its; s->done = done ? 1 : 0;
    }
}

// Banded runs: the dot totals were summed over ranks by an all-reduce on
// `pending`; apply them exactly as the single-GPU kernels' last block does.
__global__ void k_finalize(PcgBuffers b, int kind, float tol)
{
    PcgScalars* s = b.scal;
    if (kind == FINALIZE_BUILD) {
        s->rr = (float)b.pending[0];
        s->rz = (float)b.pending[1];
        s->rz_old = 0.f;
        s->pAp = 0.f;
        s->alpha = 0.f;
        s->tol = tol;
        s->its = 0;
        s->done = !((float)b.pending[0] > tol);
        return;
    }
    if (s->done) return;
    if (kind == FINALIZE_PASS1) {
        s->pAp = (float)b.pending[0];
    } else {
        const float rr = (float)b.pending[0];
        s->alpha = s->rz / s->pAp;             // what every block of pass 2 just used
        s->rz_old = s->rz;
        s->rz = (float)b.pending[1];
        s->rr = rr;
        s->its = s->its + 1;
        s->done = !(rr > s->tol);
    }
}

void launch_finalize(const PcgBuffers& b, int kind, float tol, cudaStream_t st)
{
    k_finalize<<<1, 1, 0, st>>>(b, kind, tol);
}

// u += x, v += x after a solve (:1185-1195), with the last pending x += alpha p folded in.
// After `its` iterations x holds the terms of iterations 0 .. its-2 (none when its == 1) and
// p[its & 1] is the search direction of iteration its-1.  Nothing happens when no iteration ran.
__global__ void __launch_bounds__(256)
k_update_uv(float* __restrict__ u, float* __restrict__ v, PcgBuffers b, Geom g, int ja, int jb, int* its_out, size_t ps,
            int its_stride)
{
    const PcgScalars* s = b.scal + blockIdx.z;                // pair blockIdx.z
    const int its = s->its;
    if (blockIdx.x == 0 && threadIdx.x == 0 && its_out) its_out[(size_t)blockIdx.z * its_stride] = its;
    if (its == 0) return;
    const float alpha = s->alpha;
    const float* pu = b.pu[its & 1];
    const float* pv = b.pv[its & 1];
    const int upr = g.pitch >> 2;
    const long long nunits = (long long)(jb - ja) * upr;
    for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < nunits; t += (long long)gridDim.x * 256) {
        const int jr = (int)(t / upr), i0 = (int)(t - (long long)jr * upr) * 4;
        if (i0 >= g.nx) continue;
        const size_t off = g.at(i0, ja + jr) + (size_t)blockIdx.z * ps;
        float4 a = ld4(u + off), c = ld4(v + off);
        float4 xu = make_float4(0.f, 0.f, 0.f, 0.f), xv = xu;
        if (its > 1) { xu = ld4(b.xu + off); xv = ld4(b.xv + off); }
        const float4 p_u = ld4(pu + off), p_v = ld4(pv + off);
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (i0 + k < g.nx) {
                const float x1 = fmaf(alpha, el(p_u, k), el(xu, k));     // :1172 of the last iteration
                const float x2 = fmaf(alpha, el(p_v, k), el(xv, k));
                el(a, k) = el(a, k) + x1;                                // :1187-1188
                el(c, k) = el(c, k) + x2;
            }
        st4(u + off, a);
        st4(v + off, c);
    }
}

// The same after a merged-reduction solve (pcg_fused.cu): x is brought up to date every second iteration (two terms
// at once), so after an odd number of iterations the last term alpha p is still pending; x exists from the
// second iteration on; iteration k leaves its p in pu[(k & 1) ^ 1], so the last one is in pu[its & 1] as for the
// two-pass kernels.
__global__ void __launch_bounds__(256)
k_update_uv_fused(float* __restrict__ u, float* __restrict__ v, PcgBuffers b, Geom g, int ja, int jb, int* its_out, size_t ps,
                  int its_stride)
{
    const PcgScalars* s = b.scal + blockIdx.z;                // pair blockIdx.z
    const int its = s->its;
    if (blockIdx.x == 0 && threadIdx.x == 0 && its_out) its_out[(size_t)blockIdx.z * its_stride] = its;
    if (its == 0) return;
    const bool pending = (its & 1) != 0, havex = its >= 2;
    const float alpha = s->alpha;
    const int upr = g.pitch >> 2;
    const long long nunits = (long long)(jb - ja) * upr;
    for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < nunits; t += (long long)gridDim.x * 256) {
        const int jr = (int)(t / upr), i0 = (int)(t - (long long)jr * upr) * 4;
        if (i0 >= g.nx) continue;
        const size_t off = g.at(i0, ja + jr) + (size_t)blockIdx.z * ps;
        float4 a = ld4(u + off), c = ld4(v + off);
        float4 xu = make_float4(0.f, 0.f, 0.f, 0.f), xv = xu, p_u = xu, p_v = xu;
        if (havex) { xu = ld4(b.xu + off); xv = ld4(b.xv + off); }
        if (pending) { p_u = ld4(b.pu[its & 1] + off); p_v = ld4(b.pv[its & 1] + off); }
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (i0 + k < g.nx) {
                const float x1 = pending ? fmaf(alpha, el(p_u, k), el(xu, k)) : el(xu, k);     // :1172 of the last iteration
                const float x2 = pending ? fmaf(alpha, el(p_v, k), el(xv, k)) : el(xv, k);
                el(a, k) = el(a, k) + x1;                                                        // :1187-1188
                el(c, k) = el(c, k) + x2;
            }
        st4(u + off, a);
        st4(v + off, c);
    }
}

// test hook: the reference's boundary-merged a5..a8 from the stored W, N
__global__ void __launch_bounds__(256)
k_expand_coef(PcgBuffers b, Geom g, float* a5, float* a6, float* a7, float* a8)
{
    const int i = blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
    if (i >= g.nx || j >= g.ny) return;
    const size_t l = g.at(i, j);
    const float* W = b.coef[C_W];
    const float* N = b.coef[C_N];
    a5[l] = mul_lo(i, g.nx) * (i > 0 ? W[l - 1] : 0.f);
    a7[l] = mul_hi(i, g.nx) * W[l];
    a6[l] = mul_lo(j, g.ny) * (j > g.jlo() ? N[l - g.pitch] : 0.f);
    a8[l] = mul_hi(j, g.ny) * N[l];
}

// dst(pitched rows [ja,jb)) = scale * src(dense, row 0 == ja)
__global__ void __launch_bounds__(256)
k_scale_copy(const float* __restrict__ src, float* __restrict__ dst, Geom g, int ja, int jb, float scale)
{
    const int i = blockIdx.x * 256 + threadIdx.x;
    const int j = ja + blockIdx.y;
    if (i < g.nx && j < jb) dst[g.at(i, j)] = src[(size_t)(j - ja) * g.nx + i] * scale;
}

static int pass1_rows_per_task(int nstrips, int nrows, int sm_count)
{
    // enough warp tasks to fill the machine a few times over, at most 64 rows each
    long long want = (long long)sm_count * 16 * 4;
    long long rs = ((long long)nstrips * nrows + want - 1) / want;
    if (rs < 4) rs = 4;
    if (rs > 64) rs = 64;
    return (int)rs;
}

void launch_pcg_pass1(const PcgBuffers& b, const Geom& g, int ja, int jb, int ki, int store_halo,
                      int sm_count, cudaStream_t st)
{
    P1Args a;
    a.b = b; a.g = g; a.ja = ja; a.jb = jb; a.cur = ki & 1; a.store_halo = store_halo;
    a.nstrips = (g.nx + 127) / 128;
    a.rs = pass1_rows_per_task(a.nstrips, jb - ja, sm_count);
    a.nsegs = (jb - ja + a.rs - 1) / a.rs;
    const int ntasks = a.nstrips * a.nsegs;
    int grid = (ntasks + 7) / 8;
    const int cap = sm_count * 16;
    if (grid > cap) grid = cap;
    if (grid > b.max_partial_blocks) grid = b.max_partial_blocks;
    if (ki == 0)      k_pcg_pass1<XM_NONE><<<grid, 256, 0, st>>>(a);
    else if (ki == 1) k_pcg_pass1<XM_INIT><<<grid, 256, 0, st>>>(a);
    else              k_pcg_pass1<XM_ACC><<<grid, 256, 0, st>>>(a);
}

// grid of the cooperative whole-solve kernel: enough blocks for the level's warp tasks, never more than fit on the
// device at once (2 blocks of 256 threads per SM by the launch bounds; the occupancy query has the last word)
int launch_pcg_coop(const PcgBuffers& b, const Geom& g, int ja, int jb, int iters, int sm_count, cudaStream_t st)
{
    P1Args a;
    a.b = b; a.g = g; a.ja = ja; a.jb = jb; a.cur = 0; a.store_halo = 0;
    a.nstrips = (g.nx + 127) / 128;
    a.rs = pass1_rows_per_task(a.nstrips, jb - ja, sm_count);
    a.nsegs = (jb - ja + a.rs - 1) / a.rs;
    static int per_sm = 0;
    if (!per_sm) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg_coop, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
    }
    const int ntasks = a.nstrips * a.nsegs;
    int grid = (ntasks + 7) / 8;
    const int cap = sm_count * per_sm;
    if (grid > cap) grid = cap;
    if (3 * grid > 2 * b.max_partial_blocks) grid = 2 * b.max_partial_blocks / 3;
    if (grid < 1) grid = 1;
    void* args[] = { &a, &iters };
    return cudaLaunchCooperativeKernel((const void*)k_pcg_coop, dim3(grid), dim3(256), args, 0, st) == cudaSuccess ? 0 : -1;
}

void launch_pcg_pass2(const PcgBuffers& b, const Geom& g, int ja, int jb, int sm_count, cudaStream_t st)
{
    P2Args a;
    a.b = b; a.g = g; a.ja = ja; a.jb = jb; a.cur = 0; a.store_halo = 0; a.rs = 0; a.nstrips = 0; a.nsegs = 0;
    const long long nunits = (long long)(jb - ja) * (g.pitch >> 2);
    long long grid = (nunits + 255) / 256;
    const int cap = sm_count * 16;
    if (grid > cap) grid = cap;
    if (grid > b.max_partial_blocks) grid = b.max_partial_blocks;
    k_pcg_pass2<<<(int)grid, 256, 0, st>>>(a);
}

void launch_update_uv(float* u, float* v, const PcgBuffers& b, const Geom& g, int ja, int jb,
                      int* its_out, int sm_count, cudaStream_t st, int npairs, size_t ps, int its_stride)
{
    const long long nunits = (long long)(jb - ja) * (g.pitch >> 2);
    long long grid = (nunits + 255) / 256;
    if (grid > sm_count * 16) grid = sm_count * 16;
    k_update_uv<<<dim3((unsigned)grid, 1, npairs), 256, 0, st>>>(u, v, b, g, ja, jb, its_out, ps, its_stride);
}

void launch_update_uv_fused(float* u, float* v, const PcgBuffers& b, const Geom& g, int ja, int jb,
                            int* its_out, int sm_count, cudaStream_t st, int npairs, size_t ps, int its_stride)
{
    const long long nunits = (long long)(jb - ja) * (g.pitch >> 2);
    long long grid = (nunits + 255) / 256;
    if (grid > sm_count * 16) grid = sm_count * 16;
    k_update_uv_fused<<<dim3((unsigned)grid, 1, npairs), 256, 0, st>>>(u, v, b, g, ja, jb, its_out, ps, its_stride);
}

// Blocks per pair of the batched whole-solve kernel: one per 8 warp tasks of 8 rows each, at most 8 -- a function of
// the level geometry alone.
int coop_batch_blocks(const Geom& g, int ja, int jb)
{
    const int nstrips = (g.nx + 127) / 128, nsegs = (jb - ja + 7) / 8;
    const int G = (nstrips * nsegs + 7) / 8;
    return G < 1 ? 1 : (G > 8 ? 8 : G);
}

int coop_batch_pairs_per_launch(const Geom& g, int ja, int jb, int sm_count)
{
    static int per_sm = 0;
    if (!per_sm) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg_coop_batch, 256, 0) != cudaSuccess || per_sm < 1)
            per_sm = 1;
    }
    const int n = sm_count * per_sm / coop_batch_blocks(g, ja, jb);
    return n < 1 ? 1 : n;
}

int launch_pcg_coop_batch(const PcgBuffers& b, const Geom& g, int ja, int jb, int iters, int pair0, int npairs, size_t ps,
                          double* partials, unsigned* bar, cudaStream_t st)
{
    P1Args a;
    a.b = b; a.g = g; a.ja = ja; a.jb = jb; a.cur = 0; a.store_halo = 0;
    a.nstrips = (g.nx + 127) / 128;
    a.rs = 8;
    a.nsegs = (jb - ja + a.rs - 1) / a.rs;
    CoopBatch cb;
    cb.G = coop_batch_blocks(g, ja, jb); cb.pair0 = pair0; cb.ps = ps; cb.partials = partials; cb.bar = bar;
    if (cudaMemsetAsync(bar, 0, 2 * sizeof(unsigned) * npairs, st) != cudaSuccess) return -1;
    void* args[] = { &a, &cb, &iters };
    return cudaLaunchCooperativeKernel((const void*)k_pcg_coop_batch, dim3(cb.G * npairs), dim3(256), args, 0, st) == cudaSuccess
               ? 0 : -1;
}

void launch_expand_coef(const PcgBuffers& b, const Geom& g, float* a5, float* a6, float* a7, float* a8, cudaStream_t st)
{
    dim3 grid((g.nx + 255) / 256, g.ny);
    k_expand_coef<<<grid, 256, 0, st>>>(b, g, a5, a6, a7, a8);
}

void launch_scale_copy(const float* src, float* dst, const Geom& g, int ja, int jb, float scale, cudaStream_t st)
{
    if (jb <= ja) return;
    dim3 grid((g.nx + 255) / 256, jb - ja);
    k_scale_copy<<<grid, 256, 0, st>>>(src, dst, g, ja, jb, scale);
}

}  // namespace octane
