// kernels.cuh -- host-callable launchers of the octane_b200 kernels.
#pragma once
#include "common.cuh"

namespace octane {

// Batched launches: npairs pairs whose planes lie ps floats apart (one copy of the per-pair workspace each); the
// kernels take the pair from blockIdx.z.  npairs = 1, ps = 0 is the single-pair call.
// ---- pyramid.cu
void launch_fill_gk(float* GK, float factor, int R, cudaStream_t st);
void launch_blur_decimate(const float* src, const Geom& gs, float* dst, const Geom& gd, int ja, int jb,
                          float factor, const float* GK, int R, float scale, int nc, cudaStream_t st,
                          int npairs = 1, size_t ps = 0);
// batched: pair z reads f + z * ps_in and writes gx, gy + z * ps
void launch_gradient(const float* f, float* gx, float* gy, const Geom& g, int ja, int jb, int nc, cudaStream_t st,
                     int npairs = 1, size_t ps = 0, size_t ps_in = 0);
void launch_zoom_in(const float* flow, const Geom& gc, float* out, const Geom& gf, int ja, int jb, float sf,
                    cudaStream_t st, int npairs = 1, size_t ps = 0);

// ---- build.cu
struct LevelFields {           // device planes of one level, all sharing Geom g
    const float *g1, *g1x, *g1y;                     // image 1 and its gradient   (nc planes each)
    const float *g2, *g2x, *g2y, *g2xx, *g2xy, *g2yy; // image 2 and derivatives    (nc planes each)
    float *u, *v;                                    // current flow
    const float *uh, *vh;                            // hint (first guess at this level) or nullptr
};
// Coefficient storage.  The reference's 12 CSR entries per pixel (:868-1077) hold 7 distinct
// values a1,a2,a4 (2x2 diagonal block) and a5..a8 (couplings to i-1, j-1, i+1, j+1).  The
// couplings are symmetric bit for bit -- a5(i,j) == a7(i-1,j) and a6(i,j) == a8(i,j-1), the
// half-point weights of :680-683 being the same expression with two commuted additions -- so
// only W = a7 (to i+1) and N = a8 (to j+1) are stored, unmerged; the boundary merging of
// :929-1077 (an absent neighbour's weight is added to the opposite one, which there equals
// doubling it) is applied when the stencil is evaluated.
enum { C_A1 = 0, C_A2 = 1, C_A4 = 2, C_W = 3, C_N = 4, NCOEF = 5 };
struct PcgBuffers {
    float* coef[NCOEF];        // a1, a2, a4, W, N
    float *ru, *rv;            // rhs, then residual
    float *xu, *xv;            // solution increment
    float *pu[2], *pv[2];      // search direction, ping-pong
    float *qu, *qv;            // A p
    // merged-reduction solver (pcg_fused.cu): r and p are read with row halos and rewritten by the same launch, so
    // both are double-buffered: p in pu[] / pv[] as for the two-pass kernels, r's second buffer in the planes of q
    // (that solver computes q = A p on the fly and never stores it)
    float *r2u, *r2v;
    PcgScalars* scal;          // device
    double* partials;          // device, >= 4 * max blocks
    unsigned* ticket;          // device
    int max_partial_blocks;
    double* pending;           // device [2]: rank-local dot totals awaiting the all-reduce
    int defer;                 // 1 (banded runs over NCCL): kernels leave totals in `pending`;
                               // launch_finalize applies them after the all-reduce
    P2P p2p;                   // banded runs over peer memory (world > 1): the kernels' last block
                               // exchanges the totals itself and finalises as on one GPU
    // pass 2 pushes its boundary rows of r into the neighbours' halo rows (peer memory); the
    // pointers are pre-shifted so that p[g.at(i, j)] with THIS rank's geometry lands on (i, j) there
    float *up_ru, *up_rv, *dn_ru, *dn_rv;
};
enum { FINALIZE_BUILD = 0, FINALIZE_PASS1 = 1, FINALIZE_PASS2 = 2 };
void launch_finalize(const PcgBuffers& b, int kind, float tol, cudaStream_t st);
struct BuildParams {
    double alpha, lambdadalpha, al1;
    double ralpha;             // RN(1/alpha), for the exact division shortcut of build.cu
    float lambdac;
    int dozim, nchan;
    float tol;
};
// rows [ja,jb) get coefficients + rhs; dots (b.b, b.Minv b) over rows [da,db).  Batched: pair z seeds b.scal[z] and
// uses partials region z (2 * build_partial_blocks doubles each); its image fields g1, g1x, g1y, g2, g2x, g2y lie
// z * is floats after pair 0's, every other plane z * ps.
void launch_build(const LevelFields& f, const PcgBuffers& b, const Geom& g, int ja, int jb, int da, int db,
                  const BuildParams& bp, int halo_check, cudaStream_t st, int npairs = 1, size_t ps = 0, size_t is = 0);
int build_partial_blocks(const Geom& g, int nrows);

// shared memory one block of k_blur_decimate needs for a level (pyramid.cu); levels beyond the limit are refused
// when the plan is made instead of failing at launch
constexpr size_t BLUR_DECIMATE_SMEM_LIMIT = 160 * 1024;
size_t blur_decimate_smem_bytes(float factor, int R);

// ---- pcg.cu
// One PCG iteration ki = pass1 (x += alpha_{ki-1} p_{ki-1}; p = z + beta p; q = A p; dot p.q)
// + pass2 (r -= alpha q, dots r.r and z.r, stop rule).  The x update of an iteration rides
// on the NEXT iteration's pass 1, which reads p_old anyway (saves one read of p per
// iteration); launch_update_uv applies the last pending term.  Iteration ki reads
// p[ki & 1] and writes p[(ki & 1) ^ 1].
void launch_pcg_pass1(const PcgBuffers& b, const Geom& g, int ja, int jb, int ki, int store_halo,
                      int sm_count, cudaStream_t st);
// large levels: persistent TMA-fed variant of pass 1 (pcg_tma.cu)
bool pcg_pass1_tma_usable(const Geom& g, int nrows);
// const_wn: the system comes from the first GNC stage, whose W and N planes are -1 everywhere (experimental)
void launch_pcg_pass1_tma(const PcgBuffers& b, const Geom& g, int ja, int jb, int ki, int store_halo,
                          int sm_count, cudaStream_t st, int const_wn = 0);
void launch_pcg_pass2(const PcgBuffers& b, const Geom& g, int ja, int jb, int sm_count, cudaStream_t st);
// small levels on one GPU: the whole solve (up to `iters` iterations of the same two passes, same recurrence) in one
// cooperative launch with grid-wide barriers instead of 2 x iters launches; returns 0, or -1 when the launch fails
int launch_pcg_coop(const PcgBuffers& b, const Geom& g, int ja, int jb, int iters, int sm_count, cudaStream_t st);
// small levels of a batch: pairs [pair0, pair0 + npairs) solved in one cooperative launch, coop_batch_blocks blocks
// per pair, each group with its own partials (3 G doubles) and barrier (2 unsigned, zeroed here on the stream);
// b.scal[pair] are the pairs' scalars.  Returns 0, or -1 when the launch fails.
int coop_batch_blocks(const Geom& g, int ja, int jb);
int coop_batch_pairs_per_launch(const Geom& g, int ja, int jb, int sm_count);
int launch_pcg_coop_batch(const PcgBuffers& b, const Geom& g, int ja, int jb, int iters, int pair0, int npairs, size_t ps,
                          double* partials, unsigned* bar, cudaStream_t st);
// u += x + alpha_last p_last, v likewise (:1185-1195 with the pending x term folded in).  Batched: pair z reads
// b.scal[z] and writes its_out[z * its_stride].
void launch_update_uv(float* u, float* v, const PcgBuffers& b, const Geom& g, int ja, int jb,
                      int* its_out, int sm_count, cudaStream_t st, int npairs = 1, size_t ps = 0, int its_stride = 0);
// ---- pcg_fused.cu: one launch and one reduction per iteration (merged recurrence; large levels)
bool pcg_fused_usable(const Geom& g, int nrows);
// banded runs: the neighbours' two r buffers [buffer][component] as mapped here (peer memory), shifted to this rank's
// row origin; all nullptr on one GPU and at the outer edges
struct FusedPeers {
    float *up_r[2][2], *dn_r[2][2];
};
// ki = -1: forms the first alpha (q0 = A z0, no writes); ki >= 0: iteration ki.  Reads r[ki & 1], p[ki & 1]
// (r[0] = ru / rv as the build leaves it), writes the other buffer of each pair.
// Batched: npairs pairs in one launch, the pair from blockIdx.z; pair z uses b.scal[z], its own ticket b.ticket[z] and
// partials region z (2 * b.max_partial_blocks doubles each), and its planes ps floats after pair z - 1's.  Every pair
// gets the tiling and grid of a single-pair launch, so its bits are those of a launch of that pair alone; npairs = 1 runs
// the single-pair kernels, npairs > 1 kernels compiled apart with the pair addressing.  Returns 0,
// or -1 (nothing launched) when npairs < 1 or npairs > 1 comes with banded peers.
int launch_pcg_fused(const PcgBuffers& b, const Geom& g, int ja, int jb, int ki, const FusedPeers& peers,
                     int sm_count, cudaStream_t st, int const_wn, int npairs = 1, size_t ps = 0);
// u += x (+ the pending alpha p when the iteration count is odd), after a merged-reduction solve
void launch_update_uv_fused(float* u, float* v, const PcgBuffers& b, const Geom& g, int ja, int jb,
                            int* its_out, int sm_count, cudaStream_t st, int npairs = 1, size_t ps = 0, int its_stride = 0);
// test hooks: 5-plane storage <-> the reference's 7 boundary-merged entries
void launch_expand_coef(const PcgBuffers& b, const Geom& g, float* a5, float* a6, float* a7, float* a8, cudaStream_t st);
// dense (stride nx, rows [ja,jb) starting at src row 0) <-> pitched
void launch_scale_copy(const float* src, float* dst, const Geom& g, int ja, int jb, float scale, cudaStream_t st);

// ---- nav.cu
struct NavParams {
    double pph, req, rpol, lam0;
    float xScale, xOffset, yScale, yOffset, lat1, lon1, lon0, R;
    int minX, minY;
    double t1, t2;
    int pixuv, dp, dm;
};
// tab: device scratch of pix2uv_table_doubles(nx, nrows) doubles (constants + per-column / per-row tables of the
// unmoved pixel, filled by a setup kernel on the same stream); returns the number of launches
size_t pix2uv_table_doubles(int nx, int nrows);
int launch_pix2uv(const NavParams& np, const float* u, const float* v, int nx, int row0, int nrows, double* tab,
                  short* U, short* V, short* Uraw, short* Vraw, cudaStream_t st);
// npairs whole scenes: pair b has d_navs[b] (device; the grid kind of np0 for all), dense planes b * nx * ny values
// on and its table at tab + b * pix2uv_table_doubles(nx, ny)
int launch_pix2uv_batch(const NavParams& np0, const NavParams* d_navs, int npairs, const float* u, const float* v, int nx,
                        int ny, double* tab, short* U, short* V, short* Uraw, short* Vraw, cudaStream_t st);
void launch_ctp_pack(const float* cth, short* ctp, size_t n, int ir, cudaStream_t st);


// ---- ingest.cu
struct CalParams {
    float xScale, xOffset, yScale, yOffset, radScale, radOffset;
    float rpol, req, H, lam0;                 // narrowed to float as oct_navcal_cuda's arguments are
    float fk1, fk2, bc1, bc2, kap1;
    float maxin, minin, maxout, minout;
    float subpoint_slope, subpoint_int;
    int cal, donav;
};
void launch_navcal(const short* rad, const short* x, const short* y, int nx, int ny, const CalParams& c,
                   float* data, float* lat, float* lon, cudaStream_t st);
struct Uv2PixParams {
    double secs, req, req2, rpol, rpol2, eval, lam0, pph;
    float xscale, xoffset, yscale, yoffset;
};
void launch_navcal_grid(int grid_kind, const float* data2, const short* x, const short* y, int nx, int ny, float xScale,
                        float xOffset, float yScale, float yOffset, float R, float lon0_rad, float lat1_rad, int donav,
                        float* data3, float* lat, float* lon, cudaStream_t st);
void launch_zoom_in_float(const float* in, int nx, int ny, float* out, int nxx, int nyy, int interp, cudaStream_t st);
// oct_zoom_out_float: taps == nullptr selects the copy branch (factor >= 0.999999); returns the number of launches
struct ZoomOutTaps {
    int R;
    double gk[2 * 32 + 1];
};
int launch_zoom_out_float(const float* in, int nx, int ny, float* out, int nxx, int nyy, double factor,
                          const ZoomOutTaps* taps, double* tmp_a, double* tmp_b, cudaStream_t st);
void launch_uv2pix(float* u, float* v, const float* lat, const float* lon, const short* xs, const short* ys, int nx,
                   int ny, const Uv2PixParams& q, cudaStream_t st);


// ---- post.cu
// -srsal: 37 x 37 bilateral filter of the pixel displacements, weights from the cloud-top heights
struct SrsalTaps {
    double gk[37];
    double sigpix2;
};
// u, v, cth: dense rows [e0, ...) of the scene; u_out, v_out: dense rows [o0, o1).  Every row the window of an
// output row reads (after reflection at the scene edges 0 and ny) must be present in the inputs.  Batched: npairs
// pairs, every input and output plane of pair z ps floats after pair 0's.
void launch_srsal(const float* u, const float* v, const float* cth, int nx, int ny, int e0, int o0, int o1,
                  const SrsalTaps& t, float* u_out, float* v_out, cudaStream_t st, int npairs = 1, size_t ps = 0);

}  // namespace octane
