/* octane_b200.h -- C ABI of the B200-native OCTANE dense variational
 * optical-flow path (liboctane_b200.so).
 *
 * Plain C: pointers, sizes and POD structs only; no C++ / torch types.  Every
 * entry point returns 0 on success and a negative OCTANE_E* code on failure
 * (the reference prints and exit()s, or ignores CUDA errors:
 * src/oct_variational_optical_flow.cu:1255-1266,1421,1431); nothing here ever
 * calls exit().  There is NO CPU fallback: without a CUDA device every compute
 * entry point fails with OCTANE_ENODEV.
 *
 * Reference interfaces replaced (paths relative to the reference tree):
 *   octane_variational_flow*   void oct_variational_optical_flow(Image,Image,float*CTH,
 *                              float*u,float*v,int nx,int ny,int nc,OFFlags)
 *                              src/oct_variational_optical_flow.cu:1213
 *   octane_pix2uv*             void oct_pix2uv_cuda(GOESVar&,double t2,float*u,float*v,
 *                              short*ur,short*vr,short*ur2,short*vr2,OFFlags)
 *                              src/oct_pix2uv_cuda.cu:265
 *   octane_optical_flow        int oct_optical_flow(GOESVar&,GOESVar&,OFFlags&)
 *                              src/oct_optical_flow.cc:21 (variational branch + CTP pack + navigation)
 *   octane_params              the OFFlags fields the path reads, include/offlags.h:4-72
 *                              (src/oct_variational_optical_flow.cu:1229-1241,
 *                               src/oct_pix2uv_cuda.cu:279,291-297)
 *   octane_nav                 GOESNAVVar, include/goesread.h:3-14 (fields read by
 *                              src/oct_pix2uv_cuda.cu:27-172,295)
 *   octane_navcal*             void oct_navcal_cuda(short*data2,short*data2s,short*x,short*y,short*xs,
 *                              short*ys,int nx,int ny,int minx,int maxx,int miny,int maxy,float*data3,
 *                              float*lat,float*lon,string cal,int datf,float xScale,...,int donav,OFFlags)
 *                              src/oct_navcal_cuda.cu:100 (called by oct_goesread, src/oct_fileread.cc:383)
 *   octane_uv2pix*             void oct_uv2pix(GOESVar&,float*u,float*v,double t2,OFFlags)
 *                              src/oct_pix2uv_cuda.cu:372 (first-guess winds -> pixel displacements)
 *   octane_navcal_grid         void oct_polar_navcal_cuda(float*data2,short*,short*x,short*y,short*,short*,int nx,int ny,
 *                              int,int,int,int,float*data3,float*lat,float*lon,float xScale,float xOffset,float yScale,
 *                              float yOffset,float lon0,float lat1,float R,int donav,int chan,OFFlags)
 *                              src/oct_polar_navcal_cuda.cu:69, and oct_merc_navcal_cuda(... float lon0,float R,int donav,
 *                              OFFlags) src/oct_merc_navcal_cuda.cu:51 (ingest of the -Polar / -Merc grids)
 *   octane_band_minmax         void oct_bandminmax(int,float&,float&), src/oct_normalize_geo.cc:9
 *   octane_zoom_in_float       void oct_zoom_in_float(float*flow,float*flowout,int nx,int ny,int nxx,int nyy,
 *                              int cnum,int interp), src/oct_zoom.cc:180 (cloud-top heights / extra channels
 *                              on a coarser grid, src/oct_fileread.cc:370,796)
 *   octane_zoom_out_float      void oct_zoom_out_float(float*image,float*imageout,int nx,int ny,double factor,
 *                              int verb,int cnum), src/oct_zoom.cc:51 (cloud-top heights / extra channels
 *                              on a FINER grid, src/oct_fileread.cc:379,805); octane_zoom_out_size is
 *                              oct_zoom_size, src/oct_zoom.cc:12
 *   octane_srsal*              void oct_srsal_cu(float*upix,float*vpix,float*CTHsub21,int nx,int ny,OFFlags)
 *                              src/oct_srsal_cuda.cu:73 (-srsal, called by oct_optical_flow.cc:100-105)
 * Image layout everywhere: row-major float32, index i + nx*j (+ nx*ny*c), i = x
 * (fastest), as the reference (src/oct_variational_optical_flow.cu:316-320).
 *
 * Environment variables the library reads (all optional; none changes a result):
 *   OCTANE_NCCL_LIB       path of libnccl.so.2 when neither the host process nor the loader path has one
 *   OCTANE_COMM=nccl      banded runs: per-iteration exchanges over NCCL instead of peer memory (and the two-pass kernels)
 *   OCTANE_STREAM_DEFER   0 / 1: force the copy-out schedule of octane_stream_submit (default: deferred on banded
 *                         contexts only, see there); used by the tests to run the banded schedule on one GPU
 *   OCTANE_DUMP_EVENTS    file that receives the per-launch event times of a profiled call (octane_ctx_set_profile)
 */
#ifndef OCTANE_B200_H
#define OCTANE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCTANE_ABI_VERSION 3   /* 2: octane_params.dosrsal appended; zoom-out and srsal entry points
                                  3: octane_ctx_set_solver; octane_stats.pcg_solver, finest_pass1_bytes_per_px appended */

enum {
    OCTANE_OK = 0,
    OCTANE_ENODEV = -1,   /* no CUDA device (reference: prints + exit(0)) */
    OCTANE_EINVAL = -2,   /* bad argument */
    OCTANE_ENOMEM = -3,   /* device allocation failed */
    OCTANE_ECUDA = -4,    /* CUDA runtime error (octane_last_error has the text) */
    OCTANE_EHALO = -5,    /* banded run: a warp left the band's halo (raise max_disp) */
    OCTANE_ECOMM = -6     /* NCCL missing or failed */
};

/* OFFlags subset.  Defaults = src/main.cc:53-108. */
typedef struct octane_params {
    double alpha;      /* -alpha   smoothness weight            (5)   */
    double lambda;     /* -lambda  gradient-constancy weight    (1)   */
    double lambdac;    /* -lambdac first-guess hinting weight   (0)   */
    double scaleF;     /* pyramid scale factor                  (0.5) */
    double scsig;      /* deprecated, carried for layout parity (400) */
    int kiters;        /* -kiters  pyramid levels               (4)   */
    int liters;        /* -liters  inner iterations per GNC step(3)   */
    int cgiters;       /* PCG iteration cap                     (30)  */
    int dozim;         /* Zimmer normalisation, 0 with -brox    (1)   */
    int setdevice;     /* 0-based CUDA device                   (0)   */
    int pixuv;         /* -pd: U,V = 100*pixel displacement     (0)   */
    int dopolar;       /* -Polar                                (0)   */
    int domerc;        /* -Merc                                 (0)   */
    int first_guess;   /* 1: u/v inputs hold a first guess (reference semantics of the
                          in/out arrays); 0: start from zero without reading them,
                          which is what oct_optical_flow.cc:38-48 feeds the solver */
    int max_disp;      /* banded (multi-GPU) runs: bound on |v| in full-res pixels that
                          sizes the image-2 warp halo                (64) */
    int doCTH;         /* -i1cth: pack CTP                      (0)   */
    int ir;            /* -ir: CTP = (CTH-300)*100              (0)   */
    int dosrsal;       /* -srsal: bilateral post-smoothing of the pixel displacements
                          by the dispatcher, needs cth           (0)   */
} octane_params;

/* GOESNAVVar subset (double/float split as in the reference: the float fields
 * take part in float arithmetic, src/oct_pix2uv_cuda.cu:40-41,99-100). */
typedef struct octane_nav {
    double pph, req, rpol, lam0;
    float xScale, xOffset, yScale, yOffset;
    float g2xOffset, g2yOffset;          /* file-2 offsets: sector-moved guard, :295 */
    float lat1, lon1, lon0, R;           /* polar / Mercator constants */
    int minX, minY;                      /* sector origin added to the pixel index, :192 */
} octane_nav;

/* Calibration / normalisation constants of one GOES-R L1b channel: the scalar arguments of
 * oct_navcal_cuda (src/oct_navcal_cuda.cu:100-107) that are not already in octane_nav.
 * The reference narrows req, rpol, pph+req and lam0 to float for this kernel; the library
 * does the same from octane_nav. */
typedef struct octane_cal {
    float radScale, radOffset;           /* Rad:scale_factor, Rad:add_offset */
    float fk1, fk2, bc1, bc2, kap1;      /* planck_fk1/fk2/bc1/bc2, kappa0 */
    float maxin, minin;                  /* band radiance range (octane_band_minmax) */
    float maxout, minout;                /* 255, 0 (src/oct_fileread.cc:341-342) */
    float H;                             /* pph + req summed in float (src/oct_fileread.cc:306); 0: the
                                            library forms it from octane_nav the same way */
    int cal;                             /* 0 RAW (the only mode main.cc uses), 1 TEMP, 2 REF, 3 BRIT */
    int donav;                           /* 1: fill lat/lon; 0: zeros */
} octane_cal;

/* Per-call statistics (filled by the last solve on the context). */
#define OCTANE_MAX_SOLVES 256
typedef struct octane_stats {
    int n_levels;
    int n_solves;                         /* kiters*3*liters */
    int level_nx[16], level_ny[16];
    int cg_iterations[OCTANE_MAX_SOLVES]; /* PCG iterations actually executed per solve */
    long long kernel_launches;            /* our kernels launched by the last call */
    double algorithmic_bytes;             /* DESIGN.md section 4: compulsory HBM bytes of the call on this rank */
    /* profile mode (octane_ctx_set_profile): CUDA-event timings on our stream */
    double ms_total;                      /* whole call, device side */
    double ms_pyramid, ms_build, ms_pcg_pass1, ms_pcg_pass2, ms_update, ms_nav;
    long long n_pcg_pass1, n_pcg_pass2;   /* launches that did work (not early-exited) */
    double finest_pass1_ms, finest_pass2_ms;   /* average per working launch, finest level */
    long long finest_pixels;              /* pixels one finest-level launch covers on this rank */
    int pcg_solver;                       /* kernels the finest level ran: 1 merged reduction (one launch per iteration,
                                             timed as "pass1", no pass 2), 0 the two-pass kernels */
    double finest_pass1_bytes_per_px;     /* algorithmic bytes per pixel, averaged over the launches finest_pass1_ms averages */
} octane_stats;

typedef struct octane_ctx octane_ctx;

/* library / device */
int         octane_abi_version(void);
const char* octane_last_error(void);
int         octane_device_count(void);
void        octane_params_default(octane_params* p);

/* A context owns a CUDA stream and a reusable device workspace (the reference
 * allocates and frees 37 managed buffers per call, :1268-1328,1441-1472). */
int  octane_ctx_create(octane_ctx** ctx, int device);
void octane_ctx_destroy(octane_ctx* ctx);
int  octane_ctx_set_profile(octane_ctx* ctx, int on);      /* per-stage CUDA-event timing */
int  octane_ctx_set_graphs(octane_ctx* ctx, int on);       /* CUDA-graph the PCG loop (default on) */
/* PCG kernels of the large levels.  1 (default): the merged form of the reference's recurrence -- one launch and one
 * reduction phase per iteration, 68-84 B/px; the same Krylov iterate as the reference's loop
 * (src/oct_variational_optical_flow.cu:1131-1182) up to fp32 rounding (measured: its own run-to-run noise).
 * 0: that loop literally, two launches per iteration, 100 B/px.  Small levels always run 0. */
int  octane_ctx_set_solver(octane_ctx* ctx, int solver);
int  octane_get_stats(octane_ctx* ctx, octane_stats* out);
int  octane_ctx_synchronize(octane_ctx* ctx);
void* octane_ctx_stream(octane_ctx* ctx);                  /* the cudaStream_t all work is ordered on */
size_t octane_workspace_bytes(int nx, int ny, int nc, const octane_params* p);

/* Pyramid geometry: level k has factor scaleF^(kiters-1-k) and size
 * (int)(n*factor+0.5) (src/oct_variational_optical_flow.cu:50-54,488-489). */
int octane_level_dims(int nx, int ny, const octane_params* p, int k, int* xi, int* yi);

/* ---- host-buffer entry points (blocking; copies inside) ---------------- */

/* u,v: in = first guess if p->first_guess, out = flow in pixels. */
int octane_variational_flow(octane_ctx* ctx, const float* img1, const float* img2,
                            int nx, int ny, int nc, const octane_params* p,
                            float* u_inout, float* v_inout);

/* U,V = (short)(100*m/s) (or 100*pixels with pixuv); U_raw,V_raw = (short)(100*pixels).
 * Returns 1 (not an error) when the sector-moved guard zeroed the outputs. */
int octane_pix2uv(octane_ctx* ctx, const octane_nav* nav, double t1, double t2,
                  const float* u, const float* v, int nx, int ny, const octane_params* p,
                  short* U, short* V, short* U_raw, short* V_raw, float* dT);

/* Dispatcher: solve + CTP pack + navigation with the flow kept on the device
 * between the two stages.  cth/ctp may be NULL when !p->doCTH (cth is also needed by
 * p->dosrsal, which smooths upix/vpix AFTER the navigation as oct_optical_flow.cc:91-105 does:
 * U, V, U_raw, V_raw come from the unsmoothed flow). */
int octane_optical_flow(octane_ctx* ctx, const float* img1, const float* img2, const float* cth,
                        int nx, int ny, int nc, const octane_nav* nav, double t1, double t2,
                        const octane_params* p, float* upix_inout, float* vpix_inout,
                        short* U, short* V, short* U_raw, short* V_raw, short* ctp, float* dT);

/* Ingest: Rad counts -> 0..255 normalised brightness with the limb taper, and the latitude /
 * longitude (degrees) of every pixel.  rad: ny*nx shorts; x: nx, y: ny fixed-grid counts;
 * data/lat/lon: ny*nx floats out (lat and lon may both be NULL to skip navigation). */
int octane_navcal(octane_ctx* ctx, const short* rad, const short* x, const short* y, int nx, int ny,
                  const octane_nav* nav, const octane_cal* cal, float* data, float* lat, float* lon);
/* Ingest of the projected grids: grid 1 = orthographic polar (uses nav->lon0, nav->lat1, nav->R, degrees /
 * metres as GOESNAVVar holds them), grid 2 = spherical Mercator (nav->lon1 in degrees, nav->R).  The float
 * image passes through to data_out; lat/lon (degrees) may both be NULL. */
int octane_navcal_grid(octane_ctx* ctx, int grid, const float* data, const short* x, const short* y, int nx, int ny,
                       const octane_nav* nav, int donav, float* data_out, float* lat, float* lon);
/* ABI band table: radiance range used for the normalisation; returns 0, or -2 for an unknown band
 * (the reference leaves maxch/minch uninitialised there). */
int octane_band_minmax(int band, float* maxch, float* minch);
/* First-guess winds (m/s, navigated) -> pixel displacements over t2-t1, in place.  lat/lon as
 * octane_navcal produced them; x, y the fixed-grid counts.  All zeros when the sector moved
 * (exact comparison of the offsets, src/oct_pix2uv_cuda.cu:421). */
int octane_uv2pix(octane_ctx* ctx, const octane_nav* nav, double t1, double t2,
                  const float* lat, const float* lon, const short* x, const short* y,
                  int nx, int ny, const octane_params* p, float* u_inout, float* v_inout);

/* Regrid a coarser ancillary field (nx*ny) onto the image grid (nxx*nyy >= nx*ny): bicubic when
 * interp == 1 (default of the reference, -nncth selects 0 = nearest neighbour). */
int octane_zoom_in_float(octane_ctx* ctx, const float* in, int nx, int ny, float* out, int nxx, int nyy, int interp);

/* Regrid a FINER ancillary field (nx*ny) down to the image grid: Gaussian blur (sigma = 0.6 sqrt(1/factor^2 - 1),
 * radius max(5, (int)(2 sigma)), +R tap dropped) and bicubic sampling at (ii/factor, jj/factor), all in double as
 * the reference's CPU code; factor in (0, 1], >= 0.999999 copies.  out: dense nxx*nyy plane with (nxx, nyy) from
 * octane_zoom_out_size (the reference stores it at imageout + cnum -- an element, not a plane, offset; placing the
 * plane is the caller's business here).  Bit-identical to the reference's CPU object. */
int octane_zoom_out_size(int nx, int ny, double factor, int* nxx, int* nyy);
int octane_zoom_out_float(octane_ctx* ctx, const float* in, int nx, int ny, float* out, double factor);

/* -srsal: 37 x 37 bilateral filter (spatial sigma 9 px, range sigma 20 in the units of cth) of the pixel
 * displacements, in place.  nx, ny must exceed 18 (below that the reference's reflected index leaves the array). */
int octane_srsal(octane_ctx* ctx, float* u_inout, float* v_inout, const float* cth, int nx, int ny);

/* ---- device-pointer entry points (stream-ordered on the ctx stream) ----- */
/* All pointers are device memory on the context's device, dense (stride nx). */
int octane_variational_flow_dev(octane_ctx* ctx, const float* d_img1, const float* d_img2,
                                int nx, int ny, int nc, const octane_params* p,
                                float* d_u_inout, float* d_v_inout);
int octane_pix2uv_dev(octane_ctx* ctx, const octane_nav* nav, double t1, double t2,
                      const float* d_u, const float* d_v, int nx, int ny, const octane_params* p,
                      short* d_U, short* d_V, short* d_U_raw, short* d_V_raw);
/* The dispatcher on device buffers (solve + CTP pack + navigation, nothing copied, no host synchronisation):
 * what a pipeline over many pairs calls, one context (= stream + workspace) per pair in flight.
 * d_cth / d_ctp may be NULL when !p->doCTH. */
int octane_optical_flow_dev(octane_ctx* ctx, const float* d_img1, const float* d_img2, const float* d_cth,
                            int nx, int ny, int nc, const octane_nav* nav, double t1, double t2,
                            const octane_params* p, float* d_upix_inout, float* d_vpix_inout,
                            short* d_U, short* d_V, short* d_U_raw, short* d_V_raw, short* d_ctp);
/* Many same-size pairs in one call: each pair is solved, its CTP packed and its flow navigated exactly as
 * octane_optical_flow_dev does, with one launch per stage for the whole batch.  Arrays are dense and pair-major:
 * images npairs x nc x ny x nx, d_cth and every output npairs x ny x nx; nav, t1 and t2 are host arrays of npairs.
 * Small pyramid levels solve all pairs in one cooperative launch (each pair on its own group of blocks, with its own
 * barrier and stop rule).  Large levels (nx >= 512, >= 64 rows) under the default solver (octane_ctx_set_solver 1)
 * run one PCG launch per iteration for all pairs, each pair on the grid and tiling it would get alone, with its own
 * reductions and stop rule (a converged pair's blocks exit at once), replayed from a CUDA graph; under solver 0 they
 * run the two-pass kernels pair by pair.  A pair's result does not depend on the other pairs of the call, nor on
 * their number.  Stream-ordered, no host
 * synchronisation; moved_out (host, npairs, may be NULL) gets 1 for each pair whose sector moved (its four short
 * planes are zero).  OCTANE_EINVAL for npairs < 1, a first guess, dosrsal or a banded context (a first guess and
 * -srsal go through octane_optical_flow_batch_ex_dev, which shares this call's body); OCTANE_ENOMEM when the npairs
 * workspaces do not fit.  The context stays usable after either.  octane_get_stats then reports the call's kernel
 * launches and pair 0's iteration counts. */
int octane_optical_flow_batch_dev(octane_ctx* ctx, int npairs, const float* d_img1, const float* d_img2,
                                  const float* d_cth, int nx, int ny, int nc, const octane_nav* nav,
                                  const double* t1, const double* t2, const octane_params* p,
                                  float* d_upix, float* d_vpix, short* d_U, short* d_V, short* d_U_raw,
                                  short* d_V_raw, short* d_ctp, int* moved_out);
/* octane_optical_flow_batch_dev with a first guess and -srsal: per pair, what octane_optical_flow_dev does with the
 * same flags.  With neither flag set the results are octane_optical_flow_batch_dev's, bit for bit.
 * - p->first_guess: d_fg_u / d_fg_v (npairs x ny x nx, only read; NULL otherwise) are each pair's first guess.  They
 *   may be d_upix / d_vpix themselves (octane_optical_flow_dev's in/out convention): they are copied into the
 *   workspaces before any output is written.  The hint term is built on the levels with lambdac != 0.
 * - p->dosrsal: each pair's d_upix / d_vpix is smoothed with its own heights d_cth (npairs x ny x nx), in one launch
 *   for all pairs, after the CTP pack and the navigation: the short planes and CTP come from the unsmoothed flow.
 *   A pair whose sector moved is smoothed too.
 * OCTANE_EINVAL for npairs < 1, first_guess without both fg pointers, dosrsal without d_cth or with nx or ny <= 18,
 * doCTH without d_cth / d_ctp and a banded context; OCTANE_ENOMEM when the workspaces or the -srsal staging
 * (2 x npairs x ny x nx floats) do not fit.  Every allocation is made before anything is enqueued: the context stays
 * usable after any refusal. */
int octane_optical_flow_batch_ex_dev(octane_ctx* ctx, int npairs, const float* d_img1, const float* d_img2,
                                     const float* d_fg_u, const float* d_fg_v, const float* d_cth,
                                     int nx, int ny, int nc, const octane_nav* nav,
                                     const double* t1, const double* t2, const octane_params* p,
                                     float* d_upix, float* d_vpix, short* d_U, short* d_V, short* d_U_raw,
                                     short* d_V_raw, short* d_ctp, int* moved_out);
/* A sequence of nframes same-size frames (d_frames: nframes x nc x ny x nx, dense), solved as its nframes - 1
 * consecutive pairs: pair k is (frame k, frame k + 1) with t1 = t[k], t2 = t[k + 1] (t: host array of nframes).
 * Per pair, the results are octane_optical_flow_batch_ex_dev's on those pairs, bit for bit, with the same flags,
 * refusals (OCTANE_EINVAL also for nframes < 2) and guarantees; nav (host) and moved_out have one entry per pair (pair
 * k's nav carries frame k + 1's g2xOffset / g2yOffset), and d_fg_u, d_fg_v, d_cth (image 1's heights of each pair) and
 * every output are (nframes - 1) x ny x nx.  Each frame is copied in, blurred, decimated and differentiated once
 * instead of twice, in a workspace of nframes instead of 2 (nframes - 1) image slots (octane_batch_workspace_bytes).
 * octane_batch_cg_iterations (npairs = nframes - 1) and octane_get_stats work afterwards as after a batch. */
int octane_optical_flow_sequence_dev(octane_ctx* ctx, int nframes, const float* d_frames,
                                     const float* d_fg_u, const float* d_fg_v, const float* d_cth,
                                     int nx, int ny, int nc, const octane_nav* nav, const double* t,
                                     const octane_params* p, float* d_upix, float* d_vpix, short* d_U, short* d_V,
                                     short* d_U_raw, short* d_V_raw, short* d_ctp, int* moved_out);
/* Device bytes a batched call (sequence = 0) or a sequence call (sequence = 1) of npairs pairs allocates on a fresh
 * context of a 148-SM B200: the workspace, the per-pair scalars, partial sums and iteration counts, the navigation
 * tables and, with p->dosrsal, the -srsal staging.  Host arithmetic, no device needed; 0 for invalid arguments. */
size_t octane_batch_workspace_bytes(int npairs, int sequence, int nx, int ny, int nc, const octane_params* p);
/* PCG iterations of every solve of every pair of the last batched call (any of the three above):
 * its[pair * n_solves + solve].  npairs must be that call's.  Synchronises the context's stream. */
int octane_batch_cg_iterations(octane_ctx* ctx, int* its, int npairs);

int octane_navcal_dev(octane_ctx* ctx, const short* d_rad, const short* d_x, const short* d_y, int nx, int ny,
                      const octane_nav* nav, const octane_cal* cal, float* d_data, float* d_lat, float* d_lon);
int octane_zoom_in_float_dev(octane_ctx* ctx, const float* d_in, int nx, int ny, float* d_out, int nxx, int nyy, int interp);
int octane_zoom_out_float_dev(octane_ctx* ctx, const float* d_in, int nx, int ny, float* d_out, double factor);
int octane_srsal_dev(octane_ctx* ctx, float* d_u_inout, float* d_v_inout, const float* d_cth, int nx, int ny);
int octane_uv2pix_dev(octane_ctx* ctx, const octane_nav* nav, double t1, double t2,
                      const float* d_lat, const float* d_lon, const short* d_x, const short* d_y,
                      int nx, int ny, const octane_params* p, float* d_u_inout, float* d_v_inout);

/* ---- stage entry points (device pointers; used by the parity tests) ----- */
int octane_stage_blur_decimate(octane_ctx* ctx, const float* d_img, int nx, int ny, int nc,
                               float factor, float* d_out /* nxx*nyy*nc dense */);
int octane_stage_gradient(octane_ctx* ctx, const float* d_f, int xi, int yi, int nc,
                          float* d_gx, float* d_gy);
int octane_stage_zoom_in(octane_ctx* ctx, const float* d_flow, int nx, int ny, int nxx, int nyy,
                         float sf, float* d_out);
/* coef: 7 dense planes [a1,a2,a4,a5,a6,a7,a8] = the distinct entries of the reference's CSR rows
 * with its boundary merging applied (src/oct_variational_optical_flow.cu:929-1077).  The library
 * stores 5 of them (a5, a6 are their neighbours' a7, a8); octane_stage_build expands, and
 * octane_stage_pcg expects a system of that structure (symmetric couplings, mirror-merged edges). */
int octane_stage_build(octane_ctx* ctx, const float* d_u, const float* d_v,
                       const float* d_uh, const float* d_vh,
                       const float* d_g1, const float* d_g2, int xi, int yi, int nc,
                       const octane_params* p, float lambdac_level, int gnc,
                       float* d_coef, float* d_bu, float* d_bv);
int octane_stage_pcg(octane_ctx* ctx, const float* d_coef, const float* d_bu, const float* d_bv,
                     int xi, int yi, int iters, float tol, float* d_xu, float* d_xv, int* iterations);

/* ---- row-band multi-GPU (one process per GPU) --------------------------- */
/* Rank r of `world` owns finest-level rows [own0,own1) and must supply
 * full-resolution input rows [in0,in1) (band + blur/gradient/warp overlap). */
int octane_band_plan(int nx, int ny, const octane_params* p, int rank, int world,
                     int* own0, int* own1, int* in0, int* in1);
/* NCCL bootstrap: rank 0 calls octane_comm_unique_id, the host framework
 * broadcasts the 128 bytes, every rank calls octane_comm_init. */
int octane_comm_unique_id(char id[128]);
int octane_comm_init(octane_ctx* ctx, const char id[128], int rank, int world);
int octane_comm_rank(octane_ctx* ctx, int* rank, int* world);
/* d_img*: rows [in0,in1) dense; d_u/d_v: rows [own0,own1) dense (in/out). */
int octane_variational_flow_band_dev(octane_ctx* ctx, const float* d_img1_band, const float* d_img2_band,
                                     int nx, int ny, int nc, const octane_params* p,
                                     float* d_u_band_inout, float* d_v_band_inout);
/* The same with a first guess (p->first_guess = 1, optionally p->lambdac): d_fg_u / d_fg_v hold rows [in0,in1) of the
 * first-guess displacement field (band + overlap, like the images: the hint field of every level is blurred and
 * decimated from them locally, nothing is exchanged); d_u / d_v receive rows [own0,own1) of the flow. */
int octane_variational_flow_band_fg_dev(octane_ctx* ctx, const float* d_img1_band, const float* d_img2_band,
                                        const float* d_fg_u_band, const float* d_fg_v_band,
                                        int nx, int ny, int nc, const octane_params* p,
                                        float* d_u_band_out, float* d_v_band_out);
/* rows [row0,row0+nrows) of an nx-wide scene; d_u etc. hold just those rows */
int octane_pix2uv_band_dev(octane_ctx* ctx, const octane_nav* nav, double t1, double t2,
                           const float* d_u, const float* d_v, int nx, int row0, int nrows,
                           const octane_params* p,
                           short* d_U, short* d_V, short* d_U_raw, short* d_V_raw);
/* -srsal on row bands (collective over the context's communicator): d_u / d_v (in/out) and d_cth hold the owned rows
 * [own0,own1) of octane_band_plan, dense.  Each rank stages its rows with 18 more on each side, exchanges those with
 * its neighbours and filters its own rows: the gathered result is bit for bit octane_srsal_dev on the whole scene.
 * Every band must be at least 18 rows high (else OCTANE_EINVAL on every rank) and nx, ny must exceed 18.  A rank
 * that cannot allocate its staging makes every rank return an error; the contexts stay usable.  World 1: exactly
 * octane_srsal_dev.  Synchronises the host with the context's stream (the vote on the staging). */
int octane_srsal_band_dev(octane_ctx* ctx, float* d_u_own, float* d_v_own, const float* d_cth_own, int nx, int ny);

/* ---- pipelined host-buffer dispatcher (sequences of pairs; one GPU or row bands) -------
 * The reference processes one pair per run (src/main.cc:439 -> oct_optical_flow, src/oct_optical_flow.cc:21);
 * an archive or a 1-minute mesoscale sequence is a loop over pairs.  octane_stream_submit enqueues, for one pair,
 * copy-in -> solve -> CTP pack -> navigation -> copy-out on three streams and returns; octane_stream_wait blocks
 * until that pair's outputs are in host memory.  Two pairs may be in flight (slot 0 / 1), so the copies of one
 * pair run under the solve of the other.  Host buffers must be pinned for the overlap to happen and stay valid
 * until the wait returns.  img*: rows [in0,in1) of octane_band_plan (the whole scene on one GPU); every output:
 * rows [own0,own1).  upix/vpix may both be NULL (the reference writes them only with -pd).  p->dosrsal needs cth_own
 * and upix/vpix: as in octane_optical_flow the navigation runs on the unsmoothed flow and -srsal then smooths the
 * pixel displacements (on row bands after an 18-row exchange with the neighbours, as octane_srsal_band_dev; every
 * band must be at least 18 rows high).  A first guess goes through octane_stream_submit_fg; here p->first_guess is
 * OCTANE_EINVAL.  In banded runs every rank submits the same sequence; there a pair's copy-out is enqueued by the NEXT
 * submit, to start when that pair's solve reaches its finest level (a device-to-host copy in flight slows the
 * system-scope fences of the short coarse-level iterations), or by octane_stream_wait if no submit followed.
 * Returns 1 when the sector-moved guard zeroed the navigated outputs. */
int octane_stream_submit(octane_ctx* ctx, int slot, const float* img1_band, const float* img2_band, const float* cth_own,
                         int nx, int ny, int nc, const octane_nav* nav, double t1, double t2, const octane_params* p,
                         float* upix_own, float* vpix_own, short* U, short* V, short* U_raw, short* V_raw, short* ctp_own);
/* The same with a first guess (p->first_guess = 1, optionally p->lambdac): fg_u_band / fg_v_band are host rows
 * [in0,in1) of the first-guess displacement field, like the images (and like octane_variational_flow_band_fg_dev);
 * they are only read, and must stay valid until the wait returns.  upix/vpix receive the flow. */
int octane_stream_submit_fg(octane_ctx* ctx, int slot, const float* img1_band, const float* img2_band,
                            const float* fg_u_band, const float* fg_v_band, const float* cth_own, int nx, int ny, int nc,
                            const octane_nav* nav, double t1, double t2, const octane_params* p,
                            float* upix_own, float* vpix_own, short* U, short* V, short* U_raw, short* V_raw, short* ctp_own);
int octane_stream_wait(octane_ctx* ctx, int slot);

#ifdef __cplusplus
}
#endif
#endif /* OCTANE_B200_H */
