// ctx.cu -- context, workspace, coarse-to-fine driver and the C ABI of
// include/octane_b200.h.
//
// Host-side counterpart of the reference's wrapper
// oct_variational_optical_flow (src/oct_variational_optical_flow.cu:1213-1473)
// and of the level / GNC / inner-iteration control flow that the reference
// runs inside its single cooperative kernel (:487-1210).  Here the control
// flow lives on the host as a stream of kernel launches (the PCG loop replayed
// from a CUDA graph), with every data-dependent decision (stop rule, alpha,
// beta) taken on the device, so the host never synchronises inside a solve.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/octane_b200.h"
#include "comm.h"
#include "kernels.cuh"

using namespace octane;

namespace {

thread_local char g_err[512] = "";
void set_err(const char* fmt, const char* a = "", const char* b = "")
{
    snprintf(g_err, sizeof g_err, fmt, a, b);
}

#define CUDA_OK(call)                                                                  \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            set_err("%s: %s", #call, cudaGetErrorString(e_));                          \
            return (e_ == cudaErrorMemoryAllocation) ? OCTANE_ENOMEM : OCTANE_ECUDA;   \
        }                                                                              \
    } while (0)

// ---- pyramid geometry (:50-54, :488, :521-526) -------------------------------------
float level_factor(const octane_params& p, int k)
{
    float sf = (float)p.scaleF;
    return (float)pow((double)sf, (double)(p.kiters - k - 1));
}
void zoom_size(int nx, int ny, float factor, int* nxx, int* nyy)
{
    double f = (double)factor;
    *nxx = (int)((double)nx * f + 0.5);
    *nyy = (int)((double)ny * f + 0.5);
}
int filter_radius(float factor)
{
    float sigma = (float)(1.0 / sqrt(2. * (double)factor));
    int filtsize = (int)(2 * sigma);
    if (filtsize < 5) filtsize = 5;
    return filtsize;
}

constexpr int HALO_UV = 4;   // rows of u,v kept valid beyond the owned band (3x3 build + bicubic prolongation)

struct Level {
    float factor;
    int R;
    int own0, own1;          // rows this rank solves
    Geom g;                  // local storage
    float lambdac;
    // peer-memory runs: the neighbours' r planes, shifted so that p[g.at(i, j)] with THIS rank's
    // geometry addresses (i, j) in the neighbour's plane (nullptr at the outer edges)
    float *up_ru = nullptr, *up_rv = nullptr, *dn_ru = nullptr, *dn_rv = nullptr;
    FusedPeers fp = {};      // the same for the merged-reduction solver: both buffers of r and q
};

struct Plan {
    int nx = 0, ny = 0, nc = 0, rank = 0, world = 1;
    octane_params p;
    std::vector<Level> lv;
    int in0 = 0, in1 = 0;    // full-res input rows needed (== finest level's local rows)
    size_t P = 0, Pc = 0;    // plane sizes (floats): finest, second finest
    // only what shapes the workspace, the graphs and the band geometry: a change of pixuv / doCTH / ir / dosrsal /
    // setdevice (or of struct padding) must not force a re-plan -- in banded runs a re-plan is a collective
    bool same(int nx_, int ny_, int nc_, const octane_params& q, int rank_, int world_) const
    {
        return nx == nx_ && ny == ny_ && nc == nc_ && rank == rank_ && world == world_ &&
               p.alpha == q.alpha && p.lambda == q.lambda && p.lambdac == q.lambdac && p.scaleF == q.scaleF &&
               p.kiters == q.kiters && p.liters == q.liters && p.cgiters == q.cgiters && p.dozim == q.dozim &&
               p.first_guess == q.first_guess && p.max_disp == q.max_disp;
    }
};

int make_plan(Plan& pl, int nx, int ny, int nc, const octane_params& p, int rank, int world)
{
    if (nx < 4 || ny < 4 || nc < 1 || nc > 3 || p.kiters < 1 || p.kiters > 16 || p.liters < 0 ||
        p.cgiters < 0 || !(p.scaleF > 0.0 && p.scaleF < 1.0) || !(p.alpha > 0.0) ||
        p.kiters * 3 * p.liters > OCTANE_MAX_SOLVES) {
        set_err("invalid size or parameters");
        return OCTANE_EINVAL;
    }
    pl.nx = nx; pl.ny = ny; pl.nc = nc; pl.rank = rank; pl.world = world; pl.p = p;
    const int K = p.kiters;
    pl.lv.assign(K, Level());
    const float lambdaco = (float)(p.lambdac / p.alpha);      // :1236
    int in0 = ny, in1 = 0;
    for (int k = 0; k < K; k++) {
        Level& L = pl.lv[k];
        L.factor = level_factor(p, k);
        L.R = filter_radius(L.factor);
        int xi, yi;
        zoom_size(nx, ny, L.factor, &xi, &yi);
        if (xi < 4 || yi < 4) { set_err("pyramid level smaller than 4 pixels"); return OCTANE_EINVAL; }
        if (k < K - 1 && blur_decimate_smem_bytes(L.factor, L.R) > BLUR_DECIMATE_SMEM_LIMIT) {
            // the blur stages (8-1)/factor + 2R + 2 full-resolution rows of a 32-column tile per block
            set_err("pyramid too deep: the coarsest level's blur footprint exceeds shared memory (use fewer levels)");
            return OCTANE_EINVAL;
        }
        L.lambdac = (float)((double)lambdaco * pow(0.5, k));  // :494
        L.own0 = (int)((long long)rank * yi / world);
        L.own1 = (int)((long long)(rank + 1) * yi / world);
        int lo = 0, hi = yi;
        if (world > 1) {
            // image-2 fields are gathered at (j + v): warp halo, +4 rows so the second
            // derivatives there are valid, never less than the u,v halo
            int W = (int)ceil((double)p.max_disp * L.factor) + 3;
            int H = W + 4;
            if (H < HALO_UV) H = HALO_UV;
            lo = L.own0 - H; if (lo < 0) lo = 0;
            hi = L.own1 + H; if (hi > yi) hi = yi;
            if (L.own1 - L.own0 < 2 * HALO_UV) { set_err("band thinner than the halo: fewer ranks or larger scene"); return OCTANE_EINVAL; }
        }
        L.g.nx = xi; L.g.ny = yi; L.g.pitch = round_up(xi, 32); L.g.j0 = lo; L.g.rows = hi - lo;
        // full-res rows this level's blur reads (:369-370: j2 = (int)(jj/factor))
        if (k < K - 1) {
            int a = (int)(lo / L.factor) - L.R, b = (int)((hi - 1) / L.factor) + L.R;
            if (a < in0) in0 = a;
            if (b > in1) in1 = b;
        } else {
            if (lo < in0) in0 = lo;
            if (hi > in1) in1 = hi;
        }
    }
    if (in0 < 0) in0 = 0;
    if (in1 > ny) in1 = ny;
    Level& F = pl.lv[K - 1];
    F.g.j0 = in0; F.g.rows = in1 - in0;          // the finest level IS the input band
    pl.in0 = in0; pl.in1 = in1;
    for (int k = 0; k < K; k++) pl.lv[k].g.plane = (long long)pl.lv[k].g.rows * pl.lv[k].g.pitch;
    pl.P = (size_t)F.g.plane;
    pl.Pc = (K > 1) ? (size_t)pl.lv[K - 2].g.plane : 0;
    for (int k = 0; k + 1 < K; k++)
        if ((size_t)pl.lv[k].g.plane > pl.Pc) pl.Pc = (size_t)pl.lv[k].g.plane;
    return OCTANE_OK;
}

struct Buffers {
    float *img1, *img2, *g1c, *g2c;
    float *g1x, *g1y, *g2x, *g2y, *g2xx, *g2xy, *g2yy;
    float *u, *v, *ut, *vt;
    float *uh, *vh, *hu, *hv;
    PcgBuffers pcg;
};

struct TimedEvent { cudaEvent_t a, b; int cat, level, solve, ki; };
enum { CAT_PYR = 0, CAT_BUILD, CAT_P1, CAT_P2, CAT_UPDATE, CAT_NAV, CAT_TOTAL, CAT_N };

}  // namespace

struct octane_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // host-buffer entry points: result copies that overlap the next stage
    cudaEvent_t ev_stage = nullptr;
    bool profile = false, graphs = true;
    // PCG kernels of the large levels: 1 = merged recurrence, one launch and one reduction per iteration
    // (pcg_fused.cu, the default); 0 = the reference's recurrence literally, two launches (pcg_tma.cu + pcg.cu).
    // Small levels always run the latter (octane_ctx_set_solver).
    int solver = 1;
    bool coop = true;        // small levels: one cooperative launch per solve (falls back to per-iteration launches)
    Comm comm;
    // workspace
    char* arena = nullptr;
    size_t arena_bytes = 0;
    // the layout (image slots, per-pair states; arena_layout) the workspace was last cleared for: a call with another
    // layout clears it again, so that padding and unused rows hold finite values
    int arena_slots = 0, arena_states = 0;
    // batched calls (octane_optical_flow_batch_dev, octane_optical_flow_sequence_dev): per-pair scalars, partial sums,
    // group barriers, iteration counts and navigation parameters, for up to batch_cap pairs
    PcgScalars* d_bscal = nullptr;
    double* d_bpart = nullptr;
    size_t bpart_doubles = 0;
    unsigned* d_bbar = nullptr;
    unsigned* d_bticket = nullptr;       // one grid-reduction ticket per pair (large levels, merged-reduction solver)
    int* d_bits = nullptr;
    NavParams* d_bnav = nullptr;
    int batch_cap = 0;
    int batch_npairs = 0, batch_nsolves = 0;   // of the last batched call
    Plan plan;
    bool plan_valid = false;
    Buffers buf;
    std::vector<cudaGraphExec_t> pcg_graph;   // two per level: [2 * level + (constant W / N variant)]
    // batched calls: the large levels' PCG loop of all pairs, same slots; captured for the workspace layout
    // (arena_slots, arena_states) and destroyed when it changes
    std::vector<cudaGraphExec_t> batch_graph;
    // small persistent device objects
    PcgScalars* d_scal = nullptr;
    double* d_pending = nullptr;
    double* d_vote = nullptr;      // banded runs: one double for the all-ranks vote of octane_srsal_band_dev
    unsigned* d_ticket = nullptr;
    double* d_partials = nullptr;
    int partial_blocks = 0;
    int* d_its = nullptr;
    int* h_its = nullptr;          // pinned
    PcgScalars* h_scal = nullptr;  // pinned
    float* d_gk = nullptr;
    double* d_navtab = nullptr;    // navigation: constants + per-column / per-row tables of the unmoved pixel
    size_t navtab_doubles = 0;
    // pipelined host-buffer dispatcher (octane_stream_submit / _wait): two slots of device staging, so that the
    // copies of one pair overlap the solve of the other
    struct StreamSlot {
        char* buf = nullptr;
        size_t bytes = 0;
        cudaEvent_t in_ready = nullptr, in_free = nullptr, out_ready = nullptr, done = nullptr, mid = nullptr;
        bool busy = false;
        // copy-out of the pair in this slot, not yet enqueued (see flush_copy_out)
        bool copy_pending = false;
        int ncopy = 0;
        void* dst[8] = { nullptr };
        const void* src[8] = { nullptr };
        size_t nbytes[8] = { 0 };
    } slot[2];
    int copy_out_at_finest = -1;          // slot whose pending copy-out run_levels enqueues when the finest level starts
    cudaStream_t h2d_stream = nullptr;
    // host-API staging (device)
    char* stage = nullptr;
    size_t stage_bytes = 0;
    octane_stats stats;
    long long launches = 0;
    std::vector<TimedEvent> events;
    std::vector<cudaEvent_t> event_pool;
    size_t event_next = 0;
};

namespace {

void destroy_batch_graphs(octane_ctx* c)
{
    for (auto g : c->batch_graph) if (g) cudaGraphExecDestroy(g);
    c->batch_graph.clear();
}

void destroy_graphs(octane_ctx* c)
{
    for (auto g : c->pcg_graph) if (g) cudaGraphExecDestroy(g);
    c->pcg_graph.clear();
    destroy_batch_graphs(c);
}

size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

// The workspace: nslots image slots `is` floats apart (an image at the finest level, its current coarse level and that
// level's gradients, nc planes each), then npairs per-pair states `ps` floats apart (second derivatives, flow, hint and
// PCG planes).  b gets slot 0's fields as image 1's, slot 1's as image 2's and pair 0's state.  A single-pair call is
// nslots = 2, npairs = 1; a batch of N pairs has 2N slots (pair z: slots 2z, 2z + 1), a sequence of N pairs N + 1
// (pair z: slots z, z + 1).  Returns the bytes.
size_t arena_layout(const Plan& pl, Buffers* b, char* base, int nslots = 2, int npairs = 1, size_t* is = nullptr,
                    size_t* ps = nullptr)
{
    size_t off = 0;
    auto take = [&](size_t nfloats) -> float* {
        float* p = base ? (float*)(base + off) : nullptr;
        off += align_up(nfloats * sizeof(float));
        return p;
    };
    const size_t P = pl.P, Pc = pl.Pc, nc = pl.nc;
    Buffers tmp;
    Buffers& B = b ? *b : tmp;
    B.img1 = take(P * nc); B.g1c = take(Pc * nc); B.g1x = take(P * nc); B.g1y = take(P * nc);
    const size_t slot = off;
    B.img2 = take(P * nc); B.g2c = take(Pc * nc); B.g2x = take(P * nc); B.g2y = take(P * nc);
    off = slot * nslots;
    const size_t state0 = off;
    B.g2xx = take(P * nc); B.g2xy = take(P * nc); B.g2yy = take(P * nc);
    B.u = take(P); B.v = take(P); B.ut = take(Pc); B.vt = take(Pc);
    if (pl.p.first_guess) { B.uh = take(P); B.vh = take(P); B.hu = take(Pc); B.hv = take(Pc); }
    else { B.uh = B.vh = B.hu = B.hv = nullptr; }
    for (int i = 0; i < NCOEF; i++) B.pcg.coef[i] = take(P);
    B.pcg.ru = take(P); B.pcg.rv = take(P); B.pcg.xu = take(P); B.pcg.xv = take(P);
    B.pcg.pu[0] = take(P); B.pcg.pu[1] = take(P); B.pcg.pv[0] = take(P); B.pcg.pv[1] = take(P);
    B.pcg.qu = take(P); B.pcg.qv = take(P);
    B.pcg.r2u = B.pcg.qu; B.pcg.r2v = B.pcg.qv;           // the merged-reduction solver never stores q: r's second buffer
    if (is) *is = slot / sizeof(float);
    if (ps) *ps = (off - state0) / sizeof(float);
    return state0 + (off - state0) * npairs;
}

int ensure_small(octane_ctx* c, int partial_blocks)
{
    if (!c->d_scal) {
        CUDA_OK(cudaMalloc(&c->d_scal, sizeof(PcgScalars)));
        CUDA_OK(cudaMemset(c->d_scal, 0, sizeof(PcgScalars)));
        CUDA_OK(cudaMalloc(&c->d_pending, 2 * sizeof(double)));
        CUDA_OK(cudaMemset(c->d_pending, 0, 2 * sizeof(double)));
        CUDA_OK(cudaMalloc(&c->d_ticket, sizeof(unsigned)));
        CUDA_OK(cudaMemset(c->d_ticket, 0, sizeof(unsigned)));
        CUDA_OK(cudaMalloc(&c->d_its, OCTANE_MAX_SOLVES * sizeof(int)));
        CUDA_OK(cudaMemset(c->d_its, 0, OCTANE_MAX_SOLVES * sizeof(int)));
        CUDA_OK(cudaMallocHost(&c->h_its, OCTANE_MAX_SOLVES * sizeof(int)));
        CUDA_OK(cudaMallocHost(&c->h_scal, sizeof(PcgScalars)));
        memset(c->h_scal, 0, sizeof(PcgScalars));
        CUDA_OK(cudaMalloc(&c->d_gk, 256 * sizeof(float)));
    }
    if (partial_blocks > c->partial_blocks) {
        if (c->d_partials) cudaFree(c->d_partials);
        c->d_partials = nullptr;
        CUDA_OK(cudaMalloc(&c->d_partials, (size_t)partial_blocks * 2 * sizeof(double)));
        c->partial_blocks = partial_blocks;
    }
    return OCTANE_OK;
}

// (re)build plan + workspace for this problem; cached across calls.  batched: the caller lays the workspace out itself
// (ensure_batch); otherwise it is made the single-pair layout c->buf describes.
int prepare(octane_ctx* c, int nx, int ny, int nc, const octane_params& p, bool batched = false)
{
    CUDA_OK(cudaSetDevice(c->device));
    if (c->plan_valid && c->plan.same(nx, ny, nc, p, c->comm.rank, c->comm.world)) {
        if (!batched && (c->arena_slots != 2 || c->arena_states != 1)) {     // after a batched call
            CUDA_OK(cudaMemsetAsync(c->arena, 0, arena_layout(c->plan, nullptr, nullptr), c->stream));
            c->arena_slots = 2; c->arena_states = 1;
        }
        return OCTANE_OK;
    }
    c->plan_valid = false;
    destroy_graphs(c);
    Plan pl;
    const bool p2p = c->comm.world > 1 && c->comm.p2p;
    // With a peer-memory communicator a re-plan is collective (every rank re-plans at the same
    // call) and every rank must reach the exchanges inside comm_p2p_unmap_arenas and
    // comm_p2p_map_arenas: a rank-local failure (a refused plan, no memory, a CUDA error) is
    // carried in `local` and voted on in the mapping step, never returned before it -- the
    // peers would wait for this rank forever.
    int local = make_plan(pl, nx, ny, nc, p, c->comm.rank, c->comm.world);
    if (local && !p2p) return local;
    const size_t need = local ? 0 : arena_layout(pl, nullptr, nullptr);
    if (p2p) {
        // nobody may free a workspace a peer still maps
        if (cudaStreamSynchronize(c->stream) != cudaSuccess && !local) { set_err("cudaStreamSynchronize (re-plan)"); local = OCTANE_ECUDA; }
        if (comm_p2p_unmap_arenas(&c->comm, c->stream)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    }
    if (!local && need > c->arena_bytes) {
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { set_err("cudaStreamSynchronize (workspace)"); local = OCTANE_ECUDA; }
        if (c->arena) cudaFree(c->arena);
        c->arena = nullptr; c->arena_bytes = 0;
        if (local) {
        } else if (cudaMalloc(&c->arena, need) != cudaSuccess) {
            cudaGetLastError();
            c->arena = nullptr;
            set_err("cudaMalloc (workspace): out of device memory");
            local = OCTANE_ENOMEM;
        } else c->arena_bytes = need;
    }
    // padding columns / halo rows must hold finite values (they are multiplied by zero
    // coefficients): clear the whole workspace once per plan
    if (!local && cudaMemsetAsync(c->arena, 0, need, c->stream) != cudaSuccess) { set_err("cudaMemsetAsync (workspace)"); local = OCTANE_ECUDA; }
    if (!local) arena_layout(pl, &c->buf, c->arena);
    Plan pn[2];
    if (p2p) {
        for (int side = 0; side < 2 && !local; side++) {
            const int nb = c->comm.rank + (side == 0 ? -1 : 1);
            if (nb >= 0 && nb < c->comm.world) local = make_plan(pn[side], nx, ny, nc, p, nb, c->comm.world);
        }
        // the clear must not race a neighbour's first halo store
        if (!local && cudaStreamSynchronize(c->stream) != cudaSuccess) { set_err("cudaStreamSynchronize (workspace)"); local = OCTANE_ECUDA; }
        if (comm_p2p_map_arenas(&c->comm, c->arena, local == OCTANE_OK, c->stream)) {
            if (!local) { set_err("%s", comm_last_error()); local = OCTANE_ECOMM; }
        }
    }
    if (local) return local;
    if (p2p) {
        for (int side = 0; side < 2; side++) {
            const int nb = c->comm.rank + (side == 0 ? -1 : 1);
            if (nb < 0 || nb >= c->comm.world) continue;
            Buffers bn;
            arena_layout(pn[side], &bn, (char*)c->comm.nb_arena[side]);
            for (size_t k = 0; k < pl.lv.size(); k++) {
                const long long shift = (long long)(pl.lv[k].g.j0 - pn[side].lv[k].g.j0) * pl.lv[k].g.pitch;
                if (side == 0) { pl.lv[k].up_ru = bn.pcg.ru + shift; pl.lv[k].up_rv = bn.pcg.rv + shift; }
                else { pl.lv[k].dn_ru = bn.pcg.ru + shift; pl.lv[k].dn_rv = bn.pcg.rv + shift; }
                FusedPeers& fp = pl.lv[k].fp;
                float* rb[2][2] = { { bn.pcg.ru, bn.pcg.rv }, { bn.pcg.r2u, bn.pcg.r2v } };
                for (int bi = 0; bi < 2; bi++)
                    for (int ci = 0; ci < 2; ci++) (side == 0 ? fp.up_r : fp.dn_r)[bi][ci] = rb[bi][ci] + shift;
            }
        }
    }
    int pb = c->sm_count * 16;
    const Level& F = pl.lv.back();
    int bb = build_partial_blocks(F.g, F.g.rows);
    for (auto& L : pl.lv) { int t = build_partial_blocks(L.g, L.g.rows); if (t > bb) bb = t; }
    if (bb > pb) pb = bb;
    int rc = ensure_small(c, pb);
    if (rc) return rc;
    c->buf.pcg.scal = c->d_scal;
    c->buf.pcg.partials = c->d_partials;
    c->buf.pcg.ticket = c->d_ticket;
    c->buf.pcg.max_partial_blocks = c->partial_blocks;
    c->buf.pcg.pending = c->d_pending;
    c->buf.pcg.defer = (c->comm.world > 1 && !p2p) ? 1 : 0;
    c->buf.pcg.p2p.world = p2p ? c->comm.world : 1;
    c->buf.pcg.p2p.rank = c->comm.rank;
    c->buf.pcg.p2p.peers = (P2PWindow* const*)c->comm.d_peers;
    c->buf.pcg.p2p.epoch = c->comm.d_epoch;
    c->buf.pcg.up_ru = c->buf.pcg.up_rv = c->buf.pcg.dn_ru = c->buf.pcg.dn_rv = nullptr;
    c->plan = pl;
    c->arena_slots = 2; c->arena_states = 1;
    c->pcg_graph.assign(2 * pl.lv.size(), nullptr);
    c->plan_valid = true;
    return OCTANE_OK;
}

// ---- profile-mode event helpers ------------------------------------------------------
cudaEvent_t next_event(octane_ctx* c)
{
    if (c->event_next == c->event_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->event_pool.push_back(e);
    }
    return c->event_pool[c->event_next++];
}
struct Scope {
    octane_ctx* c; TimedEvent ev; bool on;
    Scope(octane_ctx* c_, int cat, int level = -1, int solve = -1, int ki = -1) : c(c_), on(c_->profile)
    {
        if (!on) return;
        ev.cat = cat; ev.level = level; ev.solve = solve; ev.ki = ki;
        ev.a = next_event(c); ev.b = next_event(c);
        cudaEventRecord(ev.a, c->stream);
    }
    ~Scope()
    {
        if (!on) return;
        cudaEventRecord(ev.b, c->stream);
        c->events.push_back(ev);
    }
};

// ---- halo exchange of whole rows (banded runs) ------------------------------------------
int exchange_rows(octane_ctx* c, const Level& L, int nplanes, float* const* planes, int h)
{
    if (c->comm.world <= 1) return OCTANE_OK;
    const Geom& g = L.g;
    // interior cuts always have h rows of halo on both sides (make_plan); the outermost
    // ranks have no neighbour there and comm_halo_exchange skips those pointers
    float *su[8], *ru[8], *sd[8], *rd[8];
    const bool has_up = c->comm.rank > 0, has_dn = c->comm.rank + 1 < c->comm.world;
    for (int p = 0; p < nplanes; p++) {
        su[p] = planes[p] + g.at(0, L.own0);                          // my first owned rows -> rank-1's lower halo
        ru[p] = has_up ? planes[p] + g.at(0, L.own0 - h) : nullptr;   // rank-1's last owned rows -> my upper halo
        sd[p] = planes[p] + g.at(0, L.own1 - h);                      // my last owned rows -> rank+1's upper halo
        rd[p] = has_dn ? planes[p] + g.at(0, L.own1) : nullptr;       // rank+1's first owned rows -> my lower halo
    }
    if (comm_halo_exchange(&c->comm, nplanes, su, ru, sd, rd, (size_t)h * g.pitch, c->stream)) {
        set_err("%s", comm_last_error());
        return OCTANE_ECOMM;
    }
    return OCTANE_OK;
}

int allreduce_pending(octane_ctx* c, int n)
{
    if (c->comm.world <= 1) return OCTANE_OK;
    if (comm_allreduce_f64(&c->comm, c->d_pending, n, c->stream)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    return OCTANE_OK;
}

// the merged-reduction kernels serve the levels that are large enough for them, on one GPU or over peer memory
bool level_fused(const octane_ctx* c, const Level& L)
{
    return c->solver == 1 && pcg_fused_usable(L.g, L.own1 - L.own0) && (c->comm.world <= 1 || c->comm.p2p);
}

// ---- the PCG loop of one solve (:1129-1182), enqueued or captured ----------------------
int enqueue_pcg(octane_ctx* c, const Level& L, int level, int solve, int const_wn, const PcgBuffers& pb)
{
    PcgBuffers b = pb;
    const int iters = c->plan.p.cgiters;
    const bool multi = c->comm.world > 1;
    const bool p2p = multi && c->comm.p2p;
    if (level_fused(c, L)) {
        // one launch per iteration (+ one that forms the first alpha); r and q halo rows and the six sums
        // cross the band boundaries inside the kernel (peer memory)
        for (int ki = -1; ki < iters; ki++) {
            Scope s(c, CAT_P1, level, solve, ki);
            launch_pcg_fused(b, L.g, L.own0, L.own1, ki, L.fp, c->sm_count, c->stream, const_wn);
            c->launches++;
        }
        return OCTANE_OK;
    }
    // peer-memory runs: pass 2 stores its boundary rows of r straight into the neighbours' halo rows
    // and the last block of each pass sums the dots across the ranks itself (2 launches per iteration,
    // as on one GPU); otherwise NCCL: all-reduce + a scalar kernel after each pass, send/recv of r
    if (p2p) { b.up_ru = L.up_ru; b.up_rv = L.up_rv; b.dn_ru = L.dn_ru; b.dn_rv = L.dn_rv; }
    for (int ki = 0; ki < iters; ki++) {
        {
            Scope s(c, CAT_P1, level, solve, ki);
            if (pcg_pass1_tma_usable(L.g, L.own1 - L.own0))
                launch_pcg_pass1_tma(b, L.g, L.own0, L.own1, ki, multi, c->sm_count, c->stream, const_wn);
            else
                launch_pcg_pass1(b, L.g, L.own0, L.own1, ki, multi, c->sm_count, c->stream);
            c->launches++;
        }
        if (multi && !p2p) {
            int rc = allreduce_pending(c, 1); if (rc) return rc;
            launch_finalize(b, FINALIZE_PASS1, 0.f, c->stream); c->launches++;
        }
        {
            Scope s(c, CAT_P2, level, solve, ki);
            launch_pcg_pass2(b, L.g, L.own0, L.own1, c->sm_count, c->stream);
            c->launches++;
        }
        if (multi && !p2p) {
            int rc = allreduce_pending(c, 2); if (rc) return rc;
            launch_finalize(b, FINALIZE_PASS2, 0.f, c->stream); c->launches++;
            float* planes[2] = { b.ru, b.rv };            // next pass 1 rebuilds p on the halo rows from r
            rc = exchange_rows(c, L, 2, planes, 1); if (rc) return rc;
        }
    }
    return OCTANE_OK;
}

// small levels on one GPU: the whole solve in one cooperative launch (pcg.cu: k_pcg_coop)
bool level_coop(const octane_ctx* c, const Level& L)
{
    // "small" = below the size the TMA-fed kernels take (either solver)
    return c->coop && c->comm.world <= 1 && !pcg_fused_usable(L.g, L.own1 - L.own0);
}

// Capture what enqueue() puts on the stream as an executable graph (*exec); the launches it counts are not counted
// here (the caller counts each replay).
template <class F>
int capture_graph(octane_ctx* c, F enqueue, cudaGraphExec_t* exec)
{
    cudaGraph_t graph = nullptr;
    const long long before = c->launches;
    CUDA_OK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue();
    cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
    c->launches = before;
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) { set_err("cudaStreamEndCapture: %s", cudaGetErrorString(e)); return OCTANE_ECUDA; }
    e = cudaGraphInstantiate(exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { *exec = nullptr; set_err("cudaGraphInstantiate: %s", cudaGetErrorString(e)); return OCTANE_ECUDA; }
    return OCTANE_OK;
}

// const_wn: the system was built in the first GNC stage (W = N = -1 everywhere)
int run_pcg(octane_ctx* c, const Level& L, int level, int solve, int const_wn)
{
    if (c->plan.p.cgiters <= 0) return OCTANE_OK;
    if (level_coop(c, L)) {
        Scope s(c, CAT_P1, level, solve, -2);           // ki = -2: a whole solve, not an iteration
        if (launch_pcg_coop(c->buf.pcg, L.g, L.own0, L.own1, c->plan.p.cgiters, c->sm_count, c->stream) == 0) {
            c->launches++;
            return OCTANE_OK;
        }
        cudaGetLastError();                              // e.g. a device that cannot co-schedule the grid: per-iteration launches
        c->coop = false;
    }
    if (!c->graphs || c->profile) return enqueue_pcg(c, L, level, solve, const_wn, c->buf.pcg);
    const size_t slot = 2 * (size_t)level + (const_wn ? 1 : 0);
    if (!c->pcg_graph[slot]) {
        int rc = capture_graph(c, [&] { return enqueue_pcg(c, L, level, solve, const_wn, c->buf.pcg); }, &c->pcg_graph[slot]);
        if (rc) return rc;
    }
    CUDA_OK(cudaGraphLaunch(c->pcg_graph[slot], c->stream));
    if (level_fused(c, L)) c->launches += (long long)c->plan.p.cgiters + 1;
    else c->launches += (long long)c->plan.p.cgiters * ((c->comm.world > 1 && !c->comm.p2p) ? 4 : 2);
    return OCTANE_OK;
}

// ---- coarse-to-fine driver (:487-1210) ----------------------------------------------------
// Inputs are already in buf.img1/img2 (pitched, rows [in0,in1)) and, with a first guess,
// buf.uh/vh.  Output: buf.u/v at the finest level.
// Enqueue the device-to-host copies of the pair in slot k on the copy stream: after that pair's results are ready
// and, with after_here, not before the point the solve stream has reached now.
int flush_copy_out(octane_ctx* c, int k, bool after_here)
{
    auto& sl = c->slot[k];
    if (!sl.copy_pending) return OCTANE_OK;
    if (after_here) {
        CUDA_OK(cudaEventRecord(sl.mid, c->stream));
        CUDA_OK(cudaStreamWaitEvent(c->copy_stream, sl.mid, 0));
    }
    CUDA_OK(cudaStreamWaitEvent(c->copy_stream, sl.out_ready, 0));
    for (int i = 0; i < sl.ncopy; i++)
        CUDA_OK(cudaMemcpyAsync(sl.dst[i], sl.src[i], sl.nbytes[i], cudaMemcpyDeviceToHost, c->copy_stream));
    CUDA_OK(cudaEventRecord(sl.done, c->copy_stream));
    sl.copy_pending = false;
    return OCTANE_OK;
}

int run_levels(octane_ctx* c)
{
    Plan& pl = c->plan;
    Buffers& B = c->buf;
    const octane_params& p = pl.p;
    const int K = p.kiters, nc = pl.nc;
    cudaStream_t st = c->stream;
    const bool multi = c->comm.world > 1;
    const float sf = (float)p.scaleF;
    int solve = 0;
    for (int k = 0; k < K; k++) {
        const Level& L = pl.lv[k];
        const Geom& g = L.g;
        const bool finest = (k == K - 1);
        float *g1 = finest ? B.img1 : B.g1c, *g2 = finest ? B.img2 : B.g2c;
        const float *hu = nullptr, *hv = nullptr;
        if (finest && c->copy_out_at_finest >= 0) {               // pipelined dispatcher, banded: see octane_stream_submit
            int rc = flush_copy_out(c, c->copy_out_at_finest, true);
            c->copy_out_at_finest = -1;
            if (rc) return rc;
        }
        {
            Scope s(c, CAT_PYR, k);
            if (k > 0) {                                          // :498-503
                const Level& Lc = pl.lv[k - 1];
                launch_zoom_in(B.ut, Lc.g, B.u, g, L.own0, L.own1, sf, st);
                launch_zoom_in(B.vt, Lc.g, B.v, g, L.own0, L.own1, sf, st);
                c->launches += 2;
                float* planes[2] = { B.u, B.v };
                int rc = exchange_rows(c, L, 2, planes, HALO_UV); if (rc) return rc;
            }
            if (!finest) {                                        // :518-564
                const Geom& gF = pl.lv[K - 1].g;
                launch_fill_gk(c->d_gk, L.factor, L.R, st);
                launch_blur_decimate(B.img1, gF, B.g1c, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, 1.f, nc, st);
                launch_blur_decimate(B.img2, gF, B.g2c, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, 1.f, nc, st);
                c->launches += 3;
                if (p.first_guess) {
                    launch_blur_decimate(B.uh, gF, B.hu, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, L.factor, 1, st);
                    launch_blur_decimate(B.vh, gF, B.hv, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, L.factor, 1, st);
                    c->launches += 2;
                    hu = B.hu; hv = B.hv;
                }
            } else if (p.first_guess) {                           // :504-517
                hu = B.uh; hv = B.vh;
            }
            if (k == 0) {                                         // :576-585
                if (hu) {
                    CUDA_OK(cudaMemcpyAsync(B.u, hu, (size_t)g.plane * sizeof(float), cudaMemcpyDeviceToDevice, st));
                    CUDA_OK(cudaMemcpyAsync(B.v, hv, (size_t)g.plane * sizeof(float), cudaMemcpyDeviceToDevice, st));
                } else {
                    CUDA_OK(cudaMemsetAsync(B.u, 0, (size_t)g.plane * sizeof(float), st));
                    CUDA_OK(cudaMemsetAsync(B.v, 0, (size_t)g.plane * sizeof(float), st));
                }
            }
            // :587-595 (the reference's third call also writes d(g2x)/dy into g2xy, which its fourth call overwrites)
            launch_gradient(g1, B.g1x, B.g1y, g, g.jlo(), g.jhi(), nc, st);
            launch_gradient(g2, B.g2x, B.g2y, g, g.jlo(), g.jhi(), nc, st);
            launch_gradient(B.g2x, B.g2xx, nullptr, g, g.jlo(), g.jhi(), nc, st);     // its y-output would be overwritten next
            launch_gradient(B.g2y, B.g2xy, B.g2yy, g, g.jlo(), g.jhi(), nc, st);
            c->launches += 4;
        }
        LevelFields f;
        f.g1 = g1; f.g1x = B.g1x; f.g1y = B.g1y;
        f.g2 = g2; f.g2x = B.g2x; f.g2y = B.g2y; f.g2xx = B.g2xx; f.g2xy = B.g2xy; f.g2yy = B.g2yy;
        f.u = B.u; f.v = B.v;
        f.uh = (L.lambdac != 0.f) ? hu : nullptr;
        f.vh = (L.lambdac != 0.f) ? hv : nullptr;
        BuildParams bp;
        bp.alpha = p.alpha; bp.ralpha = 1.0 / p.alpha; bp.lambdadalpha = p.lambda / p.alpha; bp.lambdac = L.lambdac;
        bp.dozim = p.dozim != 0; bp.nchan = nc; bp.tol = 0.0001 * 0.0001;       // :1353
        // rows to build: owned rows plus the halo rows the PCG kernels rebuild z (and p) on -- one each side for the
        // two-pass kernels, two for the merged-reduction kernel (its second stencil reaches one row further)
        const bool fused = level_fused(c, L);
        int ba = L.own0, bb = L.own1;
        if (multi) { const int h = fused ? 2 : 1; ba = ba - h < 0 ? 0 : ba - h; bb = bb + h > g.ny ? g.ny : bb + h; }
        for (int gnc = 0; gnc < 3; gnc++) {                       // :604-608
            bp.al1 = 1. - 0.5 * gnc;
            for (int l = 0; l < p.liters; l++, solve++) {
                {
                    Scope s(c, CAT_BUILD, k, solve);
                    launch_build(f, B.pcg, g, ba, bb, L.own0, L.own1, bp, multi ? 1 : 0, st);
                    c->launches += 2;
                    if (multi && !c->comm.p2p) {
                        int rc = allreduce_pending(c, 2); if (rc) return rc;
                        launch_finalize(B.pcg, FINALIZE_BUILD, bp.tol, st); c->launches++;
                    }
                }
                // the first GNC stage's systems have W = N = -1 everywhere: those solves do not read the two planes
                int rc = run_pcg(c, L, k, solve, gnc == 0 ? 1 : 0);
                if (rc) return rc;
                {
                    Scope s(c, CAT_UPDATE, k, solve);             // :1185-1195
                    if (fused) launch_update_uv_fused(B.u, B.v, B.pcg, g, L.own0, L.own1, c->d_its + solve, c->sm_count, st);
                    else launch_update_uv(B.u, B.v, B.pcg, g, L.own0, L.own1, c->d_its + solve, c->sm_count, st);
                    c->launches++;
                    float* planes[2] = { B.u, B.v };
                    rc = exchange_rows(c, L, 2, planes, HALO_UV); if (rc) return rc;
                }
            }
        }
        if (!finest) {                                            // :1201-1205
            CUDA_OK(cudaMemcpyAsync(B.ut, B.u, (size_t)g.plane * sizeof(float), cudaMemcpyDeviceToDevice, st));
            CUDA_OK(cudaMemcpyAsync(B.vt, B.v, (size_t)g.plane * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
    }
    CUDA_OK(cudaMemcpyAsync(c->h_its, c->d_its, sizeof(int) * solve, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(c->h_scal, c->d_scal, sizeof(PcgScalars), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

// dense band rows [in0,in1) -> pitched finest-level planes
int ingest(octane_ctx* c, const float* d_img1, const float* d_img2, const float* d_u, const float* d_v)
{
    const Plan& pl = c->plan;
    const Geom& g = pl.lv.back().g;
    const size_t w = (size_t)g.nx * sizeof(float), dp = (size_t)g.pitch * sizeof(float);
    for (int ch = 0; ch < pl.nc; ch++) {
        CUDA_OK(cudaMemcpy2DAsync(c->buf.img1 + (size_t)ch * g.plane, dp, d_img1 + (size_t)ch * g.rows * g.nx, w, w,
                                  g.rows, cudaMemcpyDeviceToDevice, c->stream));
        CUDA_OK(cudaMemcpy2DAsync(c->buf.img2 + (size_t)ch * g.plane, dp, d_img2 + (size_t)ch * g.rows * g.nx, w, w,
                                  g.rows, cudaMemcpyDeviceToDevice, c->stream));
    }
    if (pl.p.first_guess) {
        CUDA_OK(cudaMemcpy2DAsync(c->buf.uh, dp, d_u, w, w, g.rows, cudaMemcpyDeviceToDevice, c->stream));
        CUDA_OK(cudaMemcpy2DAsync(c->buf.vh, dp, d_v, w, w, g.rows, cudaMemcpyDeviceToDevice, c->stream));
    }
    return OCTANE_OK;
}

int emit(octane_ctx* c, float* d_u, float* d_v)
{
    const Level& L = c->plan.lv.back();
    const Geom& g = L.g;
    const size_t w = (size_t)g.nx * sizeof(float), dp = (size_t)g.pitch * sizeof(float);
    CUDA_OK(cudaMemcpy2DAsync(d_u, w, c->buf.u + g.at(0, L.own0), dp, w, L.own1 - L.own0, cudaMemcpyDeviceToDevice, c->stream));
    CUDA_OK(cudaMemcpy2DAsync(d_v, w, c->buf.v + g.at(0, L.own0), dp, w, L.own1 - L.own0, cudaMemcpyDeviceToDevice, c->stream));
    return OCTANE_OK;
}

void begin_call(octane_ctx* c)
{
    c->launches = 0;
    c->events.clear();
    c->event_next = 0;
}

// d_fg_u / d_fg_v: the first guess over the SAME rows as the images (the whole scene on one GPU, rows [in0,in1)
// of a band), read only when p->first_guess; d_u / d_v: the owned rows of the flow, written.  On one GPU the
// two are the same in/out buffers (the reference's uarr / varr, :1330-1335,1434-1438).
int solve_dev(octane_ctx* c, const float* d_img1, const float* d_img2, int nx, int ny, int nc,
              const octane_params* p, const float* d_fg_u, const float* d_fg_v, float* d_u, float* d_v)
{
    if (!c || !d_img1 || !d_img2 || !p || !d_u || !d_v) { set_err("null argument"); return OCTANE_EINVAL; }
    if (p->first_guess && (!d_fg_u || !d_fg_v)) { set_err("first_guess is set but no first guess was given"); return OCTANE_EINVAL; }
    int rc = prepare(c, nx, ny, nc, *p);
    if (rc) return rc;
    Scope total(c, CAT_TOTAL);
    rc = ingest(c, d_img1, d_img2, d_fg_u, d_fg_v);
    if (rc) return rc;
    rc = run_levels(c);
    if (rc) return rc;
    return emit(c, d_u, d_v);
}

int ensure_stage(octane_ctx* c, size_t bytes)
{
    if (bytes <= c->stage_bytes) return OCTANE_OK;
    CUDA_OK(cudaStreamSynchronize(c->stream));
    if (c->stage) cudaFree(c->stage);
    c->stage = nullptr; c->stage_bytes = 0;
    if (cudaMalloc(&c->stage, bytes) != cudaSuccess) {
        cudaGetLastError();                    // not sticky: later calls must not see it
        c->stage = nullptr;
        set_err("cudaMalloc (staging): out of device memory");
        return OCTANE_ENOMEM;
    }
    c->stage_bytes = bytes;
    return OCTANE_OK;
}

void fill_nav(NavParams& np, const octane_nav* nav, double t1, double t2, const octane_params* p)
{
    np.pph = nav->pph; np.req = nav->req; np.rpol = nav->rpol; np.lam0 = nav->lam0;
    np.xScale = nav->xScale; np.xOffset = nav->xOffset; np.yScale = nav->yScale; np.yOffset = nav->yOffset;
    np.lat1 = nav->lat1; np.lon1 = nav->lon1; np.lon0 = nav->lon0; np.R = nav->R;
    np.minX = nav->minX; np.minY = nav->minY; np.t1 = t1; np.t2 = t2;
    np.pixuv = p->pixuv; np.dp = p->dopolar == 1; np.dm = p->domerc == 1;
}

// sector-moved guard, src/oct_pix2uv_cuda.cu:295
bool sector_moved(const octane_nav* nav)
{
    float dx = nav->xOffset - nav->g2xOffset, dy = nav->yOffset - nav->g2yOffset;
    return !(((dx * dx) < (0.00001 * 0.00001)) && ((dy * dy) < (0.00001 * 0.00001)));
}

int pix2uv_dev_rows(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* d_u, const float* d_v,
                    int nx, int row0, int nrows, const octane_params* p, short* U, short* V, short* Ur, short* Vr)
{
    if (!c || !nav || !d_u || !d_v || !p || !U || !V || !Ur || !Vr || nx <= 0 || nrows < 0) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * nrows;
    if (sector_moved(nav)) {       // :358-368: all four planes zero
        CUDA_OK(cudaMemsetAsync(U, 0, n * sizeof(short), c->stream));
        CUDA_OK(cudaMemsetAsync(V, 0, n * sizeof(short), c->stream));
        CUDA_OK(cudaMemsetAsync(Ur, 0, n * sizeof(short), c->stream));
        CUDA_OK(cudaMemsetAsync(Vr, 0, n * sizeof(short), c->stream));
        return 1;
    }
    NavParams np;
    fill_nav(np, nav, t1, t2, p);
    const size_t need = pix2uv_table_doubles(nx, nrows);
    if (need > c->navtab_doubles) {
        CUDA_OK(cudaStreamSynchronize(c->stream));
        if (c->d_navtab) cudaFree(c->d_navtab);
        c->d_navtab = nullptr; c->navtab_doubles = 0;
        CUDA_OK(cudaMalloc(&c->d_navtab, need * sizeof(double)));
        c->navtab_doubles = need;
    }
    {
        Scope s(c, CAT_NAV);
        c->launches += launch_pix2uv(np, d_u, d_v, nx, row0, nrows, c->d_navtab, U, V, Ur, Vr, c->stream);
    }
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

// algorithmic bytes per pixel of one merged-reduction launch (DESIGN.md section 4): r, p in and out, x in and out
// every second iteration, the five coefficient planes (three when W = N = -1 is known)
double fused_bytes(int ki, bool cwn)
{
    const double coef = cwn ? 12.0 : 20.0;
    if (ki < 0) return 8.0 + coef;                       // r + coefficients, nothing written
    if (ki == 0) return 8.0 + coef + 16.0;               // no p of a previous iteration yet; r, p written
    if (ki == 1) return 16.0 + coef + 24.0;              // x is started, not read
    return (ki & 1) ? 24.0 + coef + 24.0 : 16.0 + coef + 16.0;
}

void collect_stats(octane_ctx* c)
{
    octane_stats& s = c->stats;
    const Plan& pl = c->plan;
    memset(&s, 0, sizeof s);
    s.kernel_launches = c->launches;
    if (!c->plan_valid) return;             // the context has only run ingest / regridding / post stages so far
    s.n_levels = (int)pl.lv.size();
    s.n_solves = pl.p.kiters * 3 * pl.p.liters;
    double bytes = 0.0;
    int solve = 0;
    for (int k = 0; k < s.n_levels; k++) {
        const Level& L = pl.lv[k];
        s.level_nx[k] = L.g.nx; s.level_ny[k] = L.g.ny;
        const double Nk = (double)L.g.nx * (L.own1 - L.own0);
        // DESIGN.md "algorithmic bytes": pyramid 100 B/px per level; per solve the build
        // (72 B/px), pass 1 (44 / 60 / 68 B/px for iteration 0 / 1 / later), pass 2 (32 B/px)
        // for the iterations actually executed, and the u,v update (32 B/px)
        bytes += Nk * 100.0;
        const bool fused = level_fused(c, L);
        for (int q = 0; q < 3 * pl.p.liters; q++, solve++) {
            const int n = c->h_its[solve];
            s.cg_iterations[solve] = n;
            const bool cwn = q < pl.p.liters;          // first GNC stage: W, N are not read by the large-level kernels
            double per = 72.0;                          // build
            if (fused) {
                per += fused_bytes(-1, cwn);            // the launch that forms the first alpha runs whenever the solve does
                for (int ki = 0; ki < n; ki++) per += fused_bytes(ki, cwn);
                if (n >= 1) per += 8.0 + 8.0 + (n >= 2 ? 8.0 : 0.0) + ((n & 1) ? 8.0 : 0.0);     // u, v in and out, x, pending p
            } else {
                per += 32.0 * n + (n >= 1 ? 44.0 : 0.0) + (n >= 2 ? 60.0 : 0.0) + (n > 2 ? 68.0 * (n - 2) : 0.0);
                if (cwn && pcg_pass1_tma_usable(L.g, L.own1 - L.own0)) per -= 8.0 * n;
                if (n >= 1) per += 32.0;
            }
            bytes += Nk * per;
        }
    }
    s.algorithmic_bytes = bytes;
    s.kernel_launches = c->launches;
    const Level& F = pl.lv.back();
    s.finest_pixels = (long long)F.g.nx * (F.own1 - F.own0);
    double f1 = 0, f2 = 0, fb = 0; long long n1 = 0, n2 = 0;
    s.pcg_solver = level_fused(c, F) ? 1 : 0;
    // developer switch: one line per timed scope (category, level, solve, iteration, ms)
    FILE* dump = (c->profile && getenv("OCTANE_DUMP_EVENTS")) ? fopen(getenv("OCTANE_DUMP_EVENTS"), "w") : nullptr;
    for (auto& e : c->events) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, e.a, e.b) != cudaSuccess) continue;
        if (dump) fprintf(dump, "%d %d %d %d %.4f\n", e.cat, e.level, e.solve, e.ki, ms);
        switch (e.cat) {
            case CAT_PYR: s.ms_pyramid += ms; break;
            case CAT_BUILD: s.ms_build += ms; break;
            case CAT_UPDATE: s.ms_update += ms; break;
            case CAT_NAV: s.ms_nav += ms; break;
            case CAT_TOTAL: s.ms_total += ms; break;
            case CAT_P1:
            case CAT_P2: {
                // ki = -1 is the merged-reduction solver's launch that forms the first alpha: counted in the stage time,
                // not in the per-iteration average
                const bool worked = e.solve >= 0 && e.ki >= 0 && e.ki < c->h_its[e.solve];
                if (e.cat == CAT_P1) { s.ms_pcg_pass1 += ms; if (worked) s.n_pcg_pass1++; }
                else { s.ms_pcg_pass2 += ms; if (worked) s.n_pcg_pass2++; }
                if (worked && e.level == s.n_levels - 1) {
                    if (e.cat == CAT_P1) {
                        f1 += ms; n1++;
                        const int q = e.solve - (s.n_levels - 1) * 3 * pl.p.liters;
                        fb += s.pcg_solver ? fused_bytes(e.ki, q < pl.p.liters)
                                           : ((e.ki == 0 ? 44.0 : (e.ki == 1 ? 60.0 : 68.0)) - (q < pl.p.liters && pcg_pass1_tma_usable(F.g, F.own1 - F.own0) ? 8.0 : 0.0));
                    } else { f2 += ms; n2++; }
                }
            } break;
        }
    }
    if (dump) fclose(dump);
    s.finest_pass1_bytes_per_px = n1 ? fb / n1 : 0.0;
    s.finest_pass1_ms = n1 ? f1 / n1 : 0.0;
    s.finest_pass2_ms = n2 ? f2 / n2 : 0.0;
}

}  // namespace

// =========================================================================================
extern "C" {

int octane_abi_version(void) { return OCTANE_ABI_VERSION; }
const char* octane_last_error(void) { return g_err; }

int octane_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void octane_params_default(octane_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->alpha = 5.; p->lambda = 1.; p->lambdac = 0.; p->scaleF = 0.5; p->scsig = 400.;   // src/main.cc:77-87
    p->kiters = 4; p->liters = 3; p->cgiters = 30; p->dozim = 1; p->setdevice = 0;
    p->pixuv = 0; p->dopolar = 0; p->domerc = 0; p->first_guess = 0; p->max_disp = 64;
    p->doCTH = 0; p->ir = 0; p->dosrsal = 0;
}

int octane_ctx_create(octane_ctx** out, int device)
{
    if (!out) { set_err("null argument"); return OCTANE_EINVAL; }
    *out = nullptr;
    int n = octane_device_count();
    if (n == 0) { set_err("no CUDA device: octane_b200 has no CPU fallback"); return OCTANE_ENODEV; }
    if (device < 0 || device >= n) {              // reference: warning + device 0, :1260-1264
        fprintf(stderr, "octane_b200: device %d is not available (%d visible), using device 0\n", device, n);
        device = 0;
    }
    CUDA_OK(cudaSetDevice(device));
    octane_ctx* c = new octane_ctx();
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_err("cudaStreamCreate: %s", cudaGetErrorString(e)); delete c; return OCTANE_ECUDA; }
    if (cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_stage, cudaEventDisableTiming) != cudaSuccess) {
        set_err("cudaStreamCreate (copy stream)");
        cudaStreamDestroy(c->stream);
        delete c;
        return OCTANE_ECUDA;
    }
    memset(&c->stats, 0, sizeof c->stats);
    *out = c;
    return OCTANE_OK;
}

void octane_ctx_destroy(octane_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    destroy_graphs(c);
    comm_destroy(&c->comm);
    for (auto e : c->event_pool) cudaEventDestroy(e);
    if (c->arena) cudaFree(c->arena);
    if (c->stage) cudaFree(c->stage);
    if (c->d_scal) cudaFree(c->d_scal);
    if (c->d_pending) cudaFree(c->d_pending);
    if (c->d_vote) cudaFree(c->d_vote);
    if (c->d_ticket) cudaFree(c->d_ticket);
    if (c->d_partials) cudaFree(c->d_partials);
    if (c->d_its) cudaFree(c->d_its);
    if (c->d_gk) cudaFree(c->d_gk);
    if (c->d_navtab) cudaFree(c->d_navtab);
    for (void* q : { (void*)c->d_bscal, (void*)c->d_bpart, (void*)c->d_bbar, (void*)c->d_bticket, (void*)c->d_bits,
                     (void*)c->d_bnav })
        if (q) cudaFree(q);
    for (auto& sl : c->slot) {
        if (sl.done) cudaEventSynchronize(sl.done);
        if (sl.buf) cudaFree(sl.buf);
        for (cudaEvent_t e : { sl.in_ready, sl.in_free, sl.out_ready, sl.done, sl.mid }) if (e) cudaEventDestroy(e);
    }
    if (c->h2d_stream) { cudaStreamSynchronize(c->h2d_stream); cudaStreamDestroy(c->h2d_stream); }
    if (c->h_its) cudaFreeHost(c->h_its);
    if (c->h_scal) cudaFreeHost(c->h_scal);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    if (c->ev_stage) cudaEventDestroy(c->ev_stage);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int octane_ctx_set_profile(octane_ctx* c, int on) { if (!c) return OCTANE_EINVAL; c->profile = on != 0; return OCTANE_OK; }
int octane_ctx_set_graphs(octane_ctx* c, int on) { if (!c) return OCTANE_EINVAL; c->graphs = on != 0; return OCTANE_OK; }

int octane_ctx_set_solver(octane_ctx* c, int solver)
{
    if (!c || (solver != 0 && solver != 1)) { set_err("solver must be 0 (reference recurrence) or 1 (merged reduction)"); return OCTANE_EINVAL; }
    if (solver != c->solver) {
        if (c->stream) cudaStreamSynchronize(c->stream);
        destroy_graphs(c);                                   // the captured PCG loops belong to the other kernels
        if (c->plan_valid) c->pcg_graph.assign(2 * c->plan.lv.size(), nullptr);
        c->solver = solver;
    }
    return OCTANE_OK;
}

int octane_ctx_synchronize(octane_ctx* c)
{
    if (!c) return OCTANE_EINVAL;
    CUDA_OK(cudaSetDevice(c->device));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

void* octane_ctx_stream(octane_ctx* c) { return c ? (void*)c->stream : nullptr; }

int octane_get_stats(octane_ctx* c, octane_stats* out)
{
    if (!c || !out) return OCTANE_EINVAL;
    int rc = octane_ctx_synchronize(c);
    if (rc) return rc;
    collect_stats(c);
    *out = c->stats;
    return OCTANE_OK;
}

size_t octane_workspace_bytes(int nx, int ny, int nc, const octane_params* p)
{
    if (!p) return 0;
    Plan pl;
    if (make_plan(pl, nx, ny, nc, *p, 0, 1)) return 0;
    return arena_layout(pl, nullptr, nullptr);
}

int octane_level_dims(int nx, int ny, const octane_params* p, int k, int* xi, int* yi)
{
    if (!p || !xi || !yi || k < 0 || k >= p->kiters) return OCTANE_EINVAL;
    zoom_size(nx, ny, level_factor(*p, k), xi, yi);
    return OCTANE_OK;
}

int octane_variational_flow_dev(octane_ctx* c, const float* d_img1, const float* d_img2, int nx, int ny, int nc,
                                const octane_params* p, float* d_u, float* d_v)
{
    if (!c) return OCTANE_EINVAL;
    if (c->comm.world > 1) { set_err("context is banded: use octane_variational_flow_band_dev"); return OCTANE_EINVAL; }
    begin_call(c);
    return solve_dev(c, d_img1, d_img2, nx, ny, nc, p, d_u, d_v, d_u, d_v);
}

namespace {
int band_solve(octane_ctx* c, const float* d_img1, const float* d_img2, const float* d_fg_u, const float* d_fg_v,
               int nx, int ny, int nc, const octane_params* p, float* d_u, float* d_v)
{
    begin_call(c);
    // the two error flags are only ever OR-ed into on the device: clear them per call, so that a context that
    // reported OCTANE_EHALO / OCTANE_ECOMM once can be used again (e.g. after the caller raised max_disp)
    if (c->d_scal) {
        CUDA_OK(cudaSetDevice(c->device));
        CUDA_OK(cudaMemsetAsync(&c->d_scal->halo_err, 0, 2 * sizeof(int), c->stream));
    }
    int rc = solve_dev(c, d_img1, d_img2, nx, ny, nc, p, d_fg_u, d_fg_v, d_u, d_v);
    if (rc) return rc;
    if (c->comm.world > 1) {          // halo check needs the device flag
        CUDA_OK(cudaStreamSynchronize(c->stream));
        if (c->h_scal->halo_err) { set_err("warp left the band halo: raise max_disp"); return OCTANE_EHALO; }
        if (c->h_scal->comm_err) { set_err("a peer's partial sums did not arrive (peer-memory exchange timed out)"); return OCTANE_ECOMM; }
    }
    return OCTANE_OK;
}
}  // namespace

int octane_variational_flow_band_dev(octane_ctx* c, const float* d_img1, const float* d_img2, int nx, int ny, int nc,
                                     const octane_params* p, float* d_u, float* d_v)
{
    if (!c || !p) { set_err("null argument"); return OCTANE_EINVAL; }
    if (p->first_guess && c->comm.world > 1) {
        // the in/out buffers hold the owned rows only; the hint field needs the band's overlap rows too
        set_err("banded runs take the first guess through octane_variational_flow_band_fg_dev (rows [in0,in1))");
        return OCTANE_EINVAL;
    }
    return band_solve(c, d_img1, d_img2, d_u, d_v, nx, ny, nc, p, d_u, d_v);
}

int octane_variational_flow_band_fg_dev(octane_ctx* c, const float* d_img1, const float* d_img2, const float* d_fg_u,
                                        const float* d_fg_v, int nx, int ny, int nc, const octane_params* p, float* d_u,
                                        float* d_v)
{
    if (!c || !p) { set_err("null argument"); return OCTANE_EINVAL; }
    if (!p->first_guess) { set_err("octane_variational_flow_band_fg_dev needs p->first_guess"); return OCTANE_EINVAL; }
    return band_solve(c, d_img1, d_img2, d_fg_u, d_fg_v, nx, ny, nc, p, d_u, d_v);
}

int octane_variational_flow(octane_ctx* c, const float* img1, const float* img2, int nx, int ny, int nc,
                            const octane_params* p, float* u, float* v)
{
    if (!c || !img1 || !img2 || !p || !u || !v) { set_err("null argument"); return OCTANE_EINVAL; }
    if (c->comm.world > 1) { set_err("host-buffer entry points are single-GPU"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, img_bytes = n * nc * sizeof(float), uv_bytes = n * sizeof(float);
    int rc = ensure_stage(c, 2 * img_bytes + 2 * uv_bytes);
    if (rc) return rc;
    float* d_i1 = (float*)c->stage;
    float* d_i2 = (float*)(c->stage + img_bytes);
    float* d_u = (float*)(c->stage + 2 * img_bytes);
    float* d_v = (float*)(c->stage + 2 * img_bytes + uv_bytes);
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_i1, img1, img_bytes, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_i2, img2, img_bytes, cudaMemcpyHostToDevice, c->stream));
    if (p->first_guess) {
        CUDA_OK(cudaMemcpyAsync(d_u, u, uv_bytes, cudaMemcpyHostToDevice, c->stream));
        CUDA_OK(cudaMemcpyAsync(d_v, v, uv_bytes, cudaMemcpyHostToDevice, c->stream));
    }
    rc = solve_dev(c, d_i1, d_i2, nx, ny, nc, p, d_u, d_v, d_u, d_v);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(u, d_u, uv_bytes, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(v, d_v, uv_bytes, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

int octane_pix2uv_dev(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* d_u, const float* d_v,
                      int nx, int ny, const octane_params* p, short* U, short* V, short* Ur, short* Vr)
{
    return pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, 0, ny, p, U, V, Ur, Vr);
}

int octane_pix2uv_band_dev(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* d_u,
                           const float* d_v, int nx, int row0, int nrows, const octane_params* p,
                           short* U, short* V, short* Ur, short* Vr)
{
    return pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, row0, nrows, p, U, V, Ur, Vr);
}

namespace {
constexpr int SRSAL_R = 18;    // radius of the -srsal window (src/oct_srsal_cuda.cu:78-79)
int srsal_enqueue(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny, float* tmp_u, float* tmp_v,
                  int npairs = 1);
size_t srsal_band_stage_bytes(int nx, int ny, int own0, int own1);
int srsal_band_enqueue(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny, int own0, int own1, char* stage);
bool srsal_bands_ok(int ny, int world);
bool srsal_args_ok(const octane_params* p, const void* cth, int nx, int ny)
{
    if (!p->dosrsal) return true;
    if (!cth) { set_err("dosrsal needs cth"); return false; }
    if (nx <= SRSAL_R || ny <= SRSAL_R) { set_err("dosrsal needs a scene larger than 18 x 18"); return false; }
    return true;
}
}  // namespace

int octane_optical_flow_dev(octane_ctx* c, const float* d_img1, const float* d_img2, const float* d_cth, int nx, int ny, int nc,
                            const octane_nav* nav, double t1, double t2, const octane_params* p, float* d_u, float* d_v,
                            short* U, short* V, short* Ur, short* Vr, short* d_ctp)
{
    if (!c || !d_img1 || !d_img2 || !nav || !p || !d_u || !d_v || !U || !V || !Ur || !Vr) { set_err("null argument"); return OCTANE_EINVAL; }
    if (p->doCTH && (!d_cth || !d_ctp)) { set_err("doCTH needs cth and ctp"); return OCTANE_EINVAL; }
    if (!srsal_args_ok(p, d_cth, nx, ny)) return OCTANE_EINVAL;
    if (c->comm.world > 1) { set_err("context is banded: use the band entry points"); return OCTANE_EINVAL; }
    const size_t fb = align_up((size_t)nx * ny * sizeof(float));
    if (p->dosrsal) {
        int rc = ensure_stage(c, 2 * fb);
        if (rc) return rc;
    }
    begin_call(c);
    int rc = solve_dev(c, d_img1, d_img2, nx, ny, nc, p, d_u, d_v, d_u, d_v);
    if (rc) return rc;
    if (p->doCTH) {                            // src/oct_optical_flow.cc:71-88
        launch_ctp_pack(d_cth, d_ctp, (size_t)nx * ny, p->ir == 1, c->stream);
        c->launches++;
    }
    const int nrc = pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, 0, ny, p, U, V, Ur, Vr);
    if (nrc < 0 || !p->dosrsal) return nrc;
    rc = srsal_enqueue(c, d_u, d_v, d_cth, nx, ny, (float*)c->stage, (float*)(c->stage + fb));   // :100-105
    return rc ? rc : nrc;
}

// ---- batched calls: many same-size pairs, one launch per stage -----------------------------------------------------
namespace {
// doubles of partial sums per pair of a batched call: large enough for the build, a cooperative group and a
// merged-reduction launch (2 * partial_blocks doubles, the single-pair budget: a pair's grid is never capped below its
// single-pair one)
size_t batch_partials_per_pair(const Plan& pl, int partial_blocks)
{
    int bb = 0;
    for (const Level& L : pl.lv) { int t = build_partial_blocks(L.g, L.g.rows); if (t > bb) bb = t; }
    size_t per = 2 * (size_t)bb > 3 * 8 ? 2 * (size_t)bb : 3 * 8;
    if (2 * (size_t)partial_blocks > per) per = 2 * (size_t)partial_blocks;
    return per;
}

// bytes of ensure_batch's per-pair buffers for n pairs
size_t batch_buffer_bytes(int n, size_t partials_per_pair)
{
    return n * (sizeof(PcgScalars) + partials_per_pair * sizeof(double) + 3 * sizeof(unsigned) +
                OCTANE_MAX_SOLVES * sizeof(int) + sizeof(NavParams));
}

// The workspace of a batched call laid out with nslots image slots and npairs per-pair states (arena_layout) into *B
// (image strides *is, pair stride *ps floats), plus the per-pair buffers.  A failed allocation leaves the context as
// it was.
int ensure_batch(octane_ctx* c, int nslots, int npairs, Buffers* B, size_t* is, size_t* ps)
{
    const Plan& pl = c->plan;
    const size_t need = arena_layout(pl, nullptr, nullptr, nslots, npairs);
    if (need > c->arena_bytes) {
        char* na = nullptr;
        if (cudaMalloc(&na, need) != cudaSuccess) {
            cudaGetLastError();
            set_err("cudaMalloc (batch workspace): out of device memory");
            return OCTANE_ENOMEM;
        }
        CUDA_OK(cudaStreamSynchronize(c->stream));
        cudaFree(c->arena);
        c->arena = na; c->arena_bytes = need; c->arena_slots = 0; c->arena_states = 0;
        arena_layout(pl, &c->buf, c->arena);
        destroy_graphs(c);                                   // the captured PCG loops point into the old workspace
        c->pcg_graph.assign(2 * pl.lv.size(), nullptr);
    }
    const size_t pd = (size_t)npairs * batch_partials_per_pair(pl, c->partial_blocks);
    if (npairs > c->batch_cap || pd > c->bpart_doubles) {
        CUDA_OK(cudaStreamSynchronize(c->stream));
        for (void* q : { (void*)c->d_bscal, (void*)c->d_bpart, (void*)c->d_bbar, (void*)c->d_bticket, (void*)c->d_bits,
                         (void*)c->d_bnav })
            if (q) cudaFree(q);
        c->d_bscal = nullptr; c->d_bpart = nullptr; c->d_bbar = nullptr; c->d_bticket = nullptr; c->d_bits = nullptr;
        c->d_bnav = nullptr;
        c->batch_cap = 0; c->bpart_doubles = 0;
        destroy_batch_graphs(c);                             // the captured batched PCG loops point into the old buffers
        const int n = npairs > c->batch_cap ? npairs : c->batch_cap;
        if (cudaMalloc(&c->d_bscal, n * sizeof(PcgScalars)) != cudaSuccess ||
            cudaMalloc(&c->d_bpart, pd * sizeof(double)) != cudaSuccess ||
            cudaMalloc(&c->d_bbar, 2 * n * sizeof(unsigned)) != cudaSuccess ||
            cudaMalloc(&c->d_bticket, n * sizeof(unsigned)) != cudaSuccess ||
            cudaMalloc(&c->d_bits, (size_t)n * OCTANE_MAX_SOLVES * sizeof(int)) != cudaSuccess ||
            cudaMalloc(&c->d_bnav, n * sizeof(NavParams)) != cudaSuccess) {
            cudaGetLastError();
            set_err("cudaMalloc (batch buffers): out of device memory");
            return OCTANE_ENOMEM;
        }
        CUDA_OK(cudaMemsetAsync(c->d_bscal, 0, n * sizeof(PcgScalars), c->stream));
        CUDA_OK(cudaMemsetAsync(c->d_bticket, 0, n * sizeof(unsigned), c->stream));      // each launch leaves it at 0
        c->batch_cap = n; c->bpart_doubles = pd;
    }
    if (nslots != c->arena_slots || npairs != c->arena_states) {     // padding and unused rows must hold finite values
        CUDA_OK(cudaMemsetAsync(c->arena, 0, need, c->stream));
        c->arena_slots = nslots; c->arena_states = npairs;
        destroy_batch_graphs(c);                             // the captured batched PCG loops point into the old layout
    }
    *B = c->buf;                                             // the scalars, partials and flags; the planes follow
    arena_layout(pl, B, c->arena, nslots, npairs, is, ps);
    return OCTANE_OK;
}

// pair b's view of the PCG planes (the large-level loop runs the single-pair kernels on it)
PcgBuffers pair_buffers(const PcgBuffers& b0, int b, size_t ps)
{
    PcgBuffers q = b0;
    const size_t po = (size_t)b * ps;
    for (int i = 0; i < NCOEF; i++) q.coef[i] += po;
    q.ru += po; q.rv += po; q.xu += po; q.xv += po;
    q.pu[0] += po; q.pu[1] += po; q.pv[0] += po; q.pv[1] += po;
    q.qu += po; q.qv += po; q.r2u += po; q.r2v += po;
    return q;
}

// The PCG loop of one solve of every pair on a large level, merged-reduction solver: one launch per iteration (+ the
// one that forms the first alpha) for all pairs.  pb: pair 0's planes, the pairs' scalars, partials and tickets.
int enqueue_pcg_batch(octane_ctx* c, const Level& L, int level, int solve, int const_wn, const PcgBuffers& pb, int npairs,
                      size_t ps)
{
    for (int ki = -1; ki < c->plan.p.cgiters; ki++) {
        Scope s(c, CAT_P1, level, solve, ki);
        if (launch_pcg_fused(pb, L.g, L.own0, L.own1, ki, L.fp, c->sm_count, c->stream, const_wn, npairs, ps)) {
            set_err("batched merged-reduction launch refused");
            return OCTANE_EINVAL;
        }
        c->launches++;
    }
    return OCTANE_OK;
}

// enqueue_pcg_batch replayed from a graph per (level, constant-W/N variant), captured for the workspace layout of the
// call (ensure_batch destroys the graphs when it changes); without graphs or with profiling on, enqueued directly
int run_pcg_batch(octane_ctx* c, const Level& L, int level, int solve, int const_wn, const PcgBuffers& pb, int npairs,
                  size_t ps)
{
    if (!c->graphs || c->profile) return enqueue_pcg_batch(c, L, level, solve, const_wn, pb, npairs, ps);
    const size_t slot = 2 * (size_t)level + (const_wn ? 1 : 0);
    if (c->batch_graph.size() != 2 * c->plan.lv.size()) {
        destroy_batch_graphs(c);
        c->batch_graph.assign(2 * c->plan.lv.size(), nullptr);
    }
    cudaGraphExec_t& exec = c->batch_graph[slot];
    if (!exec) {
        int rc = capture_graph(c, [&] { return enqueue_pcg_batch(c, L, level, solve, const_wn, pb, npairs, ps); }, &exec);
        if (rc) return rc;
    }
    CUDA_OK(cudaGraphLaunch(exec, c->stream));
    c->launches += (long long)c->plan.p.cgiters + 1;
    return OCTANE_OK;
}

// run_levels for npairs pairs in the workspace B of ensure_batch (image slots is floats apart, per-pair states ps
// floats apart); one GPU.  A batch's pair z reads slots 2z and 2z + 1, a sequence's slots z and z + 1.  With a first
// guess, each pair's hint is in its own uh / vh planes.  Per-pixel stages are one launch for all pairs or all slots;
// small levels solve all pairs in cooperative launches with one barrier per pair (launch_pcg_coop_batch); large levels
// under the merged-reduction solver run one launch per iteration for all pairs (run_pcg_batch), under the two-pass
// solver the single-pair PCG kernels pair by pair.
int run_levels_batch(octane_ctx* c, int npairs, bool sequence, const Buffers& B, size_t is, size_t ps)
{
    const Plan& pl = c->plan;
    const octane_params& p = pl.p;
    const int K = p.kiters, nc = pl.nc;
    const int nsol = K * 3 * p.liters;
    cudaStream_t st = c->stream;
    const float sf = (float)p.scaleF;
    const size_t S = ps * sizeof(float);
    // pair z's image 1 is B's image-1 fields + z * istep, its image 2 the image-2 fields + z * istep.  The per-image
    // stages visit every slot once: a sequence's npairs + 1 slots in one launch, a batch's image-1 slots and its
    // image-2 slots in one launch each.
    const size_t istep = sequence ? is : 2 * is;
    const int runs = sequence ? 1 : 2, run_slots = sequence ? npairs + 1 : npairs;
    PcgBuffers pb = B.pcg;                       // build and update: pair z uses d_bscal[z] (and partials region z)
    pb.scal = c->d_bscal;
    pb.partials = c->d_bpart;
    pb.ticket = c->d_bticket;
    int solve = 0;
    for (int k = 0; k < K; k++) {
        const Level& L = pl.lv[k];
        const Geom& g = L.g;
        const bool finest = (k == K - 1);
        float *g1 = finest ? B.img1 : B.g1c, *g2 = finest ? B.img2 : B.g2c;
        const float *hu = nullptr, *hv = nullptr;
        if (k > 0) {
            const Level& Lc = pl.lv[k - 1];
            launch_zoom_in(B.ut, Lc.g, B.u, g, L.own0, L.own1, sf, st, npairs, ps);
            launch_zoom_in(B.vt, Lc.g, B.v, g, L.own0, L.own1, sf, st, npairs, ps);
            c->launches += 2;
        }
        if (!finest) {
            const Geom& gF = pl.lv[K - 1].g;
            launch_fill_gk(c->d_gk, L.factor, L.R, st);
            for (int r = 0; r < runs; r++)
                launch_blur_decimate(r ? B.img2 : B.img1, gF, r ? B.g2c : B.g1c, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R,
                                     1.f, nc, st, run_slots, istep);
            c->launches += 1 + runs;
            if (p.first_guess) {
                launch_blur_decimate(B.uh, gF, B.hu, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, L.factor, 1, st, npairs, ps);
                launch_blur_decimate(B.vh, gF, B.hv, g, g.jlo(), g.jhi(), L.factor, c->d_gk, L.R, L.factor, 1, st, npairs, ps);
                c->launches += 2;
                hu = B.hu; hv = B.hv;
            }
        } else if (p.first_guess) {
            hu = B.uh; hv = B.vh;
        }
        if (k == 0) {
            const size_t w = (size_t)g.plane * sizeof(float);
            if (hu) {
                CUDA_OK(cudaMemcpy2DAsync(B.u, S, hu, S, w, npairs, cudaMemcpyDeviceToDevice, st));
                CUDA_OK(cudaMemcpy2DAsync(B.v, S, hv, S, w, npairs, cudaMemcpyDeviceToDevice, st));
            } else {
                CUDA_OK(cudaMemset2DAsync(B.u, S, 0, w, npairs, st));
                CUDA_OK(cudaMemset2DAsync(B.v, S, 0, w, npairs, st));
            }
        }
        for (int r = 0; r < runs; r++)
            launch_gradient(r ? g2 : g1, r ? B.g2x : B.g1x, r ? B.g2y : B.g1y, g, g.jlo(), g.jhi(), nc, st, run_slots, istep,
                            istep);
        launch_gradient(B.g2x, B.g2xx, nullptr, g, g.jlo(), g.jhi(), nc, st, npairs, ps, istep);
        launch_gradient(B.g2y, B.g2xy, B.g2yy, g, g.jlo(), g.jhi(), nc, st, npairs, ps, istep);
        c->launches += runs + 2;
        LevelFields f;
        f.g1 = g1; f.g1x = B.g1x; f.g1y = B.g1y;
        f.g2 = g2; f.g2x = B.g2x; f.g2y = B.g2y; f.g2xx = B.g2xx; f.g2xy = B.g2xy; f.g2yy = B.g2yy;
        f.u = B.u; f.v = B.v;
        f.uh = (L.lambdac != 0.f) ? hu : nullptr;
        f.vh = (L.lambdac != 0.f) ? hv : nullptr;
        BuildParams bp;
        bp.alpha = p.alpha; bp.ralpha = 1.0 / p.alpha; bp.lambdadalpha = p.lambda / p.alpha; bp.lambdac = L.lambdac;
        bp.dozim = p.dozim != 0; bp.nchan = nc; bp.tol = 0.0001 * 0.0001;
        const bool fused = level_fused(c, L);
        const bool small = !pcg_fused_usable(L.g, L.own1 - L.own0);
        const int per_launch = small ? coop_batch_pairs_per_launch(g, L.own0, L.own1, c->sm_count) : 0;
        for (int gnc = 0; gnc < 3; gnc++) {
            bp.al1 = 1. - 0.5 * gnc;
            for (int l = 0; l < p.liters; l++, solve++) {
                launch_build(f, pb, g, L.own0, L.own1, L.own0, L.own1, bp, 0, st, npairs, ps, istep);
                c->launches += 2;
                if (p.cgiters > 0 && small) {
                    for (int p0 = 0; p0 < npairs; p0 += per_launch) {
                        const int n = npairs - p0 < per_launch ? npairs - p0 : per_launch;
                        if (launch_pcg_coop_batch(pb, g, L.own0, L.own1, p.cgiters, p0, n, ps, c->d_bpart, c->d_bbar, st)) {
                            set_err("cooperative launch of the batched PCG solver: %s", cudaGetErrorString(cudaGetLastError()));
                            return OCTANE_ECUDA;
                        }
                        c->launches++;
                    }
                } else if (p.cgiters > 0 && fused) {
                    int rc = run_pcg_batch(c, L, k, solve, gnc == 0 ? 1 : 0, pb, npairs, ps);
                    if (rc) return rc;
                } else if (p.cgiters > 0) {
                    for (int b = 0; b < npairs; b++) {
                        PcgBuffers q = pair_buffers(B.pcg, b, ps);
                        q.scal = c->d_bscal + b;
                        int rc = enqueue_pcg(c, L, k, solve, gnc == 0 ? 1 : 0, q);
                        if (rc) return rc;
                    }
                }
                if (fused) launch_update_uv_fused(B.u, B.v, pb, g, L.own0, L.own1, c->d_bits + solve, c->sm_count, st, npairs, ps, nsol);
                else launch_update_uv(B.u, B.v, pb, g, L.own0, L.own1, c->d_bits + solve, c->sm_count, st, npairs, ps, nsol);
                c->launches++;
            }
        }
        if (!finest) {
            CUDA_OK(cudaMemcpy2DAsync(B.ut, S, B.u, S, (size_t)g.plane * sizeof(float), npairs, cudaMemcpyDeviceToDevice, st));
            CUDA_OK(cudaMemcpy2DAsync(B.vt, S, B.v, S, (size_t)g.plane * sizeof(float), npairs, cudaMemcpyDeviceToDevice, st));
        }
    }
    // pair 0's counts and scalars for octane_get_stats
    CUDA_OK(cudaMemcpyAsync(c->h_its, c->d_bits, sizeof(int) * nsol, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(c->h_scal, c->d_bscal, sizeof(PcgScalars), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

// the body of octane_optical_flow_batch_ex_dev, octane_optical_flow_batch_dev (which passes no first guess) and
// octane_optical_flow_sequence_dev (sequence: d_img1 holds the npairs + 1 frames, d_img2 is unused and t2 = t1 + 1)
int optical_flow_batch(octane_ctx* c, int npairs, bool sequence, const float* d_img1, const float* d_img2,
                       const float* d_fg_u, const float* d_fg_v, const float* d_cth, int nx, int ny, int nc,
                       const octane_nav* nav, const double* t1, const double* t2, const octane_params* p, float* d_upix,
                       float* d_vpix, short* U, short* V, short* Ur, short* Vr, short* d_ctp, int* moved_out)
{
    if (!c || !d_img1 || (!sequence && !d_img2) || !nav || !t1 || !t2 || !p || !d_upix || !d_vpix || !U || !V || !Ur || !Vr) {
        set_err("null argument");
        return OCTANE_EINVAL;
    }
    if (npairs < 1) { set_err("npairs must be at least 1"); return OCTANE_EINVAL; }
    if (p->first_guess && (!d_fg_u || !d_fg_v)) { set_err("first_guess is set but no first guess was given"); return OCTANE_EINVAL; }
    if (p->doCTH && (!d_cth || !d_ctp)) { set_err("doCTH needs cth and ctp"); return OCTANE_EINVAL; }
    if (!srsal_args_ok(p, d_cth, nx, ny)) return OCTANE_EINVAL;
    if (c->comm.world > 1) { set_err("context is banded: batched calls are single-GPU"); return OCTANE_EINVAL; }
    begin_call(c);
    int rc = prepare(c, nx, ny, nc, *p, true);
    if (rc) return rc;
    if (p->kiters * 3 * p->liters > OCTANE_MAX_SOLVES) { set_err("too many solves"); return OCTANE_EINVAL; }
    const int nslots = sequence ? npairs + 1 : 2 * npairs;
    Buffers B;
    size_t is = 0, ps = 0;
    rc = ensure_batch(c, nslots, npairs, &B, &is, &ps);
    if (rc) return rc;
    const size_t n = (size_t)nx * ny;
    cudaStream_t st = c->stream;
    // every allocation of the call before its first copy or launch: a failed one leaves nothing half enqueued
    const size_t need = pix2uv_table_doubles(nx, ny) * (size_t)npairs;
    if (need > c->navtab_doubles) {
        CUDA_OK(cudaStreamSynchronize(st));
        if (c->d_navtab) cudaFree(c->d_navtab);
        c->d_navtab = nullptr; c->navtab_doubles = 0;
        if (cudaMalloc(&c->d_navtab, need * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            c->d_navtab = nullptr;
            set_err("cudaMalloc (navigation tables): out of device memory");
            return OCTANE_ENOMEM;
        }
        c->navtab_doubles = need;
    }
    const size_t sfb = align_up((size_t)npairs * n * sizeof(float));      // -srsal: two result planes per pair
    if (p->dosrsal) {
        rc = ensure_stage(c, 2 * sfb);
        if (rc) return rc;
    }
    // dense images -> pitched finest-level planes of the image slots (each frame of a sequence once); the first guess
    // is copied in before any output is written, so it may alias d_upix / d_vpix
    const Geom& g = c->plan.lv.back().g;
    const size_t w = (size_t)nx * sizeof(float), dp = (size_t)g.pitch * sizeof(float);
    for (int k = 0; k < nslots; k++) {
        const float* src = sequence ? d_img1 + (size_t)k * nc * n : (k & 1 ? d_img2 : d_img1) + (size_t)(k >> 1) * nc * n;
        for (int ch = 0; ch < nc; ch++)
            CUDA_OK(cudaMemcpy2DAsync(B.img1 + (size_t)k * is + (size_t)ch * g.plane, dp, src + (size_t)ch * n, w, w, ny,
                                      cudaMemcpyDeviceToDevice, st));
    }
    if (p->first_guess) {
        for (int b = 0; b < npairs; b++) {
            CUDA_OK(cudaMemcpy2DAsync(B.uh + (size_t)b * ps, dp, d_fg_u + b * n, w, w, ny, cudaMemcpyDeviceToDevice, st));
            CUDA_OK(cudaMemcpy2DAsync(B.vh + (size_t)b * ps, dp, d_fg_v + b * n, w, w, ny, cudaMemcpyDeviceToDevice, st));
        }
    }
    rc = run_levels_batch(c, npairs, sequence, B, is, ps);
    if (rc) return rc;
    for (int b = 0; b < npairs; b++) {
        CUDA_OK(cudaMemcpy2DAsync(d_upix + b * n, w, B.u + (size_t)b * ps, dp, w, ny, cudaMemcpyDeviceToDevice, st));
        CUDA_OK(cudaMemcpy2DAsync(d_vpix + b * n, w, B.v + (size_t)b * ps, dp, w, ny, cudaMemcpyDeviceToDevice, st));
    }
    if (p->doCTH) {                            // src/oct_optical_flow.cc:71-88, all pairs in one launch
        launch_ctp_pack(d_cth, d_ctp, (size_t)npairs * n, p->ir == 1, st);
        c->launches++;
    }
    std::vector<NavParams> np(npairs);
    for (int b = 0; b < npairs; b++) fill_nav(np[b], &nav[b], t1[b], t2[b], p);
    CUDA_OK(cudaMemcpyAsync(c->d_bnav, np.data(), npairs * sizeof(NavParams), cudaMemcpyHostToDevice, st));
    c->launches += launch_pix2uv_batch(np[0], c->d_bnav, npairs, d_upix, d_vpix, nx, ny, c->d_navtab, U, V, Ur, Vr, st);
    for (int b = 0; b < npairs; b++) {        // sector-moved guard, src/oct_pix2uv_cuda.cu:295,358-368
        const bool moved = sector_moved(&nav[b]);
        if (moved_out) moved_out[b] = moved ? 1 : 0;
        if (!moved) continue;
        for (short* q : { U, V, Ur, Vr }) CUDA_OK(cudaMemsetAsync(q + b * n, 0, n * sizeof(short), st));
    }
    if (p->dosrsal) {      // src/oct_optical_flow.cc:100-105: after the navigation, so only uPix / vPix are smoothed
        rc = srsal_enqueue(c, d_upix, d_vpix, d_cth, nx, ny, (float*)c->stage, (float*)(c->stage + sfb), npairs);
        if (rc) return rc;
    }
    CUDA_OK(cudaGetLastError());
    c->batch_npairs = npairs;
    c->batch_nsolves = p->kiters * 3 * p->liters;
    return OCTANE_OK;
}
}  // namespace

int octane_optical_flow_batch_ex_dev(octane_ctx* c, int npairs, const float* d_img1, const float* d_img2,
                                     const float* d_fg_u, const float* d_fg_v, const float* d_cth, int nx, int ny, int nc,
                                     const octane_nav* nav, const double* t1, const double* t2, const octane_params* p,
                                     float* d_upix, float* d_vpix, short* U, short* V, short* Ur, short* Vr, short* d_ctp,
                                     int* moved_out)
{
    return optical_flow_batch(c, npairs, false, d_img1, d_img2, d_fg_u, d_fg_v, d_cth, nx, ny, nc, nav, t1, t2, p, d_upix,
                              d_vpix, U, V, Ur, Vr, d_ctp, moved_out);
}

int octane_optical_flow_sequence_dev(octane_ctx* c, int nframes, const float* d_frames, const float* d_fg_u,
                                     const float* d_fg_v, const float* d_cth, int nx, int ny, int nc,
                                     const octane_nav* nav, const double* t, const octane_params* p, float* d_upix,
                                     float* d_vpix, short* U, short* V, short* Ur, short* Vr, short* d_ctp, int* moved_out)
{
    if (nframes < 2) { set_err("a sequence needs at least 2 frames"); return OCTANE_EINVAL; }
    return optical_flow_batch(c, nframes - 1, true, d_frames, nullptr, d_fg_u, d_fg_v, d_cth, nx, ny, nc, nav, t,
                              t ? t + 1 : nullptr, p, d_upix, d_vpix, U, V, Ur, Vr, d_ctp, moved_out);
}

size_t octane_batch_workspace_bytes(int npairs, int sequence, int nx, int ny, int nc, const octane_params* p)
{
    Plan pl;
    if (!p || npairs < 1 || make_plan(pl, nx, ny, nc, *p, 0, 1)) return 0;
    const int nslots = sequence ? npairs + 1 : 2 * npairs;
    // the partial-sum budget prepare gives a context on a 148-SM B200
    int pb = 148 * 16;
    for (const Level& L : pl.lv) { int t = build_partial_blocks(L.g, L.g.rows); if (t > pb) pb = t; }
    const size_t n = (size_t)nx * ny;
    size_t bytes = arena_layout(pl, nullptr, nullptr, nslots, npairs) +
                   batch_buffer_bytes(npairs, batch_partials_per_pair(pl, pb)) +
                   pix2uv_table_doubles(nx, ny) * (size_t)npairs * sizeof(double);
    if (p->dosrsal) bytes += 2 * align_up((size_t)npairs * n * sizeof(float));
    return bytes;
}

int octane_optical_flow_batch_dev(octane_ctx* c, int npairs, const float* d_img1, const float* d_img2, const float* d_cth,
                                  int nx, int ny, int nc, const octane_nav* nav, const double* t1, const double* t2,
                                  const octane_params* p, float* d_upix, float* d_vpix, short* U, short* V, short* Ur,
                                  short* Vr, short* d_ctp, int* moved_out)
{
    if (p && p->first_guess) { set_err("batched calls take no first guess: use octane_optical_flow_batch_ex_dev"); return OCTANE_EINVAL; }
    if (p && p->dosrsal) { set_err("octane_optical_flow_batch_dev does not run -srsal: use octane_optical_flow_batch_ex_dev"); return OCTANE_EINVAL; }
    return optical_flow_batch(c, npairs, false, d_img1, d_img2, nullptr, nullptr, d_cth, nx, ny, nc, nav, t1, t2, p, d_upix,
                              d_vpix, U, V, Ur, Vr, d_ctp, moved_out);
}

int octane_batch_cg_iterations(octane_ctx* c, int* its, int npairs)
{
    if (!c || !its) { set_err("null argument"); return OCTANE_EINVAL; }
    if (npairs != c->batch_npairs || npairs < 1) { set_err("npairs differs from the last batched call"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    const int ns = c->batch_nsolves;
    for (int b = 0; b < npairs; b++)
        CUDA_OK(cudaMemcpy(its + (size_t)b * ns, c->d_bits + (size_t)b * ns, ns * sizeof(int), cudaMemcpyDeviceToHost));
    return OCTANE_OK;
}

int octane_pix2uv(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* u, const float* v,
                  int nx, int ny, const octane_params* p, short* U, short* V, short* Ur, short* Vr, float* dT)
{
    if (!c || !nav || !u || !v || !p || !U || !V || !Ur || !Vr) { set_err("null argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, fb = n * sizeof(float), sb = n * sizeof(short);
    int rc = ensure_stage(c, 2 * fb + 4 * sb);
    if (rc) return rc;
    float* d_u = (float*)c->stage;
    float* d_v = (float*)(c->stage + fb);
    short* d_s = (short*)(c->stage + 2 * fb);
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_u, u, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_v, v, fb, cudaMemcpyHostToDevice, c->stream));
    rc = pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, 0, ny, p, d_s, d_s + n, d_s + 2 * n, d_s + 3 * n);
    if (rc < 0) return rc;
    CUDA_OK(cudaMemcpyAsync(U, d_s, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(V, d_s + n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(Ur, d_s + 2 * n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(Vr, d_s + 3 * n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    if (dT) *dT = (float)(t2 - t1);           // :347
    return rc;
}

int octane_optical_flow(octane_ctx* c, const float* img1, const float* img2, const float* cth, int nx, int ny, int nc,
                        const octane_nav* nav, double t1, double t2, const octane_params* p,
                        float* upix, float* vpix, short* U, short* V, short* Ur, short* Vr, short* ctp, float* dT)
{
    if (!c || !img1 || !img2 || !nav || !p || !upix || !vpix || !U || !V || !Ur || !Vr) { set_err("null argument"); return OCTANE_EINVAL; }
    if (p->doCTH && (!cth || !ctp)) { set_err("doCTH needs cth and ctp"); return OCTANE_EINVAL; }
    if (!srsal_args_ok(p, cth, nx, ny)) return OCTANE_EINVAL;
    if (c->comm.world > 1) { set_err("host-buffer entry points are single-GPU"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, ib = n * nc * sizeof(float), fb = n * sizeof(float), sb = n * sizeof(short);
    int rc = ensure_stage(c, 2 * ib + 3 * fb + 5 * sb + (p->dosrsal ? 2 * fb + 256 : 0));
    if (rc) return rc;
    char* s = c->stage;
    float* d_i1 = (float*)s; s += ib;
    float* d_i2 = (float*)s; s += ib;
    float* d_u = (float*)s; s += fb;
    float* d_v = (float*)s; s += fb;
    float* d_cth = (float*)s; s += fb;
    short* d_s = (short*)s;
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_i1, img1, ib, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_i2, img2, ib, cudaMemcpyHostToDevice, c->stream));
    if (p->first_guess) {
        CUDA_OK(cudaMemcpyAsync(d_u, upix, fb, cudaMemcpyHostToDevice, c->stream));
        CUDA_OK(cudaMemcpyAsync(d_v, vpix, fb, cudaMemcpyHostToDevice, c->stream));
    }
    rc = solve_dev(c, d_i1, d_i2, nx, ny, nc, p, d_u, d_v, d_u, d_v);
    if (rc) return rc;
    if (p->doCTH || p->dosrsal) CUDA_OK(cudaMemcpyAsync(d_cth, cth, fb, cudaMemcpyHostToDevice, c->stream));
    if (p->doCTH) {                            // src/oct_optical_flow.cc:71-88
        launch_ctp_pack(d_cth, d_s + 4 * n, n, p->ir == 1, c->stream);
        c->launches++;
        CUDA_OK(cudaMemcpyAsync(ctp, d_s + 4 * n, sb, cudaMemcpyDeviceToHost, c->stream));
    }
    // the pixel displacements are final: their copy back runs on the second stream under the
    // navigation kernel (with pinned host buffers; pageable ones simply serialise)
    CUDA_OK(cudaEventRecord(c->ev_stage, c->stream));
    CUDA_OK(cudaStreamWaitEvent(c->copy_stream, c->ev_stage, 0));
    int nrc = pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, 0, ny, p, d_s, d_s + n, d_s + 2 * n, d_s + 3 * n);
    if (nrc < 0) { cudaStreamSynchronize(c->copy_stream); return nrc; }
    if (p->dosrsal) {      // src/oct_optical_flow.cc:100-105: after the navigation, so only uPix / vPix are smoothed
        float* tmp = (float*)(((uintptr_t)(d_s + 5 * n) + 255) & ~(uintptr_t)255);
        rc = srsal_enqueue(c, d_u, d_v, d_cth, nx, ny, tmp, tmp + n);
        if (rc) { cudaStreamSynchronize(c->copy_stream); return rc; }
        CUDA_OK(cudaEventRecord(c->ev_stage, c->stream));
        CUDA_OK(cudaStreamWaitEvent(c->copy_stream, c->ev_stage, 0));
    }
    CUDA_OK(cudaMemcpyAsync(upix, d_u, fb, cudaMemcpyDeviceToHost, c->copy_stream));
    CUDA_OK(cudaMemcpyAsync(vpix, d_v, fb, cudaMemcpyDeviceToHost, c->copy_stream));
    CUDA_OK(cudaMemcpyAsync(U, d_s, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(V, d_s + n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(Ur, d_s + 2 * n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(Vr, d_s + 3 * n, sb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    CUDA_OK(cudaStreamSynchronize(c->copy_stream));
    if (dT) *dT = (float)(t2 - t1);
    return nrc;
}

// ---- ingest: calibration / normalisation / lat-lon, first-guess conversion ------------------
static void fill_cal(CalParams& c, const octane_nav* nav, const octane_cal* cal)
{
    c.xScale = nav->xScale; c.xOffset = nav->xOffset; c.yScale = nav->yScale; c.yOffset = nav->yOffset;
    c.radScale = cal->radScale; c.radOffset = cal->radOffset;
    // src/oct_fileread.cc:51,306: req, rpol, pph are read into floats, H = pph + req in float,
    // lam0 = lam0*DTOR in float; oct_navcal_cuda takes them as float arguments
    const float req = (float)nav->req, rpol = (float)nav->rpol, pph = (float)nav->pph;
    c.req = req; c.rpol = rpol; c.H = (cal->H != 0.f) ? cal->H : pph + req; c.lam0 = (float)nav->lam0;
    c.fk1 = cal->fk1; c.fk2 = cal->fk2; c.bc1 = cal->bc1; c.bc2 = cal->bc2; c.kap1 = cal->kap1;
    c.maxin = cal->maxin; c.minin = cal->minin; c.maxout = cal->maxout; c.minout = cal->minout;
    c.subpoint_slope = 1. / (0.021 - 0.0212);                       // src/oct_navcal_cuda.cu:178-179
    c.subpoint_int = 1. - 0.021 * c.subpoint_slope;
    c.cal = cal->cal; c.donav = cal->donav;
}

int octane_navcal_dev(octane_ctx* c, const short* d_rad, const short* d_x, const short* d_y, int nx, int ny,
                      const octane_nav* nav, const octane_cal* cal, float* d_data, float* d_lat, float* d_lon)
{
    if (!c || !d_rad || !d_x || !d_y || !nav || !cal || !d_data || nx <= 0 || ny <= 0 || (!d_lat != !d_lon)) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    CalParams cp;
    fill_cal(cp, nav, cal);
    launch_navcal(d_rad, d_x, d_y, nx, ny, cp, d_data, d_lat, d_lon, c->stream);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

int octane_navcal(octane_ctx* c, const short* rad, const short* x, const short* y, int nx, int ny,
                  const octane_nav* nav, const octane_cal* cal, float* data, float* lat, float* lon)
{
    if (!c || !rad || !x || !y || !nav || !cal || !data || nx <= 0 || ny <= 0 || (!lat != !lon)) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, sb = n * sizeof(short), fb = n * sizeof(float);
    const size_t xb = align_up((size_t)nx * sizeof(short)), yb = align_up((size_t)ny * sizeof(short));
    int rc = ensure_stage(c, align_up(sb) + xb + yb + 3 * fb);
    if (rc) return rc;
    char* s = c->stage;
    short* d_rad = (short*)s; s += align_up(sb);
    short* d_x = (short*)s; s += xb;
    short* d_y = (short*)s; s += yb;
    float* d_data = (float*)s; s += fb;
    float* d_lat = lat ? (float*)s : nullptr; s += fb;
    float* d_lon = lon ? (float*)s : nullptr;
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_rad, rad, sb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_x, x, (size_t)nx * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_y, y, (size_t)ny * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    rc = octane_navcal_dev(c, d_rad, d_x, d_y, nx, ny, nav, cal, d_data, d_lat, d_lon);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(data, d_data, fb, cudaMemcpyDeviceToHost, c->stream));
    if (lat) {
        CUDA_OK(cudaMemcpyAsync(lat, d_lat, fb, cudaMemcpyDeviceToHost, c->stream));
        CUDA_OK(cudaMemcpyAsync(lon, d_lon, fb, cudaMemcpyDeviceToHost, c->stream));
    }
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

int octane_navcal_grid(octane_ctx* c, int grid, const float* data, const short* x, const short* y, int nx, int ny,
                       const octane_nav* nav, int donav, float* data_out, float* lat, float* lon)
{
    if (!c || (grid != 1 && grid != 2) || !data || !x || !y || !nav || !data_out || nx <= 0 || ny <= 0 || (!lat != !lon)) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, fb = n * sizeof(float);
    const size_t xb = align_up((size_t)nx * sizeof(short)), yb = align_up((size_t)ny * sizeof(short));
    int rc = ensure_stage(c, 4 * fb + xb + yb);
    if (rc) return rc;
    char* s = c->stage;
    float* d_in = (float*)s; s += fb;
    float* d_out = (float*)s; s += fb;
    float* d_lat = lat ? (float*)s : nullptr; s += fb;
    float* d_lon = lon ? (float*)s : nullptr; s += fb;
    short* d_x = (short*)s; s += xb;
    short* d_y = (short*)s;
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_in, data, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_x, x, (size_t)nx * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_y, y, (size_t)ny * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    // the reference's wrappers convert to radians in double and pass floats (oct_polar_navcal_cuda.cu:141-143,
    // oct_merc_navcal_cuda.cu:122-124)
    const double PI = 3.14159265359, DTOR = PI / 180.;
    const float lon0 = (float)((grid == 1 ? nav->lon0 : nav->lon1) * DTOR);
    const float lat1 = (float)(nav->lat1 * DTOR);
    launch_navcal_grid(grid, d_in, d_x, d_y, nx, ny, nav->xScale, nav->xOffset, nav->yScale, nav->yOffset, nav->R, lon0, lat1,
                       donav, d_out, d_lat, d_lon, c->stream);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(data_out, d_out, fb, cudaMemcpyDeviceToHost, c->stream));
    if (lat) {
        CUDA_OK(cudaMemcpyAsync(lat, d_lat, fb, cudaMemcpyDeviceToHost, c->stream));
        CUDA_OK(cudaMemcpyAsync(lon, d_lon, fb, cudaMemcpyDeviceToHost, c->stream));
    }
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

// src/oct_normalize_geo.cc:9-88 (the table is data: ABI band radiance ranges; bands 7 and 8
// carry the reference's "meteorological" ranges)
int octane_band_minmax(int band, float* maxch, float* minch)
{
    static const float tab[16][2] = {
        { 804.03605737f, -25.93664701f }, { 628.98723908f, -20.28991094f }, { 373.16695681f, -12.03764377f },
        { 140.19342584f, -4.52236858f },  { 94.84802665f, -3.05961376f },   { 29.78947040f, -0.96095066f },
        { 2.f, 0.f },                     { 6.f, 3.f },                     { 44.998f, -0.2472f },
        { 79.831f, -0.2871f },            { 134.93f, -0.3909f },            { 108.44f, -0.4617f },
        { 185.5699f, -1.6443f },          { 198.71f, -0.5154f },            { 212.28f, -0.5262f },
        { 170.19f, -1.5726f } };
    if (!maxch || !minch || band < 1 || band > 16) { set_err("unknown ABI band"); return OCTANE_EINVAL; }
    *maxch = tab[band - 1][0];
    *minch = tab[band - 1][1];
    return OCTANE_OK;
}

int octane_zoom_in_float_dev(octane_ctx* c, const float* d_in, int nx, int ny, float* d_out, int nxx, int nyy, int interp)
{
    if (!c || !d_in || !d_out || nx <= 0 || ny <= 0 || nxx < nx || nyy < ny) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    launch_zoom_in_float(d_in, nx, ny, d_out, nxx, nyy, interp, c->stream);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

int octane_zoom_in_float(octane_ctx* c, const float* in, int nx, int ny, float* out, int nxx, int nyy, int interp)
{
    if (!c || !in || !out || nx <= 0 || ny <= 0 || nxx < nx || nyy < ny) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t ib = align_up((size_t)nx * ny * sizeof(float)), ob = (size_t)nxx * nyy * sizeof(float);
    int rc = ensure_stage(c, ib + ob);
    if (rc) return rc;
    float* d_in = (float*)c->stage;
    float* d_out = (float*)(c->stage + ib);
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_in, in, (size_t)nx * ny * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    rc = octane_zoom_in_float_dev(c, d_in, nx, ny, d_out, nxx, nyy, interp);
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(out, d_out, ob, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

// ---- oct_zoom_out_float (src/oct_zoom.cc:51-88): a finer field down to the image grid ----------
int octane_zoom_out_size(int nx, int ny, double factor, int* nxx, int* nyy)
{
    if (!nxx || !nyy || nx <= 0 || ny <= 0 || !(factor > 0.0)) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    *nxx = (int)((double)nx * factor + 0.5);       // oct_zoom_size, src/oct_zoom.cc:12-16
    *nyy = (int)((double)ny * factor + 0.5);
    return OCTANE_OK;
}

namespace {
// Taps of oct_gaussian / oct_getGaussian_1D for this factor (src/oct_zoom.cc:64, src/oct_gaussian.cc:34-56),
// evaluated on the host in double exactly as the reference does.  Returns 0 for the copy branch
// (factor >= 0.999999, :74-81), 1 with taps filled, or a negative code.
int zoom_out_taps(double factor, ZoomOutTaps* t)
{
    if (!(factor < 0.999999)) return 0;
    const double sigma = 0.6 * sqrt(1.0 / (factor * factor) - 1.0);
    int filtsize = 2 * sigma;                      // `(int) 2*sigma`: truncated on assignment
    if (filtsize < 5) filtsize = 5;
    if (filtsize > 32) { set_err("zoom-out factor below 1/27 is not supported (blur radius > 32)"); return OCTANE_EINVAL; }
    const int wk = 2 * filtsize + 1;
    const double s = 2.0 * sigma * sigma;
    double sum = 0.0;
    for (int x = -filtsize; x <= filtsize; x++) {
        const double r = x;
        t->gk[x + filtsize] = (exp(-(r * r) / s)) / (M_PI * s);
        sum += t->gk[x + filtsize];
    }
    for (int i = 0; i < wk; ++i) t->gk[i] /= sum;
    t->R = filtsize;
    return 1;
}

int zoom_out_enqueue(octane_ctx* c, const float* d_in, int nx, int ny, float* d_out, int nxx, int nyy, double factor,
                     int have_taps, const ZoomOutTaps& taps, double* tmp_a, double* tmp_b)
{
    c->launches += launch_zoom_out_float(d_in, nx, ny, d_out, nxx, nyy, factor, have_taps ? &taps : nullptr, tmp_a, tmp_b, c->stream);
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

bool zoom_out_args_ok(int nx, int ny, double factor, int* nxx, int* nyy)
{
    if (nx <= 0 || ny <= 0 || !(factor > 0.0) || factor > 1.0) return false;
    *nxx = (int)((double)nx * factor + 0.5);
    *nyy = (int)((double)ny * factor + 0.5);
    return *nxx > 0 && *nyy > 0 && *nxx <= nx && *nyy <= ny;
}
}  // namespace

int octane_zoom_out_float_dev(octane_ctx* c, const float* d_in, int nx, int ny, float* d_out, double factor)
{
    int nxx, nyy;
    if (!c || !d_in || !d_out || !zoom_out_args_ok(nx, ny, factor, &nxx, &nyy)) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    ZoomOutTaps taps;
    const int have = zoom_out_taps(factor, &taps);
    if (have < 0) return have;
    CUDA_OK(cudaSetDevice(c->device));
    const size_t db = align_up((size_t)nx * ny * sizeof(double));
    if (have) {
        int rc = ensure_stage(c, 2 * db);
        if (rc) return rc;
    }
    return zoom_out_enqueue(c, d_in, nx, ny, d_out, nxx, nyy, factor, have, taps, (double*)c->stage, (double*)(c->stage + db));
}

int octane_zoom_out_float(octane_ctx* c, const float* in, int nx, int ny, float* out, double factor)
{
    int nxx, nyy;
    if (!c || !in || !out || !zoom_out_args_ok(nx, ny, factor, &nxx, &nyy)) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    ZoomOutTaps taps;
    const int have = zoom_out_taps(factor, &taps);
    if (have < 0) return have;
    CUDA_OK(cudaSetDevice(c->device));
    const size_t db = align_up((size_t)nx * ny * sizeof(double)), ib = align_up((size_t)nx * ny * sizeof(float)),
                 ob = (size_t)nxx * nyy * sizeof(float);
    int rc = ensure_stage(c, 2 * db + ib + ob);
    if (rc) return rc;
    float* d_in = (float*)(c->stage + 2 * db);
    float* d_out = (float*)(c->stage + 2 * db + ib);
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_in, in, (size_t)nx * ny * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    rc = zoom_out_enqueue(c, d_in, nx, ny, d_out, nxx, nyy, factor, have, taps, (double*)c->stage, (double*)(c->stage + db));
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(out, d_out, ob, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

// ---- -srsal (oct_srsal_cu, src/oct_srsal_cuda.cu:73-147) ----------------------------------------
namespace {
void srsal_taps(SrsalTaps* t)
{
    const double sigpix = 20.;                      // :75-79
    t->sigpix2 = -1. / (sigpix * sigpix * 2.);
    const double filtsigma = 9;
    const int filtsize = 2 * filtsigma;
    const double s = 2.0 * filtsigma * filtsigma;   // oct_getGaussian_1D, src/oct_gaussian.cc:34-47
    double sum = 0.0;
    for (int x = -filtsize; x <= filtsize; x++) {
        const double r = x;
        t->gk[x + filtsize] = (exp(-(r * r) / s)) / (M_PI * s);
        sum += t->gk[x + filtsize];
    }
    for (int i = 0; i < 2 * filtsize + 1; ++i) t->gk[i] /= sum;
}

// u, v -> tmp (filtered) -> back into u, v, all on the context's stream.  npairs dense pair-major scenes (u, v, cth
// and each tmp plane npairs x ny x nx), filtered in one launch, each pair with its own heights.
int srsal_enqueue(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny, float* tmp_u, float* tmp_v,
                  int npairs)
{
    SrsalTaps t;
    srsal_taps(&t);
    const size_t n = (size_t)nx * ny, fb = (size_t)npairs * n * sizeof(float);
    launch_srsal(d_u, d_v, d_cth, nx, ny, 0, 0, ny, t, tmp_u, tmp_v, c->stream, npairs, n);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(d_u, tmp_u, fb, cudaMemcpyDeviceToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_v, tmp_v, fb, cudaMemcpyDeviceToDevice, c->stream));
    return OCTANE_OK;
}
}  // namespace

int octane_srsal_dev(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny)
{
    // the reflected index stays inside the scene only for nx, ny > 18 (the reference reads out of bounds below that)
    if (!c || !d_u || !d_v || !d_cth || nx <= SRSAL_R || ny <= SRSAL_R) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t fb = align_up((size_t)nx * ny * sizeof(float));
    int rc = ensure_stage(c, 2 * fb);
    if (rc) return rc;
    return srsal_enqueue(c, d_u, d_v, d_cth, nx, ny, (float*)c->stage, (float*)(c->stage + fb));
}

// ---- -srsal on row bands ------------------------------------------------------------------------
// Rank r owns rows [r*ny/world, (r+1)*ny/world), the finest level's rule of make_plan.  The 37 x 37 window of an owned
// row reaches 18 rows into each neighbour's band; the window of a row near the scene edge reflects back into the scene
// (rows 1..18 above row 0, ny-18..ny-1 below row ny-1).  With every band at least 18 rows high both come from this
// band and the two adjacent ones only: each rank stages u, v, cth over rows [max(0, own0-18), min(ny, own1+18)) and
// takes the 18 rows above and below from its neighbours in one NCCL exchange.
namespace {
void own_rows(int ny, int rank, int world, int* own0, int* own1)
{
    *own0 = (int)((long long)rank * ny / world);
    *own1 = (int)((long long)(rank + 1) * ny / world);
}

// the same answer on every rank (it depends on ny and world only): all refuse together, none enters the exchange alone
bool srsal_bands_ok(int ny, int world)
{
    for (int r = 0; r < world; r++) {
        int a, b;
        own_rows(ny, r, world, &a, &b);
        if (b - a < SRSAL_R) return false;
    }
    return true;
}

// three planes (u, v, cth) of the extended rows
size_t srsal_band_stage_bytes(int nx, int ny, int own0, int own1)
{
    const int e0 = own0 - SRSAL_R < 0 ? 0 : own0 - SRSAL_R, e1 = own1 + SRSAL_R > ny ? ny : own1 + SRSAL_R;
    return 3 * align_up((size_t)(e1 - e0) * nx * sizeof(float));
}

// d_u, d_v, d_cth: the owned rows [own0,own1), dense; stage: srsal_band_stage_bytes.  Collective on the context's
// communicator (nothing is exchanged at world 1); the result goes back into d_u, d_v.
int srsal_band_enqueue(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny, int own0, int own1, char* stage)
{
    const int e0 = own0 - SRSAL_R < 0 ? 0 : own0 - SRSAL_R, e1 = own1 + SRSAL_R > ny ? ny : own1 + SRSAL_R;
    const size_t pb = align_up((size_t)(e1 - e0) * nx * sizeof(float)), ob = (size_t)(own1 - own0) * nx * sizeof(float);
    float* ext[3] = { (float*)stage, (float*)(stage + pb), (float*)(stage + 2 * pb) };
    const float* own[3] = { d_u, d_v, d_cth };
    const size_t at_own = (size_t)(own0 - e0) * nx;
    for (int p = 0; p < 3; p++)
        CUDA_OK(cudaMemcpyAsync(ext[p] + at_own, own[p], ob, cudaMemcpyDeviceToDevice, c->stream));
    if (c->comm.world > 1) {
        // interior cuts have 18 rows of staging on both sides (every band >= 18 rows); the outermost ranks have no
        // neighbour there and comm_halo_exchange skips those pointers
        const bool has_up = c->comm.rank > 0, has_dn = c->comm.rank + 1 < c->comm.world;
        float *su[3], *ru[3], *sd[3], *rd[3];
        for (int p = 0; p < 3; p++) {
            su[p] = ext[p] + at_own;                                                // my first 18 rows -> rank-1
            ru[p] = has_up ? ext[p] : nullptr;                                      // rank-1's last 18 rows (e0 = own0-18)
            sd[p] = ext[p] + (size_t)(own1 - SRSAL_R - e0) * nx;                    // my last 18 rows -> rank+1
            rd[p] = has_dn ? ext[p] + (size_t)(own1 - e0) * nx : nullptr;           // rank+1's first 18 rows
        }
        if (comm_halo_exchange(&c->comm, 3, su, ru, sd, rd, (size_t)SRSAL_R * nx, c->stream)) {
            set_err("%s", comm_last_error());
            return OCTANE_ECOMM;
        }
    }
    SrsalTaps t;
    srsal_taps(&t);
    launch_srsal(ext[0], ext[1], ext[2], nx, ny, e0, own0, own1, t, d_u, d_v, c->stream);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}
}  // namespace

int octane_srsal_band_dev(octane_ctx* c, float* d_u, float* d_v, const float* d_cth, int nx, int ny)
{
    if (!c || !d_u || !d_v || !d_cth || nx <= SRSAL_R || ny <= SRSAL_R) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    const int world = c->comm.world;
    if (world <= 1) return octane_srsal_dev(c, d_u, d_v, d_cth, nx, ny);
    if (!srsal_bands_ok(ny, world)) {
        set_err("-srsal on row bands needs every band at least 18 rows high: fewer ranks or a taller scene");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    int own0, own1;
    own_rows(ny, c->comm.rank, world, &own0, &own1);
    // the staging is the only step that can fail on one rank alone: vote on it before the exchange, so that a rank
    // without memory returns an error on every rank instead of leaving its peers waiting in the exchange
    int local = ensure_stage(c, srsal_band_stage_bytes(nx, ny, own0, own1));
    if (local) cudaGetLastError();          // a failed allocation is not a sticky error: keep it out of later checks
    const double mine = local ? 0.0 : 1.0;
    double all = 0.0;
    CUDA_OK(cudaMemcpyAsync(c->d_vote, &mine, sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if (comm_allreduce_f64(&c->comm, c->d_vote, 1, c->stream)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    CUDA_OK(cudaMemcpyAsync(&all, c->d_vote, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    if (local) return local;
    if (all != (double)world) { set_err("-srsal on row bands: a peer could not allocate its staging"); return OCTANE_ENOMEM; }
    return srsal_band_enqueue(c, d_u, d_v, d_cth, nx, ny, own0, own1, c->stage);
}

int octane_srsal(octane_ctx* c, float* u, float* v, const float* cth, int nx, int ny)
{
    if (!c || !u || !v || !cth || nx <= SRSAL_R || ny <= SRSAL_R) { set_err("null or invalid argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t fb = align_up((size_t)nx * ny * sizeof(float)), nb = (size_t)nx * ny * sizeof(float);
    int rc = ensure_stage(c, 5 * fb);
    if (rc) return rc;
    float* d_u = (float*)(c->stage + 2 * fb);
    float* d_v = (float*)(c->stage + 3 * fb);
    float* d_c = (float*)(c->stage + 4 * fb);
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_u, u, nb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_v, v, nb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_c, cth, nb, cudaMemcpyHostToDevice, c->stream));
    rc = srsal_enqueue(c, d_u, d_v, d_c, nx, ny, (float*)c->stage, (float*)(c->stage + fb));
    if (rc) return rc;
    CUDA_OK(cudaMemcpyAsync(u, d_u, nb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(v, d_v, nb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

int octane_uv2pix_dev(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* d_lat,
                      const float* d_lon, const short* d_x, const short* d_y, int nx, int ny,
                      const octane_params* p, float* d_u, float* d_v)
{
    if (!c || !nav || !d_lat || !d_lon || !d_x || !d_y || !p || !d_u || !d_v || nx <= 0 || ny <= 0) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t fb = (size_t)nx * ny * sizeof(float);
    // src/oct_pix2uv_cuda.cu:421: exact comparison; otherwise the first guess is zero (:464-474)
    if (!((nav->xOffset == nav->g2xOffset) && (nav->yOffset == nav->g2yOffset))) {
        CUDA_OK(cudaMemsetAsync(d_u, 0, fb, c->stream));
        CUDA_OK(cudaMemsetAsync(d_v, 0, fb, c->stream));
        return 1;
    }
    Uv2PixParams q;
    q.secs = t2 - t1;
    q.req = nav->req; q.rpol = nav->rpol; q.req2 = nav->req * nav->req; q.rpol2 = nav->rpol * nav->rpol;
    double eval = sqrt((q.req2 - q.rpol2) / (q.req2));               // :417-428
    q.eval = eval * eval;
    q.lam0 = nav->lam0; q.pph = nav->pph;
    q.xscale = nav->xScale; q.xoffset = nav->xOffset; q.yscale = nav->yScale; q.yoffset = nav->yOffset;
    launch_uv2pix(d_u, d_v, d_lat, d_lon, d_x, d_y, nx, ny, q, c->stream);
    c->launches++;
    CUDA_OK(cudaGetLastError());
    return OCTANE_OK;
}

int octane_uv2pix(octane_ctx* c, const octane_nav* nav, double t1, double t2, const float* lat, const float* lon,
                  const short* x, const short* y, int nx, int ny, const octane_params* p, float* u, float* v)
{
    if (!c || !nav || !lat || !lon || !x || !y || !p || !u || !v || nx <= 0 || ny <= 0) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    const size_t n = (size_t)nx * ny, fb = n * sizeof(float);
    const size_t xb = align_up((size_t)nx * sizeof(short)), yb = align_up((size_t)ny * sizeof(short));
    int rc = ensure_stage(c, 4 * fb + xb + yb);
    if (rc) return rc;
    char* s = c->stage;
    float* d_u = (float*)s; s += fb;
    float* d_v = (float*)s; s += fb;
    float* d_lat = (float*)s; s += fb;
    float* d_lon = (float*)s; s += fb;
    short* d_x = (short*)s; s += xb;
    short* d_y = (short*)s;
    begin_call(c);
    CUDA_OK(cudaMemcpyAsync(d_u, u, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_v, v, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_lat, lat, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_lon, lon, fb, cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_x, x, (size_t)nx * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    CUDA_OK(cudaMemcpyAsync(d_y, y, (size_t)ny * sizeof(short), cudaMemcpyHostToDevice, c->stream));
    rc = octane_uv2pix_dev(c, nav, t1, t2, d_lat, d_lon, d_x, d_y, nx, ny, p, d_u, d_v);
    if (rc < 0) return rc;
    CUDA_OK(cudaMemcpyAsync(u, d_u, fb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaMemcpyAsync(v, d_v, fb, cudaMemcpyDeviceToHost, c->stream));
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return rc;
}

// ---- band planning / NCCL bootstrap ----------------------------------------------------------
int octane_band_plan(int nx, int ny, const octane_params* p, int rank, int world, int* own0, int* own1, int* in0, int* in1)
{
    if (!p || rank < 0 || world < 1 || rank >= world) { set_err("invalid argument"); return OCTANE_EINVAL; }
    Plan pl;
    int rc = make_plan(pl, nx, ny, 1, *p, rank, world);
    if (rc) return rc;
    if (own0) *own0 = pl.lv.back().own0;
    if (own1) *own1 = pl.lv.back().own1;
    if (in0) *in0 = pl.in0;
    if (in1) *in1 = pl.in1;
    return OCTANE_OK;
}

int octane_comm_unique_id(char id[128])
{
    if (!id) return OCTANE_EINVAL;
    if (comm_unique_id(id)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    return OCTANE_OK;
}

int octane_comm_init(octane_ctx* c, const char id[128], int rank, int world)
{
    if (!c || !id || rank < 0 || world < 1 || rank >= world) { set_err("invalid argument"); return OCTANE_EINVAL; }
    CUDA_OK(cudaSetDevice(c->device));
    c->plan_valid = false;
    destroy_graphs(c);
    comm_destroy(&c->comm);
    if (world == 1) return OCTANE_OK;
    // allocated once, before any collective: the vote of a later call must not itself need an allocation
    if (!c->d_vote) CUDA_OK(cudaMalloc(&c->d_vote, sizeof(double)));
    if (comm_init(&c->comm, id, rank, world)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    // per-iteration exchanges over peer memory when every rank can map its peers (else NCCL)
    if (comm_p2p_init(&c->comm, sizeof(P2PWindow), c->stream)) { set_err("%s", comm_last_error()); return OCTANE_ECOMM; }
    return OCTANE_OK;
}

int octane_comm_rank(octane_ctx* c, int* rank, int* world)
{
    if (!c) return OCTANE_EINVAL;
    if (rank) *rank = c->comm.rank;
    if (world) *world = c->comm.world;
    return OCTANE_OK;
}

// ---- pipelined host-buffer dispatcher -----------------------------------------------------------
// The reference handles one pair per process run (src/main.cc:439 -> oct_optical_flow); reprocessing an archive or a
// 1-minute mesoscale sequence is a loop over pairs.  For that loop the copies are the only part of a step the GPU
// does not need to wait for: submit() enqueues copy-in -> solve -> navigation -> copy-out of one pair on three
// streams and returns, wait() blocks until that pair's outputs are in host memory; with two slots the copies of
// pair k+1 and k-1 run under the solve of pair k.
namespace {
int slot_prepare(octane_ctx* c, int k, size_t bytes)
{
    auto& sl = c->slot[k];
    if (!c->h2d_stream) CUDA_OK(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
    if (!sl.done) {
        CUDA_OK(cudaEventCreateWithFlags(&sl.in_ready, cudaEventDisableTiming));
        CUDA_OK(cudaEventCreateWithFlags(&sl.in_free, cudaEventDisableTiming));
        CUDA_OK(cudaEventCreateWithFlags(&sl.out_ready, cudaEventDisableTiming));
        CUDA_OK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        CUDA_OK(cudaEventCreateWithFlags(&sl.mid, cudaEventDisableTiming));
    }
    if (bytes > sl.bytes) {
        if (sl.busy) CUDA_OK(cudaEventSynchronize(sl.done));
        CUDA_OK(cudaStreamSynchronize(c->stream));
        if (sl.buf) cudaFree(sl.buf);
        sl.buf = nullptr; sl.bytes = 0;
        CUDA_OK(cudaMalloc(&sl.buf, bytes));
        sl.bytes = bytes;
    }
    return OCTANE_OK;
}
}  // namespace

namespace {
// octane_stream_submit and octane_stream_submit_fg: fg_u / fg_v are host rows [in0,in1) of the first guess, read only
// when p->first_guess (the callers check which of the two may set it)
int stream_submit(octane_ctx* c, int k, const float* img1, const float* img2, const float* fg_u, const float* fg_v,
                  const float* cth, int nx, int ny, int nc, const octane_nav* nav, double t1, double t2,
                  const octane_params* p, float* upix, float* vpix, short* U, short* V, short* Ur, short* Vr, short* ctp)
{
    if (!c || (k != 0 && k != 1) || !img1 || !img2 || !nav || !p || !U || !V || !Ur || !Vr || (!upix != !vpix)) {
        set_err("null or invalid argument");
        return OCTANE_EINVAL;
    }
    if (p->doCTH && (!cth || !ctp)) { set_err("doCTH needs cth and ctp"); return OCTANE_EINVAL; }
    if (!srsal_args_ok(p, cth, nx, ny)) return OCTANE_EINVAL;
    // -srsal changes the pixel displacements only (src/oct_optical_flow.cc:91-105): a submit that does not ask for them
    // would smooth nothing it returns
    if (p->dosrsal && !upix) { set_err("dosrsal smooths upix / vpix only: the pipelined dispatcher needs them"); return OCTANE_EINVAL; }
    if (p->dosrsal && !srsal_bands_ok(ny, c->comm.world)) {
        set_err("-srsal on row bands needs every band at least 18 rows high: fewer ranks or a taller scene");
        return OCTANE_EINVAL;
    }
    CUDA_OK(cudaSetDevice(c->device));
    int rc = prepare(c, nx, ny, nc, *p);
    if (rc) return rc;
    const Level& F = c->plan.lv.back();
    const bool banded = c->comm.world > 1;
    const size_t nin = (size_t)F.g.rows * nx, nown = (size_t)(F.own1 - F.own0) * nx;
    const size_t ib = align_up(nin * nc * sizeof(float)), fb = align_up(nown * sizeof(float)), sb = align_up(nown * sizeof(short));
    const size_t gb = p->first_guess ? align_up(nin * sizeof(float)) : 0;
    // -srsal staging: two result planes on one GPU, the three extended planes of the band otherwise
    const size_t rb = !p->dosrsal ? 0 : banded ? srsal_band_stage_bytes(nx, ny, F.own0, F.own1) : 2 * fb;
    auto& sl = c->slot[k];
    if (sl.busy) {                       // resubmitting a slot implies its previous pair is finished with
        rc = flush_copy_out(c, k, false);
        if (rc) return rc;
        CUDA_OK(cudaEventSynchronize(sl.done));
        sl.busy = false;
    }
    rc = slot_prepare(c, k, 2 * ib + 3 * fb + 5 * sb + 2 * gb + rb);
    if (rc) return rc;
    // When does the copy-out of a pair run?  On one GPU right after its navigation, under the next pair's solve.
    // In a banded run the peer-memory exchanges of every PCG iteration end in system-scope fences, and those take
    // far longer while a device-to-host copy is in flight (DESIGN.md section 5): the copy-out of the pair in the
    // OTHER slot is therefore held back until this pair's solve reaches its finest level, where an iteration is
    // long and the iterations under the copy are few -- not under the hundreds of short coarse-level iterations a
    // solve starts with.  wait() enqueues it at once if no later submit() has.
    static const int defer_env = getenv("OCTANE_STREAM_DEFER") ? atoi(getenv("OCTANE_STREAM_DEFER")) : -1;   // developer switch
    const bool defer = defer_env >= 0 ? defer_env != 0 : banded;
    c->copy_out_at_finest = (defer && c->slot[k ^ 1].copy_pending) ? (k ^ 1) : -1;
    char* q = sl.buf;
    float* d_i1 = (float*)q; q += ib;
    float* d_i2 = (float*)q; q += ib;
    float* d_u = (float*)q; q += fb;
    float* d_v = (float*)q; q += fb;
    float* d_cth = (float*)q; q += fb;
    short* d_s = (short*)q; q += 5 * sb;
    float* d_fgu = p->first_guess ? (float*)q : nullptr; q += gb;
    float* d_fgv = p->first_guess ? (float*)q : nullptr; q += gb;
    char* d_srsal = q;
    const size_t sstride = sb / sizeof(short);
    // copy-in on its own stream: runs under the solve of the pair in the other slot
    CUDA_OK(cudaMemcpyAsync(d_i1, img1, nin * nc * sizeof(float), cudaMemcpyHostToDevice, c->h2d_stream));
    CUDA_OK(cudaMemcpyAsync(d_i2, img2, nin * nc * sizeof(float), cudaMemcpyHostToDevice, c->h2d_stream));
    if (p->first_guess) {
        CUDA_OK(cudaMemcpyAsync(d_fgu, fg_u, nin * sizeof(float), cudaMemcpyHostToDevice, c->h2d_stream));
        CUDA_OK(cudaMemcpyAsync(d_fgv, fg_v, nin * sizeof(float), cudaMemcpyHostToDevice, c->h2d_stream));
    }
    if (p->doCTH || p->dosrsal) CUDA_OK(cudaMemcpyAsync(d_cth, cth, nown * sizeof(float), cudaMemcpyHostToDevice, c->h2d_stream));
    CUDA_OK(cudaEventRecord(sl.in_ready, c->h2d_stream));
    // solve + navigation on the context's stream
    begin_call(c);
    if (c->d_scal) CUDA_OK(cudaMemsetAsync(&c->d_scal->halo_err, 0, 2 * sizeof(int), c->stream));
    CUDA_OK(cudaStreamWaitEvent(c->stream, sl.in_ready, 0));
    {
        Scope total(c, CAT_TOTAL);
        rc = ingest(c, d_i1, d_i2, d_fgu, d_fgv);
        if (rc) return rc;
        CUDA_OK(cudaEventRecord(sl.in_free, c->stream));
        rc = run_levels(c);
        if (rc) return rc;
        rc = emit(c, d_u, d_v);
        if (rc) return rc;
    }
    if (p->doCTH) {
        launch_ctp_pack(d_cth, d_s + 4 * sstride, nown, p->ir == 1, c->stream);
        c->launches++;
    }
    const int nrc = pix2uv_dev_rows(c, nav, t1, t2, d_u, d_v, nx, F.own0, F.own1 - F.own0, p, d_s, d_s + sstride,
                                    d_s + 2 * sstride, d_s + 3 * sstride);
    if (nrc < 0) return nrc;
    if (p->dosrsal) {      // src/oct_optical_flow.cc:100-105: after the navigation, so only uPix / vPix are smoothed
        rc = banded ? srsal_band_enqueue(c, d_u, d_v, d_cth, nx, ny, F.own0, F.own1, d_srsal)
                    : srsal_enqueue(c, d_u, d_v, d_cth, nx, ny, (float*)d_srsal, (float*)(d_srsal + fb));
        if (rc) return rc;
    }
    CUDA_OK(cudaEventRecord(sl.out_ready, c->stream));
    // copy-out
    sl.ncopy = 0;
    auto add = [&](void* dst, const void* src, size_t n) { sl.dst[sl.ncopy] = dst; sl.src[sl.ncopy] = src; sl.nbytes[sl.ncopy] = n; sl.ncopy++; };
    short* hs[4] = { U, V, Ur, Vr };
    for (int i = 0; i < 4; i++) add(hs[i], d_s + i * sstride, nown * sizeof(short));
    if (p->doCTH) add(ctp, d_s + 4 * sstride, nown * sizeof(short));
    if (upix) { add(upix, d_u, nown * sizeof(float)); add(vpix, d_v, nown * sizeof(float)); }
    sl.copy_pending = true;
    sl.busy = true;
    if (c->copy_out_at_finest >= 0) {    // a solve that never reached run_levels' hook (cannot happen today): do not lose the copy
        rc = flush_copy_out(c, c->copy_out_at_finest, false);
        c->copy_out_at_finest = -1;
        if (rc) return rc;
    }
    if (!defer) { rc = flush_copy_out(c, k, false); if (rc) return rc; }
    return nrc;
}

}  // namespace

int octane_stream_submit(octane_ctx* c, int k, const float* img1, const float* img2, const float* cth, int nx, int ny, int nc,
                         const octane_nav* nav, double t1, double t2, const octane_params* p, float* upix, float* vpix,
                         short* U, short* V, short* Ur, short* Vr, short* ctp)
{
    if (p && p->first_guess) { set_err("the pipelined dispatcher takes a first guess through octane_stream_submit_fg"); return OCTANE_EINVAL; }
    return stream_submit(c, k, img1, img2, nullptr, nullptr, cth, nx, ny, nc, nav, t1, t2, p, upix, vpix, U, V, Ur, Vr, ctp);
}

int octane_stream_submit_fg(octane_ctx* c, int k, const float* img1, const float* img2, const float* fg_u, const float* fg_v,
                            const float* cth, int nx, int ny, int nc, const octane_nav* nav, double t1, double t2,
                            const octane_params* p, float* upix, float* vpix, short* U, short* V, short* Ur, short* Vr, short* ctp)
{
    if (p && !p->first_guess) { set_err("octane_stream_submit_fg needs p->first_guess"); return OCTANE_EINVAL; }
    if (!fg_u || !fg_v) { set_err("octane_stream_submit_fg: no first guess was given"); return OCTANE_EINVAL; }
    return stream_submit(c, k, img1, img2, fg_u, fg_v, cth, nx, ny, nc, nav, t1, t2, p, upix, vpix, U, V, Ur, Vr, ctp);
}

int octane_stream_wait(octane_ctx* c, int k)
{
    if (!c || (k != 0 && k != 1)) { set_err("invalid argument"); return OCTANE_EINVAL; }
    auto& sl = c->slot[k];
    if (!sl.busy) return OCTANE_OK;
    CUDA_OK(cudaSetDevice(c->device));
    int rc = flush_copy_out(c, k, false);       // not yet enqueued by a later submit(): now
    if (rc) return rc;
    CUDA_OK(cudaEventSynchronize(sl.done));
    sl.busy = false;
    if (c->comm.world > 1) {
        if (c->h_scal->halo_err) { set_err("warp left the band halo: raise max_disp"); return OCTANE_EHALO; }
        if (c->h_scal->comm_err) { set_err("a peer's partial sums did not arrive (peer-memory exchange timed out)"); return OCTANE_ECOMM; }
    }
    return OCTANE_OK;
}

// ---- stage entry points (parity tests) -----------------------------------------------------
static Geom dense_geom(int nx, int ny)
{
    Geom g; g.nx = nx; g.ny = ny; g.pitch = nx; g.j0 = 0; g.rows = ny; g.plane = (long long)nx * ny;
    return g;
}

int octane_stage_blur_decimate(octane_ctx* c, const float* d_img, int nx, int ny, int nc, float factor, float* d_out)
{
    if (!c || !d_img || !d_out) return OCTANE_EINVAL;
    CUDA_OK(cudaSetDevice(c->device));
    int rc = ensure_small(c, c->sm_count * 16); if (rc) return rc;
    int nxx, nyy;
    zoom_size(nx, ny, factor, &nxx, &nyy);
    const int R = filter_radius(factor);
    Geom gs = dense_geom(nx, ny), gd = dense_geom(nxx, nyy);
    launch_fill_gk(c->d_gk, factor, R, c->stream);
    launch_blur_decimate(d_img, gs, d_out, gd, 0, nyy, factor, c->d_gk, R, 1.f, nc, c->stream);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

int octane_stage_gradient(octane_ctx* c, const float* d_f, int xi, int yi, int nc, float* d_gx, float* d_gy)
{
    if (!c || !d_f || !d_gx || !d_gy) return OCTANE_EINVAL;
    CUDA_OK(cudaSetDevice(c->device));
    launch_gradient(d_f, d_gx, d_gy, dense_geom(xi, yi), 0, yi, nc, c->stream);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

int octane_stage_zoom_in(octane_ctx* c, const float* d_flow, int nx, int ny, int nxx, int nyy, float sf, float* d_out)
{
    if (!c || !d_flow || !d_out) return OCTANE_EINVAL;
    CUDA_OK(cudaSetDevice(c->device));
    launch_zoom_in(d_flow, dense_geom(nx, ny), d_out, dense_geom(nxx, nyy), 0, nyy, sf, c->stream);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaStreamSynchronize(c->stream));
    return OCTANE_OK;
}

// The build and PCG stages run on the pitched workspace exactly as the full solve does:
// dense inputs are copied in, the level's kernels run, dense outputs are copied out.
static int stage_prepare(octane_ctx* c, int xi, int yi, int nc, const octane_params* p)
{
    octane_params q = *p;
    q.kiters = 1;             // a single level of size xi x yi
    return prepare(c, xi, yi, nc, q);
}

static int copy_in(octane_ctx* c, float* dst, const float* src, const Geom& g, int nplanes)
{
    const size_t w = (size_t)g.nx * sizeof(float), dp = (size_t)g.pitch * sizeof(float);
    for (int k = 0; k < nplanes; k++)
        CUDA_OK(cudaMemcpy2DAsync(dst + (size_t)k * g.plane, dp, src + (size_t)k * g.nx * g.ny, w, w, g.ny,
                                  cudaMemcpyDeviceToDevice, c->stream));
    return OCTANE_OK;
}
static int copy_out(octane_ctx* c, float* dst, const float* src, const Geom& g)
{
    const size_t w = (size_t)g.nx * sizeof(float), dp = (size_t)g.pitch * sizeof(float);
    CUDA_OK(cudaMemcpy2DAsync(dst, w, src, dp, w, g.ny, cudaMemcpyDeviceToDevice, c->stream));
    return OCTANE_OK;
}

int octane_stage_build(octane_ctx* c, const float* d_u, const float* d_v, const float* d_uh, const float* d_vh,
                       const float* d_g1, const float* d_g2, int xi, int yi, int nc, const octane_params* p,
                       float lambdac_level, int gnc, float* d_coef, float* d_bu, float* d_bv)
{
    if (!c || !d_u || !d_v || !d_g1 || !d_g2 || !p || !d_coef || !d_bu || !d_bv) return OCTANE_EINVAL;
    octane_params q = *p;
    q.first_guess = (d_uh && d_vh) ? 1 : 0;
    int rc = stage_prepare(c, xi, yi, nc, &q); if (rc) return rc;
    Buffers& B = c->buf;
    const Geom& g = c->plan.lv[0].g;
    cudaStream_t st = c->stream;
    if ((rc = copy_in(c, B.img1, d_g1, g, nc))) return rc;
    if ((rc = copy_in(c, B.img2, d_g2, g, nc))) return rc;
    if ((rc = copy_in(c, B.u, d_u, g, 1))) return rc;
    if ((rc = copy_in(c, B.v, d_v, g, 1))) return rc;
    if (q.first_guess) { if ((rc = copy_in(c, B.uh, d_uh, g, 1))) return rc; if ((rc = copy_in(c, B.vh, d_vh, g, 1))) return rc; }
    launch_gradient(B.img1, B.g1x, B.g1y, g, 0, yi, nc, st);
    launch_gradient(B.img2, B.g2x, B.g2y, g, 0, yi, nc, st);
    launch_gradient(B.g2x, B.g2xx, nullptr, g, 0, yi, nc, st);
    launch_gradient(B.g2y, B.g2xy, B.g2yy, g, 0, yi, nc, st);
    LevelFields f;
    f.g1 = B.img1; f.g1x = B.g1x; f.g1y = B.g1y;
    f.g2 = B.img2; f.g2x = B.g2x; f.g2y = B.g2y; f.g2xx = B.g2xx; f.g2xy = B.g2xy; f.g2yy = B.g2yy;
    f.u = B.u; f.v = B.v;
    f.uh = (q.first_guess && lambdac_level != 0.f) ? B.uh : nullptr;
    f.vh = (q.first_guess && lambdac_level != 0.f) ? B.vh : nullptr;
    BuildParams bp;
    bp.alpha = p->alpha; bp.ralpha = 1.0 / p->alpha; bp.lambdadalpha = p->lambda / p->alpha; bp.lambdac = lambdac_level;
    bp.dozim = p->dozim != 0; bp.nchan = nc; bp.tol = 0.0001 * 0.0001; bp.al1 = 1. - 0.5 * gnc;
    launch_build(f, B.pcg, g, 0, yi, 0, yi, bp, 0, st);
    // the 7 boundary-merged entries of the reference, expanded from the 5 stored planes
    // (scratch: the PCG vectors, which the build does not touch)
    float* e[4] = { B.pcg.pu[0], B.pcg.pv[0], B.pcg.pu[1], B.pcg.pv[1] };
    launch_expand_coef(B.pcg, g, e[0], e[1], e[2], e[3], st);
    const float* src7[7] = { B.pcg.coef[C_A1], B.pcg.coef[C_A2], B.pcg.coef[C_A4], e[0], e[1], e[2], e[3] };
    for (int k = 0; k < 7; k++) if ((rc = copy_out(c, d_coef + (size_t)k * xi * yi, src7[k], g))) return rc;
    if ((rc = copy_out(c, d_bu, B.pcg.ru, g))) return rc;
    if ((rc = copy_out(c, d_bv, B.pcg.rv, g))) return rc;
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaStreamSynchronize(st));
    return OCTANE_OK;
}

// seeds the PCG scalars from (coef, b) like the tail of the build kernel does
__global__ void k_seed_scalars(PcgBuffers b, Geom g, float tol)
{
    __shared__ double red[2 * 32];
    double acc[2] = { 0.0, 0.0 };
    for (int j = 0; j < g.ny; j++)
        for (int i = threadIdx.x; i < g.nx; i += blockDim.x) {
            const size_t l = g.at(i, j);
            const float bu = b.ru[l], bv = b.rv[l];
            const float mu = 1. / b.coef[C_A1][l], mv = 1. / b.coef[C_A4][l];
            acc[0] += (double)(bu * bu) + (double)(bv * bv);
            acc[1] += (double)(bu * (mu * bu)) + (double)(bv * (mv * bv));
        }
    block_sum<2>(acc, red);
    if (threadIdx.x == 0) {
        PcgScalars* s = b.scal;
        s->rr = (float)acc[0]; s->rz = (float)acc[1]; s->rz_old = 0.f; s->pAp = 0.f; s->alpha = 0.f;
        s->tol = tol; s->its = 0; s->done = !((float)acc[0] > tol);
    }
}

__global__ void k_unmerge_edges(PcgBuffers b, Geom g)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < g.ny) b.coef[C_W][g.at(0, t)] *= 0.5f;                       // a7(0,j) = 2 W(0,j)
    else if (t - g.ny < g.nx) b.coef[C_N][g.at(t - g.ny, 0)] *= 0.5f;    // a8(i,0) = 2 N(i,0)
}

int octane_stage_pcg(octane_ctx* c, const float* d_coef, const float* d_bu, const float* d_bv, int xi, int yi,
                     int iters, float tol, float* d_xu, float* d_xv, int* iterations)
{
    if (!c || !d_coef || !d_bu || !d_bv || !d_xu || !d_xv) return OCTANE_EINVAL;
    octane_params q;
    octane_params_default(&q);
    q.cgiters = iters;
    int rc = stage_prepare(c, xi, yi, 1, &q); if (rc) return rc;
    Buffers& B = c->buf;
    const Level& L = c->plan.lv[0];
    const Geom& g = L.g;
    cudaStream_t st = c->stream;
    // d_coef must be a system as the build produces it: symmetric couplings, mirror-merged
    // edges.  W = a7 and N = a8 with the edge doubling undone (first column / first row).
    const int src5[NCOEF] = { 0, 1, 2, 5, 6 };
    for (int k = 0; k < NCOEF; k++)
        if ((rc = copy_in(c, B.pcg.coef[k], d_coef + (size_t)src5[k] * xi * yi, g, 1))) return rc;
    k_unmerge_edges<<<(xi + yi + 255) / 256, 256, 0, st>>>(B.pcg, g);
    if ((rc = copy_in(c, B.pcg.ru, d_bu, g, 1))) return rc;
    if ((rc = copy_in(c, B.pcg.rv, d_bv, g, 1))) return rc;
    k_seed_scalars<<<1, 1024, 0, st>>>(B.pcg, g, tol);
    CUDA_OK(cudaMemsetAsync(B.u, 0, (size_t)g.plane * sizeof(float), st));
    CUDA_OK(cudaMemsetAsync(B.v, 0, (size_t)g.plane * sizeof(float), st));
    begin_call(c);
    rc = run_pcg(c, L, 0, 0, 0); if (rc) return rc;
    if (level_fused(c, L)) launch_update_uv_fused(B.u, B.v, B.pcg, g, 0, yi, c->d_its, c->sm_count, st);
    else launch_update_uv(B.u, B.v, B.pcg, g, 0, yi, c->d_its, c->sm_count, st);   // u = 0 + x
    if ((rc = copy_out(c, d_xu, B.u, g))) return rc;
    if ((rc = copy_out(c, d_xv, B.v, g))) return rc;
    CUDA_OK(cudaMemcpyAsync(c->h_its, c->d_its, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaStreamSynchronize(st));
    if (iterations) *iterations = c->h_its[0];
    return OCTANE_OK;
}

}  // extern "C"
