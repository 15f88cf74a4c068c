// sph_engine.cu — world state, step driver and the extern "C" boundary (include/sph.h) of the
// B200-native SPH step path.  The step sequence restates LiquidWorld::step_with_coupling
// (liquid_world.rs:67-158) + DFSPHSolver::step (dfsph_solver.rs:667-708) / IISPHSolver::step
// (iisph_solver.rs:643-711) as a chain of CUDA kernels on one stream; see DESIGN.md.
//
// There is no CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sph.h"
#include "sph_kernels.cuh"
#include "sph_passes.cuh"
#include "sph_tile.cuh"
#include "sph_iisph.cuh"
#include "sph_elasticity.cuh"
#include "sph_viscosity.cuh"

using namespace sphk;

namespace {

// All worlds of a process share the module's __constant__ block; API calls are serialised per process
// (GPU work of different worlds on one device would serialise anyway) and re-upload it on entry.
// recursive: host-force and coupling callbacks run inside sph_world_step and may call back into the API (reads,
// boundary rewrites, queries) on the same thread
std::recursive_mutex g_mutex;
const void* g_const_owner = nullptr;

inline uint32_t cdiv(size_t a, size_t b) { return (uint32_t)((a + b - 1) / b); }

template <class T>
struct DBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n, bool keep = false, cudaStream_t st = 0) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = std::max(n, cap + cap / 4);
        T* q = nullptr;
        cudaError_t e = cudaMalloc(&q, ncap * sizeof(T));
        if (e != cudaSuccess) return e;
        if (keep && p && cap) {
            e = cudaMemcpyAsync(q, p, cap * sizeof(T), cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
            cudaStreamSynchronize(st);
        }
        if (p) cudaFree(p);
        p = q;
        cap = ncap;
        return cudaSuccess;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct ForceRec;
}  // namespace
struct sph_world;
namespace {
constexpr int FORCE_HOST_CALLBACK = 100;  // internal kind of sph_fluid_push_host_force entries
struct ForceRec {
    sph_force_desc d;
    sph_host_force_fn host_fn = nullptr;
    sph_host_force_fn2 host_fn2 = nullptr;  // context-style callback (contacts / boundaries on request)
    uint32_t host_flags = 0;
    void* host_user = nullptr;
    ElasticityState* elastic = nullptr;  // Becker2009 rest-pose state (sph_elasticity.cuh)
    uint32_t visc_iters = 0;             // DFSPHViscosity: acceleration updates of the last solve
    float visc_err = 0.f;                // ... and its last strain-rate error
};
struct FluidRec {
    size_t n = 0, offset = 0;
    float density0 = 1000.f;
    uint32_t memberships = 1, filter = 0xFFFFFFFFu;
    std::vector<ForceRec> forces;
    std::vector<uint8_t> pending_delete;
    size_t n_pending = 0;
    float uniform_mass = 0.f;  // common particle mass if all volumes are equal, else 0
    bool alive = true;         // false after LiquidWorld::remove_fluid (liquid_world.rs:171-173); the slot is reused by the next add
    uint32_t gen = 0;          // handle = slot | gen << 16 (the reference's arena handles carry a generation too)
};
struct BoundaryRec {
    size_t n = 0, offset = 0;
    uint32_t memberships = 1, filter = 0xFFFFFFFFu;
    bool want_forces = false;
    bool alive = true;
    uint32_t gen = 0;
};

sph_status iisph_step(sph_world* w, float dt_total, const float g[3]);
sph_status slab_begin_step(sph_world* w);
sph_status slab_after_sort(sph_world* w);
sph_status slab_refresh(sph_world* w, void* array, size_t elem);
struct SlabArray {
    void* p;
    size_t elem;
};
sph_status slab_refresh_n(sph_world* w, const SlabArray* arrays, int n_arrays);
sph_status p2p_setup(sph_world* w);
sph_status post_density_refresh(sph_world* w);
sph_status slab_allreduce(sph_world* w, float* buf, size_t n);
void iisph_release(sph_world* w);
void slab_release(sph_world* w);
const float* iisph_pred(sph_world* w);
sph_status elasticity_solve(sph_world* w, uint32_t fluid, ForceRec& fr);
void elasticity_release(ForceRec& fr);
sph_status elasticity_restore(sph_world* w, ForceRec& fr, size_t n, uint32_t cap0, uint32_t stride0, const char* blob);
sph_status viscosity_solve(sph_world* w, uint32_t fluid, ForceRec& fr);
void viscosity_release(sph_world* w);
inline float __uint_as_float_host(uint32_t u) {
    float f;
    memcpy(&f, &u, sizeof f);
    return f;
}

struct P2PState {  // NVLink peer-memory exchange (sph_slab.inl)
    bool on = false;
    size_t box_bytes = 0;
    char* base = nullptr;          // my landing zones + flags + reduction table (one cudaIpc-exported allocation)
    char* peer_base[8] = {};       // the same allocation of every rank, mapped into this process ([rank] == base)
    uint32_t seq_send[2] = {0, 0}, seq_recv[2] = {0, 0}, red_seq = 0;
    DBuf<uint32_t> tickets;
};

struct SlabState {
    bool active = false, own_comm = false;
    P2PState p2p;
    int rank = 0, nranks = 1;
    int lo = INT_MIN, hi = INT_MAX;  // owned cell columns [lo, hi) in absolute cell coordinates floor(x / h)
    int has_left = 0, has_right = 0;
    void* comm = nullptr;
    DBuf<uint32_t> d_cnt, flag, gid_l, gid_r, gid_cl, gid_cr;
    uint32_t cap_out = 1u << 14, cap_col = 1u << 17;  // staging capacities (emigrants / boundary-column particles per side); grown on demand
    uint32_t sort_off = 0, sort_n = 0, sort_dead_n = 0;  // what the step's counting sort reads (set by slab_begin_step)
    DBuf<unsigned long long> d_cnt64;
    DBuf<float4> out_l[3], out_r[3], col_l[3], col_r[3];
    bool global_valid = false;
    // slot ranges of the current step (after the sort)
    uint32_t gl_count = 0, sl_begin = 0, sl_count = 0, sr_begin = 0, sr_count = 0, gr_begin = 0, gr_count = 0;
    uint32_t exp_ghost_l = 0, exp_ghost_r = 0, exp_send_l = 0, exp_send_r = 0;
    uint32_t migrated_in = 0, migrated_out = 0;
    unsigned long long global_n = 0;
};

enum { EV_START = 0, EV_GRID, EV_NBR, EV_DENS, EV_DIV, EV_FOLD, EV_FORCES, EV_INTEG, EV_PRESS, EV_END, EV_COUNT };

}  // namespace

struct sph_world {
    sph_world_desc desc;
    float h = 0.f;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    cudaEvent_t ev_lists = nullptr;  // list-capacity read-back of phase_neighbors
    std::string err;
    Consts hc;

    std::vector<FluidRec> fluids;
    std::vector<BoundaryRec> bounds;
    size_t N = 0, B = 0;   // N = fluid particles OWNED by this world
    size_t Ntot = 0;       // slots of the sorted arrays during a step: owned + ghost (== N on one GPU)
    int protect_buf = -1;    // double-buffer index ensure_fluid_buffers() must not reallocate (it is being read)
    uint32_t own_begin = 0;  // first owned slot (ghost columns of a slab world sit at both ends of the sorted arrays)
    SlabState slab;
    uint64_t stats_exchanges = 0;

    // timestep_manager.rs:21-31: dt/inv_dt are 0 until the first advance()
    float dt = 0.f, inv_dt = 0.f;
    int force_div = -1, force_press = -1;

    // host truth in ORIGINAL order while `staged` (before the first step / after structural edits)
    bool staged = true;
    std::vector<float> h_pos, h_vel, h_vc, h_vol, h_press;
    // boundaries: host copy is always kept (static data); b_dirty => re-upload
    bool b_dirty = true;
    int b_aabb[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};  // boundary cell-coordinate AABB (host side, static)
    bool b_bad = false;
    // the boundary sort / volumes are reused while the boundaries and the grid mapping are unchanged
    bool b_sorted_valid = false, b_reused = false;
    unsigned long long bb_contacts = 0;
    int b_sorted_grid[6] = {0, 0, 0, 0, 0, 0};
    std::vector<float> hb_pos, hb_vel;

    // sorted device state (double buffered for the counting sort)
    int cur = 0, bcur = 0;
    DBuf<float4> pos[2], vel[2], vc[2], bpos[2], bvel[2];
    DBuf<uint32_t> orig[2], borig[2];
    DBuf<uint32_t> gid[2];  // caller-visible particle ids (default: original index); follow particles across ranks
    std::vector<uint32_t> h_gid;
    DBuf<float> press[2];
    DBuf<float4> vs, acc, normals, dbg_acc;
    DBuf<float> dens, alpha, kappa, divv, pred, bvol, bforce;
    DBuf<uint32_t> cid, rank, perm, cstart, bcid, brank, bperm, bstart, scan_aux[3], scan_aux_k[3];
    DBuf<uint32_t> nbr_f, nbr_b, cnt_f, cnt_b;
    // gather_backend 1 (sph_tile.cuh): 16-bit tile-local fluid contact indices
    DBuf<uint16_t> nbr16;
    uint32_t tile_slots = 2048;  // widest tile halo seen by the last neighbour build (local index space size)
    uint32_t n_tiles = 0;
    bool tile = false;
    // gather_backend 0: the second per-contact gather (v* / kappa) can go through the texture pipe
    // uniform-mass packed gather records (sph_passes.cuh): pvx4 = (x,y,z,v*x), vyz2 = (v*y,v*z), pk4 = (x,y,z,kappa); their
    // gathers are split evenly over the texture and LSU pipes (even / odd contacts)
    bool unimass = false;
    DBuf<float4> pvx4, pk4;
    DBuf<float2> vyz2;
    bool nr4_valid = false;  // Akinci normals rode with a divergence evaluation (k_vel_divergence_xsph_u<2>)
    cudaTextureObject_t tex_pvx = 0, tex_vyz = 0, tex_pk = 0;
    const void* tex_pvx_ptr = nullptr;
    const void* tex_vyz_ptr = nullptr;
    const void* tex_pk_ptr = nullptr;
    DBuf<float> he_colors, he_gradc;  // He2014 colours / squared colour-gradient norms (he2014_surface_tension.rs:16-17)
    DBuf<uint32_t> q_out, q_count;     // particles_intersecting_aabb results
    DBuf<float> map_pos, map_vel;      // sph_fluid_map_positions / _velocities: ORIGINAL-order device views
    bool in_coupling = false;          // inside CouplingManager::update_boundaries: the grid holds fluids only (liquid_world.rs:90-103)
    const sph_coupling_manager* coupling = nullptr;
    // ParticlesContacts materialised for host plugins (original order CSR)
    DBuf<uint32_t> ct_cnt[2], ct_j[2], ct_model[2];
    DBuf<float> ct_w[2], ct_g[2];
    DBuf<uint32_t> d_ticket;      // last-block ticket of the in-kernel error reduction (kept at 0 between launches)
    bool errsum_ready = false;    // the last evaluation launch already reduced its partials into errsum
    bool fused_first_div = false;  // the first compute_divergences evaluation rode with the density pass
    bool xs_valid = false;    // the last divergence evaluation of this step produced the XSPH sums (k_vel_divergence_xsph_u)
    DBuf<float4> xs;
    uint32_t fused_nblk = 0;
    cudaTextureObject_t tex_vs = 0, tex_kappa = 0;
    const void* tex_vs_ptr = nullptr;
    const void* tex_kappa_ptr = nullptr;
    DBuf<float> partial, errsum;
    DBuf<int> d_scal;  // [0..6] bounds + bad flag, [7] error flag, [8..9] maxcnt
    DBuf<unsigned long long> d_cnt;  // [0] bb contacts, [1] ff+fb contacts
    DBuf<float> o_a, o_b, o_c, o_mass;  // staging, original order
    DBuf<uint32_t> o_fid;
    IisphState iisph;
    ViscosityState visc;
    float* h_pinned = nullptr;  // 64 floats of pinned host memory for small read-backs

    // fine-grained kernel timers: (slot, begin, end) event pairs accumulated into stats at step end
    struct Span { int slot; cudaEvent_t a, b; };
    std::vector<Span> spans;
    size_t n_spans = 0;

    uint32_t cap_f = 64, cap_b = 32, stride = 0;
    bool lists_valid = false;
    // cell-coordinate AABB of the positions the last step wrote (k_update_positions): sizes the next grid without a bounds pass
    bool nb_valid = false, nb_pending = false;
    int nb[7] = {0, 0, 0, 0, 0, 0, 0};
    DBuf<int> d_nb;
    int xysub = 1;              // row order (Consts::xysub, SALVA_B200_XYSUB): x / y bins per cell; one GPU, gather backend 0 only

    bool grid_ready = false;    // cstart/bstart + sorted arrays describe the last step's cell grid (AABB queries)
    bool ever_stepped = false;
    sph_step_stats stats;
    uint64_t launches = 0;

    sph_status fail(sph_status s, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return s;
    }
};

namespace {

#define CU(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return w->fail(e_ == cudaErrorMemoryAllocation ? SPH_ERR_OOM : SPH_ERR_CUDA, "%s failed: %s (%s:%d)", #call, \
                           cudaGetErrorString(e_), __FILE__, __LINE__);                            \
    } while (0)
#define TRY(call)                          \
    do {                                   \
        sph_status s_ = (call);            \
        if (s_ != SPH_OK) return s_;       \
    } while (0)
#define LAUNCH(kern, n, threads, ...)                                                  \
    do {                                                                               \
        if ((n) > 0) {                                                                 \
            kern<<<cdiv((n), (threads)), (threads), 0, w->st>>>(__VA_ARGS__);           \
            w->launches++;                                                             \
        }                                                                              \
    } while (0)

inline uint32_t make_handle(size_t slot, uint32_t gen) { return (uint32_t)slot | (gen << 16); }
// slot of a live fluid / boundary handle, or -1
inline int fluid_slot(const sph_world* w, uint32_t handle) {
    const uint32_t slot = handle & 0xFFFFu;
    if (slot >= w->fluids.size() || !w->fluids[slot].alive || (w->fluids[slot].gen & 0xFFFFu) != (handle >> 16)) return -1;
    return (int)slot;
}
inline int boundary_slot(const sph_world* w, uint32_t handle) {
    const uint32_t slot = handle & 0xFFFFu;
    if (slot >= w->bounds.size() || !w->bounds[slot].alive || (w->bounds[slot].gen & 0xFFFFu) != (handle >> 16)) return -1;
    return (int)slot;
}
#define FLUID_OR_FAIL(var, handle)                                                                   \
    const int var##_slot_ = fluid_slot(w, handle);                                                   \
    if (var##_slot_ < 0) return w->fail(SPH_ERR_INVALID, "bad fluid handle %u", (unsigned)(handle)); \
    const uint32_t var = (uint32_t)var##_slot_;
#define BOUNDARY_OR_FAIL(var, handle)                                                                   \
    const int var##_slot_ = boundary_slot(w, handle);                                                   \
    if (var##_slot_ < 0) return w->fail(SPH_ERR_INVALID, "bad boundary handle %u", (unsigned)(handle)); \
    const uint32_t var = (uint32_t)var##_slot_;

enum { SP_DIV_EVAL = 0, SP_DIV_UPD, SP_PRED, SP_PUPD, SP_COUNT };
sph_status span_begin(sph_world* w, int slot) {
    if (w->n_spans == w->spans.size()) {
        sph_world::Span s{slot, nullptr, nullptr};
        CU(cudaEventCreate(&s.a));
        CU(cudaEventCreate(&s.b));
        w->spans.push_back(s);
    }
    w->spans[w->n_spans].slot = slot;
    CU(cudaEventRecord(w->spans[w->n_spans].a, w->st));
    return SPH_OK;
}
sph_status span_end(sph_world* w) {
    CU(cudaEventRecord(w->spans[w->n_spans].b, w->st));
    w->n_spans++;
    return SPH_OK;
}

sph_status upload_consts(sph_world* w) {
    CU(cudaMemcpyToSymbolAsync(C, &w->hc, sizeof(Consts), 0, cudaMemcpyHostToDevice, w->st));
    g_const_owner = w;
    return SPH_OK;
}

sph_status enter(sph_world* w) {
    CU(cudaSetDevice(w->desc.device));
    if (g_const_owner != w) TRY(upload_consts(w));
    return SPH_OK;
}

void fill_static_consts(sph_world* w) {
    Consts& c = w->hc;
    c.h = w->h;
    c.inv_h = 1.0f / w->h;
    c.h2 = w->h * w->h;
    c.xysub = (w->tile || w->slab.active) ? 1 : w->xysub;  // slab worlds cut x into cell columns of width h: plain cells there
    c.xysub_f = (float)c.xysub;
    c.h_reach = std::nextafter(w->h * 1.00001f, INFINITY);
    c.sigma = 8.0f / (3.14159265358979323846f * w->h * w->h * w->h);
    c.dsigma = c.sigma / w->h;
    c.dsigma6 = 6.0f * c.dsigma;
    c.kw = w->desc.kernel_density;
    c.kg = w->desc.kernel_gradient;
    c.kgen = (c.kw != 0 || c.kg != 0) ? 1 : 0;
    {
        const float h = w->h, pi = 3.14159265358979323846f;
        auto powi = [](float x, int n) { float r = 1.f; for (int k = 0; k < n; ++k) r *= x; return r; };
        c.poly6_n = (float)(315.0 / 64.0) / (pi * powi(h, 9));
        c.spiky_n = 15.0f / (pi * powi(h, 6));
        c.visc_n = 15.0f / (2.0f * pi * powi(h, 3));
    }
    {
        const double a = (double)F32_EPS * (double)F32_EPS, b = 1.0e-5 * (double)w->h * 1.0e-5 * (double)w->h;
        c.g_t2 = (float)std::max(a, b);
    }
    c.n_fluid = (uint32_t)w->Ntot;
    c.i_begin = w->own_begin;
    c.n_owned = (uint32_t)w->N;
    c.n_bound = (uint32_t)w->B;
    c.n_fluids = (int)w->fluids.size();
    c.n_bounds = (int)w->bounds.size();
    for (size_t f = 0; f < w->fluids.size(); ++f)
        c.fluids[f] = {w->fluids[f].density0, w->fluids[f].memberships, w->fluids[f].filter, w->fluids[f].uniform_mass};
    for (size_t b = 0; b < w->bounds.size(); ++b) c.bounds[b] = {w->bounds[b].memberships, w->bounds[b].filter};
    c.stride = w->stride;
    c.cap_f = w->cap_f;
    c.cap_b = w->cap_b;
}

// ---- exclusive scan over n u32 (in place) -------------------------------------------------------
sph_status scan_exclusive(sph_world* w, uint32_t* data, size_t n, int level = 0) {
    if (n == 0) return SPH_OK;
    uint32_t nb = cdiv(n, SCAN_B);
    if (nb == 1) {
        k_scan_block<<<1, SCAN_T, 0, w->st>>>(data, data, (uint32_t)n, nullptr);
        w->launches++;
        return SPH_OK;
    }
    if (level >= 3) return w->fail(SPH_ERR_INVALID, "scan too deep");
    CU(w->scan_aux[level].ensure(nb));
    k_scan_block<<<nb, SCAN_T, 0, w->st>>>(data, data, (uint32_t)n, w->scan_aux[level].p);
    w->launches++;
    TRY(scan_exclusive(w, w->scan_aux[level].p, nb, level + 1));
    k_scan_add<<<nb, SCAN_T, 0, w->st>>>(data, (uint32_t)n, w->scan_aux[level].p);
    w->launches++;
    return SPH_OK;
}

// K arrays of the same length scanned together (in place, exclusive); n <= 2048 * 2048 * 2048
template <int K>
sph_status scan_exclusive_k(sph_world* w, ScanSet<K> arrays, size_t n, int level = 0) {
    if (n == 0) return SPH_OK;
    uint32_t nb = cdiv(n, SCAN_B);
    ScanSet<K> sums;
    for (int a = 0; a < K; ++a) sums.a[a] = nullptr;
    if (nb == 1) {
        k_scanK_block<K><<<1, SCAN_T, 0, w->st>>>(arrays, (uint32_t)n, sums);
        w->launches++;
        return SPH_OK;
    }
    if (level >= 3) return w->fail(SPH_ERR_INVALID, "scan too deep");
    CU(w->scan_aux_k[level].ensure((size_t)K * nb));
    for (int a = 0; a < K; ++a) sums.a[a] = w->scan_aux_k[level].p + (size_t)a * nb;
    k_scanK_block<K><<<nb, SCAN_T, 0, w->st>>>(arrays, (uint32_t)n, sums);
    w->launches++;
    TRY(scan_exclusive_k<K>(w, sums, nb, level + 1));
    k_scanK_add<K><<<nb, SCAN_T, 0, w->st>>>(arrays, (uint32_t)n, sums);
    w->launches++;
    return SPH_OK;
}

// ---- host <-> device staging --------------------------------------------------------------------
// Device holds the truth -> pull everything back into the host vectors (original order).
sph_status stage_down(sph_world* w) {
    if (w->staged) return SPH_OK;
    size_t N = w->N;
    w->h_pos.resize(3 * N);
    w->h_vel.resize(3 * N);
    w->h_vc.resize(3 * N);
    w->h_press.assign(N, 0.f);
    w->h_gid.resize(N);
    if (N) {
        int c = w->cur;
        uint32_t ob = w->own_begin;
        CU(w->o_a.ensure(3 * N));
        const float4* srcs[3] = {w->pos[c].p, w->vel[c].p, w->vc[c].p};
        float* dsts[3] = {w->h_pos.data(), w->h_vel.data(), w->h_vc.data()};
        for (int a = 0; a < 3; ++a) {
            LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + ob, srcs[a] + ob, w->o_a.p);
            CU(cudaMemcpyAsync(dsts[a], w->o_a.p, 3 * N * sizeof(float), cudaMemcpyDeviceToHost, w->st));
            CU(cudaStreamSynchronize(w->st));
        }
        LAUNCH(k_export_u32, N, 256, (uint32_t)N, w->orig[c].p + ob, w->gid[c].p + ob, reinterpret_cast<uint32_t*>(w->o_a.p));
        CU(cudaMemcpyAsync(w->h_gid.data(), w->o_a.p, N * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
        CU(cudaStreamSynchronize(w->st));
        if (w->desc.solver == SPH_SOLVER_IISPH && w->press[c].p) {
            LAUNCH(k_export1, N, 256, (uint32_t)N, w->orig[c].p + ob, w->press[c].p + ob, w->o_a.p);
            CU(cudaMemcpyAsync(w->h_press.data(), w->o_a.p, N * sizeof(float), cudaMemcpyDeviceToHost, w->st));
            CU(cudaStreamSynchronize(w->st));
        }
    }
    w->staged = true;
    w->lists_valid = false;
    w->grid_ready = false;
    w->nb_valid = false;
    return SPH_OK;
}

void recompute_offsets(sph_world* w) {
    size_t o = 0;
    for (auto& f : w->fluids) {
        f.offset = o;
        o += f.n;
    }
    w->N = o;
    o = 0;
    for (auto& b : w->bounds) {
        b.offset = o;
        o += b.n;
    }
    w->B = o;
}

sph_status ensure_fluid_buffers(sph_world* w) {
    size_t N = std::max(w->Ntot, w->N);
    for (int k = 0; k < 2; ++k) {
        if (k == w->protect_buf) continue;
        bool keep = k == w->cur;  // the live buffers may be grown while they hold particles (ghost append)
        CU(w->pos[k].ensure(N, keep, w->st));
        CU(w->vel[k].ensure(N, keep, w->st));
        CU(w->vc[k].ensure(N, keep, w->st));
        CU(w->orig[k].ensure(N, keep, w->st));
        CU(w->gid[k].ensure(N, keep, w->st));
        if (w->desc.solver == SPH_SOLVER_IISPH) CU(w->press[k].ensure(N, keep, w->st));
    }
    CU(w->vs.ensure(N));
    CU(w->pvx4.ensure(N));
    CU(w->pk4.ensure(N));
    CU(w->vyz2.ensure(N));
    CU(w->acc.ensure(N));
    CU(w->dens.ensure(N + 8));
    CU(w->alpha.ensure(N + 8));
    CU(w->kappa.ensure(N + 8));
    CU(w->divv.ensure(N + 8));
    CU(w->pred.ensure(N + 8));
    CU(w->cid.ensure(N));
    CU(w->rank.ensure(N));
    CU(w->perm.ensure(N));
    CU(w->cnt_f.ensure(N));
    CU(w->cnt_b.ensure(N));
    w->stride = (uint32_t)((N + 31) / 32 * 32);
    if (w->tile) CU(w->nbr16.ensure((size_t)w->cap_f * w->stride));
    else CU(w->nbr_f.ensure((size_t)w->cap_f * w->stride));
    CU(w->nbr_b.ensure((size_t)w->cap_b * w->stride));
    uint32_t nblk = cdiv(std::max<size_t>(N, 1), PASS_T);
    CU(w->partial.ensure((size_t)nblk * std::max<size_t>(1, w->fluids.size())));
    CU(w->errsum.ensure(MAX_FLUIDS));
    return SPH_OK;
}

// Host vectors hold the truth -> build the device state (sorted order starts as the identity).
sph_status stage_up(sph_world* w) {
    if (!w->staged) return SPH_OK;
    recompute_offsets(w);
    size_t N = w->N;
    w->Ntot = N;
    w->own_begin = 0;
    TRY(ensure_fluid_buffers(w));
    w->h_gid.resize(N);
    if (N) {
        std::vector<float> mass(N);
        std::vector<uint32_t> fid(N);
        for (size_t f = 0; f < w->fluids.size(); ++f) {
            bool uniform = w->fluids[f].n > 0;
            for (size_t i = 0; i < w->fluids[f].n; ++i) {
                size_t g = w->fluids[f].offset + i;
                mass[g] = w->h_vol[g] * w->fluids[f].density0;  // fluid.rs:183-185
                fid[g] = (uint32_t)f;
                uniform = uniform && w->h_vol[g] == w->h_vol[w->fluids[f].offset];
            }
            w->fluids[f].uniform_mass = uniform ? mass[w->fluids[f].offset] : 0.f;
        }
        CU(w->o_a.ensure(3 * N));
        CU(w->o_b.ensure(3 * N));
        CU(w->o_c.ensure(3 * N));
        CU(w->o_mass.ensure(N));
        CU(w->o_fid.ensure(N));
        CU(cudaMemcpyAsync(w->o_a.p, w->h_pos.data(), 3 * N * sizeof(float), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemcpyAsync(w->o_b.p, w->h_vel.data(), 3 * N * sizeof(float), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemcpyAsync(w->o_c.p, w->h_vc.data(), 3 * N * sizeof(float), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemcpyAsync(w->o_mass.p, mass.data(), N * sizeof(float), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemcpyAsync(w->o_fid.p, fid.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice, w->st));
        int c = w->cur;
        LAUNCH(k_iota, N, 256, (uint32_t)N, w->orig[c].p);
        CU(cudaMemcpyAsync(w->gid[c].p, w->h_gid.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemsetAsync(w->pos[c].p, 0, N * sizeof(float4), w->st));
        CU(cudaMemsetAsync(w->vel[c].p, 0, N * sizeof(float4), w->st));
        LAUNCH(k_import, N, 256, (uint32_t)N, w->orig[c].p, w->o_a.p, w->o_b.p, w->o_c.p, w->o_mass.p, w->o_fid.p, w->pos[c].p, w->vel[c].p,
               w->vc[c].p, 0u, (uint32_t)N);
        if (w->desc.solver == SPH_SOLVER_IISPH) {
            w->h_press.resize(N, 0.f);
            CU(cudaMemcpyAsync(w->press[c].p, w->h_press.data(), N * sizeof(float), cudaMemcpyHostToDevice, w->st));
        }
        CU(cudaStreamSynchronize(w->st));  // host temporaries go out of scope
    }
    w->staged = false;
    w->lists_valid = false;
    w->slab.global_valid = false;
    // a slab world takes the fast path on every rank or on none: volumes default to uniform there, and an empty
    // slab inherits the constant from its first immigrant only through the classic path -> keep it simple: require
    // particles with uniform volumes on this rank, otherwise fall back (all ranks are built by the same host code).
    w->unimass = !w->tile && w->desc.solver == SPH_SOLVER_DFSPH && w->fluids.size() == 1 && w->fluids[0].uniform_mass > 0.f;
    return SPH_OK;
}

sph_status upload_boundaries(sph_world* w) {
    if (!w->b_dirty) return SPH_OK;
    recompute_offsets(w);
    size_t B = w->B;
    for (int k = 0; k < 2; ++k) {
        CU(w->bpos[k].ensure(B));
        CU(w->bvel[k].ensure(B));
        CU(w->borig[k].ensure(B));
    }
    CU(w->bvol.ensure(B));
    CU(w->bcid.ensure(B));
    CU(w->brank.ensure(B));
    CU(w->bperm.ensure(B));
    CU(w->bforce.ensure(3 * B));
    if (B) {
        std::vector<float4> p(B), v(B);
        int aabb[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
        bool bad = false;
        for (size_t g = 0; g < B; ++g)
            for (int a = 0; a < 3; ++a) {
                float cf = floorf(w->hb_pos[3 * g + a] / w->h);  // hgrid.rs:41-43, same IEEE division as the device
                if (!(fabsf(cf) < 1.0e9f)) { bad = true; continue; }
                aabb[a] = std::min(aabb[a], (int)cf);
                aabb[3 + a] = std::max(aabb[3 + a], (int)cf);
            }
        memcpy(w->b_aabb, aabb, sizeof aabb);
        w->b_bad = bad;
        for (size_t b = 0; b < w->bounds.size(); ++b)
            for (size_t i = 0; i < w->bounds[b].n; ++i) {
                size_t g = w->bounds[b].offset + i;
                p[g] = make_float4(w->hb_pos[3 * g], w->hb_pos[3 * g + 1], w->hb_pos[3 * g + 2], 0.f);
                v[g] = make_float4(w->hb_vel[3 * g], w->hb_vel[3 * g + 1], w->hb_vel[3 * g + 2], __uint_as_float_host((uint32_t)b));
            }
        int c = w->bcur;
        CU(cudaMemcpyAsync(w->bpos[c].p, p.data(), B * sizeof(float4), cudaMemcpyHostToDevice, w->st));
        CU(cudaMemcpyAsync(w->bvel[c].p, v.data(), B * sizeof(float4), cudaMemcpyHostToDevice, w->st));
        LAUNCH(k_iota, B, 256, (uint32_t)B, w->borig[c].p);
        CU(cudaStreamSynchronize(w->st));
    }
    if (!B) {
        int none[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
        memcpy(w->b_aabb, none, sizeof none);
        w->b_bad = false;
    }
    w->b_dirty = false;
    w->b_sorted_valid = false;
    w->lists_valid = false;
    return SPH_OK;
}

// fluid.rs:88-98 apply_particles_removal (+ solver scratch filtering dfsph_solver.rs:550-559)
sph_status apply_pending_deletes(sph_world* w) {
    bool any = false;
    for (auto& f : w->fluids) any |= f.n_pending != 0;
    if (!any) return SPH_OK;
    TRY(stage_down(w));
    std::vector<float> np, nv, nc, nvol, npr;
    std::vector<uint32_t> ngid;
    np.reserve(w->h_pos.size());
    nv.reserve(w->h_pos.size());
    nc.reserve(w->h_pos.size());
    for (auto& f : w->fluids) {
        size_t kept = 0;
        for (size_t i = 0; i < f.n; ++i) {
            if (f.n_pending && f.pending_delete[i]) continue;
            size_t g = f.offset + i;
            for (int a = 0; a < 3; ++a) {
                np.push_back(w->h_pos[3 * g + a]);
                nv.push_back(w->h_vel[3 * g + a]);
                nc.push_back(w->h_vc[3 * g + a]);
            }
            nvol.push_back(w->h_vol[g]);
            ngid.push_back(g < w->h_gid.size() ? w->h_gid[g] : (uint32_t)g);
            npr.push_back(g < w->h_press.size() ? w->h_press[g] : 0.f);
            ++kept;
        }
        f.n = kept;
        f.pending_delete.assign(kept, 0);
        f.n_pending = 0;
    }
    w->h_pos.swap(np);
    w->h_vel.swap(nv);
    w->h_vc.swap(nc);
    w->h_vol.swap(nvol);
    w->h_press.swap(npr);
    w->h_gid.swap(ngid);
    recompute_offsets(w);
    return SPH_OK;
}

// ---- step phases ----------------------------------------------------------------------------------
sph_status phase_grid(sph_world* w) {
    size_t N = w->Ntot, B = w->B;  // the sort covers owned + ghost slots
    int c = w->cur, bc = w->bcur;
    // slab worlds: the prologue appended immigrants / ghosts behind the owned range of the live arrays and flagged the
    // particles that left; the sort reads [off, off + Nin) and drops the flagged slots.  Elsewhere: all N slots from 0.
    const uint32_t off = w->slab.active ? w->slab.sort_off : 0u;
    const size_t Nin = w->slab.active ? w->slab.sort_n : N;
    const uint32_t* dead = w->slab.active ? w->slab.flag.p : nullptr;
    const uint32_t n_dead = w->slab.active ? w->slab.sort_dead_n : 0u;
    int init[11] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, 0, 0, 0, 0, 0};
    CU(cudaMemcpyAsync(w->d_scal.p, init, sizeof init, cudaMemcpyHostToDevice, w->st));
    CU(cudaMemsetAsync(w->d_cnt.p, 0, 2 * sizeof(unsigned long long), w->st));
    int hb[7];
    if (w->nb_valid && !w->slab.active && N) {
        // positions are exactly what the last step's k_update_positions wrote (no host edit since): its bounds came back with
        // that step's final read-back, so this step starts without a bounds pass and without a host round trip
        memcpy(hb, w->nb, sizeof hb);
    } else {
        if (Nin) {
            k_bounds<<<std::min<uint32_t>(cdiv(Nin, 256), 296), 256, 0, w->st>>>(w->pos[c].p + off, (uint32_t)Nin, w->d_scal.p);
            w->launches++;
        }
        CU(cudaMemcpyAsync(hb, w->d_scal.p, sizeof hb, cudaMemcpyDeviceToHost, w->st));
        CU(cudaStreamSynchronize(w->st));
    }
    w->nb_valid = false;
    if (hb[6] || w->b_bad) return w->fail(SPH_ERR_INVALID, "non-finite or out-of-range particle coordinates");
    for (int a = 0; a < 3; ++a) {  // boundary AABB: static, kept on the host
        hb[a] = std::min(hb[a], w->b_aabb[a]);
        hb[3 + a] = std::max(hb[3 + a], w->b_aabb[3 + a]);
    }
    long long dims[3];
    for (int a = 0; a < 3; ++a) dims[a] = (long long)hb[3 + a] - hb[a] + 3;  // one padding cell each side
    double ncell_d = (double)dims[0] * (double)dims[1] * (double)dims[2];
    if (ncell_d > 1.0e9) return w->fail(SPH_ERR_OOM, "dense cell grid too large: %lld x %lld x %lld cells of width h", dims[0], dims[1], dims[2]);
    const int xys = (w->tile || w->slab.active) ? 1 : w->xysub;  // x / y bins per cell (row order, Consts::xysub)
    if (ncell_d * xys * xys > 2.0e9) return w->fail(SPH_ERR_OOM, "dense cell grid too large: %lld x %lld x %lld cells of width h", dims[0], dims[1], dims[2]);
    size_t ncell = (size_t)dims[0] * dims[1] * dims[2] * xys * xys;
    w->hc.ox = (hb[0] - 1) * xys;
    w->hc.oy = (hb[1] - 1) * xys;
    w->hc.oz = hb[2] - 1;
    w->hc.nx = (int)dims[0] * xys;
    w->hc.ny = (int)dims[1] * xys;
    w->hc.nz = (int)dims[2];
    w->hc.ntx = (int)((dims[0] - 2 + TILE_X - 1) / TILE_X);
    w->hc.nty = (int)((dims[1] - 2 + TILE_Y - 1) / TILE_Y);
    w->hc.ntz = (int)((dims[2] - 2 + TILE_Z - 1) / TILE_Z);
    w->n_tiles = (uint32_t)w->hc.ntx * w->hc.nty * w->hc.ntz;
    fill_static_consts(w);
    TRY(upload_consts(w));
    CU(w->cstart.ensure(ncell + 1));
    CU(w->bstart.ensure(ncell + 1));
    if (w->tile) CU(w->partial.ensure((size_t)std::max<uint32_t>(w->n_tiles, 1) * std::max<size_t>(1, w->fluids.size())));
    w->stats.grid_dims[0] = (uint32_t)dims[0];
    w->stats.grid_dims[1] = (uint32_t)dims[1];
    w->stats.grid_dims[2] = (uint32_t)dims[2];
    // fluid: counting sort by cell, then reorder every persistent array
    CU(cudaMemsetAsync(w->cstart.p, 0, (ncell + 1) * sizeof(uint32_t), w->st));
    if (xys > 1) LAUNCH(k_cell_hist_xy, Nin, 256, w->pos[c].p + off, (uint32_t)Nin, w->cid.p, w->rank.p, w->cstart.p);  // (never a slab world: no dead slots)
    else LAUNCH(k_cell_hist, Nin, 256, w->pos[c].p + off, (uint32_t)Nin, w->cid.p, w->rank.p, w->cstart.p, dead, n_dead);
    TRY(scan_exclusive(w, w->cstart.p, ncell + 1));
    LAUNCH(k_cell_scatter, Nin, 256, (uint32_t)Nin, w->cid.p, w->rank.p, w->cstart.p, w->perm.p);
    if (w->desc.deterministic)
        LAUNCH(k_cell_sort, ncell, 256, (uint32_t)ncell, w->cstart.p, w->perm.p, (const uint32_t*)w->gid[c].p + off,
               w->fluids.size() > 1 ? (const float4*)w->vel[c].p + off : (const float4*)nullptr);
    if (N) {
        GatherSet g;
        memset(&g, 0, sizeof g);
        g.in4[0] = w->pos[c].p + off; g.out4[0] = w->pos[c ^ 1].p;
        g.in4[1] = w->vel[c].p + off; g.out4[1] = w->vel[c ^ 1].p;
        g.in4[2] = w->vc[c].p + off;  g.out4[2] = w->vc[c ^ 1].p;
        g.n4 = 3;
        g.in1[0] = w->orig[c].p + off; g.out1[0] = w->orig[c ^ 1].p;  // (slab worlds overwrite orig with the identity after the sort)
        g.in1[1] = w->gid[c].p + off; g.out1[1] = w->gid[c ^ 1].p;
        g.n1 = 2;
        if (w->desc.solver == SPH_SOLVER_IISPH) {
            g.in1[2] = reinterpret_cast<const uint32_t*>(w->press[c].p);
            g.out1[2] = reinterpret_cast<uint32_t*>(w->press[c ^ 1].p);
            g.n1 = 3;
        }
        // reorder + v* = vel + vc (the divergence solve works on vel + vc carried over from the previous step, Appendix A.3.2) in one pass
        LAUNCH(k_gather_vstar, N, 256, (uint32_t)N, w->perm.p, g, w->vs.p, w->unimass ? w->pvx4.p : nullptr, w->unimass ? w->vyz2.p : nullptr);
        w->cur = c ^ 1;
    }
    // boundaries: same sort — reused while neither the boundaries nor the cell mapping changed (static tanks)
    const int gridkey[6] = {w->hc.ox, w->hc.oy, w->hc.oz, w->hc.nx, w->hc.ny, w->hc.nz};
    const bool reuse_b = w->b_sorted_valid && memcmp(gridkey, w->b_sorted_grid, sizeof gridkey) == 0;
    w->b_reused = reuse_b;
    if (!reuse_b) CU(cudaMemsetAsync(w->bstart.p, 0, (ncell + 1) * sizeof(uint32_t), w->st));
    if (B && !reuse_b) {
        if (xys > 1) LAUNCH(k_cell_hist_xy, B, 256, w->bpos[bc].p, (uint32_t)B, w->bcid.p, w->brank.p, w->bstart.p);
        else LAUNCH(k_cell_hist, B, 256, w->bpos[bc].p, (uint32_t)B, w->bcid.p, w->brank.p, w->bstart.p, (const uint32_t*)nullptr, 0u);
        TRY(scan_exclusive(w, w->bstart.p, ncell + 1));
        LAUNCH(k_cell_scatter, B, 256, (uint32_t)B, w->bcid.p, w->brank.p, w->bstart.p, w->bperm.p);
        if (w->desc.deterministic) LAUNCH(k_cell_sort, ncell, 256, (uint32_t)ncell, w->bstart.p, w->bperm.p, (const uint32_t*)nullptr, (const float4*)nullptr);
        GatherSet g;
        memset(&g, 0, sizeof g);
        g.in4[0] = w->bpos[bc].p; g.out4[0] = w->bpos[bc ^ 1].p;
        g.in4[1] = w->bvel[bc].p; g.out4[1] = w->bvel[bc ^ 1].p;
        g.n4 = 2;
        g.in1[0] = w->borig[bc].p; g.out1[0] = w->borig[bc ^ 1].p;
        g.n1 = 1;
        LAUNCH(k_gather, B, 256, (uint32_t)B, w->bperm.p, g);
        w->bcur = bc ^ 1;
    }
    if (!reuse_b) {
        memcpy(w->b_sorted_grid, gridkey, sizeof gridkey);
        w->b_sorted_valid = true;
    }
    CU(cudaGetLastError());
    if (w->slab.active) {
        TRY(slab_after_sort(w));
        fill_static_consts(w);
        TRY(upload_consts(w));
    }
    return SPH_OK;
}

// ---- tile kernel launches (gather_backend 1, sph_tile.cuh) -------------------------------------------
constexpr size_t TILE_DYN_SMEM_LIMIT = 200 * 1024;
// Number of halo slots staged in shared memory for a kernel that needs `slot_bytes` per slot.
uint32_t tile_cap(const sph_world* w, uint32_t slot_bytes) {
    uint32_t want = (w->tile_slots + 63u) / 64u * 64u;
    uint32_t fit = (uint32_t)(TILE_DYN_SMEM_LIMIT / slot_bytes) / 64u * 64u;
    return std::min(want, fit);
}
template <class K>
cudaError_t tile_prepare(K kern) {
    static std::mutex m;
    static std::vector<const void*> done;
    std::lock_guard<std::mutex> lock(m);
    const void* key = reinterpret_cast<const void*>(kern);
    for (const void* d : done)
        if (d == key) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TILE_DYN_SMEM_LIMIT);
    if (e == cudaSuccess) done.push_back(key);
    return e;
}
#define LAUNCH_TILE(kern, slot_bytes, cap, ...)                                                      \
    do {                                                                                             \
        if (w->n_tiles > 0) {                                                                        \
            CU(tile_prepare(kern));                                                                  \
            kern<<<w->n_tiles, TILE_T, (size_t)(cap) * (slot_bytes), w->st>>>(__VA_ARGS__);          \
            w->launches++;                                                                           \
        }                                                                                            \
    } while (0)
#define TDISPATCH1(kern, multi, slot_bytes, cap, ...)                               \
    do {                                                                            \
        if (multi) LAUNCH_TILE((kern<true>), slot_bytes, cap, __VA_ARGS__);         \
        else LAUNCH_TILE((kern<false>), slot_bytes, cap, __VA_ARGS__);              \
    } while (0)
#define TDISPATCH2(kern, multi, bf, slot_bytes, cap, ...)                                  \
    do {                                                                                   \
        if (multi) {                                                                       \
            if (bf) LAUNCH_TILE((kern<true, true>), slot_bytes, cap, __VA_ARGS__);         \
            else LAUNCH_TILE((kern<true, false>), slot_bytes, cap, __VA_ARGS__);           \
        } else {                                                                           \
            if (bf) LAUNCH_TILE((kern<false, true>), slot_bytes, cap, __VA_ARGS__);        \
            else LAUNCH_TILE((kern<false, false>), slot_bytes, cap, __VA_ARGS__);          \
        }                                                                                  \
    } while (0)
#define TDISPATCH3(kern, multi, bf, third, slot_bytes, cap, ...)                                          \
    do {                                                                                                  \
        if (multi) {                                                                                      \
            if (bf) LAUNCH_TILE((kern<true, true, third>), slot_bytes, cap, __VA_ARGS__);                 \
            else LAUNCH_TILE((kern<true, false, third>), slot_bytes, cap, __VA_ARGS__);                   \
        } else {                                                                                          \
            if (bf) LAUNCH_TILE((kern<false, true, third>), slot_bytes, cap, __VA_ARGS__);                \
            else LAUNCH_TILE((kern<false, false, third>), slot_bytes, cap, __VA_ARGS__);                  \
        }                                                                                                 \
    } while (0)

template <class T>
sph_status ensure_tex(sph_world* w, cudaTextureObject_t* tex, const void** cur, const T* ptr, size_t n) {
    if (*cur == ptr && *tex) return SPH_OK;
    if (*tex) cudaDestroyTextureObject(*tex);
    *tex = 0;
    cudaResourceDesc rd;
    memset(&rd, 0, sizeof rd);
    rd.resType = cudaResourceTypeLinear;
    rd.res.linear.devPtr = const_cast<T*>(ptr);
    rd.res.linear.desc = cudaCreateChannelDesc<T>();
    rd.res.linear.sizeInBytes = n * sizeof(T);
    cudaTextureDesc td;
    memset(&td, 0, sizeof td);
    td.readMode = cudaReadModeElementType;
    CU(cudaCreateTextureObject(tex, &rd, &td, nullptr));
    *cur = ptr;
    return SPH_OK;
}

// `speculative` (optional) enqueues the work that follows the neighbour search and only writes scratch (the density
// pass): it is launched BEFORE the host learns whether the lists overflowed, so the GPU is busy during that round trip;
// on overflow the lists are rebuilt with a larger capacity and the speculative work is simply enqueued again.
sph_status phase_neighbors(sph_world* w, sph_status (*speculative)(sph_world*) = nullptr) {
    size_t N = w->N, B = w->B;
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1;
    if (B) {  // compute_boundary_volumes dfsph_solver.rs:72-96: the reference recomputes them every substep; they only
              // depend on the boundary positions, so they are reused while the boundaries are unchanged
        if (!w->b_reused) {
            if (w->hc.xysub > 1) LAUNCH(k_boundary_volumes_xy, B, 128, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->bvol.p, w->d_cnt.p, w->d_scal.p + 7);
            else LAUNCH(k_boundary_volumes, B, 128, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->bvol.p, w->d_cnt.p, w->d_scal.p + 7);
            LAUNCH(k_set_w, B, 256, (uint32_t)B, w->bpos[bc].p, w->bvol.p);
        }
        for (auto& b : w->bounds)
            if (b.want_forces) {
                CU(cudaMemsetAsync(w->bforce.p, 0, 3 * B * sizeof(float), w->st));
                break;
            }
    }
    for (int attempt = 0; attempt < 8 && N; ++attempt) {
        CU(cudaMemsetAsync(w->d_scal.p + 8, 0, 3 * sizeof(int), w->st));
        uint32_t* maxcnt = reinterpret_cast<uint32_t*>(w->d_scal.p + 8);
        if (w->tile) {
            LAUNCH(k_neighbors_boundary, N, 128, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->nbr_b.p, w->cnt_b.p, maxcnt);
            uint32_t sb = multi ? 32u : 16u;
            uint32_t cap = tile_cap(w, sb);
            TDISPATCH1(k_tile_neighbors, multi, sb, cap, w->pos[c].p, w->vel[c].p, w->cstart.p, cap, w->nbr16.p, w->cnt_f.p, maxcnt);
        } else if (w->hc.xysub > 1) {  // row order
            if (multi)
                LAUNCH((k_neighbors_xy<true>), N, 128, w->pos[c].p, w->vel[c].p, w->cstart.p, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->nbr_f.p, w->nbr_b.p,
                       w->cnt_f.p, w->cnt_b.p, maxcnt);
            else
                LAUNCH((k_neighbors_xy<false>), N, 128, w->pos[c].p, w->vel[c].p, w->cstart.p, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->nbr_f.p, w->nbr_b.p,
                       w->cnt_f.p, w->cnt_b.p, maxcnt);
        } else if (multi) {
            LAUNCH((k_neighbors<true>), N, 128, w->pos[c].p, w->vel[c].p, w->cstart.p, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->nbr_f.p, w->nbr_b.p,
                   w->cnt_f.p, w->cnt_b.p, maxcnt);
        } else {
            LAUNCH((k_neighbors<false>), N, 128, w->pos[c].p, w->vel[c].p, w->cstart.p, w->bpos[bc].p, w->bvel[bc].p, w->bstart.p, w->nbr_f.p, w->nbr_b.p,
                   w->cnt_f.p, w->cnt_b.p, maxcnt);
        }
        int* hs = reinterpret_cast<int*>(w->h_pinned + 32);  // pinned: the copy is truly asynchronous
        CU(cudaMemcpyAsync(hs, w->d_scal.p + 7, 4 * sizeof(int), cudaMemcpyDeviceToHost, w->st));
        CU(cudaEventRecord(w->ev_lists, w->st));
        CU(cudaEventRecord(w->ev[EV_NBR], w->st));
        const bool early = speculative && !w->tile;  // (tile launches need this read-back's slot count)
        if (early) TRY(speculative(w));
        CU(cudaEventSynchronize(w->ev_lists));
        if (hs[0]) return w->fail(SPH_ERR_ZERO_DENSITY, "zero boundary-volume denominator (reference assert dfsph_solver.rs:92)");
        if (w->tile) {
            if ((uint32_t)hs[3] > 65535u)
                return w->fail(SPH_ERR_INVALID, "tile halo of %d particles exceeds the 16-bit contact index space", hs[3]);
            w->tile_slots = std::max<uint32_t>((uint32_t)hs[3], 64u);
        }
        w->stats.max_neighbors = (uint32_t)hs[1];
        bool grow = false;
        if ((uint32_t)hs[1] > w->cap_f) {
            w->cap_f = ((uint32_t)hs[1] + 15) / 16 * 16;
            grow = true;
        }
        if ((uint32_t)hs[2] > w->cap_b) {
            w->cap_b = ((uint32_t)hs[2] + 15) / 16 * 16;
            grow = true;
        }
        if (!grow) {
            if (speculative && !early) TRY(speculative(w));
            break;
        }
        if (early) CU(cudaMemsetAsync(w->d_scal.p + 7, 0, sizeof(int), w->st));  // error flag of the discarded speculative pass
        if (w->tile) CU(w->nbr16.ensure((size_t)w->cap_f * w->stride));
        else CU(w->nbr_f.ensure((size_t)w->cap_f * w->stride));
        CU(w->nbr_b.ensure((size_t)w->cap_b * w->stride));
        fill_static_consts(w);
        TRY(upload_consts(w));
    }
    if (!N) {  // boundaries only
        CU(cudaEventRecord(w->ev[EV_NBR], w->st));
        if (speculative) TRY(speculative(w));
    }
    if (N) {
        k_sum_u32<<<std::min<uint32_t>(cdiv(N, 256), 1184), 256, 0, w->st>>>((uint32_t)N, w->cnt_f.p + w->own_begin, w->cnt_b.p + w->own_begin,
                                                                             w->d_cnt.p + 1);
        w->launches++;
    }
    CU(cudaGetLastError());
    w->lists_valid = true;
    if (speculative) TRY(post_density_refresh(w));
    return SPH_OK;
}

// mean-per-fluid -> max over fluids (dfsph_solver.rs:153-158, :347-352)
sph_status read_error(sph_world* w, uint32_t nblk, float* out) {
    int nf = (int)w->fluids.size();
    if (!w->errsum_ready) {
        k_reduce_partials<<<nf, 256, 0, w->st>>>(w->partial.p, nblk, nf, w->errsum.p);
        w->launches++;
    }
    w->errsum_ready = false;
    TRY(slab_allreduce(w, w->errsum.p, nf));  // multi-GPU: the means are over ALL ranks' particles
    CU(cudaMemcpyAsync(w->h_pinned, w->errsum.p, nf * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    float mx = 0.f;
    for (int f = 0; f < nf; ++f) {
        double n = w->slab.active ? (double)w->slab.global_n : (double)w->fluids[f].n;
        if (n > 0) mx = std::max(mx, w->h_pinned[f] / (float)n);
    }
    *out = mx;
    return SPH_OK;
}

bool any_bforce(const sph_world* w) {
    for (auto& b : w->bounds)
        if (b.want_forces) return true;
    return false;
}

#define DISPATCH2(kern, multi, bf, n, threads, ...)                                   \
    do {                                                                              \
        if (multi) {                                                                  \
            if (bf) LAUNCH((kern<true, true>), n, threads, __VA_ARGS__);              \
            else LAUNCH((kern<true, false>), n, threads, __VA_ARGS__);                \
        } else {                                                                      \
            if (bf) LAUNCH((kern<false, true>), n, threads, __VA_ARGS__);             \
            else LAUNCH((kern<false, false>), n, threads, __VA_ARGS__);               \
        }                                                                             \
    } while (0)
#define DISPATCH1(kern, multi, n, threads, ...)                         \
    do {                                                                \
        if (multi) LAUNCH((kern<true>), n, threads, __VA_ARGS__);       \
        else LAUNCH((kern<false>), n, threads, __VA_ARGS__);            \
    } while (0)

// ---- gather passes: one wrapper per reference function, two backends ------------------------------------

// ghost refresh of v* in whichever representation the evaluations gather (one NCCL group); vs itself is included
// because the velocity fold reads vel = v* for ghosts too
sph_status refresh_vstar(sph_world* w) {
    if (!w->slab.active) return SPH_OK;
    if (w->unimass) {
        SlabArray a[3] = {{w->pvx4.p, sizeof(float4)}, {w->vyz2.p, sizeof(float2)}, {w->vs.p, sizeof(float4)}};
        return slab_refresh_n(w, a, 3);
    }
    return slab_refresh(w, w->vs.p, sizeof(float4));
}
// ghost refresh of the evaluation's output (kappa) — only needed when an update follows
sph_status refresh_kappa(sph_world* w) {
    if (!w->slab.active) return SPH_OK;
    if (w->unimass) return slab_refresh(w, w->pk4.p, sizeof(float4));
    return slab_refresh(w, w->kappa.p, sizeof(float));
}

sph_status launch_density_alpha(sph_world* w) {
    size_t N = w->N;
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1;
    if (w->tile) {
        TileLists L{w->nbr16.p, w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
        uint32_t cap = tile_cap(w, 16);
        TDISPATCH1(k_tile_density_alpha, multi, 16, cap, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->cstart.p, cap, L, w->dens.p, w->alpha.p,
                   w->d_scal.p + 7);
    } else {
        Lists L{reinterpret_cast<const uint4*>(w->nbr_f.p), w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
        DISPATCH1(k_density_alpha, multi, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, L, w->dens.p, w->alpha.p, w->d_scal.p + 7);
    }
    return SPH_OK;  // the ghost refresh of rho follows in post_density_refresh(), once the list-capacity check has passed
}
// Ghost refresh of what the density pass produced (rho; DFSPH: also kappa of the fused first divergence evaluation).  Kept out
// of the density launch itself so that the launch stays purely local: it is enqueued SPECULATIVELY behind the neighbour
// search (before the host knows whether the lists overflowed), and a rank that has to regrow its lists and repeat it must not
// leave its neighbours waiting in a collective they entered once and it enters twice.
sph_status post_density_refresh(sph_world* w) {
    if (!w->slab.active || !w->N) return SPH_OK;
    if (w->fused_first_div) {
        SlabArray a[2] = {{w->dens.p, sizeof(float)}, {w->unimass ? (void*)w->pk4.p : (void*)w->kappa.p, w->unimass ? sizeof(float4) : sizeof(float)}};
        return slab_refresh_n(w, a, 2);
    }
    return slab_refresh(w, w->dens.p, sizeof(float));  // XSPH / artificial viscosity / Akinci gather rho_j of ghosts
}
// DFSPH: densities + alphas + the first divergence evaluation in one sweep (k_density_alpha_div)
// Launch over a slot range with n = range count (kernels index rg.begin + thread)
#define LAUNCH_R(kern, rg, ...)                                                                   \
    do {                                                                                          \
        if ((rg).count > 0) {                                                                     \
            kern<<<cdiv((rg).count, PASS_T), PASS_T, 0, w->st>>>(__VA_ARGS__, (rg));              \
            w->launches++;                                                                        \
        }                                                                                         \
    } while (0)

#define BOOL2(kern, b0, b1, n, ...)                                                                \
    do {                                                                                           \
        if (b0) { if (b1) LAUNCH_R((kern<true, true>), n, __VA_ARGS__); else LAUNCH_R((kern<true, false>), n, __VA_ARGS__); }     \
        else    { if (b1) LAUNCH_R((kern<false, true>), n, __VA_ARGS__); else LAUNCH_R((kern<false, false>), n, __VA_ARGS__); }   \
    } while (0)
#define BOOL4(kern, b0, b1, b2, b3, n, ...)                                               \
    do {                                                                                           \
        if (b3) BOOL3_T(kern, b0, b1, b2, true, n, __VA_ARGS__);                          \
        else BOOL3_T(kern, b0, b1, b2, false, n, __VA_ARGS__);                            \
    } while (0)
#define BOOL3_T(kern, b0, b1, b2, B3, n, ...)                                             \
    do {                                                                                           \
        if (b0) {                                                                                  \
            if (b1) { if (b2) LAUNCH_R((kern<true, true, true, B3>), n, __VA_ARGS__); else LAUNCH_R((kern<true, true, false, B3>), n, __VA_ARGS__); } \
            else    { if (b2) LAUNCH_R((kern<true, false, true, B3>), n, __VA_ARGS__); else LAUNCH_R((kern<true, false, false, B3>), n, __VA_ARGS__); } \
        } else {                                                                                   \
            if (b1) { if (b2) LAUNCH_R((kern<false, true, true, B3>), n, __VA_ARGS__); else LAUNCH_R((kern<false, true, false, B3>), n, __VA_ARGS__); } \
            else    { if (b2) LAUNCH_R((kern<false, false, true, B3>), n, __VA_ARGS__); else LAUNCH_R((kern<false, false, false, B3>), n, __VA_ARGS__); } \
        }                                                                                          \
    } while (0)


// DFSPH: densities + alphas + the first divergence evaluation in one sweep (k_density_alpha_div)
sph_status launch_density_alpha_div(sph_world* w, uint32_t* nblk) {
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1;
    Lists L{reinterpret_cast<const uint4*>(w->nbr_f.p), w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
    if (w->unimass) {
        TRY(ensure_tex(w, &w->tex_vyz, &w->tex_vyz_ptr, w->vyz2.p, w->vyz2.cap));
        TRY(ensure_tex(w, &w->tex_pvx, &w->tex_pvx_ptr, w->pvx4.p, w->pvx4.cap));
    } else {
        TRY(ensure_tex(w, &w->tex_vs, &w->tex_vs_ptr, w->vs.p, w->vs.cap));
    }
    const Range rg{w->own_begin, (uint32_t)w->N};
    float* partial = w->partial.p;
    uint32_t* tk = w->d_ticket.p;  // one launch covers the pass -> in-kernel final reduction
    if (w->unimass)
        LAUNCH_R((k_density_alpha_div<false, true>), rg, w->pvx4.p, w->tex_pvx, w->vs.p, (cudaTextureObject_t)0, w->vyz2.p, w->tex_vyz, w->vel[c].p, w->bpos[bc].p, L,
                 w->dens.p, w->alpha.p, w->divv.p, w->kappa.p, w->pk4.p, partial, w->d_scal.p + 7, tk, w->errsum.p);
    else if (multi)
        LAUNCH_R((k_density_alpha_div<true, false>), rg, w->pos[c].p, (cudaTextureObject_t)0, w->vs.p, w->tex_vs, w->vyz2.p, (cudaTextureObject_t)0, w->vel[c].p, w->bpos[bc].p,
                 L, w->dens.p, w->alpha.p, w->divv.p, w->kappa.p, w->pk4.p, partial, w->d_scal.p + 7, tk, w->errsum.p);
    else
        LAUNCH_R((k_density_alpha_div<false, false>), rg, w->pos[c].p, (cudaTextureObject_t)0, w->vs.p, w->tex_vs, w->vyz2.p, (cudaTextureObject_t)0, w->vel[c].p, w->bpos[bc].p,
                 L, w->dens.p, w->alpha.p, w->divv.p, w->kappa.p, w->pk4.p, partial, w->d_scal.p + 7, tk, w->errsum.p);
    *nblk = cdiv(rg.count, PASS_T);
    w->errsum_ready = true;
    return SPH_OK;
}

// compute_divergences (predict = false) / compute_predicted_densities (predict = true); returns #partials.
// In a slab world refresh_kappa() exchanges the kappa ghosts afterwards, only when an update follows.
// The fluid term of the FIRST force of a single-fluid DFSPH world can ride with the divergence evaluations when it is an
// XSPHViscosity without a boundary term (see k_vel_divergence_xsph_u).
bool xsph_fusable(const sph_world* w) {
    if (w->desc.solver != SPH_SOLVER_DFSPH || w->tile || !w->unimass || w->slab.active) return false;
    if (w->fluids.size() != 1 || w->fluids[0].forces.empty()) return false;
    const sph_force_desc& d = w->fluids[0].forces[0].d;
    return d.kind == SPH_FORCE_XSPH_VISCOSITY && d.p[0] != 0.f && (d.p[1] == 0.f || w->B == 0);
}
// ... and on the default records (k_vel_divergence_xsph_u<2>, one extra 4-byte gather of rho_j): single uniform-mass fluid
bool akinci_fusable_u(const sph_world* w) {
    if (w->desc.solver != SPH_SOLVER_DFSPH || w->tile || !w->unimass || w->slab.active) return false;
    if (w->fluids.size() != 1) return false;
    for (const ForceRec& fr : w->fluids[0].forces)
        if (fr.d.kind == SPH_FORCE_AKINCI2013_TENSION) return true;
    return false;
}

sph_status launch_vel_divergence(sph_world* w, bool predict, uint32_t* nblk) {
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1;
    const bool xsf = !predict && xsph_fusable(w);
    const bool akf = !predict && !xsf && akinci_fusable_u(w);
    if (xsf) CU(w->xs.ensure(std::max(w->Ntot, w->N)));
    if (akf) CU(w->normals.ensure(std::max(w->Ntot, w->N)));
    if (w->tile) {
        TileLists L{w->nbr16.p, w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
        uint32_t cap = tile_cap(w, 32);
        TDISPATCH2(k_tile_vel_divergence, multi, predict, 32, cap, w->pos[c].p, w->vs.p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, w->cstart.p, cap, L,
                   w->dens.p, w->alpha.p, predict ? w->pred.p : w->divv.p, w->kappa.p, w->partial.p, w->dt, w->d_scal.p + 7);
        *nblk = w->n_tiles;
        w->errsum_ready = false;
        return SPH_OK;
    }
    Lists L{reinterpret_cast<const uint4*>(w->nbr_f.p), w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
    if (w->unimass) {
        TRY(ensure_tex(w, &w->tex_pvx, &w->tex_pvx_ptr, w->pvx4.p, w->pvx4.cap));
        TRY(ensure_tex(w, &w->tex_vyz, &w->tex_vyz_ptr, w->vyz2.p, w->vyz2.cap));
    } else {
        TRY(ensure_tex(w, &w->tex_vs, &w->tex_vs_ptr, w->vs.p, w->vs.cap));
    }
    float* out = predict ? w->pred.p : w->divv.p;
    const Range rg{w->own_begin, (uint32_t)w->N};
    float* partial = w->partial.p;
    uint32_t* tk = w->d_ticket.p;  // one launch covers the pass -> in-kernel final reduction
    if (!w->unimass) {
        BOOL2(k_vel_divergence, multi, predict, rg, w->pos[c].p, w->vs.p, w->tex_vs, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, L, w->dens.p,
              w->alpha.p, out, w->kappa.p, partial, w->dt, w->d_scal.p + 7, tk, w->errsum.p);
    } else if (predict) {
        LAUNCH_R((k_vel_divergence_u<true>), rg, w->pvx4.p, w->tex_pvx, w->vyz2.p, w->tex_vyz, w->bpos[bc].p, w->bvel[bc].p, L,
                 w->dens.p, w->alpha.p, out, w->pk4.p, partial, w->dt, w->d_scal.p + 7, tk, w->errsum.p);
    } else if (xsf) {
        const float cf = w->fluids[0].forces[0].d.p[0];
        LAUNCH_R((k_vel_divergence_xsph_u<1>), rg, w->pvx4.p, w->tex_pvx, w->vyz2.p, w->tex_vyz, w->bpos[bc].p, L, w->dens.p,
                 w->alpha.p, out, w->pk4.p, partial, tk, w->errsum.p, w->xs.p, cf);
        w->xs_valid = true;
    } else if (akf) {  // Akinci normals ride along: nr4 = (n, rho) for k_akinci_force_u
        LAUNCH_R((k_vel_divergence_xsph_u<2>), rg, w->pvx4.p, w->tex_pvx, w->vyz2.p, w->tex_vyz, w->bpos[bc].p, L, w->dens.p,
                 w->alpha.p, out, w->pk4.p, partial, tk, w->errsum.p, w->normals.p, 0.f);
        w->nr4_valid = true;
    } else {
        LAUNCH_R((k_vel_divergence_u<false>), rg, w->pvx4.p, w->tex_pvx, w->vyz2.p, w->tex_vyz, w->bpos[bc].p, w->bvel[bc].p, L,
                 w->dens.p, w->alpha.p, out, w->pk4.p, partial, w->dt, w->d_scal.p + 7, tk, w->errsum.p);
    }
    *nblk = cdiv(rg.count, PASS_T);
    w->errsum_ready = true;
    return SPH_OK;
}
// compute_velocity_changes_for_divergence (pressure = false) / compute_velocity_changes (pressure = true)
sph_status launch_vel_update(sph_world* w, bool pressure) {
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1, bf = any_bforce(w);
    if (w->tile) {
        TileLists L{w->nbr16.p, w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
        uint32_t cap = tile_cap(w, 20);
        if (pressure)
            TDISPATCH3(k_tile_vel_update, multi, bf, true, 20, cap, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->cstart.p, cap, L, w->kappa.p, w->vc[c].p,
                       w->vs.p, w->bforce.p, w->inv_dt);
        else
            TDISPATCH3(k_tile_vel_update, multi, bf, false, 20, cap, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->cstart.p, cap, L, w->kappa.p, w->vc[c].p,
                       w->vs.p, w->bforce.p, w->inv_dt);
        return SPH_OK;
    }
    Lists L{reinterpret_cast<const uint4*>(w->nbr_f.p), w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
    const Range rg{w->own_begin, (uint32_t)w->N};
    if (w->unimass) {
        TRY(ensure_tex(w, &w->tex_pk, &w->tex_pk_ptr, w->pk4.p, w->pk4.cap));
        BOOL2(k_vel_update_u, bf, pressure, rg, w->pk4.p, w->tex_pk, w->vel[c].p, w->bpos[bc].p, L, w->vc[c].p, w->vs.p, w->pvx4.p, w->vyz2.p,
              w->bforce.p, w->inv_dt);
    } else {
        // measured (profiles/r1_v1_*): the texture pipe helps the float4 v* gather (-12 %) but not the 4-byte kappa gather
        BOOL4(k_vel_update, multi, bf, pressure, false, rg, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, L, w->kappa.p, w->tex_kappa, w->vc[c].p, w->vs.p,
              w->bforce.p, w->inv_dt);
    }
    return refresh_vstar(w);  // the following evaluation gathers v*_j of ghosts
}

// ---- ParticlesContacts materialisation + the context-style host plugin call (nonpressure_force.rs:15-27) ---------------
struct HostContacts {
    std::vector<uint32_t> offsets, j, model;
    std::vector<float> weight, gradient;
};
// which = 0: fluid-fluid contacts, 1: fluid-boundary contacts of fluid `f`'s particles, CSR in the fluid's original order
sph_status materialise_contacts(sph_world* w, uint32_t f, int which, HostContacts* out) {
    const FluidRec& fl = w->fluids[f];
    const size_t N = w->N, Nf = fl.n;
    const int c = w->cur, bc = w->bcur;
    const uint32_t ob = w->own_begin;
    const uint32_t cap = which ? w->cap_b : w->cap_f;
    const uint32_t* cnt = which ? w->cnt_b.p : w->cnt_f.p;
    CU(w->ct_cnt[which].ensure(N + 1));
    LAUNCH(k_contacts_count, N, 256, (uint32_t)N, w->orig[c].p + ob, cnt + ob, cap, w->ct_cnt[which].p);
    CU(cudaMemsetAsync(w->ct_cnt[which].p + N, 0, sizeof(uint32_t), w->st));
    TRY(scan_exclusive(w, w->ct_cnt[which].p, N + 1));
    std::vector<uint32_t> scan(Nf + 1);
    CU(cudaMemcpyAsync(scan.data(), w->ct_cnt[which].p + fl.offset, (Nf + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
    uint32_t total = 0;
    CU(cudaMemcpyAsync(&total, w->ct_cnt[which].p + N, sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    CU(w->ct_j[which].ensure(std::max<size_t>(total, 1)));
    CU(w->ct_model[which].ensure(std::max<size_t>(total, 1)));
    CU(w->ct_w[which].ensure(std::max<size_t>(total, 1)));
    CU(w->ct_g[which].ensure(3 * std::max<size_t>(total, 1)));
    OffsetTable tab;
    memset(&tab, 0, sizeof tab);
    if (which) {
        for (size_t b = 0; b < w->bounds.size(); ++b) tab.off[b] = (uint32_t)w->bounds[b].offset;
        if (w->B)
            LAUNCH((k_contacts_fill<true>), N, 128, (uint32_t)N, w->pos[c].p, w->bpos[bc].p, w->bvel[bc].p, w->orig[c].p, w->borig[bc].p, w->nbr_b.p, cnt, cap,
                   w->ct_cnt[which].p, tab, w->ct_j[which].p, w->ct_model[which].p, w->ct_w[which].p, w->ct_g[which].p);
    } else {
        for (size_t k = 0; k < w->fluids.size(); ++k) tab.off[k] = (uint32_t)w->fluids[k].offset;
        LAUNCH((k_contacts_fill<false>), N, 128, (uint32_t)N, w->pos[c].p, w->pos[c].p, w->vel[c].p, w->orig[c].p, w->orig[c].p, w->nbr_f.p, cnt, cap,
               w->ct_cnt[which].p, tab, w->ct_j[which].p, w->ct_model[which].p, w->ct_w[which].p, w->ct_g[which].p);
    }
    const uint32_t first = scan[0], nent = scan[Nf] - scan[0];
    out->offsets.resize(Nf + 1);
    for (size_t i = 0; i <= Nf; ++i) out->offsets[i] = scan[i] - first;
    out->j.resize(nent);
    out->model.resize(nent);
    out->weight.resize(nent);
    out->gradient.resize(3 * (size_t)nent);
    if (nent) {
        CU(cudaMemcpyAsync(out->j.data(), w->ct_j[which].p + first, nent * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
        CU(cudaMemcpyAsync(out->model.data(), w->ct_model[which].p + first, nent * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
        CU(cudaMemcpyAsync(out->weight.data(), w->ct_w[which].p + first, nent * sizeof(float), cudaMemcpyDeviceToHost, w->st));
        CU(cudaMemcpyAsync(out->gradient.data(), w->ct_g[which].p + 3 * (size_t)first, 3 * (size_t)nent * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    }
    CU(cudaStreamSynchronize(w->st));
    return SPH_OK;
}

sph_status call_host_force2(sph_world* w, uint32_t f, ForceRec& fr, std::vector<float>& hp, std::vector<float>& hv, std::vector<float>& hd,
                            std::vector<float>& ha) {
    if (w->tile) return w->fail(SPH_ERR_INVALID, "host plugins with contacts need gather_backend 0");
    if (w->slab.active && (fr.host_flags & SPH_HOST_FORCE_CONTACTS))
        return w->fail(SPH_ERR_INVALID, "materialised contacts are not available in slab-decomposed worlds");
    const FluidRec& fl = w->fluids[f];
    sph_host_force_ctx ctx;
    memset(&ctx, 0, sizeof ctx);
    ctx.dt = w->dt;
    ctx.inv_dt = w->inv_dt;
    ctx.kernel_radius = w->h;
    ctx.particle_radius = w->desc.particle_radius;
    ctx.fluid = make_handle(f, fl.gen);
    ctx.fluid_index = f;
    ctx.density0 = fl.density0;
    ctx.n = fl.n;
    ctx.positions_xyz = hp.data();
    ctx.velocities_xyz = hv.data();
    ctx.densities = hd.data();
    ctx.accelerations_xyz = ha.data();
    std::vector<float> vol;
    if (!w->slab.active && w->h_vol.size() >= fl.offset + fl.n) ctx.volumes = w->h_vol.data() + fl.offset;
    HostContacts ff, fb;
    if (fr.host_flags & SPH_HOST_FORCE_CONTACTS) {
        TRY(materialise_contacts(w, f, 0, &ff));
        TRY(materialise_contacts(w, f, 1, &fb));
        ctx.ff_offsets = ff.offsets.data(); ctx.ff_j = ff.j.data(); ctx.ff_j_model = ff.model.data();
        ctx.ff_weight = ff.weight.data(); ctx.ff_gradient_xyz = ff.gradient.data();
        ctx.fb_offsets = fb.offsets.data(); ctx.fb_j = fb.j.data(); ctx.fb_j_model = fb.model.data();
        ctx.fb_weight = fb.weight.data(); ctx.fb_gradient_xyz = fb.gradient.data();
    }
    std::vector<sph_boundary_view> views;
    std::vector<float> bvol;
    if (fr.host_flags & SPH_HOST_FORCE_BOUNDARIES) {
        bvol.resize(w->B);
        if (w->B) {
            const int bc = w->bcur;
            CU(w->o_c.ensure(3 * std::max(w->N, w->B)));
            LAUNCH(k_export_w, w->B, 256, (uint32_t)w->B, w->borig[bc].p, w->bpos[bc].p, w->o_c.p);
            CU(cudaMemcpyAsync(bvol.data(), w->o_c.p, w->B * sizeof(float), cudaMemcpyDeviceToHost, w->st));
            CU(cudaStreamSynchronize(w->st));
        }
        views.resize(w->bounds.size());
        for (size_t b = 0; b < w->bounds.size(); ++b) {
            const BoundaryRec& br = w->bounds[b];
            views[b].n = br.alive ? br.n : 0;
            views[b].positions_xyz = w->hb_pos.data() + 3 * br.offset;
            views[b].velocities_xyz = w->hb_vel.data() + 3 * br.offset;
            views[b].volumes = bvol.data() + br.offset;
        }
        ctx.n_boundaries = views.size();
        ctx.boundaries = views.data();
    }
    fr.host_fn2(fr.host_user, &ctx);
    return SPH_OK;
}

// predict_advection dfsph_solver.rs:580-603: every fluid's forces in push order
sph_status phase_forces(sph_world* w) {
    size_t N = w->N;
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1, bf = any_bforce(w);
    Lists L{reinterpret_cast<const uint4*>(w->nbr_f.p), w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
    TileLists TL{w->nbr16.p, w->nbr_b.p, w->cnt_f.p, w->cnt_b.p};
    for (size_t f = 0; f < w->fluids.size(); ++f)
        for (ForceRec& fr : w->fluids[f].forces) {
            const float* p = fr.d.p;
            switch (fr.d.kind) {
                case SPH_FORCE_XSPH_VISCOSITY:
                    if (w->xs_valid && f == 0 && &fr == &w->fluids[0].forces[0]) break;  // already folded in by k_fold_velocities
                    if (w->tile) {
                        uint32_t cap = tile_cap(w, 36);
                        TDISPATCH2(k_tile_xsph, multi, bf, 36, cap, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, w->cstart.p, cap, TL,
                                   w->dens.p, w->acc.p, w->bforce.p, (uint32_t)f, p[0], p[1], w->inv_dt);
                        break;
                    }
                    DISPATCH2(k_force_xsph, multi, bf, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, L, w->dens.p, w->acc.p,
                              w->bforce.p, (uint32_t)f, p[0], p[1], w->inv_dt);
                    break;
                case SPH_FORCE_ARTIFICIAL_VISCOSITY:
                    if (w->tile) {
                        uint32_t cap = tile_cap(w, 36);
                        TDISPATCH2(k_tile_artificial, multi, bf, 36, cap, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, w->cstart.p, cap, TL,
                                   w->dens.p, w->acc.p, w->bforce.p, (uint32_t)f, p[0], p[1], p[2], p[3], p[4]);
                        break;
                    }
                    DISPATCH2(k_force_artificial, multi, bf, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->bvel[bc].p, L, w->dens.p, w->acc.p,
                              w->bforce.p, (uint32_t)f, p[0], p[1], p[2], p[3], p[4]);
                    break;
                case SPH_FORCE_AKINCI2013_TENSION: {
                    CU(w->normals.ensure(std::max(w->Ntot, w->N)));
                    float h = w->h;
                    float coh_norm = 32.0f / (3.14159265358979323846f * powf(h, 9.f));
                    float h6_64 = powf(h, 6.f) / 64.0f;
                    float adh_norm = 0.007f / powf(h, 3.25f);
                    if (w->tile) {
                        uint32_t sb1 = multi ? 36u : 20u, sb2 = multi ? 52u : 36u;
                        uint32_t cap1 = tile_cap(w, sb1), cap2 = tile_cap(w, sb2);
                        TDISPATCH1(k_tile_akinci_normals, multi, sb1, cap1, w->pos[c].p, w->vel[c].p, w->cstart.p, cap1, TL, w->dens.p, w->normals.p,
                                   (uint32_t)f);
                        TDISPATCH2(k_tile_akinci_force, multi, bf, sb2, cap2, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, w->cstart.p, cap2, TL, w->dens.p,
                                   w->normals.p, w->acc.p, w->bforce.p, (uint32_t)f, p[0], p[1], coh_norm, h6_64, adh_norm);
                        break;
                    }
                    if (w->nr4_valid && f == 0) {  // normals (and rho, in .w) came with a divergence evaluation
                        TRY(ensure_tex(w, &w->tex_pvx, &w->tex_pvx_ptr, w->pvx4.p, w->pvx4.cap));
                        if (bf) LAUNCH((k_akinci_force_u<true>), N, PASS_T, w->pvx4.p, w->tex_pvx, w->normals.p, w->bpos[bc].p, L, w->acc.p, w->bforce.p, p[0], p[1], coh_norm, h6_64, adh_norm);
                        else LAUNCH((k_akinci_force_u<false>), N, PASS_T, w->pvx4.p, w->tex_pvx, w->normals.p, w->bpos[bc].p, L, w->acc.p, w->bforce.p, p[0], p[1], coh_norm, h6_64, adh_norm);
                        break;
                    }
                    DISPATCH1(k_akinci_normals, multi, N, PASS_T, w->pos[c].p, w->vel[c].p, L, w->dens.p, w->normals.p, (uint32_t)f);
                    TRY(slab_refresh(w, w->normals.p, sizeof(float4)));
                    DISPATCH2(k_akinci_force, multi, bf, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, L, w->dens.p, w->normals.p, w->acc.p,
                              w->bforce.p, (uint32_t)f, p[0], p[1], coh_norm, h6_64, adh_norm);
                    break;
                }
                case SPH_FORCE_BECKER2009_ELASTICITY:
                    TRY(elasticity_solve(w, (uint32_t)f, fr));
                    break;
                case SPH_FORCE_HE2014_TENSION: {
                    if (w->tile) return w->fail(SPH_ERR_INVALID, "He2014SurfaceTension is not implemented by gather_backend 1");
                    CU(w->he_colors.ensure(std::max(w->Ntot, w->N)));
                    CU(w->he_gradc.ensure(std::max(w->Ntot, w->N)));
                    DISPATCH1(k_he2014_colors, multi, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, L, w->dens.p, w->he_colors.p, (uint32_t)f);
                    TRY(slab_refresh(w, w->he_colors.p, sizeof(float)));
                    DISPATCH1(k_he2014_gradc, multi, N, PASS_T, w->pos[c].p, w->vel[c].p, L, w->dens.p, w->he_colors.p, w->he_gradc.p, (uint32_t)f);
                    TRY(slab_refresh(w, w->he_gradc.p, sizeof(float)));
                    DISPATCH2(k_he2014_force, multi, bf, N, PASS_T, w->pos[c].p, w->vel[c].p, w->bpos[bc].p, L, w->dens.p, w->he_gradc.p, w->acc.p,
                              w->bforce.p, (uint32_t)f, p[0], p[1]);
                    break;
                }
                case SPH_FORCE_DFSPH_VISCOSITY:
                    TRY(viscosity_solve(w, (uint32_t)f, fr));
                    break;
                case SPH_FORCE_WCSPH_TENSION:
                    if (w->tile) return w->fail(SPH_ERR_INVALID, "WCSPHSurfaceTension is not implemented by gather_backend 1");
                    if (p[0] != 0.f) DISPATCH1(k_wcsph_force, multi, N, PASS_T, w->pos[c].p, w->vel[c].p, L, w->acc.p, (uint32_t)f, p[0]);
                    break;
                case FORCE_HOST_CALLBACK: {  // user-defined NonPressureForce::solve on the host (nonpressure_force.rs:10-30)
                    FluidRec& fl = w->fluids[f];
                    if (fl.n == 0) break;
                    const uint32_t ob = w->own_begin;
                    const size_t Nf = fl.n;
                    CU(w->o_a.ensure(3 * N));
                    CU(w->o_b.ensure(3 * N));
                    CU(w->o_c.ensure(3 * std::max(N, w->B)));
                    CU(w->o_mass.ensure(N));
                    LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + ob, w->pos[c].p + ob, w->o_a.p);
                    LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + ob, w->vel[c].p + ob, w->o_b.p);
                    LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + ob, w->acc.p + ob, w->o_c.p);
                    LAUNCH(k_export1, N, 256, (uint32_t)N, w->orig[c].p + ob, w->dens.p + ob, w->o_mass.p);
                    std::vector<float> hp(3 * Nf), hv(3 * Nf), ha(3 * Nf), hd(Nf);
                    CU(cudaMemcpyAsync(hp.data(), w->o_a.p + 3 * fl.offset, 3 * Nf * sizeof(float), cudaMemcpyDeviceToHost, w->st));
                    CU(cudaMemcpyAsync(hv.data(), w->o_b.p + 3 * fl.offset, 3 * Nf * sizeof(float), cudaMemcpyDeviceToHost, w->st));
                    CU(cudaMemcpyAsync(ha.data(), w->o_c.p + 3 * fl.offset, 3 * Nf * sizeof(float), cudaMemcpyDeviceToHost, w->st));
                    CU(cudaMemcpyAsync(hd.data(), w->o_mass.p + fl.offset, Nf * sizeof(float), cudaMemcpyDeviceToHost, w->st));
                    CU(cudaStreamSynchronize(w->st));
                    if (fr.host_fn2) TRY(call_host_force2(w, (uint32_t)f, fr, hp, hv, hd, ha));
                    else fr.host_fn(fr.host_user, w->dt, w->inv_dt, w->h, Nf, hp.data(), hv.data(), hd.data(), ha.data());
                    TRY(enter(w));  // the callback may have used another world of this process
                    CU(cudaMemcpyAsync(w->o_c.p + 3 * fl.offset, ha.data(), 3 * Nf * sizeof(float), cudaMemcpyHostToDevice, w->st));
                    LAUNCH(k_import_acc, N, 256, (uint32_t)N, w->orig[c].p + ob, w->o_c.p, (uint32_t)fl.offset, (uint32_t)(fl.offset + Nf), w->acc.p + ob);
                    CU(cudaStreamSynchronize(w->st));  // host vectors go out of scope
                    break;
                }
                default:
                    return w->fail(SPH_ERR_INVALID, "unknown force kind %d", fr.d.kind);
            }
        }
    CU(cudaGetLastError());
    return SPH_OK;
}

// timestep_manager.rs:76-88
void timestep_advance(sph_world* w, float total) {
    w->dt = total;
    w->inv_dt = total == 0.f ? 0.f : 1.0f / total;
}

// DFSPHSolver::step dfsph_solver.rs:667-708
sph_status dfsph_step(sph_world* w, float dt_total, const float g[3]) {
    size_t N = w->N;
    int c = w->cur, bc = w->bcur;
    const bool multi = w->fluids.size() > 1, bf = any_bforce(w);
    uint32_t nblk = 0;
    (void)bc; (void)multi; (void)bf;
    // divergence_solve :466-503 (uses the PREVIOUS step's inv_dt; 0 on the first step)
    w->stats.n_divergence_iter = w->stats.n_divergence_eval = 0;
    w->xs_valid = false;
    w->nr4_valid = false;
    uint32_t maxit = w->force_div >= 0 ? (uint32_t)w->force_div + 1 : w->desc.max_divergence_iter;
    for (uint32_t i = 0; i < maxit; ++i) {
        if (i == 0 && w->fused_first_div) {
            nblk = w->fused_nblk;  // evaluation 0 was computed by k_density_alpha_div
        } else {
            TRY(span_begin(w, SP_DIV_EVAL));
            TRY(launch_vel_divergence(w, false, &nblk));
            TRY(span_end(w));
        }
        w->stats.n_divergence_eval++;
        if (w->force_div >= 0) {
            if ((int)i >= w->force_div) break;
        } else if (i < w->desc.min_divergence_iter && i + 1 < maxit) {
            // the break needs `i >= min_iter` (:486): this evaluation's error cannot end the loop and the next
            // evaluation reports a fresher one, so neither the read-back (a host sync) nor the allreduce is needed
            w->errsum_ready = false;
        } else {
            float avg;
            TRY(read_error(w, nblk, &avg));
            w->stats.last_divergence_error = avg;
            float max_err = w->desc.max_divergence_error * w->inv_dt * 0.01f;
            if (avg <= max_err && i >= w->desc.min_divergence_iter) break;
        }
        if (!(i == 0 && w->fused_first_div)) TRY(refresh_kappa(w));  // the update gathers kappa_j of ghosts
        TRY(span_begin(w, SP_DIV_UPD));
        TRY(launch_vel_update(w, false));
        TRY(span_end(w));
        w->xs_valid = false;  // v* moved on: XSPH sums of the evaluation above are stale unless another evaluation follows
        w->stats.n_divergence_iter++;
    }
    CU(cudaEventRecord(w->ev[EV_DIV], w->st));
    // update_velocities :422-430, zero vc :689-691, acc += gravity :574-578
    // nothing to launch in the force phase (no plugin at all, or only the XSPH whose sums rode with the divergence loop)?  Then
    // fold, acceleration and integration are one streaming pass
    bool quiet_forces = true;
    for (size_t f = 0; f < w->fluids.size() && quiet_forces; ++f)
        for (const ForceRec& fr : w->fluids[f].forces)
            if (!(w->xs_valid && f == 0 && &fr == &w->fluids[0].forces[0] && fr.d.kind == SPH_FORCE_XSPH_VISCOSITY)) quiet_forces = false;
    if (quiet_forces) {
        const float inv_dt_old = w->inv_dt;
        CU(cudaEventRecord(w->ev[EV_FOLD], w->st));
        CU(cudaEventRecord(w->ev[EV_FORCES], w->st));
        timestep_advance(w, dt_total);  // :702
        LAUNCH(k_fold_integrate, w->Ntot, 256, w->vel[c].p, w->vc[c].p, w->vs.p, w->acc.p, g[0], g[1], g[2],
               w->xs_valid ? (const float4*)w->xs.p : (const float4*)nullptr, inv_dt_old, w->dt, w->unimass ? w->pvx4.p : nullptr,
               w->unimass ? w->vyz2.p : nullptr);
    } else {
        LAUNCH(k_fold_velocities, w->Ntot, 256, w->vel[c].p, w->vc[c].p, w->vs.p, w->acc.p, g[0], g[1], g[2],  // ghosts too (vel = v*)
               w->xs_valid ? (const float4*)w->xs.p : (const float4*)nullptr, w->inv_dt);
        CU(cudaEventRecord(w->ev[EV_FOLD], w->st));
        TRY(phase_forces(w));
        CU(cudaEventRecord(w->ev[EV_FORCES], w->st));
        timestep_advance(w, dt_total);  // :702
        LAUNCH(k_integrate_acc, N, 256, w->vel[c].p, w->vc[c].p, w->vs.p, w->acc.p, w->dt, w->unimass ? w->pvx4.p : nullptr,
               w->unimass ? w->vyz2.p : nullptr);
    }
    TRY(refresh_vstar(w));
    CU(cudaEventRecord(w->ev[EV_INTEG], w->st));
    // pressure_solve :432-464
    w->stats.n_pressure_iter = w->stats.n_pressure_eval = 0;
    maxit = w->force_press >= 0 ? (uint32_t)w->force_press + 1 : w->desc.max_pressure_iter;
    for (uint32_t i = 0; i < maxit; ++i) {
        TRY(span_begin(w, SP_PRED));
        TRY(launch_vel_divergence(w, true, &nblk));
        TRY(span_end(w));
        w->stats.n_pressure_eval++;
        if (w->force_press >= 0) {
            if ((int)i >= w->force_press) break;
        } else if (i < w->desc.min_pressure_iter && i + 1 < maxit) {
            w->errsum_ready = false;  // cannot break yet (:450): skip the read-back, as in the divergence loop
        } else {
            float avg;
            TRY(read_error(w, nblk, &avg));
            w->stats.last_density_error = avg;
            if (avg <= w->desc.max_density_error && i >= w->desc.min_pressure_iter) break;
        }
        TRY(refresh_kappa(w));
        TRY(span_begin(w, SP_PUPD));
        TRY(launch_vel_update(w, true));
        TRY(span_end(w));
        w->stats.n_pressure_iter++;
    }
    CU(cudaEventRecord(w->ev[EV_PRESS], w->st));
    {
        static const int init[7] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, 0};
        CU(w->d_nb.ensure(8));
        CU(cudaMemcpyAsync(w->d_nb.p, init, sizeof init, cudaMemcpyHostToDevice, w->st));
        LAUNCH(k_update_positions, N, 256, w->pos[c].p, w->vs.p, w->dt, w->slab.active ? (int*)nullptr : w->d_nb.p);  // :411-420
        w->nb_pending = !w->slab.active;
    }
    CU(cudaGetLastError());
    return SPH_OK;
}

sph_status world_step(sph_world* w, float dt, const float g[3], const sph_coupling_manager* coupling = nullptr) {
    TRY(enter(w));
    w->launches = 0;
    w->stats_exchanges = 0;
    w->n_spans = 0;
    w->nb_pending = false;
    memset(&w->stats, 0, sizeof w->stats);
    TRY(apply_pending_deletes(w));  // liquid_world.rs:79-81
    TRY(stage_up(w));
    TRY(upload_boundaries(w));
    size_t N = w->N;
    w->stats.n_fluid_particles = N;
    w->stats.n_boundary_particles = w->B;
    if (w->fluids.size() > (size_t)MAX_FLUIDS || w->bounds.size() > (size_t)MAX_BOUNDARIES)
        return w->fail(SPH_ERR_INVALID, "too many fluids (max %d) or boundaries (max %d)", MAX_FLUIDS, MAX_BOUNDARIES);
    if (!(dt > F32_EPS)) return SPH_OK;  // timestep_manager.rs:56-58: is_done() before the first substep
    CU(cudaEventRecord(w->ev[EV_START], w->st));
    if (w->slab.active) {
        TRY(slab_begin_step(w));
        N = w->N;
        w->stats.n_fluid_particles = N;
    } else {
        w->Ntot = N;
        w->own_begin = 0;
    }
    if (w->Ntot + w->B == 0) return SPH_OK;
    TRY(phase_grid(w));
    w->grid_ready = true;
    w->ever_stepped = true;
    if (coupling && coupling->update_boundaries) {
        // CouplingManager::update_boundaries runs after the FLUIDS of this substep are in the grid and before the boundaries
        // are (liquid_world.rs:86-103): queries issued by the callback see the fluid particles only.  The callback may rewrite
        // boundaries (count included) and fluid positions / velocities; the grid is then rebuilt from the edited state
        // (the reference keeps edited particles in their stale cells; re-binning them is the only deviation).
        CU(cudaStreamSynchronize(w->st));
        w->in_coupling = true;
        w->lists_valid = true;  // sentinel: a fluid write in the callback clears it
        coupling->update_boundaries(coupling->user, w, w->dt, w->inv_dt, w->h, w->desc.particle_radius);
        w->in_coupling = false;
        TRY(enter(w));
        if (w->staged) return w->fail(SPH_ERR_INVALID, "update_boundaries must not add / remove fluids or particles");
        if (w->b_dirty || !w->lists_valid) {
            TRY(upload_boundaries(w));
            w->stats.n_boundary_particles = w->B;
            TRY(phase_grid(w));
        }
        w->lists_valid = false;
    }
    CU(cudaEventRecord(w->ev[EV_GRID], w->st));
    // evaluate_kernels + compute_densities (liquid_world.rs:123-134) + compute_alphas (dfsph_solver.rs:679-684), enqueued
    // speculatively by the neighbour phase (EV_NBR is recorded there, between the two)
    TRY(phase_neighbors(w, [](sph_world* w) -> sph_status {
        w->fused_first_div = false;
        if (w->N) {
            if (w->desc.solver == SPH_SOLVER_DFSPH && !w->tile) {
                TRY(launch_density_alpha_div(w, &w->fused_nblk));
                w->fused_first_div = true;
            } else {
                TRY(launch_density_alpha(w));
            }
        }
        return SPH_OK;
    }));
    CU(cudaEventRecord(w->ev[EV_DENS], w->st));
    if (N) {
        if (w->desc.solver == SPH_SOLVER_DFSPH) TRY(dfsph_step(w, dt, g));
        else TRY(iisph_step(w, dt, g));
    }
    CU(cudaEventRecord(w->ev[EV_END], w->st));
    int flag = 0;
    unsigned long long cnts[2] = {0, 0};
    CU(cudaMemcpyAsync(&flag, w->d_scal.p + 7, sizeof(int), cudaMemcpyDeviceToHost, w->st));
    CU(cudaMemcpyAsync(cnts, w->d_cnt.p, sizeof cnts, cudaMemcpyDeviceToHost, w->st));
    if (w->nb_pending) CU(cudaMemcpyAsync(w->nb, w->d_nb.p, sizeof w->nb, cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    w->nb_valid = w->nb_pending;
    w->nb_pending = false;
    CU(cudaGetLastError());
    if (!w->b_reused) w->bb_contacts = cnts[0];
    w->stats.n_contacts = w->bb_contacts + cnts[1];
    w->stats.kernel_launches = w->launches;
    w->stats.n_ghost_particles = (uint32_t)(w->Ntot - w->N);
    w->stats.n_migrated = w->slab.migrated_in + w->slab.migrated_out;
    w->stats.n_exchanges = (uint32_t)w->stats_exchanges;
    auto el = [&](int a, int b) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, w->ev[a], w->ev[b]);
        return ms;
    };
    w->stats.step_ms = el(EV_START, EV_END);
    w->stats.grid_ms = el(EV_START, EV_GRID);
    w->stats.neighbors_ms = el(EV_GRID, EV_NBR);
    w->stats.density_ms = el(EV_NBR, EV_DENS);
    if (N && w->desc.solver == SPH_SOLVER_DFSPH) {
        w->stats.divergence_ms = el(EV_DENS, EV_DIV);
        w->stats.nonpressure_ms = el(EV_FOLD, EV_FORCES);
        w->stats.pressure_ms = el(EV_INTEG, EV_PRESS);
        w->stats.integrate_ms = el(EV_DIV, EV_FOLD) + el(EV_FORCES, EV_INTEG) + el(EV_PRESS, EV_END);
    } else if (N) {
        w->stats.nonpressure_ms = el(EV_DENS, EV_FORCES);
        w->stats.pressure_ms = el(EV_INTEG, EV_PRESS);
        w->stats.integrate_ms = el(EV_FORCES, EV_INTEG) + el(EV_PRESS, EV_END);
    }
    {
        float acc[SP_COUNT] = {0.f, 0.f, 0.f, 0.f};
        for (size_t k = 0; k < w->n_spans; ++k) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, w->spans[k].a, w->spans[k].b);
            acc[w->spans[k].slot] += ms;
        }
        w->stats.divergence_eval_ms = acc[SP_DIV_EVAL];
        w->stats.divergence_update_ms = acc[SP_DIV_UPD];
        w->stats.predict_density_ms = acc[SP_PRED];
        w->stats.pressure_update_ms = acc[SP_PUPD];
    }
    if (flag & 2) return w->fail(SPH_ERR_NCCL, "peer-memory ghost exchange timed out (a neighbour rank never delivered its boundary column)");
    if (flag) return w->fail(SPH_ERR_ZERO_DENSITY, "zero density (reference asserts dfsph_solver.rs:92,145,662)");
    if (coupling && coupling->transmit_forces) coupling->transmit_forces(coupling->user, w, w->dt, w->inv_dt);  // liquid_world.rs:146
    return SPH_OK;
}

}  // namespace

#include "sph_slab.inl"
#include "sph_iisph_host.inl"
#include "sph_elasticity_host.inl"
#include "sph_viscosity_host.inl"

// ===================================================================================================
// extern "C" boundary
// ===================================================================================================
extern "C" {

void sph_world_desc_default(sph_world_desc* d) {
    memset(d, 0, sizeof *d);
    d->solver = SPH_SOLVER_DFSPH;
    d->particle_radius = 0.05f;
    d->smoothing_factor = 2.0f;
    d->min_pressure_iter = 1;
    d->max_pressure_iter = 50;
    d->max_density_error = 0.05f;
    d->min_divergence_iter = 1;
    d->max_divergence_iter = 50;
    d->max_divergence_error = 0.1f;
    d->omega = 0.5f;
    d->device = 0;
    d->slab_rank = 0;
    d->slab_count = 1;
    d->deterministic = 1;
    d->gather_backend = 0;
}

sph_status sph_world_create(const sph_world_desc* desc, sph_world** out) {
    if (!desc || !out) return SPH_ERR_INVALID;
    *out = nullptr;
    if (!(desc->particle_radius > 0.f) || !(desc->smoothing_factor > 0.f)) return SPH_ERR_INVALID;
    if (desc->solver != SPH_SOLVER_DFSPH && desc->solver != SPH_SOLVER_IISPH) return SPH_ERR_INVALID;
    if (desc->kernel_density < 0 || desc->kernel_density > SPH_KERNEL_VISCOSITY || desc->kernel_gradient < 0 || desc->kernel_gradient > SPH_KERNEL_VISCOSITY)
        return SPH_ERR_INVALID;
#if !SPH_GENERIC_KERNELS
    // this build monomorphises the solver on CubicSplineKernel; libsalva_b200_kernels.so carries the other kernels
    if (desc->kernel_density != SPH_KERNEL_CUBIC_SPLINE || desc->kernel_gradient != SPH_KERNEL_CUBIC_SPLINE) return SPH_ERR_INVALID;
#endif
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || desc->device < 0 || desc->device >= ndev) return SPH_ERR_CUDA;
    if (cudaSetDevice(desc->device) != cudaSuccess) return SPH_ERR_CUDA;
    sph_world* w = new sph_world();
    w->desc = *desc;
    w->h = desc->particle_radius * desc->smoothing_factor * 2.0f;  // liquid_world.rs:44
    w->tile = desc->gather_backend == 1 && desc->solver == SPH_SOLVER_DFSPH;  // the tile backend covers the DFSPH passes only
    if (const char* t = getenv("SALVA_B200_XYSUB")) w->xysub = std::min(4, std::max(1, atoi(t)));
    memset(&w->hc, 0, sizeof w->hc);
    memset(&w->stats, 0, sizeof w->stats);
    bool ok = cudaStreamCreateWithFlags(&w->st, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < EV_COUNT; ++i) ok = cudaEventCreate(&w->ev[i]) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&w->ev_lists, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMallocHost(&w->h_pinned, 64 * sizeof(float)) == cudaSuccess;
    ok = ok && w->d_scal.ensure(16) == cudaSuccess && w->d_cnt.ensure(2) == cudaSuccess;
    ok = ok && w->d_ticket.ensure(4) == cudaSuccess && cudaMemset(w->d_ticket.p, 0, 4 * sizeof(uint32_t)) == cudaSuccess;
    if (!ok) {
        delete w;
        return SPH_ERR_CUDA;
    }
    fill_static_consts(w);
    *out = w;
    return SPH_OK;
}

void sph_world_destroy(sph_world* w) {
    if (!w) return;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    cudaSetDevice(w->desc.device);
    if (w->st) cudaStreamSynchronize(w->st);
    for (int k = 0; k < 2; ++k) {
        w->pos[k].release(); w->vel[k].release(); w->vc[k].release(); w->bpos[k].release(); w->bvel[k].release();
        w->orig[k].release(); w->borig[k].release(); w->press[k].release(); w->gid[k].release();
    }
    w->vs.release(); w->acc.release(); w->normals.release(); w->dbg_acc.release();
    w->dens.release(); w->alpha.release(); w->kappa.release(); w->divv.release(); w->pred.release(); w->bvol.release(); w->bforce.release();
    w->cid.release(); w->rank.release(); w->perm.release(); w->cstart.release(); w->bcid.release(); w->brank.release(); w->bperm.release();
    w->bstart.release();
    for (auto& a : w->scan_aux) a.release();
    for (auto& a : w->scan_aux_k) a.release();
    w->nbr_f.release(); w->nbr16.release(); w->nbr_b.release(); w->cnt_f.release(); w->cnt_b.release();
    w->partial.release(); w->errsum.release(); w->d_scal.release(); w->d_cnt.release();
    w->o_a.release(); w->o_b.release(); w->o_c.release(); w->o_mass.release(); w->o_fid.release();
    iisph_release(w);
    viscosity_release(w);
    slab_release(w);
    for (auto& f : w->fluids)
        for (auto& fr : f.forces) elasticity_release(fr);
    for (cudaTextureObject_t t : {w->tex_pvx, w->tex_vyz, w->tex_pk})
        if (t) cudaDestroyTextureObject(t);
    w->pvx4.release(); w->pk4.release(); w->vyz2.release();
    if (w->tex_vs) cudaDestroyTextureObject(w->tex_vs);
    if (w->tex_kappa) cudaDestroyTextureObject(w->tex_kappa);
    for (auto& s : w->spans) {
        cudaEventDestroy(s.a);
        cudaEventDestroy(s.b);
    }
    if (w->h_pinned) cudaFreeHost(w->h_pinned);
    w->d_ticket.release();
    w->d_nb.release();
    w->xs.release(); w->he_colors.release(); w->he_gradc.release(); w->q_out.release(); w->q_count.release();
    for (auto& e : w->ev)
        if (e) cudaEventDestroy(e);
    if (w->ev_lists) cudaEventDestroy(w->ev_lists);
    if (w->st) cudaStreamDestroy(w->st);
    if (g_const_owner == w) g_const_owner = nullptr;
    delete w;
}

sph_status sph_fluid_add(sph_world* w, const float* pos, const float* vel, const float* volumes, size_t n, float density0, uint32_t memberships,
                         uint32_t filter, uint32_t* handle) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (n && !pos) return w->fail(SPH_ERR_INVALID, "sph_fluid_add: null positions");
    size_t slot = w->fluids.size();
    for (size_t k = 0; k < w->fluids.size(); ++k)
        if (!w->fluids[k].alive) { slot = k; break; }
    if (slot >= (size_t)MAX_FLUIDS) return w->fail(SPH_ERR_INVALID, "too many fluids (max %d)", MAX_FLUIDS);
    TRY(enter(w));
    TRY(stage_down(w));
    FluidRec f;
    if (slot < w->fluids.size()) f.gen = w->fluids[slot].gen + 1;
    f.n = n;
    f.density0 = density0;
    f.memberships = memberships;
    f.filter = filter;
    f.pending_delete.assign(n, 0);
    float r = w->desc.particle_radius;
    float pv = r * r * r * (float)(8.0 * 0.8);  // fluid.rs:110-120
    // the host arrays are ordered by slot: a reused slot's (empty) range sits at its offset
    if (slot == w->fluids.size()) w->fluids.push_back(FluidRec());
    w->fluids[slot].n = 0;
    recompute_offsets(w);
    const size_t at = w->fluids[slot].offset;
    w->h_press.resize(w->h_vol.size(), 0.f);
    w->h_gid.resize(w->h_vol.size());
    w->h_pos.insert(w->h_pos.begin() + 3 * at, pos, pos + 3 * n);
    if (vel) w->h_vel.insert(w->h_vel.begin() + 3 * at, vel, vel + 3 * n);
    else w->h_vel.insert(w->h_vel.begin() + 3 * at, 3 * n, 0.f);
    w->h_vc.insert(w->h_vc.begin() + 3 * at, 3 * n, 0.f);
    if (volumes) w->h_vol.insert(w->h_vol.begin() + at, volumes, volumes + n);
    else w->h_vol.insert(w->h_vol.begin() + at, n, pv);
    w->h_press.insert(w->h_press.begin() + at, n, 0.f);
    {
        std::vector<uint32_t> ids(n);
        for (size_t i = 0; i < n; ++i) ids[i] = (uint32_t)i;
        w->h_gid.insert(w->h_gid.begin() + at, ids.begin(), ids.end());
    }
    w->fluids[slot] = f;
    recompute_offsets(w);
    if (handle) *handle = make_handle(slot, f.gen);
    return SPH_OK;
}

sph_status sph_fluid_push_force(sph_world* w, uint32_t fluid_h, const sph_force_desc* force) {
    if (!w || !force) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    if (force->kind < 0 || force->kind > SPH_FORCE_DFSPH_VISCOSITY) return w->fail(SPH_ERR_INVALID, "unknown force kind %d", force->kind);
    if (force->kind == SPH_FORCE_WCSPH_TENSION && force->p[1] != 0.f)
        return w->fail(SPH_ERR_INVALID,
                       "WCSPHSurfaceTension: boundary coefficient must be 0 (the reference's boundary loop indexes boundaries with fluid "
                       "contacts, wcsph_surface_tension.rs:66-83)");
    if (force->kind == SPH_FORCE_DFSPH_VISCOSITY && !(force->p[0] >= 0.f && force->p[0] <= 1.f))
        return w->fail(SPH_ERR_INVALID, "The viscosity coefficient must be between 0.0 and 1.0. (dfsph_viscosity.rs:106-110)");
    ForceRec fr;
    fr.d = *force;
    w->fluids[fluid].forces.push_back(fr);
    return SPH_OK;
}

sph_status sph_fluid_push_host_force(sph_world* w, uint32_t fluid_h, sph_host_force_fn fn, void* user) {
    if (!w || !fn) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    ForceRec fr;
    memset(&fr.d, 0, sizeof fr.d);
    fr.d.kind = FORCE_HOST_CALLBACK;
    fr.host_fn = fn;
    fr.host_user = user;
    w->fluids[fluid].forces.push_back(fr);
    return SPH_OK;
}

// Fluid::add_particles fluid.rs:126-150 — appended at the end of the fluid's index range.
sph_status sph_fluid_append(sph_world* w, uint32_t fluid_h, const float* pos, const float* vel, size_t n) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    if (n == 0) return SPH_OK;
    if (!pos) return w->fail(SPH_ERR_INVALID, "sph_fluid_append: null positions");
    TRY(enter(w));
    TRY(stage_down(w));
    FluidRec& f = w->fluids[fluid];
    size_t at = f.offset + f.n;
    float r = w->desc.particle_radius;
    float pv = r * r * r * (float)(8.0 * 0.8);
    w->h_pos.insert(w->h_pos.begin() + 3 * at, pos, pos + 3 * n);
    if (vel) w->h_vel.insert(w->h_vel.begin() + 3 * at, vel, vel + 3 * n);
    else w->h_vel.insert(w->h_vel.begin() + 3 * at, 3 * n, 0.f);
    w->h_vc.insert(w->h_vc.begin() + 3 * at, 3 * n, 0.f);
    w->h_vol.insert(w->h_vol.begin() + at, n, pv);
    w->h_press.resize(w->h_vol.size() - n, 0.f);
    w->h_press.insert(w->h_press.begin() + at, n, 0.f);
    w->h_gid.resize(w->h_vol.size() - n);
    {
        std::vector<uint32_t> ids(n);
        for (size_t i = 0; i < n; ++i) ids[i] = (uint32_t)(f.n + i);
        w->h_gid.insert(w->h_gid.begin() + at, ids.begin(), ids.end());
    }
    f.n += n;
    f.pending_delete.resize(f.n, 0);
    recompute_offsets(w);
    return SPH_OK;
}

sph_status sph_fluid_delete(sph_world* w, uint32_t fluid_h, const uint8_t* mask, size_t n) {
    if (!w || !mask) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    if (n != f.n) return w->fail(SPH_ERR_INVALID, "sph_fluid_delete: mask length %zu != particle count %zu", n, f.n);
    for (size_t i = 0; i < n; ++i)
        if (mask[i] && !f.pending_delete[i]) {
            f.pending_delete[i] = 1;
            f.n_pending++;
        }
    return SPH_OK;
}

sph_status sph_fluid_count(sph_world* w, uint32_t fluid_h, size_t* n) {
    if (!w || !n) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    *n = w->fluids[fluid].n;
    return SPH_OK;
}

sph_status sph_fluid_write(sph_world* w, uint32_t fluid_h, const float* pos, const float* vel, size_t n) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    if (n != f.n) return w->fail(SPH_ERR_INVALID, "sph_fluid_write: length %zu != particle count %zu", n, f.n);
    if (n == 0 || (!pos && !vel)) return SPH_OK;
    if (w->staged) {
        if (pos) memcpy(w->h_pos.data() + 3 * f.offset, pos, 3 * n * sizeof(float));
        if (vel) memcpy(w->h_vel.data() + 3 * f.offset, vel, 3 * n * sizeof(float));
        return SPH_OK;
    }
    TRY(enter(w));
    size_t N = w->N;
    int c = w->cur;
    CU(w->o_a.ensure(3 * N));
    CU(w->o_b.ensure(3 * N));
    if (pos) CU(cudaMemcpyAsync(w->o_a.p + 3 * f.offset, pos, 3 * n * sizeof(float), cudaMemcpyHostToDevice, w->st));
    if (vel) CU(cudaMemcpyAsync(w->o_b.p + 3 * f.offset, vel, 3 * n * sizeof(float), cudaMemcpyHostToDevice, w->st));
    {
        uint32_t ob = w->own_begin;
        LAUNCH(k_import, N, 256, (uint32_t)N, w->orig[c].p + ob, pos ? w->o_a.p : nullptr, vel ? w->o_b.p : nullptr, (const float*)nullptr,
               (const float*)nullptr, (const uint32_t*)nullptr, w->pos[c].p + ob, w->vel[c].p + ob, w->vc[c].p + ob, (uint32_t)f.offset,
               (uint32_t)(f.offset + n));
    }
    CU(cudaStreamSynchronize(w->st));
    w->lists_valid = false;
    if (pos) w->nb_valid = false;  // the cached bounds describe the positions the last step wrote
    return SPH_OK;
}

sph_status sph_fluid_read(sph_world* w, uint32_t fluid_h, float* pos, float* vel, size_t cap, size_t* n_out) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    if (n_out) *n_out = f.n;
    if (cap < f.n) return w->fail(SPH_ERR_INVALID, "sph_fluid_read: capacity %zu < particle count %zu", cap, f.n);
    if (f.n == 0 || (!pos && !vel)) return SPH_OK;
    if (w->staged) {
        if (pos) memcpy(pos, w->h_pos.data() + 3 * f.offset, 3 * f.n * sizeof(float));
        if (vel) memcpy(vel, w->h_vel.data() + 3 * f.offset, 3 * f.n * sizeof(float));
        return SPH_OK;
    }
    TRY(enter(w));
    size_t N = w->N;
    int c = w->cur;
    CU(w->o_a.ensure(3 * N));
    CU(w->o_b.ensure(3 * N));
    if (pos) {
        LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + w->own_begin, w->pos[c].p + w->own_begin, w->o_a.p);
        CU(cudaMemcpyAsync(pos, w->o_a.p + 3 * f.offset, 3 * f.n * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    }
    if (vel) {
        LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + w->own_begin, w->vel[c].p + w->own_begin, w->o_b.p);
        CU(cudaMemcpyAsync(vel, w->o_b.p + 3 * f.offset, 3 * f.n * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    }
    CU(cudaStreamSynchronize(w->st));
    return SPH_OK;
}

sph_status sph_boundary_add(sph_world* w, const float* pos, const float* vel, size_t n, uint32_t memberships, uint32_t filter, int want_forces,
                            uint32_t* handle) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (n && !pos) return w->fail(SPH_ERR_INVALID, "sph_boundary_add: null positions");
    size_t slot = w->bounds.size();
    for (size_t k = 0; k < w->bounds.size(); ++k)
        if (!w->bounds[k].alive) { slot = k; break; }
    if (slot >= (size_t)MAX_BOUNDARIES) return w->fail(SPH_ERR_INVALID, "too many boundaries (max %d)", MAX_BOUNDARIES);
    BoundaryRec b;
    if (slot < w->bounds.size()) b.gen = w->bounds[slot].gen + 1;
    b.n = n;
    b.memberships = memberships;
    b.filter = filter;
    b.want_forces = want_forces != 0;
    if (slot == w->bounds.size()) w->bounds.push_back(BoundaryRec());
    w->bounds[slot].n = 0;
    recompute_offsets(w);
    const size_t at = w->bounds[slot].offset;
    w->hb_pos.insert(w->hb_pos.begin() + 3 * at, pos, pos + 3 * n);
    if (vel) w->hb_vel.insert(w->hb_vel.begin() + 3 * at, vel, vel + 3 * n);
    else w->hb_vel.insert(w->hb_vel.begin() + 3 * at, 3 * n, 0.f);
    w->bounds[slot] = b;
    recompute_offsets(w);
    w->b_dirty = true;
    if (handle) *handle = make_handle(slot, b.gen);
    return SPH_OK;
}

sph_status sph_boundary_write(sph_world* w, uint32_t boundary_h, const float* pos, const float* vel, size_t n) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    BOUNDARY_OR_FAIL(boundary, boundary_h)
    BoundaryRec& b = w->bounds[boundary];
    if (n != b.n) return w->fail(SPH_ERR_INVALID, "sph_boundary_write: length %zu != particle count %zu", n, b.n);
    if (pos) memcpy(w->hb_pos.data() + 3 * b.offset, pos, 3 * n * sizeof(float));
    if (vel) memcpy(w->hb_vel.data() + 3 * b.offset, vel, 3 * n * sizeof(float));
    w->b_dirty = true;
    return SPH_OK;
}

static sph_status boundary_export(sph_world* w, uint32_t boundary_h, float* out, size_t cap, bool forces) {
    BOUNDARY_OR_FAIL(boundary, boundary_h)
    BoundaryRec& b = w->bounds[boundary];
    if (cap < b.n) return w->fail(SPH_ERR_INVALID, "capacity %zu < boundary particle count %zu", cap, b.n);
    if (b.n == 0) return SPH_OK;
    size_t width = forces ? 3 : 1;
    if (w->b_dirty || (forces && !b.want_forces)) {
        memset(out, 0, width * b.n * sizeof(float));
        return SPH_OK;
    }
    TRY(enter(w));
    size_t B = w->B;
    int bc = w->bcur;
    CU(w->o_c.ensure(3 * std::max(B, w->N)));
    if (forces) {
        // bforce is indexed by SORTED boundary index; reuse k_export3 through a float4 view is not possible -> small loop kernel
        LAUNCH(k_export_rows3, B, 256, (uint32_t)B, w->borig[bc].p, w->bforce.p, w->o_c.p);
    } else {
        LAUNCH(k_export_w, B, 256, (uint32_t)B, w->borig[bc].p, w->bpos[bc].p, w->o_c.p);
    }
    CU(cudaMemcpyAsync(out, w->o_c.p + width * b.offset, width * b.n * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    return SPH_OK;
}

sph_status sph_boundary_read_forces(sph_world* w, uint32_t boundary, float* f_xyz, size_t cap) {
    if (!w || !f_xyz) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    return boundary_export(w, boundary, f_xyz, cap, true);
}
sph_status sph_boundary_read_volumes(sph_world* w, uint32_t boundary, float* volumes, size_t cap) {
    if (!w || !volumes) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    return boundary_export(w, boundary, volumes, cap, false);
}

// Shared runner of particles_intersecting_aabb / particles_intersecting_shape: the cells [key(mins), key(maxs)] of the last
// step's grid (hgrid.rs:122-133), every particle in them tested by query_near().
static sph_status run_query(sph_world* w, AabbQuery q, const float mins[3], const float maxs[3], uint32_t* kinds, uint32_t* handles, uint32_t* indices,
                            size_t cap, size_t* n) {
    *n = 0;
    if (!w->grid_ready) {
        if (!w->ever_stepped) return SPH_OK;  // no step yet: the reference's grid is empty
        return w->fail(SPH_ERR_INVALID, "particle query: host edits are pending; the last step's cell grid no longer describes the particles");
    }
    if (w->b_dirty && !w->in_coupling) return w->fail(SPH_ERR_INVALID, "particle query: a boundary rewrite is pending; step first");
    for (int a = 0; a < 3; ++a)
        if (std::isnan(mins[a]) || std::isnan(maxs[a])) return w->fail(SPH_ERR_INVALID, "particle query: NaN bounds");
    TRY(enter(w));
    const Consts& hc = w->hc;
    int lo[3], hi[3];
    const int xs = hc.xysub > 0 ? hc.xysub : 1;  // the grid counts x, y in bins of h / xysub; the query box is in cells
    const int go[3] = {hc.ox / xs, hc.oy / xs, hc.oz}, gn[3] = {hc.nx / xs, hc.ny / xs, hc.nz};
    for (int a = 0; a < 3; ++a) {  // hgrid.rs:41-52 keys, clipped IN FLOAT to the dense grid (cells outside hold nothing; +-inf / FLT_MAX bounds are legal)
        const float flo = std::floor(mins[a] / w->h), fhi = std::floor(maxs[a] / w->h);
        if (fhi < (float)go[a] || flo > (float)(go[a] + gn[a] - 1)) return SPH_OK;
        lo[a] = (int)std::fmax(flo, (float)go[a]);
        hi[a] = (int)std::fmin(fhi, (float)(go[a] + gn[a] - 1));
        if (hi[a] < lo[a]) return SPH_OK;
    }
    q.lx = lo[0] * xs; q.ly = lo[1] * xs; q.lz = lo[2];
    q.dx = (hi[0] - lo[0] + 1) * xs; q.dy = (hi[1] - lo[1] + 1) * xs; q.dz = hi[2] - lo[2] + 1;
    for (int a = 0; a < 3; ++a) { q.mins[a] = mins[a]; q.maxs[a] = maxs[a]; }
    q.radius = w->desc.particle_radius;
    q.slot_lo = w->own_begin;
    q.slot_hi = w->own_begin + (uint32_t)w->N;
    const size_t cells = (size_t)q.dx * q.dy * q.dz;
    int c = w->cur, bc = w->bcur;
    const bool with_bounds = w->B && !w->in_coupling;  // during update_boundaries the grid holds fluids only (liquid_world.rs:90-103)
    CU(w->q_count.ensure(1));
    size_t qcap = std::max<size_t>(w->q_out.cap / 2, 4096);
    uint32_t found = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        CU(w->q_out.ensure(2 * qcap));
        CU(cudaMemsetAsync(w->q_count.p, 0, sizeof(uint32_t), w->st));
        LAUNCH(k_aabb_query, cells, 128, q, w->N ? w->pos[c].p : nullptr, w->cstart.p, w->orig[c].p, with_bounds ? w->bpos[bc].p : nullptr, w->bstart.p,
               w->borig[bc].p, w->q_out.p, (uint32_t)qcap, w->q_count.p);
        CU(cudaMemcpyAsync(&found, w->q_count.p, sizeof found, cudaMemcpyDeviceToHost, w->st));
        CU(cudaStreamSynchronize(w->st));
        if (found <= qcap) break;
        qcap = found;
    }
    std::vector<uint32_t> raw(2 * (size_t)found);
    if (found) CU(cudaMemcpy(raw.data(), w->q_out.p, raw.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    struct Hit {
        uint32_t kind, handle, index;
    };
    std::vector<Hit> hits(found);
    for (uint32_t k = 0; k < found; ++k) {
        uint32_t kind = raw[2 * (size_t)k], g = raw[2 * (size_t)k + 1];
        Hit h{kind, 0u, g};
        if (kind == 0) {
            for (size_t f = 0; f < w->fluids.size(); ++f)
                if (g >= w->fluids[f].offset && g < w->fluids[f].offset + w->fluids[f].n) { h.handle = make_handle(f, w->fluids[f].gen); h.index = g - (uint32_t)w->fluids[f].offset; }
        } else {
            for (size_t b = 0; b < w->bounds.size(); ++b)
                if (g >= w->bounds[b].offset && g < w->bounds[b].offset + w->bounds[b].n) { h.handle = make_handle(b, w->bounds[b].gen); h.index = g - (uint32_t)w->bounds[b].offset; }
        }
        hits[k] = h;
    }
    std::sort(hits.begin(), hits.end(), [](const Hit& a, const Hit& b) {
        return a.kind != b.kind ? a.kind < b.kind : a.handle != b.handle ? a.handle < b.handle : a.index < b.index;
    });
    *n = found;
    for (size_t k = 0; k < hits.size() && k < cap; ++k) {
        kinds[k] = hits[k].kind;
        handles[k] = hits[k].handle;
        indices[k] = hits[k].index;
    }
    return SPH_OK;
}

// LiquidWorld::particles_intersecting_aabb liquid_world.rs:211-243
sph_status sph_world_particles_in_aabb(sph_world* w, const float mins[3], const float maxs[3], uint32_t* kinds, uint32_t* handles, uint32_t* indices,
                                       size_t cap, size_t* n) {
    if (!w || !mins || !maxs || !n || (cap && (!kinds || !handles || !indices))) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    AabbQuery q;
    memset(&q, 0, sizeof q);
    q.kind = 0;
    return run_query(w, q, mins, maxs, kinds, handles, indices, cap, n);
}

// LiquidWorld::particles_intersecting_shape liquid_world.rs:246-281 for the shapes a C ABI can name: ball, cuboid, capsule
// (parry's Shape trait objects cannot cross the boundary).  The cells come from the shape's AABB under `pos`, exactly
// as `shape.compute_aabb(pos)` feeds cells_intersecting_aabb; the test is distance_to_point(pos, p, solid) <= particle_radius.
sph_status sph_world_particles_in_shape(sph_world* w, const sph_shape* shape, const float translation[3], const float rotation_rowmajor[9], uint32_t* kinds,
                                        uint32_t* handles, uint32_t* indices, size_t cap, size_t* n) {
    if (!w || !shape || !translation || !n || (cap && (!kinds || !handles || !indices))) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    AabbQuery q;
    memset(&q, 0, sizeof q);
    static const float ident[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    const float* R = rotation_rowmajor ? rotation_rowmajor : ident;
    for (int k = 0; k < 9; ++k) q.rot[k] = R[k];
    for (int a = 0; a < 3; ++a) q.t[a] = translation[a];
    float ext[3];  // half extents of the posed shape's AABB
    switch (shape->kind) {
        case SPH_SHAPE_BALL:
            if (!(shape->p[0] >= 0.f)) return w->fail(SPH_ERR_INVALID, "ball radius must be >= 0");
            q.kind = 1;
            q.sp[0] = shape->p[0];
            ext[0] = ext[1] = ext[2] = shape->p[0];
            break;
        case SPH_SHAPE_CUBOID:
            q.kind = 2;
            for (int a = 0; a < 3; ++a) q.sp[a] = shape->p[a];
            for (int a = 0; a < 3; ++a) ext[a] = std::fabs(R[3 * a]) * shape->p[0] + std::fabs(R[3 * a + 1]) * shape->p[1] + std::fabs(R[3 * a + 2]) * shape->p[2];
            break;
        case SPH_SHAPE_CAPSULE:
            q.kind = 3;
            q.sp[0] = shape->p[0];
            q.sp[1] = shape->p[1];
            for (int a = 0; a < 3; ++a) ext[a] = std::fabs(R[3 * a + 1]) * shape->p[0] + shape->p[1];  // segment along local y, swept by the radius
            break;
        default:
            return w->fail(SPH_ERR_INVALID, "unknown shape kind %d", shape->kind);
    }
    float mins[3], maxs[3];
    for (int a = 0; a < 3; ++a) {
        mins[a] = translation[a] - ext[a];
        maxs[a] = translation[a] + ext[a];
    }
    return run_query(w, q, mins, maxs, kinds, handles, indices, cap, n);
}

sph_status sph_world_step(sph_world* w, float dt, const float gravity[3]) {
    if (!w || !gravity) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "sph_world_step called from inside a coupling callback");
    sph_status s = world_step(w, dt, gravity);
    if (s != SPH_OK) cudaStreamSynchronize(w->st);
    return s;
}

// LiquidWorld::step_with_coupling liquid_world.rs:67-158
sph_status sph_world_step_with_coupling(sph_world* w, float dt, const float gravity[3], const sph_coupling_manager* coupling) {
    if (!w || !gravity) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "sph_world_step_with_coupling called from inside a coupling callback");
    if (coupling && w->slab.active) return w->fail(SPH_ERR_INVALID, "coupling callbacks are not supported in slab-decomposed worlds");
    sph_status s = world_step(w, dt, gravity, coupling);
    w->in_coupling = false;
    if (s != SPH_OK) cudaStreamSynchronize(w->st);
    return s;
}

sph_status sph_world_force_iterations(sph_world* w, int32_t n_div, int32_t n_press) {
    if (!w) return SPH_ERR_INVALID;
    w->force_div = n_div;
    w->force_press = n_press;
    return SPH_OK;
}

sph_status sph_world_stats(sph_world* w, sph_step_stats* out) {
    if (!w || !out) return SPH_ERR_INVALID;
    *out = w->stats;
    return SPH_OK;
}

float sph_world_h(const sph_world* w) { return w ? w->h : 0.f; }
float sph_world_particle_radius(const sph_world* w) { return w ? w->desc.particle_radius : 0.f; }

sph_status sph_debug_read(sph_world* w, uint32_t fluid_h, int what, float* out, size_t cap) {
    if (!w || !out) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    bool vec = what == SPH_DBG_VELOCITY_CHANGE || what == SPH_DBG_ACCELERATION;
    size_t width = vec ? 3 : 1;
    if (cap < f.n) return w->fail(SPH_ERR_INVALID, "sph_debug_read: capacity %zu < particle count %zu", cap, f.n);
    if (f.n == 0) return SPH_OK;
    if (w->staged) {
        if (what == SPH_DBG_VELOCITY_CHANGE) memcpy(out, w->h_vc.data() + 3 * f.offset, 3 * f.n * sizeof(float));
        else memset(out, 0, width * f.n * sizeof(float));
        return SPH_OK;
    }
    TRY(enter(w));
    size_t N = w->N;
    int c = w->cur;
    CU(w->o_c.ensure(3 * std::max(N, w->B)));
    const float* s1 = nullptr;
    switch (what) {
        case SPH_DBG_DENSITY: s1 = w->dens.p; break;
        case SPH_DBG_ALPHA: s1 = w->alpha.p; break;
        case SPH_DBG_DIVERGENCE: s1 = w->divv.p; break;
        case SPH_DBG_PREDICTED_DENSITY: s1 = w->desc.solver == SPH_SOLVER_IISPH ? iisph_pred(w) : w->pred.p; break;
        case SPH_DBG_PRESSURE: s1 = w->press[c].p; break;
        default: break;
    }
    const uint32_t ob = w->own_begin;
    const uint32_t* og = w->orig[c].p + ob;
    if (s1) LAUNCH(k_export1, N, 256, (uint32_t)N, og, s1 + ob, w->o_c.p);
    else if (what == SPH_DBG_VELOCITY_CHANGE) LAUNCH(k_export3, N, 256, (uint32_t)N, og, w->vc[c].p + ob, w->o_c.p);
    else if (what == SPH_DBG_ACCELERATION) LAUNCH(k_export3, N, 256, (uint32_t)N, og, w->acc.p + ob, w->o_c.p);
    else if (what == SPH_DBG_NUM_FLUID_CONTACTS) LAUNCH(k_export1u, N, 256, (uint32_t)N, og, w->cnt_f.p + ob, w->o_c.p);
    else if (what == SPH_DBG_NUM_BOUNDARY_CONTACTS) LAUNCH(k_export1u, N, 256, (uint32_t)N, og, w->cnt_b.p + ob, w->o_c.p);
    else return w->fail(SPH_ERR_INVALID, "sph_debug_read: unknown selector %d", what);
    CU(cudaMemcpyAsync(out, w->o_c.p + width * f.offset, width * f.n * sizeof(float), cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    return SPH_OK;
}

const char* sph_last_error(const sph_world* w) { return w ? w->err.c_str() : "null world"; }
const char* sph_version(void) {
#if SPH_GENERIC_KERNELS
    return "salva_b200 0.2 (sm_100a, kernels: cubic-spline poly6 spiky viscosity)";
#else
    return "salva_b200 0.2 (sm_100a, kernels: cubic-spline)";
#endif
}

sph_status sph_nccl_unique_id(char out[128]) {
    if (!out) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    std::string err;
    if (!nccl_load(&err)) return SPH_ERR_NCCL;
    nccl_uid id;
    if (g_nccl.GetUniqueId(&id) != 0) return SPH_ERR_NCCL;
    memcpy(out, id.internal, 128);
    return SPH_OK;
}

static sph_status slab_attach(sph_world* w, void* comm, bool own, int rank, int nranks) {
    if (rank < 0 || nranks < 1 || rank >= nranks) return w->fail(SPH_ERR_INVALID, "bad rank %d of %d", rank, nranks);
    SlabState& S = w->slab;
    S.comm = comm;
    S.own_comm = own;
    S.rank = rank;
    S.nranks = nranks;
    S.has_left = rank > 0;
    S.has_right = rank + 1 < nranks;
    S.active = nranks > 1;
    w->desc.deterministic = 1;  // ghost-column order agreement relies on the stable in-cell order
    CU(S.d_cnt.ensure(32));
    CU(S.d_cnt64.ensure(1));
    if (S.active) TRY(p2p_setup(w));
    return SPH_OK;
}

sph_status sph_world_attach_nccl(sph_world* w, void* nccl_comm, int rank, int nranks) {
    if (!w || !nccl_comm) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (!nccl_load(&w->err)) return SPH_ERR_NCCL;
    TRY(enter(w));
    return slab_attach(w, nccl_comm, false, rank, nranks);
}

sph_status sph_world_create_nccl(sph_world* w, const char unique_id[128], int rank, int nranks) {
    if (!w || !unique_id) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (!nccl_load(&w->err)) return SPH_ERR_NCCL;
    TRY(enter(w));
    nccl_uid id;
    memcpy(id.internal, unique_id, 128);
    void* comm = nullptr;
    NC(g_nccl.CommInitRank(&comm, nranks, id, rank));
    return slab_attach(w, comm, true, rank, nranks);
}

sph_status sph_world_set_slab(sph_world* w, int32_t cell_lo, int32_t cell_hi) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if ((long long)cell_hi - (long long)cell_lo < 2) return w->fail(SPH_ERR_INVALID, "a slab must be at least 2 cell columns wide");
    w->slab.lo = cell_lo;
    w->slab.hi = cell_hi;
    return SPH_OK;
}

sph_status sph_fluid_set_ids(sph_world* w, uint32_t fluid_h, const uint32_t* ids, size_t n) {
    if (!w || !ids) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    if (n != f.n) return w->fail(SPH_ERR_INVALID, "sph_fluid_set_ids: length %zu != particle count %zu", n, f.n);
    TRY(enter(w));
    TRY(stage_down(w));
    w->h_gid.resize(w->N);
    memcpy(w->h_gid.data() + f.offset, ids, n * sizeof(uint32_t));
    return SPH_OK;
}

sph_status sph_fluid_read_ids(sph_world* w, uint32_t fluid_h, uint32_t* ids, size_t cap) {
    if (!w || !ids) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    FluidRec& f = w->fluids[fluid];
    if (cap < f.n) return w->fail(SPH_ERR_INVALID, "sph_fluid_read_ids: capacity %zu < particle count %zu", cap, f.n);
    if (f.n == 0) return SPH_OK;
    if (w->staged) {
        memcpy(ids, w->h_gid.data() + f.offset, f.n * sizeof(uint32_t));
        return SPH_OK;
    }
    TRY(enter(w));
    size_t N = w->N;
    int c = w->cur;
    CU(w->o_c.ensure(3 * std::max(N, w->B)));
    LAUNCH(k_export_u32, N, 256, (uint32_t)N, w->orig[c].p + w->own_begin, w->gid[c].p + w->own_begin, reinterpret_cast<uint32_t*>(w->o_c.p));
    CU(cudaMemcpyAsync(ids, reinterpret_cast<uint32_t*>(w->o_c.p) + f.offset, f.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
    CU(cudaStreamSynchronize(w->st));
    return SPH_OK;
}


// fluid.nonpressure_forces.push(Box<dyn NonPressureForce>) with the FULL solve() argument list (nonpressure_force.rs:15-27):
// timestep, kernel radius, fluid-fluid and fluid-boundary contacts, the fluid, the boundaries, the densities.
sph_status sph_fluid_push_host_force2(sph_world* w, uint32_t fluid_h, sph_host_force_fn2 fn, void* user, uint32_t flags) {
    if (!w || !fn) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    ForceRec fr;
    memset(&fr.d, 0, sizeof fr.d);
    fr.d.kind = FORCE_HOST_CALLBACK;
    fr.host_fn2 = fn;
    fr.host_flags = flags;
    fr.host_user = user;
    w->fluids[fluid].forces.push_back(fr);
    return SPH_OK;
}

// LiquidWorld::remove_fluid liquid_world.rs:171-173.  The handle dies; other handles stay valid (arena semantics).
sph_status sph_fluid_remove(sph_world* w, uint32_t fluid_h) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "fluids cannot be removed from inside a coupling callback");
    if (w->slab.active) return w->fail(SPH_ERR_INVALID, "sph_fluid_remove is not supported in slab-decomposed worlds");
    TRY(enter(w));
    TRY(stage_down(w));
    FluidRec& f = w->fluids[fluid];
    const size_t at = f.offset, n = f.n;
    w->h_press.resize(w->h_vol.size(), 0.f);
    w->h_gid.resize(w->h_vol.size());
    w->h_pos.erase(w->h_pos.begin() + 3 * at, w->h_pos.begin() + 3 * (at + n));
    w->h_vel.erase(w->h_vel.begin() + 3 * at, w->h_vel.begin() + 3 * (at + n));
    w->h_vc.erase(w->h_vc.begin() + 3 * at, w->h_vc.begin() + 3 * (at + n));
    w->h_vol.erase(w->h_vol.begin() + at, w->h_vol.begin() + at + n);
    w->h_press.erase(w->h_press.begin() + at, w->h_press.begin() + at + n);
    w->h_gid.erase(w->h_gid.begin() + at, w->h_gid.begin() + at + n);
    for (auto& fr : f.forces) elasticity_release(fr);
    f.forces.clear();
    f.pending_delete.clear();
    f.n_pending = 0;
    f.n = 0;
    f.alive = false;
    recompute_offsets(w);
    return SPH_OK;
}

// LiquidWorld::remove_boundary liquid_world.rs:176-178
sph_status sph_boundary_remove(sph_world* w, uint32_t boundary_h) {
    if (!w) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    BOUNDARY_OR_FAIL(boundary, boundary_h)
    BoundaryRec& b = w->bounds[boundary];
    w->hb_pos.erase(w->hb_pos.begin() + 3 * b.offset, w->hb_pos.begin() + 3 * (b.offset + b.n));
    w->hb_vel.erase(w->hb_vel.begin() + 3 * b.offset, w->hb_vel.begin() + 3 * (b.offset + b.n));
    b.n = 0;
    b.alive = false;
    b.want_forces = false;
    recompute_offsets(w);
    w->b_dirty = true;
    return SPH_OK;
}

// A coupled collider re-samples its boundary every step (positions.clear(); push(..) — fluids_pipeline.rs:175-245): the
// particle COUNT changes, which sph_boundary_write cannot express.
sph_status sph_boundary_set_particles(sph_world* w, uint32_t boundary_h, const float* pos, const float* vel, size_t n) {
    if (!w || (n && !pos)) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    BOUNDARY_OR_FAIL(boundary, boundary_h)
    BoundaryRec& b = w->bounds[boundary];
    w->hb_pos.erase(w->hb_pos.begin() + 3 * b.offset, w->hb_pos.begin() + 3 * (b.offset + b.n));
    w->hb_vel.erase(w->hb_vel.begin() + 3 * b.offset, w->hb_vel.begin() + 3 * (b.offset + b.n));
    w->hb_pos.insert(w->hb_pos.begin() + 3 * b.offset, pos, pos + 3 * n);
    if (vel) w->hb_vel.insert(w->hb_vel.begin() + 3 * b.offset, vel, vel + 3 * n);
    else w->hb_vel.insert(w->hb_vel.begin() + 3 * b.offset, 3 * n, 0.f);
    b.n = n;
    recompute_offsets(w);
    w->b_dirty = true;
    return SPH_OK;
}

sph_status sph_boundary_count(sph_world* w, uint32_t boundary_h, size_t* n) {
    if (!w || !n) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    BOUNDARY_OR_FAIL(boundary, boundary_h)
    *n = w->bounds[boundary].n;
    return SPH_OK;
}

// Zero-copy read-back for renderers (testbed_plugin.rs:361-376 copies fluid.positions every frame): a DEVICE pointer to the
// fluid's positions / velocities as packed xyz f32 in ORIGINAL index order.  Valid until the next call on this world.
static sph_status fluid_map(sph_world* w, uint32_t fluid_h, bool velocities, const float** dev, size_t* n) {
    FLUID_OR_FAIL(fluid, fluid_h)
    TRY(enter(w));
    if (w->staged) {  // nothing on the device yet: build the device state (what the next step would do first)
        TRY(apply_pending_deletes(w));
        TRY(stage_up(w));
    }
    const FluidRec& f = w->fluids[fluid];
    DBuf<float>& buf = velocities ? w->map_vel : w->map_pos;
    const size_t N = w->N;
    CU(buf.ensure(3 * std::max<size_t>(N, 1)));
    const int c = w->cur;
    LAUNCH(k_export3, N, 256, (uint32_t)N, w->orig[c].p + w->own_begin, (velocities ? w->vel[c].p : w->pos[c].p) + w->own_begin, buf.p);
    CU(cudaStreamSynchronize(w->st));
    *dev = buf.p + 3 * f.offset;
    *n = f.n;
    return SPH_OK;
}
sph_status sph_fluid_map_positions(sph_world* w, uint32_t fluid_h, const float** dev_xyz, size_t* n) {
    if (!w || !dev_xyz || !n) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    return fluid_map(w, fluid_h, false, dev_xyz, n);
}
sph_status sph_fluid_map_velocities(sph_world* w, uint32_t fluid_h, const float** dev_xyz, size_t* n) {
    if (!w || !dev_xyz || !n) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    return fluid_map(w, fluid_h, true, dev_xyz, n);
}

// Replaces the whole particle set of a fluid: positions, velocities, velocity_changes (dfsph_solver.rs:44 — the part of the
// velocity the solver carries between steps) and caller-visible ids; volumes return to the default, IISPH pressures to 0.
// This is what a slab world's plane re-balancing needs (salva_b200/slab.py: particles move between ranks wholesale).
sph_status sph_fluid_replace_particles(sph_world* w, uint32_t fluid_h, const float* pos, const float* vel, const float* vc, const uint32_t* ids,
                                       size_t n) {
    if (!w || (n && !pos)) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    FLUID_OR_FAIL(fluid, fluid_h)
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "particles cannot be replaced from inside a coupling callback");
    TRY(enter(w));
    TRY(stage_down(w));
    FluidRec& f = w->fluids[fluid];
    const size_t at = f.offset, old = f.n;
    const float r = w->desc.particle_radius, pv = r * r * r * (float)(8.0 * 0.8);
    w->h_press.resize(w->h_vol.size(), 0.f);
    w->h_gid.resize(w->h_vol.size());
    auto splice3 = [&](std::vector<float>& v, const float* src) {
        v.erase(v.begin() + 3 * at, v.begin() + 3 * (at + old));
        if (src) v.insert(v.begin() + 3 * at, src, src + 3 * n);
        else v.insert(v.begin() + 3 * at, 3 * n, 0.f);
    };
    splice3(w->h_pos, pos);
    splice3(w->h_vel, vel);
    splice3(w->h_vc, vc);
    w->h_vol.erase(w->h_vol.begin() + at, w->h_vol.begin() + at + old);
    w->h_vol.insert(w->h_vol.begin() + at, n, pv);
    w->h_press.erase(w->h_press.begin() + at, w->h_press.begin() + at + old);
    w->h_press.insert(w->h_press.begin() + at, n, 0.f);
    w->h_gid.erase(w->h_gid.begin() + at, w->h_gid.begin() + at + old);
    {
        std::vector<uint32_t> g(n);
        for (size_t i = 0; i < n; ++i) g[i] = ids ? ids[i] : (uint32_t)i;
        w->h_gid.insert(w->h_gid.begin() + at, g.begin(), g.end());
    }
    f.n = n;
    f.pending_delete.assign(n, 0);
    f.n_pending = 0;
    for (auto& fr : f.forces) elasticity_release(fr);  // a rest pose belongs to the particle set it was captured from
    recompute_offsets(w);
    w->slab.global_valid = false;
    return SPH_OK;
}

// ---- snapshot / restore of the state the solver carries across steps ----------------------------------------------------
// velocity_changes (dfsph_solver.rs:44, carried :704-706), the lagging dt / inv_dt (timestep_manager.rs:29-30), IISPH
// warm-start pressures (iisph_solver.rs:673-677), Becker-2009 rest pose + rotations (becker2009_elasticity.rs:84-135),
// particle ids, volumes, slab planes.  The blob restores into a world with the SAME fluids / forces / boundaries pushed in
// the same order (scene description is the caller's); particle counts may differ from the world's current ones.
namespace {
constexpr uint32_t SNAP_MAGIC = 0x53485053u;  // "SPHS"
struct SnapHeader {
    uint32_t magic, version, solver, n_fluid_slots;
    float dt, inv_dt;
    int32_t slab_lo, slab_hi;
    uint64_t n_particles, total_bytes;
};
struct SnapFluid {
    uint64_t n;
    uint32_t alive, n_forces;
};
struct SnapElastic {
    uint64_t n;
    uint32_t cap0, stride0;
};
struct Writer {
    char* p;
    size_t cap, off = 0;
    void put(const void* src, size_t bytes) {
        if (p && off + bytes <= cap) memcpy(p + off, src, bytes);
        off += bytes;
    }
};
// walks the blob layout; with a null buffer it only measures.  Device-resident pieces (elasticity) are downloaded here.
sph_status snapshot_write(sph_world* w, Writer& wr) {
    SnapHeader h;
    memset(&h, 0, sizeof h);
    h.magic = SNAP_MAGIC;
    h.version = 1;
    h.solver = (uint32_t)w->desc.solver;
    h.n_fluid_slots = (uint32_t)w->fluids.size();
    h.dt = w->dt;
    h.inv_dt = w->inv_dt;
    h.slab_lo = w->slab.lo;
    h.slab_hi = w->slab.hi;
    h.n_particles = w->N;
    const size_t header_at = wr.off;
    wr.put(&h, sizeof h);
    for (auto& f : w->fluids) {
        SnapFluid sf{f.n, f.alive ? 1u : 0u, (uint32_t)f.forces.size()};
        wr.put(&sf, sizeof sf);
    }
    const size_t N = w->N;
    wr.put(w->h_pos.data(), 3 * N * sizeof(float));
    wr.put(w->h_vel.data(), 3 * N * sizeof(float));
    wr.put(w->h_vc.data(), 3 * N * sizeof(float));
    wr.put(w->h_vol.data(), N * sizeof(float));
    wr.put(w->h_press.data(), N * sizeof(float));
    wr.put(w->h_gid.data(), N * sizeof(uint32_t));
    for (auto& f : w->fluids)
        for (auto& fr : f.forces) {
            SnapElastic se{0, 0, 0};
            const ElasticityState* E = fr.elastic;
            if (fr.d.kind == SPH_FORCE_BECKER2009_ELASTICITY && E && E->n) se = SnapElastic{E->n, E->cap0, E->stride0};
            wr.put(&se, sizeof se);
            if (!se.n) continue;
            const size_t n = E->n, nl = (size_t)E->cap0 * E->stride0;
            const size_t bytes = n * sizeof(float4) + n * sizeof(uint32_t) + nl * sizeof(uint32_t) + 9 * n * sizeof(float);
            if (wr.p && wr.off + bytes <= wr.cap) {
                char* dst = wr.p + wr.off;
                CU(cudaMemcpyAsync(dst, E->pos0, n * sizeof(float4), cudaMemcpyDeviceToHost, w->st));
                dst += n * sizeof(float4);
                CU(cudaMemcpyAsync(dst, E->cnt0, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
                dst += n * sizeof(uint32_t);
                CU(cudaMemcpyAsync(dst, E->nbr0, nl * sizeof(uint32_t), cudaMemcpyDeviceToHost, w->st));
                dst += nl * sizeof(uint32_t);
                CU(cudaMemcpyAsync(dst, E->rot, 9 * n * sizeof(float), cudaMemcpyDeviceToHost, w->st));
                CU(cudaStreamSynchronize(w->st));
            }
            wr.off += bytes;
        }
    if (wr.p && header_at + sizeof h <= wr.cap) {
        h.total_bytes = wr.off - header_at;
        memcpy(wr.p + header_at, &h, sizeof h);
    }
    return SPH_OK;
}
}  // namespace

sph_status sph_world_snapshot_size(sph_world* w, size_t* bytes) {
    if (!w || !bytes) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "snapshots cannot be taken from inside a coupling callback");
    TRY(enter(w));
    TRY(apply_pending_deletes(w));
    TRY(stage_down(w));  // host vectors = truth in original order; the next step re-uploads (same results: the sorted order is canonical)
    Writer wr{nullptr, 0};
    TRY(snapshot_write(w, wr));
    *bytes = wr.off;
    return SPH_OK;
}

sph_status sph_world_snapshot_save(sph_world* w, void* buffer, size_t capacity, size_t* written) {
    if (!w || !buffer) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "snapshots cannot be taken from inside a coupling callback");
    TRY(enter(w));
    TRY(apply_pending_deletes(w));
    TRY(stage_down(w));
    Writer wr{static_cast<char*>(buffer), capacity};
    TRY(snapshot_write(w, wr));
    if (written) *written = wr.off;
    if (wr.off > capacity) return w->fail(SPH_ERR_INVALID, "snapshot needs %zu bytes, buffer holds %zu", wr.off, capacity);
    return SPH_OK;
}

sph_status sph_world_snapshot_load(sph_world* w, const void* buffer, size_t length) {
    if (!w || !buffer) return SPH_ERR_INVALID;
    std::lock_guard<std::recursive_mutex> lock(g_mutex);
    if (w->in_coupling) return w->fail(SPH_ERR_INVALID, "snapshots cannot be loaded from inside a coupling callback");
    const char* p = static_cast<const char*>(buffer);
    size_t off = 0;
    auto need = [&](size_t bytes) { return off + bytes <= length; };
    SnapHeader h;
    if (!need(sizeof h)) return w->fail(SPH_ERR_INVALID, "snapshot truncated");
    memcpy(&h, p, sizeof h);
    off += sizeof h;
    if (h.magic != SNAP_MAGIC || h.version != 1) return w->fail(SPH_ERR_INVALID, "not a salva_b200 snapshot (magic %08x version %u)", h.magic, h.version);
    if (h.total_bytes > length) return w->fail(SPH_ERR_INVALID, "snapshot truncated: %llu bytes expected, %zu given", (unsigned long long)h.total_bytes, length);
    if (h.solver != (uint32_t)w->desc.solver || h.n_fluid_slots != w->fluids.size())
        return w->fail(SPH_ERR_INVALID, "snapshot was taken from a differently configured world (solver %u, %u fluids)", h.solver, h.n_fluid_slots);
    std::vector<SnapFluid> sf(h.n_fluid_slots);
    if (!need(sf.size() * sizeof(SnapFluid))) return w->fail(SPH_ERR_INVALID, "snapshot truncated");
    memcpy(sf.data(), p + off, sf.size() * sizeof(SnapFluid));
    off += sf.size() * sizeof(SnapFluid);
    uint64_t total = 0;
    for (size_t k = 0; k < sf.size(); ++k) {
        if ((sf[k].alive != 0) != w->fluids[k].alive || sf[k].n_forces != w->fluids[k].forces.size())
            return w->fail(SPH_ERR_INVALID, "snapshot fluid %zu does not match the world (alive %u, %u forces)", k, sf[k].alive, sf[k].n_forces);
        total += sf[k].n;
    }
    if (total != h.n_particles) return w->fail(SPH_ERR_INVALID, "snapshot particle counts are inconsistent");
    const size_t N = (size_t)h.n_particles;
    if (!need((3 * 3 + 2) * N * sizeof(float) + N * sizeof(uint32_t))) return w->fail(SPH_ERR_INVALID, "snapshot truncated");
    TRY(enter(w));
    TRY(stage_down(w));  // flips the world to "host vectors are the truth"; their content is replaced below
    auto take = [&](void* dst, size_t bytes) {
        memcpy(dst, p + off, bytes);
        off += bytes;
    };
    w->h_pos.resize(3 * N); take(w->h_pos.data(), 3 * N * sizeof(float));
    w->h_vel.resize(3 * N); take(w->h_vel.data(), 3 * N * sizeof(float));
    w->h_vc.resize(3 * N);  take(w->h_vc.data(), 3 * N * sizeof(float));
    w->h_vol.resize(N);     take(w->h_vol.data(), N * sizeof(float));
    w->h_press.resize(N);   take(w->h_press.data(), N * sizeof(float));
    w->h_gid.resize(N);     take(w->h_gid.data(), N * sizeof(uint32_t));
    for (size_t k = 0; k < sf.size(); ++k) {
        w->fluids[k].n = (size_t)sf[k].n;
        w->fluids[k].pending_delete.assign((size_t)sf[k].n, 0);
        w->fluids[k].n_pending = 0;
    }
    recompute_offsets(w);
    w->dt = h.dt;
    w->inv_dt = h.inv_dt;
    if (w->slab.active) {
        w->slab.lo = h.slab_lo;
        w->slab.hi = h.slab_hi;
        w->slab.global_valid = false;
    }
    w->Ntot = w->N;
    w->own_begin = 0;
    for (auto& f : w->fluids)
        for (auto& fr : f.forces) {
            SnapElastic se;
            if (!need(sizeof se)) return w->fail(SPH_ERR_INVALID, "snapshot truncated");
            take(&se, sizeof se);
            elasticity_release(fr);
            if (!se.n) continue;
            const size_t n = (size_t)se.n, nl = (size_t)se.cap0 * se.stride0;
            if (!need(n * sizeof(float4) + n * sizeof(uint32_t) + nl * sizeof(uint32_t) + 9 * n * sizeof(float))) return w->fail(SPH_ERR_INVALID, "snapshot truncated");
            TRY(elasticity_restore(w, fr, n, se.cap0, se.stride0, p + off));
            off += n * sizeof(float4) + n * sizeof(uint32_t) + nl * sizeof(uint32_t) + 9 * n * sizeof(float);
        }
    w->lists_valid = false;
    w->grid_ready = false;
    return SPH_OK;
}

}  // extern "C"
