// sph_kernels.cuh — sm_100a CUDA kernels of the SPH step path.
//
// Data layout (all per-particle arrays are in SORTED order: x-major cell order, z fastest, so the
// 27-cell stencil of a particle is 9 contiguous runs of the sorted arrays):
//   pos4  : x, y, z, mass          (mass = volume * density0 of the particle's fluid, fluid.rs:183-185)
//   vel4  : vx, vy, vz, fluid id   (bit pattern of the fluid index in .w)
//   vc4   : velocity_changes       (dfsph_solver.rs:44)
//   vs4   : v* = vel + vc          (materialised so gather passes read ONE vector per neighbour)
//   bpos4 : boundary x, y, z, volume (dfsph_solver.rs:72-96);  bvel4: boundary velocity, boundary id
// Neighbour lists ("contacts", contacts.rs:83-87) are index-only and column-major:
//   nbr_f[((k / 4) * stride + i) * 4 + k % 4] = sorted index of the k-th fluid neighbour of i (self included,
//   ascending j): groups of 4 contacts are interleaved so a thread fetches 4 indices with one coalesced LDG.128;
//   nbr_b[k * stride + i] likewise (scalar) for boundary particles; W and grad W are recomputed from pos4 in
//   every pass (cheaper than streaming cached 16-byte contacts from HBM: see DESIGN.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sphk {

constexpr int MAX_FLUIDS = 16;
constexpr int MAX_BOUNDARIES = 64;
constexpr float F32_EPS = 1.1920929e-07f;

struct FluidParams {  // per fluid, in __constant__ memory
    float density0;
    uint32_t memberships, filter;
    float mass;  // the particles' common mass when every particle of the fluid has the same volume, else 0
};
struct BoundaryParams {
    uint32_t memberships, filter;
};
struct Consts {
    float h, inv_h, h2;          // h2 = h*h rounded once (contacts.rs:285 `h * h`)
    float sigma;                 // 8 / (pi h^3)            cubic_spline_kernel.rs:18
    float dsigma;                // sigma / h               cubic_spline_kernel.rs:79
    float dsigma6;               // 6 sigma / h
    float g_t2;                  // gradient is zero unless |x_ij|^2 > g_t2 = max(eps^2, (1e-5 h)^2)  (kernel.rs:19 + cubic_spline_kernel.rs:64)
    // DFSPHSolver<KernelDensity, KernelGradient> / IISPHSolver<..> type parameters (dfsph_solver.rs:17-20): 0 = CubicSpline
    // (default, the lean path), 1 = Poly6, 2 = Spiky, 3 = Viscosity; kgen != 0 <=> any of the two is not the cubic spline
    int kw, kg, kgen;
    float poly6_n, spiky_n, visc_n;  // 315/(64 pi h^9), 15/(pi h^6), 15/(2 pi h^3)
    int ox, oy, oz;              // grid origin in cell coordinates (one padding cell each side)
    int nx, ny, nz;
    float h_reach;               // h * (1 + 1e-5): covers every |dx| the f32 test d^2 <= h^2 can accept
    // "row order" (SALVA_B200_XYSUB, one GPU, gather backend 0): x and y are binned `xysub` times finer than h (ox, oy, nx, ny then
    // count BINS), z stays the run direction.  With xysub = 2 and the usual spacing h/2 every (x, y) bin column holds ONE line of
    // particles along z, so the 32 lanes of a warp are 32 consecutive particles of a line and their k-th contacts are consecutive
    // particles of a neighbouring line: a warp-wide gather touches ~4 cache lines instead of ~17 data-pipe wavefronts
    // (profiles/r2_l1tex_wavefront_model.md).  Contact SETS are unchanged (arun clips the rows to the reference's stencil).
    int xysub;
    float xysub_f;
    int ntx, nty, ntz;           // tile grid (sph_tile.cuh): 2 x 2 cell columns x TILE_Z cells per tile
    uint32_t n_fluid, n_bound;   // particle totals (n_fluid counts owned + ghost slots of the sorted arrays)
    uint32_t i_begin, n_owned;   // owned slots [i_begin, i_begin + n_owned): everything on one GPU; the slab between the
                                 // two ghost columns in a multi-GPU world (x-major order keeps ghosts at both ends)
    uint32_t stride;             // neighbour-list column stride (>= n_fluid, multiple of 32)
    uint32_t cap_f, cap_b;       // list capacities (rows)
    int n_fluids, n_bounds;      // object counts
    FluidParams fluids[MAX_FLUIDS];
    BoundaryParams bounds[MAX_BOUNDARIES];
};

__constant__ Consts C;

// ------------------------------------------------------------------------------------------------
// geometry helpers
// ------------------------------------------------------------------------------------------------
// hgrid.rs:41-52: cell = floor(x / h), IEEE division exactly as the reference.
__device__ __forceinline__ int cell_coord(float x) { return (int)floorf(__fdiv_rn(x, C.h)); }

__device__ __forceinline__ int cell_id(int cx, int cy, int cz) { return ((cx - C.ox) * C.ny + (cy - C.oy)) * C.nz + (cz - C.oz); }
// Row order (Consts::xysub): bin of a coordinate, reference cell floor(v / h) (same IEEE division) times `sub` plus the slice
// inside the cell.  Monotone non-decreasing in v (correctly rounded division, exact q - floor(q)), and every bin lies inside
// ONE reference cell.
__device__ __forceinline__ int abin(float v, int sub, float subf) {
    const float q = __fdiv_rn(v, C.h), fl = floorf(q);
    return (int)fl * sub + min(sub - 1, (int)((q - fl) * subf));
}
// Bins [lo, hi] of the row a particle at v (reference cell c) has to scan: everything within h_reach of v, clipped to the three
// reference cells c-1..c+1 the reference's 27-cell stencil looks at.  A pair that passes the f32 test d^2 <= h^2 has
// |v_i - v_j| <= h (1 + 2^-22) < h_reach; the bounds are rounded outwards, and abin is monotone, so no accepted pair of
// adjacent reference cells is ever cut off: the contact sets stay exactly the reference's.
__device__ __forceinline__ void arun(float v, int c, int sub, float subf, int& lo, int& hi) {
    lo = max(abin(__fsub_rd(v, C.h_reach), sub, subf), (c - 1) * sub);
    hi = min(abin(__fadd_ru(v, C.h_reach), sub, subf), (c + 2) * sub - 1);
}

// contacts.rs:285,322,366: (dx*dx + dy*dy) + dz*dz <= h*h with no contraction (rustc never fuses).
__device__ __forceinline__ float dist2_exact(float dx, float dy, float dz) {
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
// cubic_spline_kernel.rs:12-33: W(r) for q = r/h.
__device__ __forceinline__ float kernel_w(float r) {
    float q = r * C.inv_h;
    float q2 = q * q;
    float a = 1.0f + (q2 * q - q2) * 6.0f;
    float t = 1.0f - q;
    float b = (t * t * t) * 2.0f;
    float rhs = q <= 0.5f ? a : (q <= 1.0f ? b : 0.0f);
    return C.sigma * rhs;
}
// MUFU.RSQ without the denormal-rescue sequence rsqrtf() compiles to (3 extra instructions per contact): operands
// here are squared distances >= g_t2 ~ 1e-14 or exactly 0 (self contact: +inf, masked by the d2 > g_t2 select).
__device__ __forceinline__ float rsqrt_ftz(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// kernel/poly6_kernel.rs:12-40, spiky_kernel.rs:12-40, viscosity_kernel.rs:12-51 (dim3), evaluated like the reference
// (IEEE sqrt / division, powi as repeated products); kind 0 falls through to the cubic spline.
__device__ __forceinline__ float kernel_w_kind(int kind, float r) {
    const float h = C.h;
    if (kind == 1) {
        const float t = h * h - r * r;
        return r <= h ? C.poly6_n * (t * t * t) : 0.f;
    }
    if (kind == 2) {
        const float t = h - r;
        return r <= h ? C.spiky_n * (t * t * t) : 0.f;
    }
    if (kind == 3) {
        if (!(r > 0.f && r <= h)) return 0.f;
        const float rr_hh = __fdiv_rn(r * r, h * h);
        return C.visc_n * (rr_hh * (1.0f - __fdiv_rn(r, 2.0f * h)) + __fdiv_rn(h, 2.0f * r) - 1.0f);
    }
    return kernel_w(r);
}
__device__ __forceinline__ float kernel_dw_kind(int kind, float r) {  // scalar_apply_diff
    const float h = C.h;
    if (kind == 1) {
        const float t = h * h - r * r;
        return r <= h ? C.poly6_n * (t * t) * r * -6.0f : 0.f;
    }
    if (kind == 2) {
        const float t = h - r;
        return r <= h ? -C.spiky_n * (t * t) * 3.0f : 0.f;
    }
    if (kind == 3) {
        if (!(r > 0.f && r <= h)) return 0.f;
        const float rr = r * r, hh = h * h;
        return C.visc_n * (__fdiv_rn(-3.0f * rr, 2.0f * (hh * h)) + __fdiv_rn(2.0f * r, hh) - __fdiv_rn(h, 2.0f * rr));
    }
    const float q = __fdiv_rn(r, h);  // cubic_spline_kernel.rs:55-80
    const float t = 1.0f - q;
    const float rhs = (q > 1.0f || q <= 1.0e-5f) ? 0.f : (q <= 0.5f ? (q * 3.0f - 2.0f) * q * 6.0f : -t * t * 6.0f);
    return __fdiv_rn(C.sigma * rhs, h);
}

// The solver's KernelDensity / KernelGradient are COMPILE-TIME type parameters in the reference (monomorphised per solver
// type).  Here likewise: libsalva_b200.so is built with SPH_GENERIC_KERNELS = 0 (cubic spline only, no branch in the pair
// evaluation: the uniform `if (C.kgen)` inside the 4-way unrolled contact loops cost 6-8 % of the whole step,
// profiles/r2_exp_a_variants.md); libsalva_b200_kernels.so is the same source built with SPH_GENERIC_KERNELS = 1 and
// serves worlds whose solver names Poly6 / Spiky / Viscosity kernels.  Same C ABI in both.
#ifndef SPH_GENERIC_KERNELS
#define SPH_GENERIC_KERNELS 0
#endif
__device__ __forceinline__ float2 pair_generic(float d2, int need_w, int need_g) {
    const float r = __fsqrt_rn(d2);
    float2 o;
    o.x = need_w ? kernel_w_kind(C.kw, r) : 0.f;
    o.y = (need_g && d2 > F32_EPS * F32_EPS) ? __fdiv_rn(kernel_dw_kind(C.kg, r), r) : 0.f;
    return o;
}

struct Pair {        // geometry of one (i, j) contact
    float dx, dy, dz;  // x_i - x_j
    float d2, r;
    float w;           // contact.weight
    float g;           // contact.gradient = g * (dx, dy, dz)
};
// CUBIC_ONLY: force plugins with their OWN kernel type parameters (Becker2009Elasticity<CubicSplineKernel, ..>) do not
// follow the solver's kernels.
template <bool NEED_W, bool NEED_G, bool CUBIC_ONLY = false>
__device__ __forceinline__ Pair make_pair(const float4& pi, const float4& pj) {
    Pair p;
    p.dx = pi.x - pj.x;
    p.dy = pi.y - pj.y;
    p.dz = pi.z - pj.z;
    p.d2 = fmaf(p.dz, p.dz, fmaf(p.dy, p.dy, p.dx * p.dx));
    if (SPH_GENERIC_KERNELS && !CUBIC_ONLY && C.kgen) {  // non-default solver kernels: uniform branch, off the default path
        const float2 o = pair_generic(p.d2, NEED_W, NEED_G);
        p.r = __fsqrt_rn(p.d2);
        p.w = o.x;
        p.g = o.y;
        return p;
    }
    // Lean evaluation (about half the instructions of a guarded rsqrtf one): contacts come from lists built with
    // d^2 <= h^2, so q <= 1 up to rounding (where (1 - q)^2 ~ 1e-14 anyway), and the two "zero gradient" guards of the
    // reference (|x_ij|^2 > eps^2, q > 1e-5) collapse into one select on d2.  d2 == 0 gives inv_r = +inf and NaNs in
    // r / q, all discarded by the selects (never multiplied).
    const float inv_r = rsqrt_ftz(p.d2);
    const bool nz = p.d2 > C.g_t2;
    p.r = nz ? p.d2 * inv_r : 0.f;
    const float q = p.r * C.inv_h;
    const float t = 1.0f - q;
    const bool inner = q <= 0.5f;
    if (NEED_W) {
        const float q2 = q * q;
        const float a = fmaf(fmaf(q2, q, -q2), 6.0f, 1.0f);
        const float b = (t * t) * (t * 2.0f);
        p.w = C.sigma * (inner ? a : b);
    } else {
        p.w = 0.f;
    }
    if (NEED_G) {
        const float a = fmaf(q, 3.0f, -2.0f) * q;
        const float b = -t * t;
        p.g = nz ? (C.dsigma6 * inv_r) * (inner ? a : b) : 0.f;
    } else {
        p.g = 0.f;
    }
    return p;
}

// index of the owned particle handled by this thread (returns from the kernel when out of range)
#define SPH_OWNED_INDEX(i)                                   \
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;      \
    if (i >= C.n_owned) return;                              \
    i += C.i_begin;

__device__ __forceinline__ uint32_t fid_of(const float4& v) { return __float_as_uint(v.w); }

// interaction_groups.rs:64-69
__device__ __forceinline__ bool groups_test(uint32_t m1, uint32_t f1, uint32_t m2, uint32_t f2) {
    return (m1 & f2) != 0 && (m2 & f1) != 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Deterministic block sum (fixed tree); result valid in thread 0.
__device__ __forceinline__ float block_sum(float v, float* sm /* >= 32 floats */) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sm[wid] = v;
    __syncthreads();
    if (wid == 0) {
        int nw = (blockDim.x + 31) >> 5;
        v = lane < nw ? sm[lane] : 0.f;
        v = warp_sum(v);
    }
    return v;
}

// ------------------------------------------------------------------------------------------------
// K0: bounds (cell-coordinate AABB) — replaces the unbounded HashMap of hgrid.rs:22-25 by a dense
// grid over the occupied region.
// ------------------------------------------------------------------------------------------------
__global__ void k_bounds(const float4* __restrict__ pos, uint32_t n, int* __restrict__ out /* minx,miny,minz,maxx,maxy,maxz,bad */) {
    int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
    int bad = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 p = pos[i];
        float c[3] = {floorf(__fdiv_rn(p.x, C.h)), floorf(__fdiv_rn(p.y, C.h)), floorf(__fdiv_rn(p.z, C.h))};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(fabsf(c[a]) < 1.0e9f)) { bad = 1; continue; }  // NaN / inf / absurd coordinates
            int v = (int)c[a];
            mn[a] = min(mn[a], v);
            mx[a] = max(mx[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        for (int o = 16; o > 0; o >>= 1) {
            mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
    }
    bad = __any_sync(0xffffffffu, bad);
    __shared__ int s_mn[3][8], s_mx[3][8], s_bad[8];
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            s_mn[a][wid] = mn[a];
            s_mx[a][wid] = mx[a];
        }
        s_bad[wid] = bad;
    }
    __syncthreads();
    if (threadIdx.x < 3) {  // one atomic pair per axis per block
        int a = threadIdx.x, nw = (blockDim.x + 31) >> 5;
        int m0 = INT_MAX, m1 = INT_MIN;
        for (int k = 0; k < nw; ++k) {
            m0 = min(m0, s_mn[a][k]);
            m1 = max(m1, s_mx[a][k]);
        }
        atomicMin(&out[a], m0);
        atomicMax(&out[3 + a], m1);
        if (a == 0) {
            int b = 0;
            for (int k = 0; k < nw; ++k) b |= s_bad[k];
            if (b) atomicOr(&out[6], 1);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K1: counting sort by cell (replaces HGrid::insert hgrid.rs:60-63 / insert_*_to_grid contacts.rs:133-151
// and the dead z_order.rs sort).
// ------------------------------------------------------------------------------------------------
// dead (optional): dead[i] != 0 for i < n_dead marks an input slot that must not enter the sorted arrays (a particle that left
// this rank's slab, sph_slab.inl); such slots get cid = 0xFFFFFFFF and are skipped by the scatter.
__global__ void k_cell_hist(const float4* __restrict__ pos, uint32_t n, uint32_t* __restrict__ cid, uint32_t* __restrict__ rank,
                            uint32_t* __restrict__ count, const uint32_t* __restrict__ dead, uint32_t n_dead) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (dead && i < n_dead && dead[i]) {
        cid[i] = 0xFFFFFFFFu;
        return;
    }
    float4 p = pos[i];
    uint32_t id = (uint32_t)cell_id(cell_coord(p.x), cell_coord(p.y), cell_coord(p.z));
    cid[i] = id;
    rank[i] = atomicAdd(&count[id], 1u);
}

// row order (Consts::xysub > 1): x and y binned finer than h
__global__ void k_cell_hist_xy(const float4* __restrict__ pos, uint32_t n, uint32_t* __restrict__ cid, uint32_t* __restrict__ rank,
                               uint32_t* __restrict__ count) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = pos[i];
    uint32_t id = (uint32_t)cell_id(abin(p.x, C.xysub, C.xysub_f), abin(p.y, C.xysub, C.xysub_f), cell_coord(p.z));
    cid[i] = id;
    rank[i] = atomicAdd(&count[id], 1u);
}

__global__ void k_cell_scatter(uint32_t n, const uint32_t* __restrict__ cid, const uint32_t* __restrict__ rank,
                               const uint32_t* __restrict__ start, uint32_t* __restrict__ perm) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t c = cid[i];
    if (c == 0xFFFFFFFFu) return;
    perm[start[c] + rank[i]] = i;
}

// Deterministic mode: atomics hand out in-cell ranks in arbitrary order; sort each cell's slice of perm so the sorted
// order (and every f32 summation order downstream) is reproducible.  The in-cell order is CANONICAL — ascending
// (fluid, particle id), a pure function of the particle set — so a world restored from a snapshot, a world whose state
// went through the host, and the ranks of a slab decomposition (ghost columns!) all see the same order and produce
// bit-identical sums.  key == nullptr (boundaries): ascending previous slot, i.e. insertion order.
__device__ __forceinline__ unsigned long long sort_key(uint32_t src, const uint32_t* __restrict__ gid, const float4* __restrict__ vel) {
    if (!gid) return src;
    const uint32_t f = vel ? fid_of(vel[src]) : 0u;
    return ((unsigned long long)f << 32) | gid[src];
}
__global__ void k_cell_sort(uint32_t ncell, const uint32_t* __restrict__ start, uint32_t* __restrict__ perm, const uint32_t* __restrict__ gid,
                            const float4* __restrict__ vel) {
    uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    uint32_t s = start[c], e = start[c + 1];
    for (uint32_t a = s + 1; a < e; ++a) {
        const uint32_t v = perm[a];
        const unsigned long long kv = sort_key(v, gid, vel);
        uint32_t b = a;
        while (b > s) {
            const uint32_t u = perm[b - 1];
            const unsigned long long ku = sort_key(u, gid, vel);
            if (ku < kv || (ku == kv && u < v)) break;
            perm[b] = u;
            --b;
        }
        perm[b] = v;
    }
}

struct GatherSet {  // arrays reordered together by the counting sort
    const float4* in4[6];
    float4* out4[6];
    const uint32_t* in1[4];
    uint32_t* out1[4];
    int n4, n1;
};
__global__ void k_gather(uint32_t n, const uint32_t* __restrict__ perm, GatherSet g) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t src = perm[s];
#pragma unroll
    for (int a = 0; a < 6; ++a)
        if (a < g.n4) g.out4[a][s] = g.in4[a][src];
#pragma unroll
    for (int a = 0; a < 4; ++a)
        if (a < g.n1) g.out1[a][s] = g.in1[a][src];
}

// exclusive scan, 2048 items per block (256 threads x 8)
constexpr int SCAN_T = 256, SCAN_I = 8, SCAN_B = SCAN_T * SCAN_I;
__global__ void k_scan_block(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t warp_tot[SCAN_T / 32];
    uint32_t base = blockIdx.x * SCAN_B + threadIdx.x * SCAN_I;
    uint32_t v[SCAN_I];
    uint32_t tsum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_I; ++k) {
        v[k] = (base + k < n) ? in[base + k] : 0u;
        tsum += v[k];
    }
    uint32_t incl = tsum;
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < SCAN_T / 32 ? warp_tot[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        if (lane < SCAN_T / 32) warp_tot[lane] = wi - w;
        if (lane == SCAN_T / 32 - 1 && block_sums) block_sums[blockIdx.x] = wi;
    }
    __syncthreads();
    uint32_t run = warp_tot[wid] + incl - tsum;
#pragma unroll
    for (int k = 0; k < SCAN_I; ++k) {
        if (base + k < n) out[base + k] = run;
        run += v[k];
    }
}
__global__ void k_scan_add(uint32_t* __restrict__ out, uint32_t n, const uint32_t* __restrict__ block_offsets) {
    uint32_t i = blockIdx.x * SCAN_B + threadIdx.x;
    uint32_t off = block_offsets[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_I; ++k) {
        uint32_t j = i + k * SCAN_T;
        if (j < n) out[j] += off;
    }
}

// K-way exclusive scan: the same 2048-item blocks, K independent arrays scanned by one launch (slab prologue: the five
// classification flag arrays are compacted together instead of by five 3-kernel scans).
template <int K>
struct ScanSet {
    uint32_t* a[K];
};
template <int K>
__global__ void k_scanK_block(ScanSet<K> io, uint32_t n, ScanSet<K> block_sums) {
    __shared__ uint32_t warp_tot[K][SCAN_T / 32];
    const uint32_t base = blockIdx.x * SCAN_B + threadIdx.x * SCAN_I;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < K; ++a) {
        uint32_t v[SCAN_I];
        uint32_t tsum = 0;
#pragma unroll
        for (int k = 0; k < SCAN_I; ++k) {
            v[k] = (base + k < n) ? io.a[a][base + k] : 0u;
            tsum += v[k];
        }
        uint32_t incl = tsum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_tot[a][wid] = incl;
        __syncthreads();
        if (wid == 0) {
            uint32_t w = lane < SCAN_T / 32 ? warp_tot[a][lane] : 0u;
            uint32_t wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += t;
            }
            if (lane < SCAN_T / 32) warp_tot[a][lane] = wi - w;
            if (lane == SCAN_T / 32 - 1 && block_sums.a[a]) block_sums.a[a][blockIdx.x] = wi;
        }
        __syncthreads();
        uint32_t run = warp_tot[a][wid] + incl - tsum;
#pragma unroll
        for (int k = 0; k < SCAN_I; ++k) {
            if (base + k < n) io.a[a][base + k] = run;
            run += v[k];
        }
    }
}
template <int K>
__global__ void k_scanK_add(ScanSet<K> io, uint32_t n, ScanSet<K> block_offsets) {
    uint32_t i = blockIdx.x * SCAN_B + threadIdx.x;
#pragma unroll
    for (int a = 0; a < K; ++a) {
        uint32_t off = block_offsets.a[a][blockIdx.x];
#pragma unroll
        for (int k = 0; k < SCAN_I; ++k) {
            uint32_t j = i + k * SCAN_T;
            if (j < n) io.a[a][j] += off;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2: neighbour search (contacts.rs:154-400).  One thread per particle walks the 9 z-runs of its
// 27-cell stencil and keeps the indices that pass the reference's exact `d^2 <= h*h` test.
// Only ~15 % of the candidates pass, but in a warp SOME lane passes for nearly every candidate, so a store inside the
// candidate loop is executed (predicated off) by the whole warp almost every iteration.  The candidate loop therefore
// only records hits in a 32-bit mask per chunk of 32 candidates; the (short) emit loop then walks the set bits in
// ascending order, which keeps every list in the same order as a plain scan.
// ------------------------------------------------------------------------------------------------
template <class Accept, class Emit>
__device__ __forceinline__ void scan_run(const float4& pi, const float4* __restrict__ P, uint32_t s, uint32_t e, Accept accept, Emit emit) {
    for (uint32_t base = s; base < e; base += 32u) {
        const uint32_t n = min(32u, e - base);
        const float4* __restrict__ q = P + base;
        uint32_t rej = 0u;  // candidate t of the chunk ends up in bit n - 1 - t; set = rejected
#pragma unroll 4
        for (uint32_t t = 0; t < n; ++t) {
            const float4 pj = __ldg(&q[t]);
            const float d2 = dist2_exact(pi.x - pj.x, pi.y - pj.y, pi.z - pj.z);
            // d2 <= h*h  <=>  the sign bit of (h*h - d2) is clear (a float difference is zero only for equal operands;
            // NaN positions never get here, k_bounds rejects them): shift that bit into the mask with one funnel shift
            rej = __funnelshift_l(__float_as_uint(__fsub_rn(C.h2, d2)), rej, 1);
        }
        uint32_t m = ~rej & (n == 32u ? 0xffffffffu : (1u << n) - 1u);
        while (m) {
            const uint32_t b = 31u - (uint32_t)__clz((int)m);  // highest set bit = earliest candidate
            m &= ~(1u << b);
            const uint32_t j = base + (n - 1u - b);
            if (accept(j)) emit(j);
        }
    }
}

// Minimum blocks per SM: left to itself ptxas gives these kernels 40 registers and spills a cell coordinate across the slow
// path of the IEEE division in cell_coord(); the bounds below keep every instantiation spill-free at no higher register count.
template <bool MULTI>
__global__ void __launch_bounds__(128, MULTI ? 12 : 10)
k_neighbors(const float4* __restrict__ pos, const float4* __restrict__ vel, const uint32_t* __restrict__ cstart,
            const float4* __restrict__ bpos, const float4* __restrict__ bvel, const uint32_t* __restrict__ bstart,
            uint32_t* __restrict__ nbr_f, uint32_t* __restrict__ nbr_b, uint32_t* __restrict__ cnt_f, uint32_t* __restrict__ cnt_b,
            uint32_t* __restrict__ maxcnt /* [0]=fluid,[1]=boundary */) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t nf = 0, nb = 0;
    const bool owned = i < C.n_owned;
    i += C.i_begin;
    if (owned) {
        float4 pi = pos[i];
        uint32_t fi = MULTI ? fid_of(vel[i]) : 0u;
        int cx = cell_coord(pi.x), cy = cell_coord(pi.y), cz = cell_coord(pi.z);
        const int zlo = cz - 1, zhi = cz + 1;
        // entry k of particle i lives at ((k >> 2) * stride + i) * 4 + (k & 3): walked with a running pointer
        uint32_t* wp = nbr_f + (size_t)i * 4;                  // slot 0 of group 0 of this particle's column
        const size_t gstep = (size_t)C.stride * 4 - 4;         // from behind slot 3 of a group to slot 0 of the next one
        for (int ax = -1; ax <= 1; ++ax)
            for (int ay = -1; ay <= 1; ++ay) {
                const int lo = cell_id(cx + ax, cy + ay, zlo), hi = lo + (zhi - zlo) + 1;
                scan_run(
                    pi, pos, cstart[lo], cstart[hi],
                    [&](uint32_t j) {
                        if (!MULTI) return true;
                        uint32_t fj = fid_of(__ldg(&vel[j]));  // contacts.rs:355-362: different fluids need the groups test
                        return fi == fj || groups_test(C.fluids[fi].memberships, C.fluids[fi].filter, C.fluids[fj].memberships, C.fluids[fj].filter);
                    },
                    [&](uint32_t j) {
                        // (one 4-byte store per hit: collecting four hits in registers and storing 16-byte groups was measured
                        //  SLOWER, 1.66 -> 1.80 ms at C3 — the shift-in costs more issue slots than the stores save)
                        if (nf < C.cap_f) *wp = j;
                        ++nf;
                        ++wp;
                        if ((nf & 3u) == 0u) wp += gstep;
                    });
                if (C.n_bound)
                    scan_run(
                        pi, bpos, bstart[lo], bstart[hi],
                        [&](uint32_t j) {  // contacts.rs:347-352
                            uint32_t bj = fid_of(__ldg(&bvel[j]));
                            return groups_test(C.fluids[fi].memberships, C.fluids[fi].filter, C.bounds[bj].memberships, C.bounds[bj].filter);
                        },
                        [&](uint32_t j) {
                            if (nb < C.cap_b) nbr_b[(size_t)nb * C.stride + i] = j;
                            ++nb;
                        });
            }
        for (uint32_t t = nf; t < ((nf + 3u) & ~3u) && t < C.cap_f; ++t) *wp++ = i;  // pad the last group
        cnt_f[i] = nf;
        cnt_b[i] = nb;
    }
    uint32_t mf = nf, mb = nb;
    for (int o = 16; o > 0; o >>= 1) {
        mf = max(mf, __shfl_xor_sync(0xffffffffu, mf, o));
        mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (mf) atomicMax(&maxcnt[0], mf);
        if (mb) atomicMax(&maxcnt[1], mb);
    }
}

// Row order (Consts::xysub > 1): the same search over the bin rows within reach in x and y (5 x 5 rows of width h / 2 at xysub = 2
// instead of 3 x 3 of width h; arun() clips to the reference's stencil, so the contact sets are the reference's).  A separate kernel so that
// the default path above stays byte for byte what was validated.
template <bool MULTI>
__global__ void __launch_bounds__(128, MULTI ? 0 : 10)  // (see k_neighbors; 0: no minimum)
k_neighbors_xy(const float4* __restrict__ pos, const float4* __restrict__ vel, const uint32_t* __restrict__ cstart,
               const float4* __restrict__ bpos, const float4* __restrict__ bvel, const uint32_t* __restrict__ bstart,
               uint32_t* __restrict__ nbr_f, uint32_t* __restrict__ nbr_b, uint32_t* __restrict__ cnt_f, uint32_t* __restrict__ cnt_b,
               uint32_t* __restrict__ maxcnt /* [0]=fluid,[1]=boundary */) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t nf = 0, nb = 0;
    const bool owned = i < C.n_owned;
    i += C.i_begin;
    if (owned) {
        float4 pi = pos[i];
        uint32_t fi = MULTI ? fid_of(vel[i]) : 0u;
        const int cx = cell_coord(pi.x), cy = cell_coord(pi.y), cz = cell_coord(pi.z);
        int xlo, xhi, ylo, yhi;
        arun(pi.x, cx, C.xysub, C.xysub_f, xlo, xhi);
        arun(pi.y, cy, C.xysub, C.xysub_f, ylo, yhi);
        const int zlo = cz - 1, zhi = cz + 1;
        uint32_t* wp = nbr_f + (size_t)i * 4;
        const size_t gstep = (size_t)C.stride * 4 - 4;
        for (int bx = xlo; bx <= xhi; ++bx)
            for (int by = ylo; by <= yhi; ++by) {
                const int lo = cell_id(bx, by, zlo), hi = lo + (zhi - zlo) + 1;
                scan_run(
                    pi, pos, cstart[lo], cstart[hi],
                    [&](uint32_t j) {
                        if (!MULTI) return true;
                        uint32_t fj = fid_of(__ldg(&vel[j]));
                        return fi == fj || groups_test(C.fluids[fi].memberships, C.fluids[fi].filter, C.fluids[fj].memberships, C.fluids[fj].filter);
                    },
                    [&](uint32_t j) {
                        if (nf < C.cap_f) *wp = j;
                        ++nf;
                        ++wp;
                        if ((nf & 3u) == 0u) wp += gstep;
                    });
                if (C.n_bound)
                    scan_run(
                        pi, bpos, bstart[lo], bstart[hi],
                        [&](uint32_t j) {
                            uint32_t bj = fid_of(__ldg(&bvel[j]));
                            return groups_test(C.fluids[fi].memberships, C.fluids[fi].filter, C.bounds[bj].memberships, C.bounds[bj].filter);
                        },
                        [&](uint32_t j) {
                            if (nb < C.cap_b) nbr_b[(size_t)nb * C.stride + i] = j;
                            ++nb;
                        });
            }
        for (uint32_t t = nf; t < ((nf + 3u) & ~3u) && t < C.cap_f; ++t) *wp++ = i;  // pad the last group
        cnt_f[i] = nf;
        cnt_b[i] = nb;
    }
    uint32_t mf = nf, mb = nb;
    for (int o = 16; o > 0; o >>= 1) {
        mf = max(mf, __shfl_xor_sync(0xffffffffu, mf, o));
        mb = max(mb, __shfl_xor_sync(0xffffffffu, mb, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (mf) atomicMax(&maxcnt[0], mf);
        if (mb) atomicMax(&maxcnt[1], mb);
    }
}
// boundary volumes in row order: every bin of the 3 x 3 x 3 reference cells around the particle
__global__ void __launch_bounds__(128)
k_boundary_volumes_xy(const float4* __restrict__ bpos, const float4* __restrict__ bvel, const uint32_t* __restrict__ bstart, float* __restrict__ bvol,
                      unsigned long long* __restrict__ ncontacts, int* __restrict__ err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cnt = 0;
    if (i < C.n_bound) {
        float4 pi = bpos[i];
        uint32_t bi = fid_of(bvel[i]);
        const int cx = cell_coord(pi.x), cy = cell_coord(pi.y), cz = cell_coord(pi.z);
        float den = 0.f;
        for (int bx = (cx - 1) * C.xysub; bx < (cx + 2) * C.xysub; ++bx)
            for (int by = (cy - 1) * C.xysub; by < (cy + 2) * C.xysub; ++by) {
                const int base = cell_id(bx, by, cz - 1);
                const uint32_t s = bstart[base], e = bstart[base + 3];
                for (uint32_t j = s; j < e; ++j) {
                    float4 pj = __ldg(&bpos[j]);
                    float dx = pi.x - pj.x, dy = pi.y - pj.y, dz = pi.z - pj.z;
                    float d2 = dist2_exact(dx, dy, dz);
                    if (d2 <= C.h2) {
                        uint32_t bj = fid_of(__ldg(&bvel[j]));
                        if (bi == bj || groups_test(C.bounds[bi].memberships, C.bounds[bi].filter, C.bounds[bj].memberships, C.bounds[bj].filter)) {
                            den += C.kgen ? kernel_w_kind(C.kw, __fsqrt_rn(d2)) : kernel_w(sqrtf(d2));
                            ++cnt;
                        }
                    }
                }
            }
        if (den == 0.f) atomicOr(err, 1);
        bvol[i] = 1.0f / den;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(ncontacts, (unsigned long long)cnt);
}

// a4: compute_boundary_volumes dfsph_solver.rs:72-96 — vol_b = 1 / sum_{b'} W_bb' over boundary-boundary
// contacts (same boundary, or other boundaries passing the groups test; self included).
__global__ void __launch_bounds__(128)
k_boundary_volumes(const float4* __restrict__ bpos, const float4* __restrict__ bvel, const uint32_t* __restrict__ bstart, float* __restrict__ bvol,
                   unsigned long long* __restrict__ ncontacts, int* __restrict__ err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t cnt = 0;
    if (i < C.n_bound) {
        float4 pi = bpos[i];
        uint32_t bi = fid_of(bvel[i]);
        int cx = cell_coord(pi.x), cy = cell_coord(pi.y), cz = cell_coord(pi.z);
        float den = 0.f;
        for (int ax = -1; ax <= 1; ++ax)
            for (int ay = -1; ay <= 1; ++ay) {
                int base = cell_id(cx + ax, cy + ay, cz - 1);  // the three cells cz-1..cz+1
                uint32_t s = bstart[base], e = bstart[base + 3];
                for (uint32_t j = s; j < e; ++j) {
                    float4 pj = __ldg(&bpos[j]);
                    float dx = pi.x - pj.x, dy = pi.y - pj.y, dz = pi.z - pj.z;
                    float d2 = dist2_exact(dx, dy, dz);
                    if (d2 <= C.h2) {
                        uint32_t bj = fid_of(__ldg(&bvel[j]));
                        if (bi == bj || groups_test(C.bounds[bi].memberships, C.bounds[bi].filter, C.bounds[bj].memberships, C.bounds[bj].filter)) {
                            den += C.kgen ? kernel_w_kind(C.kw, __fsqrt_rn(d2)) : kernel_w(sqrtf(d2));
                            ++cnt;
                        }
                    }
                }
            }
        if (den == 0.f) atomicOr(err, 1);  // assert!(!denominator.is_zero()) dfsph_solver.rs:92
        bvol[i] = 1.0f / den;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(ncontacts, (unsigned long long)cnt);
}
__global__ void k_set_w(uint32_t n, float4* __restrict__ a, const float* __restrict__ w) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i].w = w[i];
}

// ------------------------------------------------------------------------------------------------
// Error reduction + elementwise (streaming) kernels.  The neighbour-gather passes live in sph_passes.cuh
// (default backend) and sph_tile.cuh (tile/TMA backend).
// ------------------------------------------------------------------------------------------------
// One block per fluid: fixed-order sum of the per-block partials.
__global__ void k_reduce_partials(const float* __restrict__ partial, uint32_t nblocks, int n_fluids, float* __restrict__ out) {
    __shared__ float sm[32];
    int f = blockIdx.x;
    float s = 0.f;
    for (uint32_t b = threadIdx.x; b < nblocks; b += blockDim.x) s += partial[(size_t)b * n_fluids + f];
    s = block_sum(s, sm);
    if (threadIdx.x == 0) out[f] = s;
}

#ifndef SPH_PASS_T
#define SPH_PASS_T 128
#endif
#ifndef SPH_PASS_MINB
#define SPH_PASS_MINB 9   // Jacobi-loop / density kernels: 56 registers, 9 blocks of 128 per SM (measured best, profiles/r1_v2_*)
#endif
#ifndef SPH_FORCE_MINB
#define SPH_FORCE_MINB 8  // force kernels gather more per contact: 64 registers avoid spills
#endif
constexpr int PASS_T = SPH_PASS_T;  // threads per block of the gather passes

// The fluid reorder fused with k_make_vstar: the sorted pos / vel / vc are in registers anyway, so v* = vel + vc and the packed
// gather records are written by the same pass (saves re-reading 48 B per particle and a launch).  g.in4 / out4 [0..2] = pos, vel, vc.
__global__ void k_gather_vstar(uint32_t n, const uint32_t* __restrict__ perm, GatherSet g, float4* __restrict__ vs, float4* __restrict__ pvx,
                               float2* __restrict__ vyz) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t src = perm[s];
    const float4 p = g.in4[0][src], v = g.in4[1][src], c = g.in4[2][src];
    g.out4[0][s] = p;
    g.out4[1][s] = v;
    g.out4[2][s] = c;
#pragma unroll
    for (int a = 0; a < 4; ++a)
        if (a < g.n1) g.out1[a][s] = g.in1[a][src];
    const float sx = v.x + c.x, sy = v.y + c.y, sz = v.z + c.z;
    vs[s] = make_float4(sx, sy, sz, 0.f);
    if (pvx) {
        pvx[s] = make_float4(p.x, p.y, p.z, sx);
        vyz[s] = make_float2(sy, sz);
    }
}

// v* = vel + vc after the reorder (the divergence solve works on vel + vc carried over from the previous step, Appendix A.3.2)
__global__ void k_make_vstar(const float4* __restrict__ vel, const float4* __restrict__ vc, float4* __restrict__ vs, const float4* __restrict__ pos,
                             float4* __restrict__ pvx, float2* __restrict__ vyz) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_fluid) return;
    float4 v = vel[i], c = vc[i];
    float sx = v.x + c.x, sy = v.y + c.y, sz = v.z + c.z;
    vs[i] = make_float4(sx, sy, sz, 0.f);
    if (pvx) {  // uniform-mass packed records (sph_passes.cuh)
        float4 p = pos[i];
        pvx[i] = make_float4(p.x, p.y, p.z, sx);
        vyz[i] = make_float2(sy, sz);
    }
}

// a10: update_velocities dfsph_solver.rs:422-430 + zero vc :689-691 + acc = gravity (predict_advection :574-578).
// vel += vc is written as vel = v*: v* was materialised as vel + vc by the producer, so the result is bitwise the
// same for owned particles, and ghost particles (multi-GPU) only carry an up-to-date v*.
// xs (optional): XSPH sums of the divergence loop's last evaluation (k_vel_divergence_xsph_u): acc = g + xs * inv_dt,
// rounded like k_force_xsph's `acc += f * inv_dt` on top of the gravity written here.
__global__ void k_fold_velocities(float4* __restrict__ vel, float4* __restrict__ vc, const float4* __restrict__ vs, float4* __restrict__ acc, float gx, float gy,
                                  float gz, const float4* __restrict__ xs, float inv_dt) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_fluid) return;
    float4 v = vel[i], s = vs[i];
    vel[i] = make_float4(s.x, s.y, s.z, v.w);
    vc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    float ax = gx, ay = gy, az = gz;
    if (xs) {
        float4 f = xs[i];
        ax = __fadd_rn(gx, __fmul_rn(f.x, inv_dt));
        ay = __fadd_rn(gy, __fmul_rn(f.y, inv_dt));
        az = __fadd_rn(gz, __fmul_rn(f.z, inv_dt));
    }
    acc[i] = make_float4(ax, ay, az, 0.f);
}
// update_velocities + the gravity / folded-XSPH acceleration + integrate_and_clear_accelerations in ONE pass, for steps whose force
// phase launches nothing (no plugin, or only the XSPH whose sums rode with the divergence loop): same arithmetic, in the same
// order, as k_fold_velocities followed by k_integrate_acc.  Ghost slots (multi-GPU) only take the fold part.
__global__ void k_fold_integrate(float4* __restrict__ vel, float4* __restrict__ vc, float4* __restrict__ vs, float4* __restrict__ acc, float gx, float gy,
                                 float gz, const float4* __restrict__ xs, float inv_dt_old, float dt_new, float4* __restrict__ pvx, float2* __restrict__ vyz) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_fluid) return;
    const float4 v = vel[i], s = vs[i];
    const float4 nv = make_float4(s.x, s.y, s.z, v.w);
    vel[i] = nv;
    const bool owned = i >= C.i_begin && i < C.i_begin + C.n_owned;
    float ax = gx, ay = gy, az = gz;
    if (xs) {
        const float4 f = xs[i];
        ax = __fadd_rn(gx, __fmul_rn(f.x, inv_dt_old));
        ay = __fadd_rn(gy, __fmul_rn(f.y, inv_dt_old));
        az = __fadd_rn(gz, __fmul_rn(f.z, inv_dt_old));
    }
    acc[i] = make_float4(ax, ay, az, 0.f);
    if (!owned) {
        vc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    const float cx = __fmul_rn(ax, dt_new), cy = __fmul_rn(ay, dt_new), cz = __fmul_rn(az, dt_new);  // vc = 0 + acc * dt
    vc[i] = make_float4(cx, cy, cz, 0.f);
    const float sx = nv.x + cx, sy = nv.y + cy, sz = nv.z + cz;
    vs[i] = make_float4(sx, sy, sz, 0.f);
    if (pvx) {
        pvx[i].w = sx;
        vyz[i] = make_float2(sy, sz);
    }
}
// IISPH variant: accelerations += gravity only (vc is already zero, velocities untouched).
__global__ void k_set_gravity(const float4* __restrict__ vel, float4* __restrict__ vs, float4* __restrict__ acc, float gx, float gy, float gz) {
    SPH_OWNED_INDEX(i)
    float4 v = vel[i];
    vs[i] = make_float4(v.x, v.y, v.z, 0.f);
    acc[i] = make_float4(gx, gy, gz, 0.f);
}

// a18: integrate_and_clear_accelerations dfsph_solver.rs:505-518 (+ v* = vel + vc).  The accelerations are NOT cleared here:
// the next step's k_fold_velocities / k_set_gravity overwrites them with gravity before any force adds to them, so the
// array doubles as the SPH_DBG_ACCELERATION view and the pass saves 32 B per particle of stores.
__global__ void k_integrate_acc(const float4* __restrict__ vel, float4* __restrict__ vc, float4* __restrict__ vs, const float4* __restrict__ acc, float dt,
                                float4* __restrict__ pvx, float2* __restrict__ vyz) {
    SPH_OWNED_INDEX(i)
    float4 a = acc[i], c = vc[i], v = vel[i];
    c.x += a.x * dt; c.y += a.y * dt; c.z += a.z * dt;
    vc[i] = c;
    float sx = v.x + c.x, sy = v.y + c.y, sz = v.z + c.z;
    vs[i] = make_float4(sx, sy, sz, 0.f);
    if (pvx) {
        pvx[i].w = sx;  // xyz already hold the position
        vyz[i] = make_float2(sy, sz);
    }
}

// a22: update_positions dfsph_solver.rs:411-420: pos += (vel + vc) * dt.  bounds_out (optional): the cell-coordinate AABB of
// the NEW positions (what k_bounds computes), so the next step's grid is sized without a bounds pass and its host round trip.
__global__ void k_update_positions(float4* __restrict__ pos, const float4* __restrict__ vs, float dt, int* __restrict__ bounds_out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < C.n_owned;
    i += C.i_begin;
    int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
    int bad = 0;
    if (valid) {
        float4 p = pos[i], v = vs[i];
        p.x += v.x * dt; p.y += v.y * dt; p.z += v.z * dt;
        pos[i] = p;
        if (bounds_out) {
            const float c[3] = {floorf(__fdiv_rn(p.x, C.h)), floorf(__fdiv_rn(p.y, C.h)), floorf(__fdiv_rn(p.z, C.h))};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (!(fabsf(c[a]) < 1.0e9f)) { bad = 1; continue; }  // NaN / inf / absurd coordinates
                mn[a] = mx[a] = (int)c[a];
            }
        }
    }
    if (!bounds_out) return;
#pragma unroll
    for (int a = 0; a < 3; ++a)
        for (int o = 16; o > 0; o >>= 1) {
            mn[a] = min(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = max(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
    bad = __any_sync(0xffffffffu, bad);
    __shared__ int s_mn[3][8], s_mx[3][8], s_bad[8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            s_mn[a][wid] = mn[a];
            s_mx[a][wid] = mx[a];
        }
        s_bad[wid] = bad;
    }
    __syncthreads();
    if (threadIdx.x < 3) {  // one atomic pair per axis per block
        const int a = threadIdx.x, nw = (blockDim.x + 31) >> 5;
        int m0 = INT_MAX, m1 = INT_MIN;
        for (int k = 0; k < nw; ++k) {
            m0 = min(m0, s_mn[a][k]);
            m1 = max(m1, s_mx[a][k]);
        }
        if (m0 <= m1) {
            atomicMin(&bounds_out[a], m0);
            atomicMax(&bounds_out[3 + a], m1);
        }
        if (a == 0) {
            int b = 0;
            for (int k = 0; k < nw; ++k) b |= s_bad[k];
            if (b) atomicOr(&bounds_out[6], 1);
        }
    }
}

__device__ __forceinline__ float powi3(float x) { return x * x * x; }
// akinci2013_surface_tension.rs:71-88
__device__ __forceinline__ float cohesion_kernel(float r, float coh_norm, float h6_64) {
    float hr = powi3(C.h - r) * powi3(r);
    float c = r <= C.h * 0.5f ? 2.0f * hr - h6_64 : (r <= C.h ? hr : 0.f);
    return coh_norm * c;
}

// akinci2013_surface_tension.rs:90-111
__device__ __forceinline__ float adhesion_kernel(float r, float adh_norm) {
    if (r > C.h * 0.5f && r <= C.h) {
        float x = fmaxf(-4.0f * r * r / C.h + 6.0f * r - 2.0f * C.h, 0.f);
        return adh_norm * sqrtf(sqrtf(x));  // powf(0.25)
    }
    return 0.f;
}

// ------------------------------------------------------------------------------------------------
// Host <-> sorted-order marshalling (Fluid/Boundary host SoA: fluid.rs:12-34, boundary.rs:11-24)
// ------------------------------------------------------------------------------------------------
// staging (original order, packed xyz) -> sorted arrays.  Any pointer may be null.
__global__ void k_import(uint32_t n, const uint32_t* __restrict__ orig, const float* __restrict__ o_pos, const float* __restrict__ o_vel,
                         const float* __restrict__ o_vc, const float* __restrict__ o_mass, const uint32_t* __restrict__ o_fid, float4* __restrict__ pos,
                         float4* __restrict__ vel, float4* __restrict__ vc, uint32_t lo, uint32_t hi) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t g = orig[s];
    if (g < lo || g >= hi) return;
    if (o_pos) {
        float4 p = pos[s];
        p.x = o_pos[3 * (size_t)g]; p.y = o_pos[3 * (size_t)g + 1]; p.z = o_pos[3 * (size_t)g + 2];
        if (o_mass) p.w = o_mass[g];
        pos[s] = p;
    }
    if (o_vel) {
        float4 v = vel[s];
        v.x = o_vel[3 * (size_t)g]; v.y = o_vel[3 * (size_t)g + 1]; v.z = o_vel[3 * (size_t)g + 2];
        if (o_fid) v.w = __uint_as_float(o_fid[g]);
        vel[s] = v;
    }
    if (o_vc) vc[s] = make_float4(o_vc[3 * (size_t)g], o_vc[3 * (size_t)g + 1], o_vc[3 * (size_t)g + 2], 0.f);
}
// sorted float4 array -> staging (original order, packed xyz)
__global__ void k_export3(uint32_t n, const uint32_t* __restrict__ orig, const float4* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t g = orig[s];
    float4 v = src[s];
    dst[3 * (size_t)g] = v.x; dst[3 * (size_t)g + 1] = v.y; dst[3 * (size_t)g + 2] = v.z;
}
// rows of 3 floats indexed by sorted index -> original order
__global__ void k_export_rows3(uint32_t n, const uint32_t* __restrict__ orig, const float* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t g = orig[s];
    dst[3 * (size_t)g] = src[3 * (size_t)s]; dst[3 * (size_t)g + 1] = src[3 * (size_t)s + 1]; dst[3 * (size_t)g + 2] = src[3 * (size_t)s + 2];
}
__global__ void k_export_w(uint32_t n, const uint32_t* __restrict__ orig, const float4* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    dst[orig[s]] = src[s].w;
}
__global__ void k_export_w_plain(uint32_t n, const float4* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) dst[s] = src[s].w;
}
__global__ void k_export1(uint32_t n, const uint32_t* __restrict__ orig, const float* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    dst[orig[s]] = src[s];
}
__global__ void k_export1u(uint32_t n, const uint32_t* __restrict__ orig, const uint32_t* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    dst[orig[s]] = (float)src[s];
}
// accelerations back from a host force callback: acc[s].xyz = src[orig[s]] for the particles of one fluid
__global__ void k_import_acc(uint32_t n, const uint32_t* __restrict__ orig, const float* __restrict__ src, uint32_t lo, uint32_t hi, float4* __restrict__ acc) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t g = orig[s];
    if (g < lo || g >= hi) return;
    acc[s] = make_float4(src[3 * (size_t)g], src[3 * (size_t)g + 1], src[3 * (size_t)g + 2], 0.f);
}
__global__ void k_import1(uint32_t n, const uint32_t* __restrict__ orig, const float* __restrict__ src, float* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    dst[s] = src[orig[s]];
}
__global__ void k_iota(uint32_t n, uint32_t* __restrict__ a) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) a[s] = s;
}
// ------------------------------------------------------------------------------------------------
// Slab decomposition helpers (sph_slab.inl): classification by cell column, stream compaction.
// ------------------------------------------------------------------------------------------------
// Owned slots [ob, ob + on) are classified by their CURRENT cell column in ONE pass.  Nothing is compacted: particles that
// left the slab are only flagged `dead` (the counting sort that follows drops them), and the few particles the neighbours
// need — emigrants and the kept particles of my two boundary columns — are appended to small staging buffers with one
// atomic per warp.  Their order inside the buffers is arbitrary; the receiver's sort orders every cell by particle id.
// counts[1..5] = #left, #right, #col-left, #col-right, #particles that jumped > 1 column.
struct SlabOut {  // staging arrays of k_slab_classify
    float4 *pos, *vel, *vc;
    uint32_t* gid;
};
__device__ __forceinline__ uint32_t warp_append(bool pred, uint32_t* counter) {
    const unsigned m = __ballot_sync(0xffffffffu, pred);
    if (!m) return 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, leader = __ffs((int)m) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    return pred ? base + (uint32_t)__popc(m & ((1u << lane) - 1u)) : 0xFFFFFFFFu;
}
__global__ void k_slab_classify(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ vc, const uint32_t* __restrict__ gid,
                                uint32_t ob, uint32_t on, int lo, int hi, int has_left, int has_right, uint32_t* __restrict__ dead, SlabOut out_l, SlabOut out_r,
                                SlabOut col_l, SlabOut col_r, uint32_t cap_out, uint32_t cap_col, uint32_t* __restrict__ counts) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = t < on;
    const uint32_t s = ob + (in ? t : 0u);
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    bool left = false, right = false, cl = false, cr = false, jumped = false;
    if (in) {
        p = pos[s];
        const int cx = cell_coord(p.x);
        left = has_left && cx < lo;
        right = has_right && cx >= hi;
        cl = !left && !right && has_left && cx == lo;
        cr = !left && !right && has_right && cx == hi - 1;
        jumped = (left && cx < lo - 1) || (right && cx > hi);
        dead[t] = (left || right) ? 1u : 0u;
    }
    const uint32_t kl = warp_append(left, &counts[1]), kr = warp_append(right, &counts[2]);
    const uint32_t kcl = warp_append(cl, &counts[3]), kcr = warp_append(cr, &counts[4]);
    warp_append(jumped, &counts[5]);
    if (!(left || right || cl || cr)) return;
    const float4 v = vel[s], c = vc[s];
    const uint32_t g = gid[s];
    if (left && kl < cap_out) { out_l.pos[kl] = p; out_l.vel[kl] = v; out_l.vc[kl] = c; out_l.gid[kl] = g; }
    if (right && kr < cap_out) { out_r.pos[kr] = p; out_r.vel[kr] = v; out_r.vc[kr] = c; out_r.gid[kr] = g; }
    if (cl && kcl < cap_col) { col_l.pos[kcl] = p; col_l.vel[kcl] = v; col_l.vc[kcl] = c; col_l.gid[kcl] = g; }
    if (cr && kcr < cap_col) { col_r.pos[kcr] = p; col_r.vel[kcr] = v; col_r.vc[kcr] = c; col_r.gid[kcr] = g; }
}
// counts[8..9] = {#emigrants left, #col-left}, counts[10..11] = {#emigrants right, #col-right}: the two 8-byte messages
__global__ void k_slab_pack_counts(uint32_t* __restrict__ counts) {
    if (threadIdx.x == 0) {
        counts[8] = counts[1]; counts[9] = counts[3];
        counts[10] = counts[2]; counts[11] = counts[4];
    }
}
__global__ void k_iota_from(uint32_t n, uint32_t start, uint32_t* __restrict__ a) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) a[s] = start + s;
}
__global__ void k_export_u32(uint32_t n, const uint32_t* __restrict__ orig, const uint32_t* __restrict__ src, uint32_t* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) dst[orig[s]] = src[s];
}
__global__ void k_import_u32(uint32_t n, const uint32_t* __restrict__ orig, const uint32_t* __restrict__ src, uint32_t* __restrict__ dst) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) dst[s] = src[orig[s]];
}

// ------------------------------------------------------------------------------------------------
// Ghost exchange over NVLink peer memory (sph_slab.inl).  Every rank maps its two neighbours' landing zones ("boxes",
// cudaIpc) and the producer side WRITES its boundary columns straight into the neighbour's box with plain st.global
// over NVLink, then publishes a sequence number (release, system scope); the consumer side spins on its own flag
// (acquire, system scope) and copies box -> ghost slots.  No NCCL, no host involvement, ~10 us per exchange.
// ------------------------------------------------------------------------------------------------
struct P2PSeg {           // one contiguous array range travelling in a message
    const char* src;      // sender: local source; receiver: unused
    char* dst;            // receiver: local ghost range; sender: unused
    uint32_t box_off;     // byte offset inside the box (16-byte aligned)
    uint32_t bytes;       // multiple of 4
};
struct P2PMsg {           // one direction (to / from one neighbour)
    char* box;            // sender: the NEIGHBOUR's box (peer pointer); receiver: my own box
    uint32_t* flag;       // sender: the neighbour's flag (peer pointer); receiver: my own flag
    P2PSeg seg[4];
    int n_seg;
    uint32_t total_words;  // sum of bytes / 4
};
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// bounded spin (a peer that never arrives must not hang the GPU): ~2 s of SM clock, then the (sticky) error flag
__device__ __forceinline__ bool p2p_wait(const uint32_t* flag, uint32_t seq, int* err) {
    if (*reinterpret_cast<volatile int*>(err) & 2) return false;  // an earlier exchange of this step already timed out: do not wait again
    const long long t0 = clock64();
    while ((int)(ld_acquire_sys(flag) - seq) < 0) {
        if (clock64() - t0 > 4000000000LL) {
            atomicOr(err, 2);
            return false;
        }
        __nanosleep(64);
    }
    return true;
}
// blockIdx.y = direction (0: left neighbour, 1: right neighbour)
__global__ void k_p2p_push(P2PMsg m0, P2PMsg m1, uint32_t seq0, uint32_t seq1, uint32_t* __restrict__ tickets) {
    const P2PMsg& m = blockIdx.y ? m1 : m0;
    if (!m.box) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (int s = 0; s < m.n_seg; ++s) {
        const uint32_t* __restrict__ src = reinterpret_cast<const uint32_t*>(m.seg[s].src);
        uint32_t* dst = reinterpret_cast<uint32_t*>(m.box + m.seg[s].box_off);
        const uint32_t nw = m.seg[s].bytes >> 2;
        const uint32_t n4 = nw >> 2;  // ranges start 16-byte aligned on both sides whenever the element size is a multiple of 16
        if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) {
            const uint4* s4 = reinterpret_cast<const uint4*>(src);
            uint4* d4 = reinterpret_cast<uint4*>(dst);
            for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += stride) d4[k] = s4[k];
            for (uint32_t k = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; k < nw; k += stride) dst[k] = src[k];
        } else {
            for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nw; k += stride) dst[k] = src[k];
        }
    }
    __threadfence_system();
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&tickets[blockIdx.y], 1u) == gridDim.x - 1;
    __syncthreads();
    if (last && threadIdx.x == 0) {
        tickets[blockIdx.y] = 0;
        __threadfence_system();
        st_release_sys(m.flag, blockIdx.y ? seq1 : seq0);
    }
}
__global__ void k_p2p_pull(P2PMsg m0, P2PMsg m1, uint32_t seq0, uint32_t seq1, int* __restrict__ err) {
    const P2PMsg& m = blockIdx.y ? m1 : m0;
    if (!m.box) return;
    __shared__ bool ok;
    if (threadIdx.x == 0) ok = p2p_wait(m.flag, blockIdx.y ? seq1 : seq0, err);
    __syncthreads();
    if (!ok) return;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (int s = 0; s < m.n_seg; ++s) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(m.box + m.seg[s].box_off);
        uint32_t* dst = reinterpret_cast<uint32_t*>(m.seg[s].dst);
        const uint32_t nw = m.seg[s].bytes >> 2;
        const uint32_t n4 = nw >> 2;
        if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0) {
            const uint4* s4 = reinterpret_cast<const uint4*>(src);
            uint4* d4 = reinterpret_cast<uint4*>(dst);
            for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += stride) d4[k] = __ldcv(&s4[k]);  // written by a peer: bypass L1
            for (uint32_t k = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; k < nw; k += stride) dst[k] = __ldcv(&src[k]);
        } else {
            for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nw; k += stride) dst[k] = __ldcv(&src[k]);
        }
    }
}
// All-ranks sum of a few floats (Jacobi error means) through peer memory: rank r writes its values into slot r of EVERY
// rank's table, publishes, waits for all slots and sums them in rank order (deterministic, same result on every rank).
struct P2PPeers {
    float* red[8];         // red[p]: rank p's table  [buf][rank][MAX_FLUIDS]
    uint32_t* red_flag[8]; // rank p's flags          [buf][rank]
};
__global__ void k_p2p_allreduce(float* __restrict__ vals, int n, int rank, int nranks, P2PPeers P, uint32_t seq, int* __restrict__ err) {
    const int buf = (int)(seq & 1u);
    const int t = threadIdx.x;
    // thread (p, f): write vals[f] into rank p's table
    for (int k = t; k < nranks * n; k += blockDim.x) {
        const int p = k / n, f = k % n;
        P.red[p][((size_t)buf * 8 + rank) * MAX_FLUIDS + f] = vals[f];
    }
    __threadfence_system();
    __syncthreads();
    for (int p = t; p < nranks; p += blockDim.x) st_release_sys(&P.red_flag[p][buf * 8 + rank], seq);
    __shared__ int ok;
    if (t == 0) ok = 1;
    __syncthreads();
    for (int p = t; p < nranks; p += blockDim.x)
        if (!p2p_wait(&P.red_flag[rank][buf * 8 + p], seq, err)) ok = 0;
    __syncthreads();
    if (!ok) return;
    for (int f = t; f < n; f += blockDim.x) {
        float s = 0.f;
        for (int p = 0; p < nranks; ++p) s += __ldcv(&P.red[rank][((size_t)buf * 8 + p) * MAX_FLUIDS + f]);
        vals[f] = s;
    }
}

// LiquidWorld::particles_intersecting_aabb liquid_world.rs:211-243 over HGrid::cells_intersecting_aabb hgrid.rs:122-133.
// One thread per cell of the (clipped) cell box [key(mins), key(maxs)] of the grid built by the last step; the CURRENT
// positions are tested (Aabb::distance_to_point, solid: norm of the per-axis excess) against particle_radius.
// out[2k] = kind (0 fluid, 1 boundary), out[2k+1] = original index; order is whatever the atomics give (host sorts).
struct AabbQuery {
    int lx, ly, lz, dx, dy, dz;  // first cell and extent (cells) of the box
    float mins[3], maxs[3], radius;
    uint32_t slot_lo, slot_hi;   // owned fluid slots (ghost copies of a slab world are skipped)
    // particles_intersecting_shape (liquid_world.rs:246-281): kind 0 = the box itself (distance < radius, :224),
    // 1 = ball, 2 = cuboid, 3 = capsule (segment along local y), each posed by the isometry (rot, t): point p is hit
    // when shape.distance_to_point(pos, p, solid) <= radius (:263)
    int kind;
    float rot[9], t[3];          // world = rot * local + t (row-major rotation)
    float sp[3];                 // ball: radius; cuboid: half extents; capsule: half height, radius
};
__device__ __forceinline__ bool query_near(const AabbQuery& q, const float4& p) {
    if (q.kind == 0) {
        float ex = fmaxf(fmaxf(q.mins[0] - p.x, p.x - q.maxs[0]), 0.f);
        float ey = fmaxf(fmaxf(q.mins[1] - p.y, p.y - q.maxs[1]), 0.f);
        float ez = fmaxf(fmaxf(q.mins[2] - p.z, p.z - q.maxs[2]), 0.f);
        return __fsqrt_rn(dist2_exact(ex, ey, ez)) < q.radius;
    }
    // local point = rot^T (p - t)
    const float wx = p.x - q.t[0], wy = p.y - q.t[1], wz = p.z - q.t[2];
    const float lx = q.rot[0] * wx + q.rot[3] * wy + q.rot[6] * wz;
    const float ly = q.rot[1] * wx + q.rot[4] * wy + q.rot[7] * wz;
    const float lz = q.rot[2] * wx + q.rot[5] * wy + q.rot[8] * wz;
    float d;
    if (q.kind == 1) {
        d = fmaxf(__fsqrt_rn(dist2_exact(lx, ly, lz)) - q.sp[0], 0.f);
    } else if (q.kind == 2) {
        float ex = fmaxf(fabsf(lx) - q.sp[0], 0.f), ey = fmaxf(fabsf(ly) - q.sp[1], 0.f), ez = fmaxf(fabsf(lz) - q.sp[2], 0.f);
        d = __fsqrt_rn(dist2_exact(ex, ey, ez));
    } else {
        float cy = fminf(fmaxf(ly, -q.sp[0]), q.sp[0]);  // closest point of the segment
        d = fmaxf(__fsqrt_rn(dist2_exact(lx, ly - cy, lz)) - q.sp[1], 0.f);
    }
    return d <= q.radius;
}
__global__ void k_aabb_query(AabbQuery q, const float4* __restrict__ pos, const uint32_t* __restrict__ cstart, const uint32_t* __restrict__ orig,
                             const float4* __restrict__ bpos, const uint32_t* __restrict__ bstart, const uint32_t* __restrict__ borig,
                             uint32_t* __restrict__ out, uint32_t cap, uint32_t* __restrict__ count) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint32_t)(q.dx * q.dy * q.dz)) return;
    int cz = q.lz + (int)(t % (uint32_t)q.dz);
    int cy = q.ly + (int)((t / (uint32_t)q.dz) % (uint32_t)q.dy);
    int cx = q.lx + (int)(t / (uint32_t)(q.dz * q.dy));
    int c = cell_id(cx, cy, cz);
    if (pos) {
        uint32_t s = max(cstart[c], q.slot_lo), e = min(cstart[c + 1], q.slot_hi);
        for (uint32_t j = s; j < e; ++j)
            if (query_near(q, pos[j])) {
                uint32_t k = atomicAdd(count, 1u);
                if (k < cap) {
                    out[2 * (size_t)k] = 0u;
                    out[2 * (size_t)k + 1] = orig[j];
                }
            }
    }
    if (bpos) {
        for (uint32_t j = bstart[c]; j < bstart[c + 1]; ++j)
            if (query_near(q, bpos[j])) {
                uint32_t k = atomicAdd(count, 1u);
                if (k < cap) {
                    out[2 * (size_t)k] = 1u;
                    out[2 * (size_t)k + 1] = borig[j];
                }
            }
    }
}

// ------------------------------------------------------------------------------------------------
// ParticlesContacts materialisation for host NonPressureForce plugins (nonpressure_force.rs:15-27 hands
// `fluid_fluid_contacts` / `fluid_boundaries_contacts` to solve(); Contact = {i_model, j_model, i, j, weight, gradient},
// contacts.rs:12-27).  CSR in ORIGINAL particle order; entries of a particle keep the list order (ascending sorted j).
// ------------------------------------------------------------------------------------------------
struct OffsetTable {
    uint32_t off[MAX_FLUIDS > MAX_BOUNDARIES ? MAX_FLUIDS + 1 : MAX_BOUNDARIES + 1];
};
__global__ void k_contacts_count(uint32_t n, const uint32_t* __restrict__ orig, const uint32_t* __restrict__ cnt, uint32_t cap, uint32_t* __restrict__ out) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) out[orig[s]] = min(cnt[s], cap);
}
// one thread per sorted slot: writes its particle's contacts at scan[orig[s]]..
template <bool BOUNDARY>
__global__ void k_contacts_fill(uint32_t n, const float4* __restrict__ pos, const float4* __restrict__ other_pos, const float4* __restrict__ other_vel,
                                const uint32_t* __restrict__ orig, const uint32_t* __restrict__ other_orig, const uint32_t* __restrict__ nbr,
                                const uint32_t* __restrict__ cnt, uint32_t cap, const uint32_t* __restrict__ scan, OffsetTable tab, uint32_t* __restrict__ out_j,
                                uint32_t* __restrict__ out_model, float* __restrict__ out_w, float* __restrict__ out_g) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t i = s + C.i_begin;
    const float4 pi = pos[i];
    const uint32_t m = min(cnt[i], cap);
    size_t base = scan[orig[i]];
    for (uint32_t k = 0; k < m; ++k) {
        const uint32_t j = BOUNDARY ? nbr[(size_t)k * C.stride + i] : nbr[((size_t)(k >> 2) * C.stride + i) * 4 + (k & 3)];
        const float4 pj = other_pos[j];
        const Pair p = make_pair<true, true>(pi, pj);
        const uint32_t model = fid_of(other_vel[j]);
        out_j[base + k] = other_orig[j] - tab.off[model];
        out_model[base + k] = model;
        out_w[base + k] = p.w;
        out_g[3 * (base + k) + 0] = p.g * p.dx;
        out_g[3 * (base + k) + 1] = p.g * p.dy;
        out_g[3 * (base + k) + 2] = p.g * p.dz;
    }
}

__global__ void k_sum_u32(uint32_t n, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, unsigned long long* __restrict__ out) {
    unsigned long long s = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += (unsigned long long)a[i] + b[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

}  // namespace sphk
