// sph_passes.cuh — neighbour-gather passes, default backend: one thread per particle walks its index-only
// contact list and gathers neighbour data from global memory through L1 (and, for the second per-contact vector,
// optionally through the TEXTURE pipe, whose data path is separate from the LSU one: profiles/r1_v0_* show the
// LSU data pipe — two float4 gathers per contact — is what bounds these kernels, not DRAM).
//
// Contacts are consumed in groups of four: one coalesced LDG.128 brings 4 list indices per thread (the next group is
// prefetched before the current one is used), then 4 position gathers + 4 auxiliary gathers are issued back to back
// and only then the 4 pair evaluations run, so 8+ independent loads are in flight per thread.
#pragma once
#include <type_traits>

#include "sph_kernels.cuh"

namespace sphk {

struct Lists {
    const uint4* nbr_f;     // nbr_f[(k / 4) * stride + i] = contacts 4*(k/4) .. 4*(k/4)+3 of particle i (sorted indices);
                            // tail slots of the last group hold i itself (a self contact has zero gradient)
    const uint32_t* nbr_b;  // nbr_b[k * stride + i]
    const uint32_t* cnt_f;
    const uint32_t* cnt_b;
};

struct NoAux {};

// Gather lambdas may take the contact's position u in its group of four as a second argument: kernels use it to send the
// gathers of even and odd contacts through DIFFERENT L1TEX front ends (texture pipe / LSU pipe).  ncu on the round-1 kernels
// (profiles/r2_ncu_pair_c3.md): the update pass ran at 88 % of the LSU data-pipe wavefront peak with the texture pipe idle, the
// evaluation at 60 % TEX / 44 % LSU; splitting every gather stream over both pipes is worth 10-15 % of those passes.
template <class F>
__device__ __forceinline__ auto call_gather(F& f, uint32_t j, int u) {
    if constexpr (std::is_invocable_v<F, uint32_t, int>) return f(j, u);
    else return f(j);
}

// Slot range a launch covers: the owned slots [begin, begin + count).
struct Range {
    uint32_t begin, count;
};

// The contact lists are streamed exactly once per pass: load them with the evict-first policy so they do not push the
// gathered particle data out of L1/L2.
__device__ __forceinline__ uint4 ld_list(const uint4* p) { return __ldcs(p); }

// ldpos(j) -> float4 whose xyz is the neighbour position (w = whatever the array packs there); ld(j) -> Aux loads
// whatever else the pass needs from neighbour j; ff(j, pair, posrec_j, aux) consumes one contact.
template <bool W, bool G, class LP, class LD, class FF>
__device__ __forceinline__ void for_fluid_contacts_g(uint32_t i, const float4& pi, const Lists& L, LP ldpos, LD ld, FF ff) {
    const uint32_t n = min(L.cnt_f[i], C.cap_f);
    const uint32_t nq = (n + 3u) >> 2;
    const uint4* col = L.nbr_f + i;
    uint4 J = nq ? ld_list(col) : make_uint4(i, i, i, i);
    for (uint32_t q = 0; q < nq; ++q) {
        uint4 Jn = J;
        if (q + 1 < nq) Jn = ld_list(col + (size_t)(q + 1) * C.stride);  // fetch the next group of indices early
        uint32_t j[4] = {J.x, J.y, J.z, J.w};
        const uint32_t k0 = q * 4u;
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            ok[u] = k0 + u < n;
            if (!ok[u]) j[u] = i;  // unwritten tail slots of the last group: point at self, masked below
        }
        float4 pj[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) pj[u] = call_gather(ldpos, j[u], u);
        decltype(call_gather(ld, 0u, 0)) aux[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) aux[u] = call_gather(ld, j[u], u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (ok[u]) {
                Pair p = make_pair<W, G>(pi, pj[u]);
                ff(j[u], p, pj[u], aux[u]);
            }
        }
        J = Jn;
    }
}
// Gradient-only passes.  Contacts are consumed in groups of four: the group's 4 position gathers and 4 auxiliary
// gathers are issued back to back before any arithmetic, and the next group's list indices are prefetched.
// (A deeper software pipeline — gathers one group ahead — was measured SLOWER: 80-96 registers halve the occupancy,
// C2 predicted-density pass 0.127 ms vs 0.099 ms; profiles/r1_v1_batching_tex_c2.md.)
// No tail masking: padded slots are (j = i) and a self contact has zero gradient.
template <bool NEED_W = false, class LP, class LD, class FF>
__device__ __forceinline__ void for_fluid_grads(uint32_t i, const float4& pi, const Lists& L, LP ldpos, LD ld, FF ff) {
    const uint32_t n = min(L.cnt_f[i], C.cap_f);
    const uint32_t nq = (n + 3u) >> 2;
    if (nq == 0) return;
    const uint4* col = L.nbr_f + i;
    uint4 J = ld_list(col);
    for (uint32_t q = 0; q < nq; ++q) {
        uint4 Jn = J;
        if (q + 1 < nq) Jn = ld_list(col + (size_t)(q + 1) * C.stride);  // fetch the next group early
        const uint32_t j[4] = {J.x, J.y, J.z, J.w};
        float4 pj[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) pj[u] = call_gather(ldpos, j[u], u);
        decltype(call_gather(ld, 0u, 0)) aux[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) aux[u] = call_gather(ld, j[u], u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            Pair p = make_pair<NEED_W, true>(pi, pj[u]);
            ff(j[u], p, pj[u], aux[u]);
        }
        J = Jn;
    }
}
template <class LD, class FF>
__device__ __forceinline__ void for_fluid_grads_pos(uint32_t i, const float4& pi, const Lists& L, const float4* __restrict__ pos, LD ld, FF ff) {
    for_fluid_grads(i, pi, L, [&](uint32_t j) { return __ldg(&pos[j]); }, ld, ff);
}

template <bool W, bool G, class LD, class FF>
__device__ __forceinline__ void for_fluid_contacts(uint32_t i, const float4& pi, const Lists& L, const float4* __restrict__ pos, LD ld, FF ff) {
    for_fluid_contacts_g<W, G>(i, pi, L, [&](uint32_t j) { return __ldg(&pos[j]); }, ld, ff);
}
template <bool W, bool G, class FB>
__device__ __forceinline__ void for_boundary_contacts(uint32_t i, const float4& pi, const Lists& L, const float4* __restrict__ bpos, FB fb) {
    uint32_t n = min(L.cnt_b[i], C.cap_b);
    const uint32_t* col = L.nbr_b + i;
    for (uint32_t k = 0; k < n; ++k) {
        uint32_t j = col[(size_t)k * C.stride];
        float4 pj = __ldg(&bpos[j]);
        Pair p = make_pair<W, G>(pi, pj);
        fb(j, p, pj);
    }
}

template <bool TEX>
__device__ __forceinline__ float4 fetch4(const float4* __restrict__ a, cudaTextureObject_t t, uint32_t j) {
    if (TEX) return tex1Dfetch<float4>(t, (int)j);
    return __ldg(&a[j]);
}
template <bool TEX>
__device__ __forceinline__ float fetch1(const float* __restrict__ a, cudaTextureObject_t t, uint32_t j) {
    if (TEX) return tex1Dfetch<float>(t, (int)j);
    return __ldg(&a[j]);
}

// Per-fluid deterministic error reduction: partial[block * n_fluids + f].
// With a ticket counter the LAST block to finish also sums the partials of the whole launch in index order into
// errsum[f] (saves a separate k_reduce_partials launch per evaluation; same fixed summation tree every run).
template <bool MULTI>
__device__ __forceinline__ void reduce_error(float e, uint32_t fi, bool valid, float* __restrict__ partial, float* sm, uint32_t* __restrict__ ticket = nullptr,
                                             float* __restrict__ errsum = nullptr) {
    const int nf = MULTI ? C.n_fluids : 1;
    if (!MULTI) {
        float s = block_sum(valid ? e : 0.f, sm);
        if (threadIdx.x == 0) partial[blockIdx.x] = s;
    } else {
        for (int f = 0; f < nf; ++f) {
            float s = block_sum((valid && fi == (uint32_t)f) ? e : 0.f, sm);
            if (threadIdx.x == 0) partial[(size_t)blockIdx.x * nf + f] = s;
        }
    }
    if (ticket) {
        __shared__ bool s_last;
        __threadfence();
        if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
        __syncthreads();
        if (s_last) {
            for (int f = 0; f < nf; ++f) {
                float s = 0.f;
                for (uint32_t b = threadIdx.x; b < gridDim.x; b += blockDim.x) s += __ldcg(&partial[(size_t)b * nf + f]);
                s = block_sum(s, sm);
                if (threadIdx.x == 0) errsum[f] = s;
            }
            if (threadIdx.x == 0) *ticket = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3: densities (dfsph_solver.rs:628-665) fused with alphas (dfsph_solver.rs:165-216) and the per-contact
// kernel evaluation of helper.rs:9-65.
// ------------------------------------------------------------------------------------------------
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_density_alpha(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L,
                float* __restrict__ dens, float* __restrict__ alpha, int* __restrict__ err) {
    SPH_OWNED_INDEX(i)
    float4 pi = pos[i];
    float rho0 = C.fluids[MULTI ? fid_of(vel[i]) : 0].density0;
    float rho = 0.f, sq = 0.f, gx = 0.f, gy = 0.f, gz = 0.f;
    {
        const uint32_t n = min(L.cnt_f[i], C.cap_f);
        const uint32_t nq = (n + 3u) >> 2;
        const uint4* col = L.nbr_f + i;
        uint4 J = nq ? ld_list(col) : make_uint4(i, i, i, i);
        for (uint32_t q = 0; q < nq; ++q) {
            uint4 Jn = J;
            if (q + 1 < nq) Jn = ld_list(col + (size_t)(q + 1) * C.stride);
            const uint32_t j[4] = {J.x, J.y, J.z, J.w};
            float4 pj[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) pj[u] = __ldg(&pos[j[u]]);  // tail slots point at i itself
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool ok = q * 4u + u < n;
                Pair p = make_pair<true, true>(pi, pj[u]);
                if (ok) {
                    rho = fmaf(pj[u].w, p.w, rho);
                    float s = p.g * pj[u].w;  // m_j * gradient
                    float ax = s * p.dx, ay = s * p.dy, az = s * p.dz;
                    sq += ax * ax + ay * ay + az * az;
                    gx += ax; gy += ay; gz += az;
                }
            }
            J = Jn;
        }
    }
    for_boundary_contacts<true, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
        float mb = pj.w * rho0;  // boundary pseudo mass: vol_b * rho0_i
        rho = fmaf(mb, p.w, rho);
        float s = p.g * mb;
        float ax = s * p.dx, ay = s * p.dy, az = s * p.dz;
        sq += ax * ax + ay * ay + az * az;
        gx += ax; gy += ay; gz += az;
    });
    if (rho == 0.f) atomicOr(err, 1);  // assert!(!density.is_zero()) dfsph_solver.rs:662
    float den = sq + (gx * gx + gy * gy + gz * gz);
    dens[i] = rho;
    alpha[i] = den <= 1.0e-5f ? 0.f : 1.0f / den;  // dfsph_solver.rs:209-213
}

// ------------------------------------------------------------------------------------------------
// K3 + first K4a fused (DFSPH): densities, alphas AND the first compute_divergences evaluation in ONE gather pass.
// The first divergence evaluation of divergence_solve (dfsph_solver.rs:474-480) reads the same neighbour positions
// and the step-start v* = vel + vc, and needs alpha_i only for kappa_i = div_i * alpha_i at the very end, so it can
// ride along with the density pass: one full neighbour sweep less per step.  Arithmetic per quantity is unchanged.
// UNI: uniform-mass packed records (positions from pvx4, v* from pvx4.w + vyz2), else pos4 / vs4.
// ------------------------------------------------------------------------------------------------
struct Vel3 {
    float x, y, z;
};
template <bool MULTI, bool UNI>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_density_alpha_div(const float4* __restrict__ posrec /* pos4 or pvx4 */, cudaTextureObject_t tposrec, const float4* __restrict__ vs, cudaTextureObject_t tvs,
                    const float2* __restrict__ vyz, cudaTextureObject_t tvyz, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L,
                    float* __restrict__ dens, float* __restrict__ alpha, float* __restrict__ divv, float* __restrict__ kappa,
                    float4* __restrict__ pk4, float* __restrict__ partial, int* __restrict__ err, uint32_t* __restrict__ ticket,
                    float* __restrict__ errsum, Range rg) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < rg.count;
    i += rg.begin;
    float e = 0.f;
    uint32_t fi = 0;
    if (valid) {
        const float4 a = posrec[i];
        const float4 pi = make_float4(a.x, a.y, a.z, a.w);
        fi = MULTI ? fid_of(vel[i]) : 0u;
        const float rho0 = C.fluids[fi].density0;
        const float umass = C.fluids[0].mass;
        Vel3 vi;
        if (UNI) {
            float2 b = vyz[i];
            vi = Vel3{a.w, b.x, b.y};
        } else {
            float4 s = vs[i];
            vi = Vel3{s.x, s.y, s.z};
        }
        float rho = 0.f, sq = 0.f, gx = 0.f, gy = 0.f, gz = 0.f, d = 0.f;
        const uint32_t n = min(L.cnt_f[i], C.cap_f);
        const uint32_t nq = (n + 3u) >> 2;
        const uint4* col = L.nbr_f + i;
        uint4 J = nq ? ld_list(col) : make_uint4(i, i, i, i);
        for (uint32_t q = 0; q < nq; ++q) {
            uint4 Jn = J;
            if (q + 1 < nq) Jn = ld_list(col + (size_t)(q + 1) * C.stride);
            const uint32_t j[4] = {J.x, J.y, J.z, J.w};
            float4 pj[4];
            Vel3 vj[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) pj[u] = (UNI && (u & 1)) ? tex1Dfetch<float4>(tposrec, (int)j[u]) : __ldg(&posrec[j[u]]);  // tail slots point at i itself
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (UNI) {  // even contacts: (record via LSU, velocity via TEX), odd ones the other way round
                    float2 b = (u & 1) ? __ldg(&vyz[j[u]]) : tex1Dfetch<float2>(tvyz, (int)j[u]);
                    vj[u] = Vel3{pj[u].w, b.x, b.y};
                } else {
                    float4 s = tex1Dfetch<float4>(tvs, (int)j[u]);
                    vj[u] = Vel3{s.x, s.y, s.z};
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool ok = q * 4u + u < n;
                Pair p = make_pair<true, true>(pi, pj[u]);
                if (ok) {
                    const float mj = UNI ? umass : pj[u].w;
                    rho = fmaf(mj, p.w, rho);
                    float s = p.g * mj;  // m_j * gradient
                    float ax = s * p.dx, ay = s * p.dy, az = s * p.dz;
                    sq += ax * ax + ay * ay + az * az;
                    gx += ax; gy += ay; gz += az;
                    float dv = (vi.x - vj[u].x) * p.dx + (vi.y - vj[u].y) * p.dy + (vi.z - vj[u].z) * p.dz;
                    d = fmaf(dv * p.g, mj, d);
                }
            }
            J = Jn;
        }
        for_boundary_contacts<true, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
            float mb = pj.w * rho0;  // boundary pseudo mass: vol_b * rho0_i
            rho = fmaf(mb, p.w, rho);
            float s = p.g * mb;
            float ax = s * p.dx, ay = s * p.dy, az = s * p.dz;
            sq += ax * ax + ay * ay + az * az;
            gx += ax; gy += ay; gz += az;
            float dv = vi.x * p.dx + vi.y * p.dy + vi.z * p.dz;  // boundary velocity ignored (dfsph_solver.rs:336-338)
            d = fmaf(dv * p.g, mb, d);
        });
        if (rho == 0.f) atomicOr(err, 1);  // assert!(!density.is_zero()) dfsph_solver.rs:662
        float den = sq + (gx * gx + gy * gy + gz * gz);
        float al = den <= 1.0e-5f ? 0.f : 1.0f / den;  // dfsph_solver.rs:209-213
        dens[i] = rho;
        alpha[i] = al;
        if (L.cnt_f[i] + L.cnt_b[i] < 20u) d = 0.f;  // min_neighbors_for_divergence_solve :62,301-314
        d = fmaxf(d, 0.f);
        divv[i] = d;
        if (UNI) pk4[i] = make_float4(a.x, a.y, a.z, d * al);
        else kappa[i] = d * al;
        e = d / rho0;
    }
    reduce_error<MULTI>(e, fi, valid, partial, sm, ticket, errsum);
}

// ------------------------------------------------------------------------------------------------
// K4a / K8a: compute_divergences dfsph_solver.rs:279-356 (PREDICT = false) and compute_predicted_densities
// dfsph_solver.rs:98-162 (PREDICT = true) share one kernel: sum_j m_j (v*_i - v*_j) . gradW_ij.
//   PREDICT: out = rho*_i, kappa = max((rho* - rho0) alpha, 0), boundary term uses the boundary velocity (:136-141);
//   else   : out = div_i (0 below 20 contacts, :62,301-314), kappa = div * alpha, boundary velocity ignored (:336-338).
// ------------------------------------------------------------------------------------------------
// The v*_j gather goes through the texture pipe: 12 % faster than through LSU (profiles/r1_v1_*).
template <bool MULTI, bool PREDICT>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_vel_divergence(const float4* __restrict__ pos, const float4* __restrict__ vs, cudaTextureObject_t tvs, const float4* __restrict__ vel,
                 const float4* __restrict__ bpos, const float4* __restrict__ bvel, Lists L, const float* __restrict__ dens,
                 const float* __restrict__ alpha, float* __restrict__ out, float* __restrict__ kappa, float* __restrict__ partial, float dt,
                 int* __restrict__ err, uint32_t* __restrict__ ticket, float* __restrict__ errsum, Range rg) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < rg.count;
    i += rg.begin;
    float e = 0.f;
    uint32_t fi = 0;
    if (valid) {
        float4 pi = pos[i];
        float4 vi = vs[i];
        fi = MULTI ? fid_of(vel[i]) : 0u;
        float rho0 = C.fluids[fi].density0;
        float d = 0.f;
        if (PREDICT || L.cnt_f[i] + L.cnt_b[i] >= 20u) {
            for_fluid_grads_pos(
                i, pi, L, pos, [&](uint32_t j) { return tex1Dfetch<float4>(tvs, (int)j); },
                [&](uint32_t, const Pair& p, const float4& pj, const float4& vj) {
                    float dv = (vi.x - vj.x) * p.dx + (vi.y - vj.y) * p.dy + (vi.z - vj.z) * p.dz;
                    d = fmaf(dv * p.g, pj.w, d);
                });
            for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
                float dv;
                if (PREDICT) {
                    float4 vj = __ldg(&bvel[j]);
                    dv = (vi.x - vj.x) * p.dx + (vi.y - vj.y) * p.dy + (vi.z - vj.z) * p.dz;
                } else {
                    dv = vi.x * p.dx + vi.y * p.dy + vi.z * p.dz;
                }
                d = fmaf(dv * p.g, pj.w * rho0, d);
            });
        }
        if (PREDICT) {
            float pd = fmaf(d, dt, dens[i]);
            if (pd == 0.f) atomicOr(err, 1);  // assert dfsph_solver.rs:145
            out[i] = pd;
            kappa[i] = fmaxf((pd - rho0) * alpha[i], 0.f);
            e = pd < rho0 ? 0.f : pd / rho0 - 1.0f;
        } else {
            d = fmaxf(d, 0.f);
            out[i] = d;
            kappa[i] = d * alpha[i];
            e = d / rho0;
        }
    }
    reduce_error<MULTI>(e, fi, valid, partial, sm, ticket, errsum);
}

// ------------------------------------------------------------------------------------------------
// K4b / K8b: compute_velocity_changes_for_divergence dfsph_solver.rs:358-409 (PRESSURE = false) and
// compute_velocity_changes dfsph_solver.rs:218-277 (PRESSURE = true):
//   vc_i -= scale * [ sum_j (k_i + k_j) m_j gradW_ij + sum_b k_i vol_b rho0 gradW_ib ],  v* = vel + vc.
// PRESSURE: k = kappa+ (>= 0), scale = inv_dt, boundary term only if k_i > 0 (:257); else k = div*alpha, scale = 1.
// ------------------------------------------------------------------------------------------------
template <bool MULTI, bool BFORCE, bool PRESSURE, bool TEX>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_vel_update(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ kappa,
             cudaTextureObject_t tkappa, float4* __restrict__ vc, float4* __restrict__ vs, float* __restrict__ bforce, float inv_dt, Range rg) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rg.count) return;
    i += rg.begin;
    float4 pi = pos[i];
    float4 v = vel[i];
    float rho0 = C.fluids[MULTI ? fid_of(v) : 0].density0;
    float ki = kappa[i];
    const float scale = PRESSURE ? inv_dt : 1.0f;
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return fetch1<TEX>(kappa, tkappa, j); },
        [&](uint32_t, const Pair& p, const float4& pj, float kj) {
            float c = (ki + kj) * pj.w * scale * p.g;
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    if (!PRESSURE || ki > 0.f) {
        for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float c = ki * pj.w * rho0 * scale * p.g;
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
            if (BFORCE) {  // :269-272 / :403-405 both reduce to +c * inv_dt * m_i * x_ij on the boundary particle
                float s = c * inv_dt * pi.w;
                atomicAdd(&bforce[3 * (size_t)j + 0], s * p.dx);
                atomicAdd(&bforce[3 * (size_t)j + 1], s * p.dy);
                atomicAdd(&bforce[3 * (size_t)j + 2], s * p.dz);
            }
        });
    }
    float4 c4 = vc[i];
    c4.x -= ax; c4.y -= ay; c4.z -= az;
    vc[i] = c4;
    vs[i] = make_float4(v.x + c4.x, v.y + c4.y, v.z + c4.z, 0.f);
}

// ------------------------------------------------------------------------------------------------
// Uniform-mass fast path (one fluid whose particles all have the same volume — every default-constructed Fluid,
// fluid.rs:110-120): the mass is a constant, so the per-contact gathers shrink to packed records
//   pvx4 = (x, y, z, v*x), vyz2 = (v*y, v*z)   for the evaluations  (24 B instead of 32 B per contact)
//   pk4  = (x, y, z, kappa)                     for the updates      (16 B instead of 20 B per contact)
// and the two records of an evaluation travel through DIFFERENT data pipes (LSU / TEX).  The records are written
// by the kernels that produce v* / kappa.  Same arithmetic as k_vel_divergence / k_vel_update.
// ------------------------------------------------------------------------------------------------
template <bool PREDICT>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_vel_divergence_u(const float4* __restrict__ pvx, cudaTextureObject_t tpvx, const float2* __restrict__ vyz, cudaTextureObject_t tvyz,
                   const float4* __restrict__ bpos, const float4* __restrict__ bvel, Lists L, const float* __restrict__ dens,
                   const float* __restrict__ alpha, float* __restrict__ out, float4* __restrict__ pk4, float* __restrict__ partial, float dt,
                   int* __restrict__ err, uint32_t* __restrict__ ticket, float* __restrict__ errsum, Range rg) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < rg.count;
    i += rg.begin;
    float e = 0.f;
    if (valid) {
        const float4 a = pvx[i];
        const float2 b = vyz[i];
        const float4 pi = make_float4(a.x, a.y, a.z, 0.f);
        const float vix = a.w, viy = b.x, viz = b.y;
        const float rho0 = C.fluids[0].density0, mass = C.fluids[0].mass;
        float d = 0.f;
        if (PREDICT || L.cnt_f[i] + L.cnt_b[i] >= 20u) {
            // even contacts fetch (pvx via TEX, vyz via LSU), odd ones the other way round, so both pipes carry the same load
            for_fluid_grads(
                i, pi, L, [&](uint32_t j, int u) { return !(u & 1) ? tex1Dfetch<float4>(tpvx, (int)j) : __ldg(&pvx[j]); },
                [&](uint32_t j, int u) { return !(u & 1) ? __ldg(&vyz[j]) : tex1Dfetch<float2>(tvyz, (int)j); },
                [&](uint32_t, const Pair& p, const float4& pj, const float2& wj) {
                    float dv = (vix - pj.w) * p.dx + (viy - wj.x) * p.dy + (viz - wj.y) * p.dz;
                    d = fmaf(dv * p.g, mass, d);
                });
            for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
                float dv;
                if (PREDICT) {
                    float4 vj = __ldg(&bvel[j]);
                    dv = (vix - vj.x) * p.dx + (viy - vj.y) * p.dy + (viz - vj.z) * p.dz;
                } else {
                    dv = vix * p.dx + viy * p.dy + viz * p.dz;
                }
                d = fmaf(dv * p.g, pj.w * rho0, d);
            });
        }
        float kap;
        if (PREDICT) {
            float pd = fmaf(d, dt, dens[i]);
            if (pd == 0.f) atomicOr(err, 1);
            out[i] = pd;
            kap = fmaxf((pd - rho0) * alpha[i], 0.f);
            e = pd < rho0 ? 0.f : pd / rho0 - 1.0f;
        } else {
            d = fmaxf(d, 0.f);
            out[i] = d;
            kap = d * alpha[i];
            e = d / rho0;
        }
        pk4[i] = make_float4(a.x, a.y, a.z, kap);
    }
    reduce_error<false>(e, 0u, valid, partial, sm, ticket, errsum);
}

// compute_divergences (a7) + the fluid term of XSPHViscosity::solve (a12, xsph_viscosity.rs:52-69) in ONE sweep.
// XSPH is evaluated on `fluid.velocities` right after update_velocities folded vc into them (dfsph_solver.rs:688-697),
// i.e. on exactly the v* the divergence loop's LAST evaluation gathers; so every stand-alone evaluation also accumulates
// the XSPH sums (one extra 4-byte gather of rho_j and the kernel value per contact) and the last one's are used:
// k_fold_velocities adds xs * inv_dt to the gravity it writes and the separate XSPH pass is skipped.  Same per-contact
// arithmetic and summation order as k_force_xsph; padded self slots contribute c * (v_i - v_i) = 0.
struct VyzRho {
    float2 v;
    float rho;
};
// EXTRA = 1: XSPH sums (above) -> xs.   EXTRA = 2: Akinci2013 compute_normals (akinci2013_surface_tension.rs:43-68) rides along
// instead: n_i = h sum_j (m_j / rho_j) grad W_ij needs positions and densities only, so ANY stand-alone evaluation of the
// step may produce it; the output record nr4 = (n_x, n_y, n_z, rho_i) is what k_akinci_force_u gathers (one float4 instead
// of a normal and a density), and the separate normals pass is skipped.
template <int EXTRA>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)  // 64 registers: the extra sums spill at 56
k_vel_divergence_xsph_u(const float4* __restrict__ pvx, cudaTextureObject_t tpvx, const float2* __restrict__ vyz, cudaTextureObject_t tvyz,
                        const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens, const float* __restrict__ alpha,
                        float* __restrict__ out, float4* __restrict__ pk4, float* __restrict__ partial, uint32_t* __restrict__ ticket,
                        float* __restrict__ errsum, float4* __restrict__ xs, float cf, Range rg) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < rg.count;
    i += rg.begin;
    float e = 0.f;
    if (valid) {
        const float4 a = pvx[i];
        const float2 b = vyz[i];
        const float4 pi = make_float4(a.x, a.y, a.z, 0.f);
        const float vix = a.w, viy = b.x, viz = b.y;
        const float rho0 = C.fluids[0].density0, mass = C.fluids[0].mass;
        const bool gated = L.cnt_f[i] + L.cnt_b[i] < 20u;  // dfsph_solver.rs:301-314
        float d = 0.f, fx = 0.f, fy = 0.f, fz = 0.f;
        for_fluid_grads<EXTRA == 1>(
            i, pi, L, [&](uint32_t j, int u) { return !(u & 1) ? tex1Dfetch<float4>(tpvx, (int)j) : __ldg(&pvx[j]); },
            [&](uint32_t j, int u) { return VyzRho{!(u & 1) ? __ldg(&vyz[j]) : tex1Dfetch<float2>(tvyz, (int)j), __ldg(&dens[j])}; },
            [&](uint32_t, const Pair& p, const float4& pj, const VyzRho& wj) {
                float dv = (vix - pj.w) * p.dx + (viy - wj.v.x) * p.dy + (viz - wj.v.y) * p.dz;
                d = fmaf(dv * p.g, mass, d);
                if (EXTRA == 1) {
                    float c = cf * p.w * mass / wj.rho;  // coeff * W * (vol_j * rho0) / rho_j
                    fx = fmaf(c, pj.w - vix, fx); fy = fmaf(c, wj.v.x - viy, fy); fz = fmaf(c, wj.v.y - viz, fz);
                } else {
                    float c = p.g * (mass / wj.rho);
                    fx = fmaf(c, p.dx, fx); fy = fmaf(c, p.dy, fy); fz = fmaf(c, p.dz, fz);
                }
            });
        if (gated) {
            d = 0.f;
        } else {
            for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
                float dv = vix * p.dx + viy * p.dy + viz * p.dz;
                d = fmaf(dv * p.g, pj.w * rho0, d);
            });
        }
        d = fmaxf(d, 0.f);
        out[i] = d;
        e = d / rho0;
        pk4[i] = make_float4(a.x, a.y, a.z, d * alpha[i]);
        if (EXTRA == 1) xs[i] = make_float4(fx, fy, fz, 0.f);
        else xs[i] = make_float4(fx * C.h, fy * C.h, fz * C.h, dens[i]);
    }
    reduce_error<false>(e, 0u, valid, partial, sm, ticket, errsum);
}

// a14 pass 2 for a single uniform-mass fluid on the records of the fused pass: positions from pvx4 (texture pipe) and
// nr4 = (n_x, n_y, n_z, rho) (LSU pipe): two gathers per contact instead of three.  Akinci2013SurfaceTension::solve
// akinci2013_surface_tension.rs:113-192.
template <bool BFORCE>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_akinci_force_u(const float4* __restrict__ pvx, cudaTextureObject_t tpvx, const float4* __restrict__ nr4, const float4* __restrict__ bpos, Lists L,
                 float4* __restrict__ acc, float* __restrict__ bforce, float gamma, float adh, float coh_norm, float h6_64, float adh_norm) {
    SPH_OWNED_INDEX(i)
    const float4 a = pvx[i];
    const float4 ni = nr4[i];
    const float rho0 = C.fluids[0].density0, mass = C.fluids[0].mass;
    const float4 pi = make_float4(a.x, a.y, a.z, mass);
    const float rho_i = ni.w;
    float ax = 0.f, ay = 0.f, az = 0.f;
    if (gamma != 0.f)
        for_fluid_contacts_g<false, false>(
            i, pi, L, [&](uint32_t j) { return tex1Dfetch<float4>(tpvx, (int)j); }, [&](uint32_t j) { return __ldg(&nr4[j]); },
            [&](uint32_t, const Pair& p, const float4&, const float4& nj) {
                // cohesion_vec = dir * C(dist) if |dpos|^2 > eps^2 (Unit::try_new_and_get)
                float coh = p.d2 > F32_EPS * F32_EPS ? cohesion_kernel(p.r, coh_norm, h6_64) / p.r : 0.f;
                float cm = coh * (-gamma * mass);
                float kij = 2.0f * rho0 / (rho_i + nj.w);
                ax += (-gamma * (ni.x - nj.x) + cm * p.dx) * kij;
                ay += (-gamma * (ni.y - nj.y) + cm * p.dy) * kij;
                az += (-gamma * (ni.z - nj.z) + cm * p.dz) * kij;
            });
    if (adh != 0.f)
        for_boundary_contacts<false, false>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float ad = p.d2 > F32_EPS * F32_EPS ? adhesion_kernel(p.r, adh_norm) / p.r : 0.f;
            float c = ad * adh * (pj.w * rho0);
            ax -= c * p.dx; ay -= c * p.dy; az -= c * p.dz;
            if (BFORCE) {  // apply_force(c.j, adhesion_acc * m_i) :188
                atomicAdd(&bforce[3 * (size_t)j + 0], c * p.dx * mass);
                atomicAdd(&bforce[3 * (size_t)j + 1], c * p.dy * mass);
                atomicAdd(&bforce[3 * (size_t)j + 2], c * p.dz * mass);
            }
        });
    float4 o = acc[i];
    o.x += ax; o.y += ay; o.z += az;
    acc[i] = o;
}

// The (x, y, z, kappa) gathers of every group of four contacts are split between the two L1TEX front ends: contacts 0 and 2
// through the texture pipe, 1 and 3 through the LSU pipe, so both carry half the wavefronts.
template <bool BFORCE, bool PRESSURE>
__global__ void __launch_bounds__(PASS_T, SPH_PASS_MINB)
k_vel_update_u(const float4* __restrict__ pk4, cudaTextureObject_t tpk, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L,
               float4* __restrict__ vc, float4* __restrict__ vs, float4* __restrict__ pvx, float2* __restrict__ vyz, float* __restrict__ bforce,
               float inv_dt, Range rg) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rg.count) return;
    i += rg.begin;
    const float4 a = pk4[i];
    const float4 pi = make_float4(a.x, a.y, a.z, 0.f);
    const float ki = a.w;
    const float4 v = vel[i];
    const float rho0 = C.fluids[0].density0, mass = C.fluids[0].mass;
    const float scale = (PRESSURE ? inv_dt : 1.0f) * mass;
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads(
        i, pi, L, [&](uint32_t j, int u) { return !(u & 1) ? tex1Dfetch<float4>(tpk, (int)j) : __ldg(&pk4[j]); }, [](uint32_t) { return NoAux{}; },
        [&](uint32_t, const Pair& p, const float4& pj, NoAux) {
            float c = (ki + pj.w) * scale * p.g;
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    if (!PRESSURE || ki > 0.f) {
        const float bscale = PRESSURE ? inv_dt : 1.0f;
        for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float c = ki * pj.w * rho0 * bscale * p.g;
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
            if (BFORCE) {
                float s = c * inv_dt * mass;
                atomicAdd(&bforce[3 * (size_t)j + 0], s * p.dx);
                atomicAdd(&bforce[3 * (size_t)j + 1], s * p.dy);
                atomicAdd(&bforce[3 * (size_t)j + 2], s * p.dz);
            }
        });
    }
    float4 c4 = vc[i];
    c4.x -= ax; c4.y -= ay; c4.z -= az;
    vc[i] = c4;
    const float sx = v.x + c4.x, sy = v.y + c4.y, sz = v.z + c4.z;
    vs[i] = make_float4(sx, sy, sz, 0.f);
    pvx[i] = make_float4(a.x, a.y, a.z, sx);
    vyz[i] = make_float2(sy, sz);
}

// ------------------------------------------------------------------------------------------------
// Nonpressure forces (predict_advection dfsph_solver.rs:565-604).  Only contacts of the SAME fluid
// count (c.i_model == c.j_model); `which` selects the fluid a force instance belongs to.
// ------------------------------------------------------------------------------------------------
struct VelRho {
    float4 v;
    float rho;
};
// a12: XSPHViscosity::solve xsph_viscosity.rs:30-95
template <bool MULTI, bool BFORCE>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_force_xsph(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, const float4* __restrict__ bvel, Lists L,
             const float* __restrict__ dens, float4* __restrict__ acc, float* __restrict__ bforce, uint32_t which, float cf, float cb, float inv_dt) {
    SPH_OWNED_INDEX(i)
    float4 vi = vel[i];
    if (MULTI && fid_of(vi) != which) return;
    float4 pi = pos[i];
    float rho0 = C.fluids[which].density0;
    float fx = 0.f, fy = 0.f, fz = 0.f, bx = 0.f, by = 0.f, bz = 0.f;
    if (cf != 0.f)
        for_fluid_contacts<true, false>(
            i, pi, L, pos, [&](uint32_t j) { return VelRho{__ldg(&vel[j]), __ldg(&dens[j])}; },
            [&](uint32_t, const Pair& p, const float4& pj, const VelRho& a) {
                if (MULTI && fid_of(a.v) != which) return;
                float c = cf * p.w * pj.w / a.rho;  // coeff * W * (vol_j * rho0) / rho_j
                fx = fmaf(c, a.v.x - vi.x, fx); fy = fmaf(c, a.v.y - vi.y, fy); fz = fmaf(c, a.v.z - vi.z, fz);
            });
    if (cb != 0.f) {
        float rho_i = dens[i];
        for_boundary_contacts<true, false>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float4 vj = __ldg(&bvel[j]);
            float c = cb * p.w * pj.w * rho0 / rho_i;
            float dx = c * (vj.x - vi.x), dy = c * (vj.y - vi.y), dz = c * (vj.z - vi.z);
            bx += dx; by += dy; bz += dz;
            if (BFORCE) {  // apply_force(c.j, delta * (-m_i * inv_dt)) :87-88
                float s = -pi.w * inv_dt;
                atomicAdd(&bforce[3 * (size_t)j + 0], s * dx);
                atomicAdd(&bforce[3 * (size_t)j + 1], s * dy);
                atomicAdd(&bforce[3 * (size_t)j + 2], s * dz);
            }
        });
    }
    float4 a = acc[i];
    a.x += fx * inv_dt + bx * inv_dt; a.y += fy * inv_dt + by * inv_dt; a.z += fz * inv_dt + bz * inv_dt;
    acc[i] = a;
}

// a13: ArtificialViscosity::solve artificial_viscosity.rs:40-124
template <bool MULTI, bool BFORCE>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_force_artificial(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, const float4* __restrict__ bvel, Lists L,
                   const float* __restrict__ dens, float4* __restrict__ acc, float* __restrict__ bforce, uint32_t which, float cf, float cb, float alpha,
                   float beta, float cs) {
    SPH_OWNED_INDEX(i)
    float4 vi = vel[i];
    if (MULTI && fid_of(vi) != which) return;
    float4 pi = pos[i];
    float rho0 = C.fluids[which].density0;
    float rho_i = dens[i];
    float eta2 = C.h * C.h * 0.01f;
    float fx = 0.f, fy = 0.f, fz = 0.f, bx = 0.f, by = 0.f, bz = 0.f;
    if (cf != 0.f)
        for_fluid_grads_pos(
            i, pi, L, pos, [&](uint32_t j) { return VelRho{__ldg(&vel[j]), __ldg(&dens[j])}; },
            [&](uint32_t, const Pair& p, const float4& pj, const VelRho& a) {
                if (MULTI && fid_of(a.v) != which) return;
                float vr = p.dx * (vi.x - a.v.x) + p.dy * (vi.y - a.v.y) + p.dz * (vi.z - a.v.z);
                if (vr < 0.f) {
                    float davg = (rho_i + a.rho) * 0.5f;
                    float mu = C.h * vr / (p.d2 + eta2);
                    float c = cf * (cs * alpha * mu - beta * mu * mu) * (pj.w / davg) * p.g;
                    fx = fmaf(c, p.dx, fx); fy = fmaf(c, p.dy, fy); fz = fmaf(c, p.dz, fz);
                }
            });
    if (cb != 0.f)
        for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float4 vj = __ldg(&bvel[j]);
            float vr = p.dx * (vi.x - vj.x) + p.dy * (vi.y - vj.y) + p.dz * (vi.z - vj.z);
            if (vr < 0.f) {
                float mu = C.h * vr / (p.d2 + eta2);
                float c = cb * (cs * alpha * mu - beta * mu * mu) * (pj.w * rho0 / rho_i) * p.g;
                bx = fmaf(c, p.dx, bx); by = fmaf(c, p.dy, by); bz = fmaf(c, p.dz, bz);
                if (BFORCE) {  // apply_force(c.j, boundary_acc * -m_i): the RUNNING sum, as the reference (:117)
                    atomicAdd(&bforce[3 * (size_t)j + 0], -pi.w * bx);
                    atomicAdd(&bforce[3 * (size_t)j + 1], -pi.w * by);
                    atomicAdd(&bforce[3 * (size_t)j + 2], -pi.w * bz);
                }
            }
        });
    float4 a = acc[i];
    a.x += fx + bx; a.y += fy + by; a.z += fz + bz;
    acc[i] = a;
}

struct FidRho {
    uint32_t fid;
    float rho;
};
// a14 pass 1: Akinci2013 compute_normals akinci2013_surface_tension.rs:43-68
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_akinci_normals(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, const float* __restrict__ dens, float4* __restrict__ normals,
                 uint32_t which) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    float nx = 0.f, ny = 0.f, nz = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return FidRho{MULTI ? fid_of(__ldg(&vel[j])) : 0u, __ldg(&dens[j])}; },
        [&](uint32_t, const Pair& p, const float4& pj, const FidRho& a) {
            if (MULTI && a.fid != which) return;
            float c = p.g * (pj.w / a.rho);
            nx = fmaf(c, p.dx, nx); ny = fmaf(c, p.dy, ny); nz = fmaf(c, p.dz, nz);
        });
    normals[i] = make_float4(nx * C.h, ny * C.h, nz * C.h, 0.f);
}

struct NrmRho {
    float4 n;
    float rho;
    uint32_t fid;
};
// a14 pass 2: Akinci2013SurfaceTension::solve akinci2013_surface_tension.rs:113-192
template <bool MULTI, bool BFORCE>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_akinci_force(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
               const float4* __restrict__ normals, float4* __restrict__ acc, float* __restrict__ bforce, uint32_t which, float gamma, float adh,
               float coh_norm, float h6_64, float adh_norm) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    float rho0 = C.fluids[which].density0;
    float rho_i = dens[i];
    float4 ni = normals[i];
    float ax = 0.f, ay = 0.f, az = 0.f;
    if (gamma != 0.f)
        for_fluid_contacts<false, false>(
            i, pi, L, pos, [&](uint32_t j) { return NrmRho{__ldg(&normals[j]), __ldg(&dens[j]), MULTI ? fid_of(__ldg(&vel[j])) : 0u}; },
            [&](uint32_t, const Pair& p, const float4& pj, const NrmRho& a) {
                if (MULTI && a.fid != which) return;
                // cohesion_vec = dir * C(dist) if |dpos|^2 > eps^2 (Unit::try_new_and_get)
                float coh = p.d2 > F32_EPS * F32_EPS ? cohesion_kernel(p.r, coh_norm, h6_64) / p.r : 0.f;
                float cm = coh * (-gamma * pj.w);
                float kij = 2.0f * rho0 / (rho_i + a.rho);
                ax += (-gamma * (ni.x - a.n.x) + cm * p.dx) * kij;
                ay += (-gamma * (ni.y - a.n.y) + cm * p.dy) * kij;
                az += (-gamma * (ni.z - a.n.z) + cm * p.dz) * kij;
            });
    if (adh != 0.f)
        for_boundary_contacts<false, false>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float ad = p.d2 > F32_EPS * F32_EPS ? adhesion_kernel(p.r, adh_norm) / p.r : 0.f;
            float c = ad * adh * (pj.w * rho0);
            ax -= c * p.dx; ay -= c * p.dy; az -= c * p.dz;
            if (BFORCE) {  // apply_force(c.j, adhesion_acc * m_i) :188
                atomicAdd(&bforce[3 * (size_t)j + 0], c * p.dx * pi.w);
                atomicAdd(&bforce[3 * (size_t)j + 1], c * p.dy * pi.w);
                atomicAdd(&bforce[3 * (size_t)j + 2], c * p.dz * pi.w);
            }
        });
    float4 a = acc[i];
    a.x += ax; a.y += ay; a.z += az;
    acc[i] = a;
}

// ------------------------------------------------------------------------------------------------
// He2014SurfaceTension (surface_tension/he2014_surface_tension.rs): colours -> squared colour-gradient norms -> forces.
// ------------------------------------------------------------------------------------------------
// pass 1: compute_colors :40-75
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_he2014_colors(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
                float* __restrict__ colors, uint32_t which) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    float color = 0.f;
    for_fluid_contacts<true, false>(
        i, pi, L, pos, [&](uint32_t j) { return FidRho{MULTI ? fid_of(__ldg(&vel[j])) : 0u, __ldg(&dens[j])}; },
        [&](uint32_t, const Pair& p, const float4& pj, const FidRho& a) {
            if (MULTI && a.fid != which) return;
            color += p.w * pj.w / a.rho;  // c.weight * m_j / rho_j
        });
    for_boundary_contacts<true, false>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) { color += p.w * pj.w; });  // W * vol_b
    colors[i] = color;
}

struct FidRhoVal {
    uint32_t fid;
    float rho, val;
};
// pass 2: compute_gradc :77-105 -> |sum_j grad W_ij c_j m_j / rho_j / c_i|^2
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_he2014_gradc(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, const float* __restrict__ dens, const float* __restrict__ colors,
               float* __restrict__ gradc, uint32_t which) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    float gx = 0.f, gy = 0.f, gz = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return FidRhoVal{MULTI ? fid_of(__ldg(&vel[j])) : 0u, __ldg(&dens[j]), __ldg(&colors[j])}; },
        [&](uint32_t, const Pair& p, const float4& pj, const FidRhoVal& a) {
            if (MULTI && a.fid != which) return;
            float c = p.g * a.val * pj.w / a.rho;
            gx = fmaf(c, p.dx, gx); gy = fmaf(c, p.dy, gy); gz = fmaf(c, p.dz, gz);
        });
    float ci = colors[i];
    float qx = gx / ci, qy = gy / ci, qz = gz / ci;
    gradc[i] = (qx * qx + qy * qy) + qz * qz;
}

// pass 3: forces :131-178
template <bool MULTI, bool BFORCE>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_he2014_force(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
               const float* __restrict__ gradc, float4* __restrict__ acc, float* __restrict__ bforce, uint32_t which, float cf, float cb) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    const float rho0 = C.fluids[which].density0;
    const float mi = pi.w, rho_i = dens[i], gi = gradc[i];
    float ax = 0.f, ay = 0.f, az = 0.f;
    if (cf != 0.f) {
        const float k = cf / (2.0f * mi);
        for_fluid_grads_pos(
            i, pi, L, pos, [&](uint32_t j) { return FidRhoVal{MULTI ? fid_of(__ldg(&vel[j])) : 0u, __ldg(&dens[j]), __ldg(&gradc[j])}; },
            [&](uint32_t, const Pair& p, const float4& pj, const FidRhoVal& a) {
                if (MULTI && a.fid != which) return;
                float s = p.g * (mi / rho_i * pj.w / a.rho * (gi + a.val) / 2.0f);
                ax += s * p.dx * k; ay += s * p.dy * k; az += s * p.dz * k;
            });
    }
    if (cb != 0.f)
        for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
            float mj = pj.w * rho0;
            float s = p.g * (mi / rho_i * mj / rho0 * gi * cb * 0.25f);
            float fx = s * p.dx, fy = s * p.dy, fz = s * p.dz;
            ax += fx / mi; ay += fy / mi; az += fz / mi;
            if (BFORCE) {  // apply_force(c.j, -f) :175
                atomicAdd(&bforce[3 * (size_t)j + 0], -fx);
                atomicAdd(&bforce[3 * (size_t)j + 1], -fy);
                atomicAdd(&bforce[3 * (size_t)j + 2], -fz);
            }
        });
    float4 a = acc[i];
    a.x += ax; a.y += ay; a.z += az;
    acc[i] = a;
}

// WCSPHSurfaceTension fluid term (surface_tension/wcsph_surface_tension.rs:45-63): a_i -= k W_ij m_j / m_i x_ij
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T, SPH_FORCE_MINB)
k_wcsph_force(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, float4* __restrict__ acc, uint32_t which, float cf) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    float4 pi = pos[i];
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_contacts<true, false>(
        i, pi, L, pos, [&](uint32_t j) { return MULTI ? fid_of(__ldg(&vel[j])) : 0u; },
        [&](uint32_t, const Pair& p, const float4& pj, uint32_t fj) {
            if (MULTI && fj != which) return;
            float c = -cf * p.w * pj.w / pi.w;
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    float4 a = acc[i];
    a.x += ax; a.y += ay; a.z += az;
    acc[i] = a;
}

}  // namespace sphk
