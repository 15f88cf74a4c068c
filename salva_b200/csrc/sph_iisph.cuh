// sph_iisph.cuh — IISPH pressure solver kernels (iisph_solver.rs), default gather backend.
//
// Per-contact gathers are minimised by pre-combining per-particle quantities in the producing kernel:
//   prho_j = p_j / rho_j^2                        (gathered by compute_dij_pjl and compute_velocity_changes)
//   s_j    = dii_j * p_j + dij_pjl_j              (the only neighbour vector compute_next_pressures needs:
//            factor = dij_pjl_i - dii_j p_j - (dij_pjl_j - d_ji p_i) = dij_pjl_i - s_j + d_ji p_i, iisph_solver.rs:307-312)
#pragma once
#include "sph_passes.cuh"

struct IisphState {
    float4* dii = nullptr;      // iisph_solver.rs:32
    float4* dij_pjl = nullptr;  // iisph_solver.rs:34
    float4* s = nullptr;        // dii * p + dij_pjl
    float* aii = nullptr;       // iisph_solver.rs:33
    float* next_p = nullptr;    // iisph_solver.rs:38
    float* prho = nullptr;      // p / rho^2
    float* next_prho = nullptr;
    size_t cap = 0;
    cudaTextureObject_t tex_s = 0;
};

namespace sphk {

// pressures *= 0.5 (iisph_solver.rs:673-677) and prho = p / rho^2
__global__ void k_iisph_warm_start(float* __restrict__ p, const float* __restrict__ dens, float* __restrict__ prho) {
    SPH_OWNED_INDEX(i)
    float v = p[i] * 0.5f;
    float r = dens[i];
    p[i] = v;
    prho[i] = v / (r * r);
}

// compute_dii iisph_solver.rs:144-186
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T)
k_iisph_dii(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
            float4* __restrict__ dii, float dt) {
    SPH_OWNED_INDEX(i)
    float4 pi = pos[i];
    float rho0 = C.fluids[MULTI ? fid_of(vel[i]) : 0].density0;
    float rhoi = dens[i];
    float factor = -dt * dt / (rhoi * rhoi);
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [](uint32_t) { return NoAux{}; },
        [&](uint32_t, const Pair& p, const float4& pj, NoAux) {
            float c = p.g * (pj.w * factor);
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
        float c = p.g * (pj.w * rho0 * factor);
        ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
    });
    dii[i] = make_float4(ax, ay, az, 0.f);
}

// compute_aii iisph_solver.rs:188-233
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T)
k_iisph_aii(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
            const float4* __restrict__ dii, float* __restrict__ aii, float dt) {
    SPH_OWNED_INDEX(i)
    float4 pi = pos[i];
    float rho0 = C.fluids[MULTI ? fid_of(vel[i]) : 0].density0;
    float rhoi = dens[i];
    float4 di = dii[i];
    float factor = dt * dt * pi.w / (rhoi * rhoi);
    float a = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [](uint32_t) { return NoAux{}; },
        [&](uint32_t, const Pair& p, const float4& pj, NoAux) {
            float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;  // gradient; d_ji = gradient * factor
            a = fmaf(pj.w, (di.x - gx * factor) * gx + (di.y - gy * factor) * gy + (di.z - gz * factor) * gz, a);
        });
    for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
        float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;
        a = fmaf(pj.w * rho0, (di.x - gx * factor) * gx + (di.y - gy * factor) * gy + (di.z - gz * factor) * gz, a);
    });
    aii[i] = a;
}

// compute_dij_pjl iisph_solver.rs:235-268 (+ s_i = dii_i p_i + dij_pjl_i for the next kernel's gather)
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T)
k_iisph_dij_pjl(const float4* __restrict__ pos, Lists L, const float* __restrict__ prho, const float* __restrict__ press, const float4* __restrict__ dii,
                float4* __restrict__ dij_pjl, float4* __restrict__ s, float dt) {
    SPH_OWNED_INDEX(i)
    float4 pi = pos[i];
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return __ldg(&prho[j]); },
        [&](uint32_t, const Pair& p, const float4& pj, float prj) {
            float c = p.g * (-pj.w * prj);
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    float dt2 = dt * dt;
    ax *= dt2; ay *= dt2; az *= dt2;
    dij_pjl[i] = make_float4(ax, ay, az, 0.f);
    float4 di = dii[i];
    float p = press[i];
    s[i] = make_float4(fmaf(di.x, p, ax), fmaf(di.y, p, ay), fmaf(di.z, p, az), 0.f);
}

// compute_next_pressures iisph_solver.rs:270-353
template <bool MULTI, bool TEX>
__global__ void __launch_bounds__(PASS_T)
k_iisph_next_pressures(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L, const float* __restrict__ dens,
                       const float* __restrict__ pred, const float* __restrict__ aii, const float* __restrict__ press, const float4* __restrict__ dij_pjl,
                       const float4* __restrict__ s, cudaTextureObject_t ts, float* __restrict__ next_p, float* __restrict__ next_prho,
                       float* __restrict__ partial, float dt, float omega) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < C.n_owned;
    i += C.i_begin;
    float e = 0.f;
    uint32_t fi = 0;
    if (valid) {
        fi = MULTI ? fid_of(vel[i]) : 0u;
        float rho0 = C.fluids[fi].density0;
        float a = aii[i];
        float np = 0.f;
        float rhoi = dens[i];
        if (fabsf(a) > 1.0e-9f) {
            float4 pi = pos[i];
            float p_i = press[i];
            float4 dj = dij_pjl[i];
            float dji_f = dt * dt * pi.w / (rhoi * rhoi) * p_i;  // d_ji p_i = gradient * dji_f
            float derr = rho0 - pred[i];
            float sum = 0.f;
            for_fluid_grads_pos(
                i, pi, L, pos, [&](uint32_t j) { return fetch4<TEX>(s, ts, j); },
                [&](uint32_t, const Pair& p, const float4& pj, const float4& sj) {
                    float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;
                    float fx = dj.x - sj.x + gx * dji_f, fy = dj.y - sj.y + gy * dji_f, fz = dj.z - sj.z + gz * dji_f;
                    sum = fmaf(pj.w, fx * gx + fy * gy + fz * gz, sum);
                });
            for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t, const Pair& p, const float4& pj) {
                sum = fmaf(pj.w * rho0, p.g * (dj.x * p.dx + dj.y * p.dy + dj.z * p.dz), sum);
            });
            np = (1.0f - omega) * p_i + omega * (derr - sum) / a;
            if (np > 0.f) e = (-sum - a * np) / rho0;
            else np = 0.f;  // clamp negative pressures (:338-342)
        }
        next_p[i] = np;
        next_prho[i] = np / (rhoi * rhoi);
    }
    reduce_error<MULTI>(e, fi, valid, partial, sm);
}

// compute_velocity_changes iisph_solver.rs:355-404
template <bool MULTI, bool BFORCE>
__global__ void __launch_bounds__(PASS_T)
k_iisph_velocity_changes(const float4* __restrict__ pos, const float4* __restrict__ vel, const float4* __restrict__ bpos, Lists L,
                         const float* __restrict__ prho, float4* __restrict__ vc, float* __restrict__ bforce, float dt) {
    SPH_OWNED_INDEX(i)
    float4 pi = pos[i];
    float rho0 = C.fluids[MULTI ? fid_of(vel[i]) : 0].density0;
    float pri = prho[i];
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return __ldg(&prho[j]); },
        [&](uint32_t, const Pair& p, const float4& pj, float prj) {
            float c = p.g * (dt * pj.w * (pri + prj));
            ax = fmaf(c, p.dx, ax); ay = fmaf(c, p.dy, ay); az = fmaf(c, p.dz, az);
        });
    for_boundary_contacts<false, true>(i, pi, L, bpos, [&](uint32_t j, const Pair& p, const float4& pj) {
        float c = p.g * (pj.w * rho0 * pri);  // acc = gradient * (m_b p_i / rho_i^2)
        ax = fmaf(c * dt, p.dx, ax); ay = fmaf(c * dt, p.dy, ay); az = fmaf(c * dt, p.dz, az);
        if (BFORCE) {  // apply_force(c.j, acc * m_i) :399-401
            atomicAdd(&bforce[3 * (size_t)j + 0], c * p.dx * pi.w);
            atomicAdd(&bforce[3 * (size_t)j + 1], c * p.dy * pi.w);
            atomicAdd(&bforce[3 * (size_t)j + 2], c * p.dz * pi.w);
        }
    });
    float4 c4 = vc[i];
    c4.x -= ax; c4.y -= ay; c4.z -= az;
    vc[i] = c4;
}

// update_velocities_and_positions iisph_solver.rs:406-420 + zero vc :707-709
__global__ void k_iisph_update(float4* __restrict__ pos, float4* __restrict__ vel, float4* __restrict__ vc, float dt) {
    SPH_OWNED_INDEX(i)
    float4 p = pos[i], v = vel[i], c = vc[i];
    v.x += c.x; v.y += c.y; v.z += c.z;
    p.x += v.x * dt; p.y += v.y * dt; p.z += v.z * dt;
    vel[i] = v;
    pos[i] = p;
    vc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

}  // namespace sphk
