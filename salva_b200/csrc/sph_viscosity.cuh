// sph_viscosity.cuh — DFSPHViscosity (viscosity/dfsph_viscosity.rs, SURVEY row a16), default gather backend.
//
// Per solve: betas (one gather pass + a 6x6 LU inverse per particle), strain-rate targets (one pass), then the
// reference's Jacobi loop: strain-rate errors (one pass + error mean) / accelerations (one pass).  Per-contact gathers are
// pre-combined per particle: vv = vel + acc * dt (strain rates) and u = beta * error / rho^2 (accelerations; the
// reference recomputes u_j per contact from the 36-float beta_j).
// The 6x6 inverse restates nalgebra 0.33's LU (partial pivoting, reciprocal-scaled multipliers, unfused axpy updates),
// exactly as oracle/oracle.cpp does, with __fmul_rn/__fadd_rn so that nvcc cannot contract what the reference keeps apart.
#pragma once
#include "sph_passes.cuh"

struct ViscosityState {
    float* beta = nullptr;    // beta[(r * 6 + c) * stride + i]
    float* target = nullptr;  // target[k * stride + i]            dfsph_viscosity.rs:24
    float4* vv = nullptr;     // vel + acc * dt
    float4* u4 = nullptr;     // u[0..3]
    float2* u2 = nullptr;     // u[4..5]
    size_t cap = 0;
};

namespace sphk {

__global__ void k_visc_vv(const float4* __restrict__ vel, const float4* __restrict__ acc, float dt, float4* __restrict__ vv) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C.n_fluid) return;  // ghosts included (a slab world would need them; single-GPU worlds have none)
    float4 v = vel[i], a = acc[i];
    vv[i] = make_float4(fmaf(a.x, dt, v.x), fmaf(a.y, dt, v.y), fmaf(a.z, dt, v.z), v.w);
}

// nalgebra LU::new + determinant + try_inverse on a 6x6 (see oracle.cpp lu6_*).  Returns false => beta = 0.
__device__ inline bool lu6_inverse(float a[6][6], float out[6][6]) {
    int sw_a[6], sw_b[6], nsw = 0;
    for (int i = 0; i < 6; ++i) {
        int piv = i;
        float best = fabsf(a[i][i]);
        for (int r = i + 1; r < 6; ++r)
            if (fabsf(a[r][i]) > best) {
                best = fabsf(a[r][i]);
                piv = r;
            }
        float diag = a[piv][i];
        if (diag == 0.f) continue;
        if (piv != i) {
            sw_a[nsw] = i;
            sw_b[nsw] = piv;
            ++nsw;
            for (int c = 0; c < 6; ++c) {
                float t = a[i][c];
                a[i][c] = a[piv][c];
                a[piv][c] = t;
            }
        }
        float inv_diag = __fdiv_rn(1.0f, diag);
        for (int r = i + 1; r < 6; ++r) a[r][i] = __fmul_rn(a[r][i], inv_diag);
        for (int k = i + 1; k < 6; ++k) {
            float mp = -a[i][k];
            for (int r = i + 1; r < 6; ++r) a[r][k] = __fadd_rn(__fmul_rn(mp, a[r][i]), a[r][k]);
        }
    }
    float det = 1.f;
    for (int i = 0; i < 6; ++i) det = __fmul_rn(det, a[i][i]);
    if (fabsf(det) < 1.0e-6f) return false;  // dfsph_viscosity.rs:187
    for (int r = 0; r < 6; ++r)
        for (int c = 0; c < 6; ++c) out[r][c] = r == c ? 1.f : 0.f;
    for (int s = 0; s < nsw; ++s)
        for (int c = 0; c < 6; ++c) {
            float t = out[sw_a[s]][c];
            out[sw_a[s]][c] = out[sw_b[s]][c];
            out[sw_b[s]][c] = t;
        }
    for (int k = 0; k < 6; ++k)
        for (int i = 0; i < 5; ++i) {
            float coeff = out[i][k];
            for (int r = i + 1; r < 6; ++r) out[r][k] = __fadd_rn(__fmul_rn(-coeff, a[r][i]), out[r][k]);
        }
    for (int k = 0; k < 6; ++k)
        for (int i = 5; i >= 0; --i) {
            float diag = a[i][i];
            if (diag == 0.f) return false;
            float coeff = __fdiv_rn(out[i][k], diag);
            out[i][k] = coeff;
            for (int r = 0; r < i; ++r) out[r][k] = __fadd_rn(__fmul_rn(-coeff, a[r][i]), out[r][k]);
        }
    return true;
}

// rows of compute_gradient_matrix(g) * s (dfsph_viscosity.rs:59-82): r0 = (a,0,0) r1 = (0,b,0) r2 = (0,0,c)
// r3 = (Y,X,0) r4 = (Z,0,X) r5 = (0,Z,Y) with a = 2 gx s ... X = gx s ...; M M^T has 15 structurally non-zero unique entries.
struct Sym15 {
    float e00, e03, e04, e11, e13, e15, e22, e24, e25, e33, e34, e35, e44, e45, e55;
};
__device__ __forceinline__ void outer15(float a, float b, float c, float X, float Y, float Z, float rho, Sym15& s) {
    // every entry is (sum over k of products) / rho_i, accumulated (dfsph_viscosity.rs:150-151)
    s.e00 += __fdiv_rn(a * a, rho);
    s.e03 += __fdiv_rn(a * Y, rho);
    s.e04 += __fdiv_rn(a * Z, rho);
    s.e11 += __fdiv_rn(b * b, rho);
    s.e13 += __fdiv_rn(b * X, rho);
    s.e15 += __fdiv_rn(b * Z, rho);
    s.e22 += __fdiv_rn(c * c, rho);
    s.e24 += __fdiv_rn(c * X, rho);
    s.e25 += __fdiv_rn(c * Y, rho);
    s.e33 += __fdiv_rn(__fadd_rn(__fmul_rn(Y, Y), __fmul_rn(X, X)), rho);
    s.e34 += __fdiv_rn(Y * Z, rho);
    s.e35 += __fdiv_rn(X * Z, rho);
    s.e44 += __fdiv_rn(__fadd_rn(__fmul_rn(Z, Z), __fmul_rn(X, X)), rho);
    s.e45 += __fdiv_rn(X * Y, rho);
    s.e55 += __fdiv_rn(__fadd_rn(__fmul_rn(Z, Z), __fmul_rn(Y, Y)), rho);
}

// compute_betas dfsph_viscosity.rs:133-201
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T)
k_visc_betas(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, const float* __restrict__ dens, float* __restrict__ beta,
             uint32_t which) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    const float4 pi = pos[i];
    const float rho_i = dens[i];
    Sym15 sq = {};
    float A = 0.f, B = 0.f, Cz = 0.f, SX = 0.f, SY = 0.f, SZ = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return MULTI ? fid_of(__ldg(&vel[j])) : 0u; },
        [&](uint32_t, const Pair& p, const float4& pj, uint32_t fj) {
            if (MULTI && fj != which) return;
            const float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;
            const float s = pj.w / (2.0f * rho_i);
            const float a = (gx * 2.f) * s, b = (gy * 2.f) * s, c = (gz * 2.f) * s, X = gx * s, Y = gy * s, Z = gz * s;
            outer15(a, b, c, X, Y, Z, rho_i, sq);
            A += a; B += b; Cz += c; SX += X; SY += Y; SZ += Z;
        });
    Sym15 gg = {};
    outer15(A, B, Cz, SX, SY, SZ, rho_i, gg);  // grad_sum * grad_sum^T / rho_i :157
    float d[6][6];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < 6; ++c) d[r][c] = 0.f;
    d[0][0] = sq.e00 + gg.e00; d[0][3] = d[3][0] = sq.e03 + gg.e03; d[0][4] = d[4][0] = sq.e04 + gg.e04;
    d[1][1] = sq.e11 + gg.e11; d[1][3] = d[3][1] = sq.e13 + gg.e13; d[1][5] = d[5][1] = sq.e15 + gg.e15;
    d[2][2] = sq.e22 + gg.e22; d[2][4] = d[4][2] = sq.e24 + gg.e24; d[2][5] = d[5][2] = sq.e25 + gg.e25;
    d[3][3] = sq.e33 + gg.e33; d[3][4] = d[4][3] = sq.e34 + gg.e34; d[3][5] = d[5][3] = sq.e35 + gg.e35;
    d[4][4] = sq.e44 + gg.e44; d[4][5] = d[5][4] = sq.e45 + gg.e45;
    d[5][5] = sq.e55 + gg.e55;
    float inv_diag[6];  // "Preconditionner" :162-174: only the first SPATIAL_DIM columns are scaled
    for (int k = 0; k < 6; ++k) inv_diag[k] = fabsf(d[k][k]) < 1.0e-6f ? 1.f : __fdiv_rn(1.f, d[k][k]);
    for (int c = 0; c < 3; ++c)
        for (int r = 0; r < 6; ++r) d[r][c] = __fmul_rn(d[r][c], inv_diag[r]);
    float inv[6][6];
    const bool ok = lu6_inverse(d, inv);
    for (int r = 0; r < 6; ++r)
        for (int c = 0; c < 6; ++c) {
            float v = ok ? inv[r][c] : 0.f;
            if (c < 3) v = __fmul_rn(v, inv_diag[c]);  // :193-196
            beta[(size_t)(r * 6 + c) * C.stride + i] = v;
        }
}

struct FidV {
    uint32_t fid;
    float4 v;
};
// compute_strain_rates dfsph_viscosity.rs:203-252; ERR: also u_i = beta_i * error_i / rho_i^2 for the next pass (:268)
template <bool MULTI, bool ERR>
__global__ void __launch_bounds__(PASS_T)
k_visc_rates(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, const float* __restrict__ dens, const float4* __restrict__ vv,
             float* __restrict__ target, const float* __restrict__ beta, float4* __restrict__ u4, float2* __restrict__ u2, float* __restrict__ partial,
             uint32_t which, float visc) {
    __shared__ float sm[32];
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < C.n_owned;
    i += C.i_begin;
    if (valid && MULTI && fid_of(vel[i]) != which) valid = false;
    float e = 0.f;
    if (valid) {
        const float4 pi = pos[i];
        const float rho_i = dens[i];
        const float4 vi = vv[i];
        float r0 = 0.f, r1 = 0.f, r2 = 0.f, r3 = 0.f, r4 = 0.f, r5 = 0.f;
        for_fluid_grads_pos(
            i, pi, L, pos, [&](uint32_t j) { return __ldg(&vv[j]); },
            [&](uint32_t, const Pair& p, const float4& pj, const float4& vj) {
                if (MULTI && fid_of(vj) != which) return;
                const float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;
                const float vx = vj.x - vi.x, vy = vj.y - vi.y, vz = vj.z - vi.z;
                const float s = pj.w / (2.0f * rho_i);
                r0 += (2.f * vx * gx) * s;
                r1 += (2.f * vy * gy) * s;
                r2 += (2.f * vz * gz) * s;
                r3 += (vx * gy + vy * gx) * s;
                r4 += (vx * gz + vz * gx) * s;
                r5 += (vy * gz + vz * gy) * s;
            });
        const float rate[6] = {r0, r1, r2, r3, r4, r5};
        if (!ERR) {
            for (int k = 0; k < 6; ++k) target[(size_t)k * C.stride + i] = rate[k] * (1.0f - visc);
        } else {
            float err[6], l1 = 0.f;
            for (int k = 0; k < 6; ++k) {
                err[k] = rate[k] - target[(size_t)k * C.stride + i];
                l1 += fabsf(err[k]);
            }
            e = l1 / 6.0f;
            float u[6];
            const float rr = rho_i * rho_i;
            for (int r = 0; r < 6; ++r) {
                float acc = __fmul_rn(beta[(size_t)(r * 6) * C.stride + i], err[0]);
                for (int k = 1; k < 6; ++k) acc = __fadd_rn(acc, __fmul_rn(beta[(size_t)(r * 6 + k) * C.stride + i], err[k]));
                u[r] = __fdiv_rn(acc, rr);
            }
            u4[i] = make_float4(u[0], u[1], u[2], u[3]);
            u2[i] = make_float2(u[4], u[5]);
        }
    }
    if (ERR) reduce_error<MULTI>(e, which, valid, partial, sm);
}

struct U6 {
    float4 a;
    float2 b;
    uint32_t fid;
};
// compute_accelerations dfsph_viscosity.rs:254-289
template <bool MULTI>
__global__ void __launch_bounds__(PASS_T)
k_visc_accel(const float4* __restrict__ pos, const float4* __restrict__ vel, Lists L, const float4* __restrict__ u4, const float2* __restrict__ u2,
             float4* __restrict__ acc, uint32_t which, float inv_dt) {
    SPH_OWNED_INDEX(i)
    if (MULTI && fid_of(vel[i]) != which) return;
    const float4 pi = pos[i];
    const float4 ua = u4[i];
    const float2 ub = u2[i];
    const float k = pi.w * inv_dt;  // volumes[c.i] * density0 * inv_dt
    float ax = 0.f, ay = 0.f, az = 0.f;
    for_fluid_grads_pos(
        i, pi, L, pos, [&](uint32_t j) { return U6{__ldg(&u4[j]), __ldg(&u2[j]), MULTI ? fid_of(__ldg(&vel[j])) : 0u}; },
        [&](uint32_t, const Pair& p, const float4& pj, const U6& uj) {
            if (MULTI && uj.fid != which) return;
            const float gx = p.g * p.dx, gy = p.g * p.dy, gz = p.g * p.dz;
            const float hm = pj.w / 2.0f;
            const float c0 = (ua.x + uj.a.x) * hm, c1 = (ua.y + uj.a.y) * hm, c2 = (ua.z + uj.a.z) * hm, c3 = (ua.w + uj.a.w) * hm,
                        c4 = (ub.x + uj.b.x) * hm, c5 = (ub.y + uj.b.y) * hm;
            ax += ((gx * 2.f) * c0 + gy * c3 + gz * c4) * k;
            ay += ((gy * 2.f) * c1 + gx * c3 + gz * c5) * k;
            az += ((gz * 2.f) * c2 + gx * c4 + gy * c5) * k;
        });
    float4 a = acc[i];
    a.x += ax; a.y += ay; a.z += az;
    acc[i] = a;
}

}  // namespace sphk
