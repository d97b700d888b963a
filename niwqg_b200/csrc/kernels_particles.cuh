// kernels_particles.cuh -- Lagrangian particles (drifters) advected with the model's own ETDRK4 stage velocities
// (DESIGN.md section 3.4).
//
// A particle is a point (x, y) in metres, stored unwrapped; grid values sit at the cell centres x_i = (i + 1/2) dx.
// Velocities are interpolated with the periodic tensor-product 4-point (cubic) Lagrange stencil: s = x/dx - 1/2,
// i = floor(s), a = s - i, nodes i-1 .. i+2 (mod N).  The 4 columns of each row are summed with the x weights, then
// the 4 rows with the y weights, both in index order (tests/particles_ref.py does exactly the same).
//
// Time stepping is classical RK4 whose four stages are the four stages of the model's ETDRK4 step: stage 1 reads the
// state at t_n, stages 2 and 3 the states a and b at t_n + dt/2, stage 4 the state c at t_n + dt.  k_particles<s>
// runs once per stage, where the model's uv (and phi) buffers hold that stage's fields.  No atomics: every particle
// belongs to one thread, so runs are bitwise repeatable.
#pragma once
#include "common.cuh"

struct PartArgs {
    const cd* uv;         // [B][npts] packed u + i v of the stage (device x order)
    const cd* phi;        // [B][npts] back-rotated wave velocity, or null: no wave velocity
    double2* xn;          // [B][P] positions at t_n (unwrapped)
    double2* xs;          // [B][P] position of the next stage
    double2* acc;         // [B][P] k1 + 2 k2 + 2 k3
    double* clk;          // [2] particle clock: clk[0] = t_n; clk[1] = t_n + dt, written at stage 1, read at stage 4
    const double* mcoef;  // [B][MC_COUNT]: the member's U and f
    size_t npts;          // N * N
    int P, N;
    int dshift, dM;       // device x order: natural x lives at position (x & ((1 << dshift) - 1)) * dM + (x >> dshift)
    double L, dx, dt;
};

// stencil of one coordinate: the 4 wrapped node indices and their weights
struct Stencil1 { int i[4]; double w[4]; };

__device__ __forceinline__ Stencil1 stencil1(double x, double L, double dx, int N) {
    // reduce the unwrapped position mod L first, so that a = s - floor(s) keeps its precision far from the origin
    const double xr = __dsub_rn(x, __dmul_rn(floor(x / L), L));
    const double s = xr / dx - 0.5;
    const double fi = floor(s);
    const double a = s - fi;
    const int i0 = (int)fi;
    Stencil1 st;
#pragma unroll
    for (int k = 0; k < 4; ++k) st.i[k] = (i0 - 1 + k) & (N - 1);
    st.w[0] = -a * (a - 1.0) * (a - 2.0) / 6.0;
    st.w[1] = (a + 1.0) * (a - 1.0) * (a - 2.0) / 2.0;
    st.w[2] = -(a + 1.0) * a * (a - 2.0) / 2.0;
    st.w[3] = (a + 1.0) * a * (a - 1.0) / 6.0;
    return st;
}

// offsets of the 16 stencil points of position p in one member's physical array (device x order)
__device__ __forceinline__ void stencil_offsets(const PartArgs& a, double2 p, double (&wx)[4], double (&wy)[4], int (&off)[16]) {
    const Stencil1 sx = stencil1(p.x, a.L, a.dx, a.N), sy = stencil1(p.y, a.L, a.dx, a.N);
    int col[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        col[k] = (sx.i[k] & ((1 << a.dshift) - 1)) * a.dM + (sx.i[k] >> a.dshift);
        wx[k] = sx.w[k];
        wy[k] = sy.w[k];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) off[4 * j + k] = sy.i[j] * a.N + col[k];
}

__device__ __forceinline__ double lerp4(const double (&w)[4], double v0, double v1, double v2, double v3) {
    return w[0] * v0 + w[1] * v1 + w[2] * v2 + w[3] * v3;
}
__device__ __forceinline__ cd lerp4(const double (&w)[4], cd v0, cd v1, cd v2, cd v3) {
    return make_double2(w[0] * v0.x + w[1] * v1.x + w[2] * v2.x + w[3] * v3.x,
                        w[0] * v0.y + w[1] * v1.y + w[2] * v2.y + w[3] * v3.y);
}
// the 16 gathered values g[4*row + col] -> interpolated value (rows with wx, then the rows with wy)
template <typename T>
__device__ __forceinline__ T interp16(const T (&g)[16], const double (&wx)[4], const double (&wy)[4]) {
    const T r0 = lerp4(wx, g[0], g[1], g[2], g[3]), r1 = lerp4(wx, g[4], g[5], g[6], g[7]);
    const T r2 = lerp4(wx, g[8], g[9], g[10], g[11]), r3 = lerp4(wx, g[12], g[13], g[14], g[15]);
    return lerp4(wy, r0, r1, r2, r3);
}

// One RK4 stage for every particle of every member (member = blockIdx.y).  The gathers of a particle (16 of uv, 16
// more of phi with WAVES) are all issued before any arithmetic that depends on them: a random gather costs a full
// HBM round trip, and only independent loads in flight hide it (DESIGN.md section 3).
template <int STAGE, bool WAVES>
__global__ void __launch_bounds__(128) k_particles(PartArgs a) {
    const int m = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    // the clock: stage 1 reads clk[0] and writes clk[1]; stage 4 reads clk[1] and writes clk[0] (no kernel reads the
    // slot it writes, so the update is race-free, and a CUDA graph that replays the step advances it by dt each time)
    if (STAGE == 1 && j == 0 && m == 0) a.clk[1] = a.clk[0] + a.dt;
    if (STAGE == 4 && j == 0 && m == 0) a.clk[0] = a.clk[1];
    if (j >= a.P) return;
    const size_t pi = (size_t)m * a.P + j;
    const double2 p = (STAGE == 1) ? a.xn[pi] : a.xs[pi];
    double wx[4], wy[4];
    int off[16];
    stencil_offsets(a, p, wx, wy, off);
    const cd* uv = a.uv + (size_t)m * a.npts;
    cd gu[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) gu[k] = __ldg(uv + off[k]);
    cd gp[16];
    if (WAVES) {
        const cd* phi = a.phi + (size_t)m * a.npts;
#pragma unroll
        for (int k = 0; k < 16; ++k) gp[k] = __ldg(phi + off[k]);
    }
    const double* mc = a.mcoef + (size_t)m * MC_COUNT;
    const cd u = interp16(gu, wx, wy);
    double vx = mc[MC_U] + u.x, vy = u.y;
    if (WAVES) {
        // u_w + i v_w = exp(-i f t) phi at the stage time
        const double t = (STAGE == 1) ? a.clk[0] : (STAGE == 4) ? a.clk[1] : a.clk[0] + 0.5 * a.dt;
        double sn, cs;
        sincos(mc[MC_F] * t, &sn, &cs);
        const cd ph = interp16(gp, wx, wy);
        vx = vx + (cs * ph.x + sn * ph.y);
        vy = vy + (cs * ph.y - sn * ph.x);
    }
    const double dt = a.dt;
    if (STAGE == 4) {
        const double2 c = a.acc[pi], x0 = a.xn[pi];
        a.xn[pi] = make_double2(x0.x + (dt / 6.0) * (c.x + vx), x0.y + (dt / 6.0) * (c.y + vy));
        return;
    }
    const double2 x0 = (STAGE == 1) ? p : a.xn[pi];
    double2 c;
    if (STAGE == 1) c = make_double2(vx, vy);
    else { c = a.acc[pi]; c.x = c.x + 2.0 * vx; c.y = c.y + 2.0 * vy; }
    a.acc[pi] = c;
    const double h = (STAGE == 3) ? dt : 0.5 * dt;
    a.xs[pi] = make_double2(x0.x + h * vx, x0.y + h * vy);
}

// niwqg_particles_sample: one field (real: [B][npts] doubles, complex: [B][npts] cd) interpolated at x_n
template <typename T>
__global__ void __launch_bounds__(128) k_particles_sample(PartArgs a, const T* __restrict__ f, T* __restrict__ out) {
    const int m = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.P) return;
    const size_t pi = (size_t)m * a.P + j;
    double wx[4], wy[4];
    int off[16];
    stencil_offsets(a, a.xn[pi], wx, wy, off);
    const T* fm = f + (size_t)m * a.npts;
    T g[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) g[k] = __ldg(fm + off[k]);
    out[pi] = interp16(g, wx, wy);
}
