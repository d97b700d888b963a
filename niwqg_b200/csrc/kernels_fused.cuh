// kernels_fused.cuh -- spectral kernels of the Coupled / UnCoupled step FUSED with the streaming radix stage of the split
// transforms (fft_split.cuh), so that the stage costs no launch and no trip through HBM of its own:
//
//   k_fstage_q    [forward combine of fft(uq + i vq)]  ->  J(psi,q) spectral part, ETDRK4 update of qh
//                                                           (Kernel.py:324-328, :346-347, :363-364, :380-383, :471-486)
//   k_fstage_phi  [forward combine of fft(P2)]         ->  ETDRK4 update of phih + the stage's spectral budget sums
//                                                           (Kernel.py:330-334, ..., :629-652)  ->  [inverse radix stage of
//                                                           phi, phix, phiy from the NEW phih]
//   k_finvert     [forward combine of fft(|phi|^2 + i J(phi*,phi))]  ->  wave PV, inversion, ep_psi sums
//                                                           (CoupledModel.py:75-97, :145-152; UnCoupledModel.py:54-64)
//                                                           ->  [inverse radix stage of u + i v and of q + i qw]
//
// Thread shape = that of k_split_p: one thread holds the 16 spectral values (ky = fam + M q, q = 0..15) of one column;
// lanes l and l + 16 of a warp hold the columns n and n + N/2 and do the x butterfly with shuffles.  The kernels that
// need the value at -K (Hermitian projection, split of a packed pair) get it through shared memory: a work unit of 256
// threads is closed under K -> -K (first half: family fam, 64 columns; second half: family M - fam, the mirrored
// columns), every thread computes ITS OWN element only.  All sums are per element (no pair weights), reduced per CTA of
// a persistent grid in a fixed order.
#pragma once
#include "fft_split.cuh"
#include "kernels_family.cuh"

template <int N> struct FusedGeom {
    static constexpr int R = 16, M = N / R, Nh = N / 2;
    static constexpr int NB = Nh / 64;                  // 64-column chunks of the half spectrum
    static constexpr int UNITS = (M / 2) * NB;          // work units of 256 threads x 16 elements
    static constexpr size_t XSMEM = (size_t)R * 256 * sizeof(cd);   // pair exchange buffer
};

struct FusedThread {
    int fam;        // row family: rows fam + M q
    int n;          // column of the pair's first half (n < N/2)
    int side;       // 0: column n, 1: column n + N/2
    int col;
    int ptid;       // thread of this unit that holds -K
    int kzero;      // family 0: -K of row M q is row M (16 - q); else row family M - fam, q' = 15 - q
};

template <int N>
__host__ __device__ __forceinline__ void fused_thread(int unit, int tid, const cd* __restrict__ twc, FusedThread& t) {
    using G = FusedGeom<N>;
    const int kk = unit / G::NB;
    int b = unit % G::NB, k;
    bool self;
    if (kk == 0) { self = true; if (b < G::NB / 2) k = 0; else { k = G::M / 2; b -= G::NB / 2; } }
    else { self = false; k = kk; }
    const int half = tid >> 7, wq = (tid >> 5) & 3, lane = tid & 31;
    t.side = lane >> 4;
    const int n0 = 64 * b + 16 * wq + (lane & 15);
    if (half == 0) { t.fam = k; t.n = n0; }
    else {
        t.fam = (G::M - k) % G::M;
        t.n = (n0 == 0) ? (self ? G::Nh / 2 : 0) : G::Nh - n0;
    }
    if (n0 != 0) t.ptid = tid ^ 128 ^ 16;               // other half, other side
    else if (!self) t.ptid = tid ^ 128;                  // column 0 / N/2 mirrors onto itself: other half, same side
    else t.ptid = half ? (tid ^ 16) : tid;               // self-paired family: column 0 -> same thread, column N/4 -> other side
    t.kzero = (t.fam == 0);
    t.col = t.n + t.side * G::Nh;
}
__host__ __device__ __forceinline__ int fused_qp(const FusedThread& t, int q) { return t.kzero ? ((16 - q) & 15) : 15 - q; }

__device__ __forceinline__ cd shfl16(cd v) {
    return make_double2(__shfl_xor_sync(0xffffffffu, v.x, 16), __shfl_xor_sync(0xffffffffu, v.y, 16));
}

// forward combine (decimation in time, see k_split_p<DIT>): T holds E_r[fam] as row r M + fam; u[q] = X[fam + M q][col]
template <int N>
__device__ __forceinline__ void fused_combine(const cd* __restrict__ T, const cd* __restrict__ twc, const FusedThread& t, cd (&u)[16]) {
    constexpr int M = N / 16;
    cd v[16];
    const cd wx = __ldg(&twc[t.n]), wy = __ldg(&twc[t.fam]);            // w_N^n, w_N^fam
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = __ldg(&T[(size_t)(r * M + t.fam) * N + t.col]);
    if (t.side) {
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = cmul(v[r], wx);
    }
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const cd o2 = shfl16(v[r]);
        v[r] = t.side ? csub(o2, v[r]) : cadd(v[r], o2);
    }
    fftc::apply_twiddles<16, 1>(v, wy);
    fftc::dft<16, 1>(v);
#pragma unroll
    for (int p = 0; p < 16; ++p) u[fftc::outidx<16>(p)] = v[p];
}

// inverse radix stage (decimation in frequency, see k_split_p<DIF>) of the 16 spectral values v[r] = s[fam + M r][col]:
// prologue, conj, x butterfly, radix 16, twiddles; stored as row q M + fam of `out`
template <int N>
__device__ __forceinline__ void fused_produce(cd (&v)[16], const cd* __restrict__ twc, const FusedThread& t, int pro, double dk,
                                              cd* __restrict__ out) {
    constexpr int M = N / 16;
    const cd wx = __ldg(&twc[t.n]), wy = __ldg(&twc[t.fam]);
#define NIWQG_PRO_CASE(P)                                                                     \
    case P:                                                                                   \
        _Pragma("unroll") for (int r = 0; r < 16; ++r) v[r] = split_prologue<N, P>(dk, t.fam + M * r, t.col, v[r]); \
        break;
    switch (pro) {
        NIWQG_PRO_CASE(PRO_IK)
        NIWQG_PRO_CASE(PRO_IL)
        NIWQG_PRO_CASE(PRO_UV)
        default: break;
    }
#undef NIWQG_PRO_CASE
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r].y = -v[r].y;
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const cd o2 = shfl16(v[r]);
        v[r] = t.side ? cmul(csub(o2, v[r]), wx) : cadd(v[r], o2);
    }
    fftc::dft<16, 1>(v);
    cd u[16];
#pragma unroll
    for (int p = 0; p < 16; ++p) u[fftc::outidx<16>(p)] = v[p];
    fftc::apply_twiddles<16, 1>(u, wy);
#pragma unroll
    for (int q = 0; q < 16; ++q) out[(size_t)(q * M + t.fam) * N + t.col] = u[q];
}

struct FStageArgs {
    StageArgs s;
    const cd* T;       // M-point column transforms (block layout) of the forward transform this kernel consumes
    cd* out[3];        // k_fstage_phi: radix-stage intermediates of phi, phix, phiy
    int nout;
    const cd* twc;
    double dk;
};

// Everything one element of an ETDRK4 stage update reads from global memory.  The loop over a thread's 16 elements is
// software-pipelined on these: the loads of element q + 1 are issued before element q is computed and stored, which
// keeps two elements' worth of bytes in flight per thread (at 512 threads per SM one is not enough to cover HBM latency).
// Arrays this launch only reads go through the read-only path (__ldg).
struct EqIn { cd y0, cur, F0, Fab, y1, c0, c1, c2, c3; double fl; };

template <int ST, bool PHI>
__device__ __forceinline__ void eq_load(EqIn& in, const cd* __restrict__ y0, const cd* y, const cd* __restrict__ y1,
                                        const cd* __restrict__ F0, const cd* Fab, const TableSet& t,
                                        const double* __restrict__ filtr, size_t i) {
    in.y0 = __ldg(&y0[i]);
    if (PHI && ST >= 2) in.cur = (ST == 2) ? __ldg(&y1[i]) : y[i];     // stage 2: the stage-1 result lives in y1
    if (ST >= 3) { in.F0 = __ldg(&F0[i]); in.Fab = (ST == 4) ? __ldg(&Fab[i]) : Fab[i]; }
    if (ST == 3) in.y1 = __ldg(&y1[i]);
    if (ST <= 3) { in.c0 = __ldg(&t.E2[i]); in.c1 = __ldg(&t.Q[i]); }
    else { in.c0 = __ldg(&t.E[i]); in.c1 = __ldg(&t.f0[i]); in.c2 = __ldg(&t.fab[i]); in.c3 = __ldg(&t.fc[i]); }
    in.fl = __ldg(&filtr[i]);
}
// register pipeline depth of the element loop per stage: as deep as 128 registers allow
template <int ST> struct FusedDepth { static constexpr int Q = ST <= 2 ? 4 : 3, PHI = ST <= 2 ? 4 : (ST == 3 ? 3 : 2), INV = 6; };
// etd_update (kernels_family.cuh) on preloaded operands; F0 / Fab come back as what the stage stores
template <int ST>
__device__ __forceinline__ cd eq_update(const EqIn& in, cd y0, cd Fn, cd& F0, cd& Fab) {
    cd r;
    if (ST == 1 || ST == 2) {
        r = cadd(cmul(in.c0, y0), cmul(Fn, in.c1));
        if (ST == 1) F0 = Fn; else Fab = Fn;
    } else if (ST == 3) {
        F0 = in.F0;
        const cd c = make_double2(2.0 * Fn.x - F0.x, 2.0 * Fn.y - F0.y);
        r = cadd(cmul(in.c0, in.y1), cmul(c, in.c1));
        Fab = cadd(in.Fab, Fn);
    } else {
        const cd ab2 = make_double2(2.0 * in.Fab.x, 2.0 * in.Fab.y);
        r = cadd(cadd(cadd(cmul(in.c0, y0), cmul(in.F0, in.c1)), cmul(ab2, in.c2)), cmul(Fn, in.c3));
    }
    return make_double2(r.x * in.fl, r.y * in.fl);
}

// ---- q equation
template <int N, int ST>
__global__ void __launch_bounds__(256, 2) k_fstage_q(FStageArgs a) {
    using G = FusedGeom<N>;
    constexpr int M = G::M;
    extern __shared__ __align__(16) unsigned char fused_smem[];
    cd* xs = reinterpret_cast<cd*>(fused_smem);
    const int tid = threadIdx.x;
    for (int unit = blockIdx.x; unit < G::UNITS; unit += gridDim.x) {
        FusedThread t;
        fused_thread<N>(unit, tid, a.twc, t);
        {
            cd u[16];
            fused_combine<N>(a.T, a.twc, t, u);
#pragma unroll
            for (int q = 0; q < 16; ++q) xs[q * 256 + tid] = u[q];      // parked: own value and the partner's come from here
        }
        __syncthreads();
        const double k1 = a.dk * (double)sidx(t.col, N);
        const size_t i0 = (size_t)t.fam * N + t.col;
        constexpr int D = FusedDepth<ST>::Q;
        EqIn in[D];
        // (units that hold the Nyquist column N/2 take the element-by-element path: the signed wavenumber of that
        // column is -N/2 for K and -K alike, so the reference is not conjugate-symmetric on it; same for row family 0)
        const int ub = unit % G::NB;
        const bool nyq = (ub == 0) || (unit < G::NB && ub == G::NB / 2);
        if (a.s.hsym && !t.kzero && !nyq) {
            // q is real: every array of the q equation is Hermitian (y(-K) = conj y(K)) and so are its tables and the
            // (symmetric) filter, hence the element at -K is the conjugate of the one at K.  -K of (this thread, q) is
            // (partner thread, 15 - q): the thread updates its EVEN q and stores both elements, which halves the
            // operand reads of the stage (y0 / F0 / Fab / y1 / tables: 28-60 B per grid point).
            const int colp = (N - t.col) & (N - 1);
#pragma unroll
            for (int p = 0; p < D - 1; ++p) eq_load<ST, false>(in[p], a.s.y0q, a.s.yq, a.s.y1q, a.s.F0q, a.s.Fabq, a.s.tq, a.s.filtr, i0 + (size_t)(2 * p) * M * N);
#pragma unroll
            for (int qq = 0; qq < 8; ++qq) {
                const int q = 2 * qq;
                const int ky = t.fam + M * q;
                const size_t i1 = i0 + (size_t)q * M * N;
                const size_t ip = (size_t)(N - ky) * N + colp;
                if (qq + D - 1 < 8) eq_load<ST, false>(in[(qq + D - 1) % D], a.s.y0q, a.s.yq, a.s.y1q, a.s.F0q, a.s.Fabq, a.s.tq, a.s.filtr, i1 + (size_t)(2 * (D - 1)) * M * N);
                const cd p1 = xs[q * 256 + tid], p2 = xs[(15 - q) * 256 + t.ptid];
                const double l1 = a.dk * (double)sidx(ky, N);
                const cd A = make_double2(0.5 * (p1.x + p2.x), 0.5 * (p1.y - p2.y));
                const cd B = make_double2(0.5 * (p1.y + p2.y), -0.5 * (p1.x - p2.x));
                const cd F1 = make_double2(k1 * A.y + l1 * B.y, -(k1 * A.x + l1 * B.x));
                const EqIn& e = in[qq % D];
                cd F0a, Faba;
                const cd n1 = eq_update<ST>(e, e.y0, F1, F0a, Faba);
                const cd n1c = make_double2(n1.x, -n1.y);
                a.s.yq[i1] = n1; a.s.yq[ip] = n1c;
                if (ST == 1) {
                    a.s.F0q[i1] = F0a; a.s.F0q[ip] = make_double2(F0a.x, -F0a.y);
                    if (a.s.y1q != a.s.yq) { a.s.y1q[i1] = n1; a.s.y1q[ip] = n1c; }
                }
                if (ST == 2 || ST == 3) { a.s.Fabq[i1] = Faba; a.s.Fabq[ip] = make_double2(Faba.x, -Faba.y); }
            }
            __syncthreads();
            continue;
        }
#pragma unroll
        for (int p = 0; p < D - 1; ++p) eq_load<ST, false>(in[p], a.s.y0q, a.s.yq, a.s.y1q, a.s.F0q, a.s.Fabq, a.s.tq, a.s.filtr, i0 + (size_t)p * M * N);
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int ky = t.fam + M * q;
            const size_t i1 = i0 + (size_t)q * M * N;
            if (q + D - 1 < 16) eq_load<ST, false>(in[(q + D - 1) % D], a.s.y0q, a.s.yq, a.s.y1q, a.s.F0q, a.s.Fabq, a.s.tq, a.s.filtr, i1 + (size_t)(D - 1) * M * N);
            const cd p1 = xs[q * 256 + tid], p2 = xs[fused_qp(t, q) * 256 + t.ptid];
            const double l1 = a.dk * (double)sidx(ky, N);
            // A = fft(u q)(K) = 0.5 (P(K) + conj P(-K)),  B = fft(v q)(K) = -0.5 i (P(K) - conj P(-K));  Fn = -(i k A + i l B)
            const cd A = make_double2(0.5 * (p1.x + p2.x), 0.5 * (p1.y - p2.y));
            const cd B = make_double2(0.5 * (p1.y + p2.y), -0.5 * (p1.x - p2.x));
            cd F1 = make_double2(k1 * A.y + l1 * B.y, -(k1 * A.x + l1 * B.x));
            if (ky == 0 && t.col == 0) F1 = make_double2(0.0, 0.0);
            const EqIn& e = in[q % D];
            cd F0a, Faba;
            const cd n1 = eq_update<ST>(e, e.y0, F1, F0a, Faba);
            a.s.yq[i1] = n1;
            if (ST == 1) { a.s.F0q[i1] = F0a; if (a.s.y1q != a.s.yq) a.s.y1q[i1] = n1; }
            if (ST == 2 || ST == 3) a.s.Fabq[i1] = Faba;
        }
        __syncthreads();
    }
}

// ---- phi equation + spectral budget sums + the inverse radix stage of phi (phix, phiy) from the new phih
template <int N, int ST>
__global__ void __launch_bounds__(256, 2) k_fstage_phi(FStageArgs a) {
    using G = FusedGeom<N>;
    constexpr int M = G::M;
    extern __shared__ __align__(16) unsigned char fused_smem[];
    cd* xs = reinterpret_cast<cd*>(fused_smem);
    const int tid = threadIdx.x;
    __shared__ double ssum[SE_COUNT][256];     // per-thread running sums live here, not in registers, across the radix stages
#pragma unroll
    for (int k = 0; k < SE_COUNT; ++k) ssum[k][tid] = 0.0;
    const bool specb = (a.s.flags & MF_SPEC_BUDGET) != 0;
    for (int unit = blockIdx.x; unit < G::UNITS; unit += gridDim.x) {
        FusedThread t;
        fused_thread<N>(unit, tid, a.twc, t);
        {
            cd u[16];
            fused_combine<N>(a.T, a.twc, t, u);
#pragma unroll
            for (int q = 0; q < 16; ++q) xs[q * 256 + tid] = u[q];      // parked (only this thread reads them back)
        }
        // no data dependence (only this thread reads xs back): a scheduling boundary, so that the operand loads below are
        // not hoisted into the combine, where the 16 values are still live (that spills past 128 registers)
        __syncwarp();
        const double k1 = a.dk * (double)sidx(t.col, N);
        const size_t i0 = (size_t)t.fam * N + t.col;
        double s[SE_COUNT];
#pragma unroll
        for (int k = 0; k < SE_COUNT; ++k) s[k] = 0.0;
        constexpr int D = FusedDepth<ST>::PHI;
        EqIn in[D];
#pragma unroll
        for (int p = 0; p < D - 1; ++p) eq_load<ST, true>(in[p], a.s.y0p, a.s.yp, a.s.y1p, a.s.F0p, a.s.Fabp, a.s.tp, a.s.filtr, i0 + (size_t)p * M * N);
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int ky = t.fam + M * q;
            const size_t i1 = i0 + (size_t)q * M * N;
            if (q + D - 1 < 16) eq_load<ST, true>(in[(q + D - 1) % D], a.s.y0p, a.s.yp, a.s.y1p, a.s.F0p, a.s.Fabp, a.s.tp, a.s.filtr, i1 + (size_t)(D - 1) * M * N);
            const EqIn& e = in[q % D];
            cd F1 = xs[q * 256 + tid];
            const cd cur1 = (ST == 1) ? e.y0 : e.cur;
            if (specb || (a.s.flags & MF_HAS_LAP2)) {     // |phih|^2 moments on the pre-update phih (Kernel.py:629-652)
                const double l1 = a.dk * (double)sidx(ky, N);
                const double wv2 = k1 * k1 + l1 * l1, w4 = wv2 * wv2;
                const double m2 = cur1.x * cur1.x + cur1.y * cur1.y;
                s[SE_LAP2] += w4 * m2;
                s[SE_WV6PHI] += w4 * wv2 * m2;
                if (specb) {                              // raw transform, before the (0,0) fix
                    const double zr = cur1.x * F1.x + cur1.y * F1.y, zi = cur1.y * F1.x - cur1.x * F1.y;
                    s[SE_T0R] += zr; s[SE_T0I] += zi;
                    s[SE_T1R] += wv2 * zr; s[SE_T1I] += wv2 * zi;
                    s[SE_T2R] += w4 * zr; s[SE_T2I] += w4 * zi;
                }
            }
            if ((a.s.flags & MF_FIX00) && ky == 0 && t.col == 0) { F1.x += a.s.sumsD[SD_J_R]; F1.y += a.s.sumsD[SD_J_I]; }
            cd F0a, Faba;
            const cd n1 = eq_update<ST>(e, e.y0, F1, F0a, Faba);
            a.s.yp[i1] = n1;
            if (ST == 1) { a.s.F0p[i1] = F0a; if (a.s.y1p != a.s.yp) a.s.y1p[i1] = n1; }
            if (ST == 2 || ST == 3) a.s.Fabp[i1] = Faba;
        }
#pragma unroll
        for (int k = 0; k < SE_COUNT; ++k) ssum[k][tid] += s[k];
        // self.phi = ifft(phih) (+ phix, phiy of jacobian_phic_phi) start here: Kernel.py:337, CoupledModel.py:70
        for (int o = 0; o < a.nout; ++o) {
            cd v[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = a.s.yp[i0 + (size_t)r * M * N];   // this thread's own stores
            fused_produce<N>(v, a.twc, t, o == 0 ? PRO_NONE : o == 1 ? PRO_IK : PRO_IL, a.dk, a.out[o]);
        }
    }
    double s[SE_COUNT];
#pragma unroll
    for (int k = 0; k < SE_COUNT; ++k) s[k] = ssum[k][tid];
    block_reduce_store<SE_COUNT>(s, a.s.partials);
}

struct FInvertArgs {
    InvertArgs i;
    const cd* T;       // M-point column transforms (block layout) of fft(|phi|^2 + i J): MF_WAVE_PV only
    cd *out_uv, *out_qs;
    const cd* twc;
    double dk;
};

struct InvIn { cd q1, q2; double fl, flp; };

// ---- _invert + _calc_rel_vorticity in spectral space + the inverse radix stage of u + i v and q + i qw
template <int N, bool HASW>
__global__ void __launch_bounds__(256, 2) k_finvert(FInvertArgs a) {
    using G = FusedGeom<N>;
    constexpr int M = G::M;
    extern __shared__ __align__(16) unsigned char fused_smem[];
    cd* xs = reinterpret_cast<cd*>(fused_smem);
    const int tid = threadIdx.x;
    __shared__ double ssum[SI_COUNT][256];
#pragma unroll
    for (int k = 0; k < SI_COUNT; ++k) ssum[k][tid] = 0.0;
    for (int unit = blockIdx.x; unit < G::UNITS; unit += gridDim.x) {
        FusedThread t;
        fused_thread<N>(unit, tid, a.twc, t);
        if (HASW) {
            cd u[16];
            fused_combine<N>(a.T, a.twc, t, u);
#pragma unroll
            for (int q = 0; q < 16; ++q) xs[q * 256 + tid] = u[q];
            __syncthreads();
        }
        cd u[16];
        double s[SI_COUNT] = {0.0, 0.0, 0.0};
        const double k1 = a.dk * (double)sidx(t.col, N);
        const int colp = (N - t.col) & (N - 1);
        const size_t i0 = (size_t)t.fam * N + t.col;
        auto load = [&](InvIn& in, int q) {
            const int ky = t.fam + M * q, kyp = (N - ky) & (N - 1);
            in.q1 = __ldg(&a.i.qh[i0 + (size_t)q * M * N]);
            in.q2 = __ldg(&a.i.qh[(size_t)kyp * N + colp]);
            if (HASW) {
                in.fl = __ldg(&a.i.filtr[i0 + (size_t)q * M * N]);
                in.flp = a.i.filtr_sym ? in.fl : __ldg(&a.i.filtr[(size_t)kyp * N + colp]);
            }
        };
        constexpr int D = FusedDepth<1>::INV;
        InvIn in[D];
#pragma unroll
        for (int p = 0; p < D - 1; ++p) load(in[p], p);
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int ky = t.fam + M * q;
            const size_t i1 = i0 + (size_t)q * M * N;
            if (q + D - 1 < 16) load(in[(q + D - 1) % D], q + D - 1);
            const InvIn& e = in[q % D];
            const double l1 = a.dk * (double)sidx(ky, N);
            const double wv2 = __dadd_rn(__dmul_rn(k1, k1), __dmul_rn(l1, l1));
            const double wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
            const cd Hq = make_double2(0.5 * (e.q1.x + e.q2.x), 0.5 * (e.q1.y - e.q2.y));   // Herm(qh)(K)
            cd qw = make_double2(0.0, 0.0), qwr = qw;      // Hermitian part (enters p, qw) / raw element (stored as qwh)
            if (HASW) {
                const cd W1 = xs[q * 256 + tid], W2 = xs[fused_qp(t, q) * 256 + t.ptid];
                const cd A = make_double2(0.5 * (W1.x + W2.x), 0.5 * (W1.y - W2.y));     // fft(|phi|^2)(K)
                cd Jc = make_double2(a.i.inv_jscale * 0.5 * (W1.y + W2.y), a.i.inv_jscale * -0.5 * (W1.x - W2.x));
                if (ky == 0 && t.col == 0) Jc = make_double2(0.0, 0.0);
                const double bx = 0.5 * (0.5 * (-wv2 * A.x) + Jc.x) / a.i.f, by = 0.5 * (0.5 * (-wv2 * A.y) + Jc.y) / a.i.f;
                const double fs = 0.5 * (e.fl + e.flp);
                qw.x = bx * fs; qw.y = by * fs;
                qwr.x = bx * e.fl; qwr.y = by * e.fl;
            }
            const cd ph1 = make_double2(wv2i * qw.x - wv2i * Hq.x, wv2i * qw.y - wv2i * Hq.y);
            {
                const double r = Hq.x * ph1.x + Hq.y * ph1.y;      // Re(Hq conj ph)(K); the sum runs over every K
                s[SI_QLAP2PSI] += wv2 * wv2 * r;
                s[SI_PLAPQ] += -wv2 * r;
                s[SI_PQ] += r;
            }
            a.i.ph[i1] = ph1;
            if (a.i.qwh) a.i.qwh[i1] = qwr;
            u[q] = make_double2(Hq.x - qw.y, Hq.y + qw.x);         // qs(K) = Herm(qh) + i qwh
        }
        if (HASW) __syncthreads();
#pragma unroll
        for (int k = 0; k < SI_COUNT; ++k) ssum[k][tid] += s[k];
        fused_produce<N>(u, a.twc, t, PRO_NONE, a.dk, a.out_qs);
#pragma unroll
        for (int r = 0; r < 16; ++r) u[r] = a.i.ph[i0 + (size_t)r * M * N];        // this thread's own stores
        fused_produce<N>(u, a.twc, t, PRO_UV, a.dk, a.out_uv);
    }
    double s[SI_COUNT];
#pragma unroll
    for (int k = 0; k < SI_COUNT; ++k) s[k] = ssum[k][tid];
    block_reduce_store<SI_COUNT>(s, a.i.partials);
}

template <int N>
static cudaError_t fused_set_attrs() {
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 64 && attr_set[dev]) return cudaSuccess;
    const int sm = (int)FusedGeom<N>::XSMEM;
    cudaError_t e;
#define NIWQG_ATTR(K) if ((e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, sm)) != cudaSuccess) return e;
    NIWQG_ATTR((k_fstage_q<N, 1>)) NIWQG_ATTR((k_fstage_q<N, 2>)) NIWQG_ATTR((k_fstage_q<N, 3>)) NIWQG_ATTR((k_fstage_q<N, 4>))
    NIWQG_ATTR((k_fstage_phi<N, 1>)) NIWQG_ATTR((k_fstage_phi<N, 2>)) NIWQG_ATTR((k_fstage_phi<N, 3>)) NIWQG_ATTR((k_fstage_phi<N, 4>))
    NIWQG_ATTR((k_finvert<N, true>))
#undef NIWQG_ATTR
    if (dev < 64) attr_set[dev] = true;
    return cudaSuccess;
}

template <int N>
static cudaError_t launch_fstage(const FStageArgs& a, bool phi, int grid, cudaStream_t st) {
    cudaError_t e = fused_set_attrs<N>();
    if (e != cudaSuccess) return e;
    const size_t sm = FusedGeom<N>::XSMEM;
    if (phi) {
        switch (a.s.stage) {
            case 1: k_fstage_phi<N, 1><<<grid, 256, sm, st>>>(a); break;
            case 2: k_fstage_phi<N, 2><<<grid, 256, sm, st>>>(a); break;
            case 3: k_fstage_phi<N, 3><<<grid, 256, sm, st>>>(a); break;
            default: k_fstage_phi<N, 4><<<grid, 256, sm, st>>>(a); break;
        }
    } else {
        switch (a.s.stage) {
            case 1: k_fstage_q<N, 1><<<grid, 256, sm, st>>>(a); break;
            case 2: k_fstage_q<N, 2><<<grid, 256, sm, st>>>(a); break;
            case 3: k_fstage_q<N, 3><<<grid, 256, sm, st>>>(a); break;
            default: k_fstage_q<N, 4><<<grid, 256, sm, st>>>(a); break;
        }
    }
    return cudaGetLastError();
}

template <int N>
static cudaError_t launch_finvert(const FInvertArgs& a, bool has_w, int grid, cudaStream_t st) {
    cudaError_t e = fused_set_attrs<N>();
    if (e != cudaSuccess) return e;
    if (has_w) k_finvert<N, true><<<grid, 256, FusedGeom<N>::XSMEM, st>>>(a);
    else k_finvert<N, false><<<grid, 256, 0, st>>>(a);
    return cudaGetLastError();
}
