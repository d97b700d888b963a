// kernels_family.cuh -- pointwise / reduction kernels of the NIW-QG kernel family
// (CoupledModel, UnCoupledModel, YBJModel, repaired QLModel; complex c2c spectra).
//
// Spectral kernels process (K, -K) index pairs in one thread: that makes the
// reference's "`.real` after an inverse transform" (= Hermitian projection of the
// spectrum) and the split of one packed forward transform into two real-field
// spectra exact, at one read and one write per element.
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------- model flags
enum {
    MF_WAVE_PV   = 1 << 0,   // Coupled / QL: wave PV feeds the inversion (CoupledModel.py:75-97)
    MF_QL_ADV    = 1 << 1,   // QL: wave advected by the vortex flow only (QLModel.py:65-67)
    MF_YBJ       = 1 << 2,   // YBJ: phi-only step in a frozen flow (YBJModel.py:52-87)
    MF_FIX00     = 1 << 3,   // zero mode (0,0) of fft(J(psi,phi)) (Kernel.py:468); not for YBJ/QL
    MF_HAS_LAP2  = 1 << 4,   // nu4w != 0: lap2phi is needed (Kernel.py:688-689)
    MF_NO_WRITE  = 1 << 5,   // diagnostics tick: sums only
    MF_SKIP_P1   = 1 << 6,   // [D] second half of a QL stage: P2 only, no sums
    MF_SKIP_P2   = 1 << 7,   // [D] first half of a QL stage: P1 + sums only
    MF_SPEC_BUDGET = 1 << 8, // Coupled / UnCoupled: the stage budgets' lapphi terms are evaluated in spectral space
                             // (Parseval, see k_spec_stage), so lapphi / lap2phi are not transformed during a step
    MF_P1_BY_LOADER = 1 << 9,   // k_phys_rhs does not store P1 = (uq, vq): P1's forward row pass forms it itself (LD_UQVQ)
};

// Grid (N, dk, local spectral columns, slab ownership) and the column maps grid_kx / grid_partner: common.cuh

// ======================================================================
// ETDRK4 tables + filter (Kernel.py:267-284, :400-454; YBJModel.py:89-121)
// ======================================================================
__device__ __forceinline__ cd cexp_d(cd z) {
    double s, c;
    sincos(z.y, &s, &c);
    const double e = exp(z.x);
    return make_double2(e * c, e * s);
}
__device__ __forceinline__ cd cdiv_d(cd a, cd b) {
    // Smith's algorithm (what numpy's complex division uses)
    if (fabs(b.x) >= fabs(b.y)) {
        const double r = b.y / b.x, d = b.x + b.y * r;
        return make_double2((a.x + a.y * r) / d, (a.y - a.x * r) / d);
    } else {
        const double r = b.x / b.y, d = b.x * r + b.y;
        return make_double2((a.x * r + a.y) / d, (a.y * r - a.x) / d);
    }
}

// Kassam-Trefethen contour means for one exponent ch = c*dt (Kernel.py:424-433)
__device__ void etdrk4_point(cd ch, double dt, cd& E, cd& E2, cd& Q, cd& f0, cd& fab, cd& fc) {
    E = cexp_d(ch);
    E2 = cexp_d(make_double2(0.5 * ch.x, 0.5 * ch.y));
    cd sQ = make_double2(0, 0), s0 = sQ, sab = sQ, sc = sQ;
    for (int jj = 1; jj <= 32; ++jj) {
        double sr, cr;
        sincospi(2.0 * (double)jj / 32.0, &sr, &cr);
        const cd LR = make_double2(ch.x + cr, ch.y + sr);
        const cd LR2 = cmul(LR, LR), LR3 = cmul(LR2, LR);
        const cd eh = cexp_d(make_double2(0.5 * LR.x, 0.5 * LR.y));
        const cd e1 = cexp_d(LR);
        sQ = cadd(sQ, cdiv_d(make_double2(eh.x - 1.0, eh.y), LR));
        // (-4 - LR + e^LR (4 - 3 LR + LR2)) / LR3
        cd t = cmul(e1, make_double2(4.0 - 3.0 * LR.x + LR2.x, -3.0 * LR.y + LR2.y));
        s0 = cadd(s0, cdiv_d(make_double2(-4.0 - LR.x + t.x, -LR.y + t.y), LR3));
        // (2 + LR + e^LR (-2 + LR)) / LR3
        t = cmul(e1, make_double2(-2.0 + LR.x, LR.y));
        sab = cadd(sab, cdiv_d(make_double2(2.0 + LR.x + t.x, LR.y + t.y), LR3));
        // (-4 - 3 LR - LR2 + e^LR (4 - LR)) / LR3
        t = cmul(e1, make_double2(4.0 - LR.x, -LR.y));
        sc = cadd(sc, cdiv_d(make_double2(-4.0 - 3.0 * LR.x - LR2.x + t.x, -3.0 * LR.y - LR2.y + t.y), LR3));
    }
    const double s = dt / 32.0;
    Q = cscale(sQ, s); f0 = cscale(s0, s); fab = cscale(sab, s); fc = cscale(sc, s);
}

struct TableSet { cd *E, *E2, *Q, *f0, *fab, *fc; };

// Per-member coefficients the kernels read by value of blockIdx.y: mcoef[member][MC_COUNT] (equal rows when the
// members share their parameters).  MC_PW_SEED = 0.25 / (N^2 kappa2), the Pw of set_phi per unit grad^2 sum.
// MC_U: the uniform mean flow U (the -ikU of the linear operator), which Lagrangian particles add to u.
enum { MC_F = 0, MC_HSLASH, MC_KAPPA2, MC_NU4, MC_NU, MC_MU, MC_NU4W, MC_NUW, MC_MUW, MC_NU4C, MC_MUC, MC_PW_SEED,
       MC_U, MC_COUNT };

// coefficients of one equation's exponent c (see InitArgs), per member for k_init_tables
enum { IC_RE_A4 = 0, IC_RE_A2, IC_RE_A0, IC_IM_WV2, IC_BETA, IC_U, IC_COUNT };

struct InitArgs {
    Grid g;                  // slab column map (kernel family); g.sym == 0 for the natural layout
    int N, nk;               // nk = local spectral columns: N (c2c), N/P (slab) or N/2+1 (QG half spectrum)
    int half;                // 1: QG wavenumber convention (k = dk*col, col<=N/2)
    double dk, dt, dx;
    double U;
    double re_a4, re_a2, re_a0;   // real part of c:  -a4*wv4 - a2*wv2 - a0
    double im_wv2;                // imag part of c: -k*U - im_wv2*wv2  (+ beta*k/wv2 when beta_on)
    double beta;
    int use_filter, dealias;
    TableSet t;
    double* filtr;               // may be null
    const double* mc;            // null: one table set from the scalars above; else [gridDim.y][IC_COUNT], one set per
                                 // member (blockIdx.y) at offset member * N * nk of every table
};

__global__ void k_init_tables(InitArgs a) {
    const size_t total = (size_t)a.N * a.nk;
    double re_a4 = a.re_a4, re_a2 = a.re_a2, re_a0 = a.re_a0, im_wv2 = a.im_wv2, beta = a.beta, U = a.U;
    size_t mo = 0;
    if (a.mc) {
        const double* c = a.mc + (size_t)blockIdx.y * IC_COUNT;
        re_a4 = c[IC_RE_A4]; re_a2 = c[IC_RE_A2]; re_a0 = c[IC_RE_A0]; im_wv2 = c[IC_IM_WV2]; beta = c[IC_BETA]; U = c[IC_U];
        mo = (size_t)blockIdx.y * total;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / a.nk), col = (int)(i % a.nk);
        const double k = a.dk * (double)(a.half ? col : sidx(grid_kx(a.g, col), a.N));
        const double l = a.dk * (double)sidx(row, a.N);
        const double wv2 = __dadd_rn(__dmul_rn(k, k), __dmul_rn(l, l));
        const double wv4 = __dmul_rn(wv2, wv2);
        double cre = __dsub_rn(__dsub_rn(__dmul_rn(-re_a4, wv4), __dmul_rn(re_a2, wv2)), re_a0);
        double cim = __dsub_rn(-__dmul_rn(k, U), __dmul_rn(im_wv2, wv2));
        if (beta != 0.0 && wv2 != 0.0) cim += beta * k * (1.0 / wv2);   // QGModel.py:428
        cd E, E2, Q, f0, fab, fc;
        etdrk4_point(make_double2(cre * a.dt, cim * a.dt), a.dt, E, E2, Q, f0, fab, fc);
        const size_t j = mo + i;
        a.t.E[j] = E; a.t.E2[j] = E2; a.t.Q[j] = Q; a.t.f0[j] = f0; a.t.fab[j] = fab; a.t.fc[j] = fc;
        if (a.filtr && blockIdx.y == 0) {
            double fl = 1.0;
            if (a.use_filter) {
                const double cphi = 0.65 * 3.14159265358979323846;
                const double wvx = sqrt((k * a.dx) * (k * a.dx) + (l * a.dx) * (l * a.dx));
                if (wvx > cphi) { const double d = wvx - cphi; fl = exp(-23.6 * (d * d) * (d * d)); }
            } else if (a.dealias) {
                const int lo = a.N / 3, hi = 2 * a.N / 3, kxi = a.half ? col : grid_kx(a.g, col);
                if ((row >= lo && row < hi) || (kxi >= lo && kxi < hi)) fl = 0.0;
            }
            a.filtr[i] = fl;
        }
    }
}

// ======================================================================
// [B] wave-PV products in physical space (CoupledModel.py:69-71, :83-84):
//     W = |phi|^2 + i * Re( i (conj(phix) phiy - conj(phiy) phix) )
// ======================================================================
// The Jacobian part is many orders of magnitude smaller than the variations of |phi|^2, so it is packed
// scaled by jscale ~ 1/k_mid^2 (a power of two): otherwise the transform's rounding noise, which is
// relative to the larger partner, swamps it and the error grows coherently in time (DESIGN.md "packing").
__global__ void k_phys_wavepv(const cd* __restrict__ phi, const cd* __restrict__ phix,
                              const cd* __restrict__ phiy, cd* __restrict__ W, size_t npts, double jscale) {
    const size_t mb = (size_t)blockIdx.y * npts;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd p = phi[mb + i], px = phix[mb + i], py = phiy[mb + i];
        // conj(px)*py - conj(py)*px = 2i*Im(conj(px)*py);  i*that = -2*Im(conj(px) py)
        const double im = px.x * py.y - px.y * py.x;
        W[mb + i] = make_double2(p.x * p.x + p.y * p.y, jscale * (-2.0 * im));
    }
}

// ======================================================================
// [C] inversion in spectral space, (K,-K) pairs.
//  Coupled/QL (CoupledModel.py:75-97, :145-152):
//     A = fft(|phi|^2), Jc = fft(J(phi*,phi)) split from W; Jc[0,0]=0
//     qwh = 0.5*(0.5*(-wv2*A) + Jc)/f * filtr
//     ph  = fft(Re ifft(wv2i*qwh) + Re ifft(-wv2i*qh)) = wv2i*qwh - wv2i*Herm(qh)
//     qs  = Herm(qh) + i*qwh            (inverse transform -> q + i*qw)
//  UnCoupled (UnCoupledModel.py:54-64): qwh = 0.
//  YBJ (YBJModel.py:141-146): ph = -wv2i*qh (no projection); uv = packed spectrum of
//     Re ifft(-il ph) + i Re ifft(ik ph) (Kernel.py:534).
//  QL additionally: uvq = the same packing for ph_q = -wv2i*qh (QLModel.py:65-66).
// ======================================================================
struct InvertArgs {
    Grid g;
    int flags;
    double f;
    double inv_jscale;   // undoes k_phys_wavepv's scaling of the Jacobian partner
    int filtr_sym;       // filtr(K) == filtr(-K) everywhere (the exponential filter; NOT the 2/3-rule mask, whose band
                         // [N/3, 2N/3) holds index N/3 but not its mirror 2N/3): spares the second filter load
    const cd* W;      // forward transform of the [B] products (MF_WAVE_PV)
    const cd* qh;
    const double* filtr;
    cd *qwh, *ph, *qs, *uvgen;   // uvgen: general packed (u + i v) spectrum (YBJ: from ph; QL: from ph_q)
    double* partials;            // [member][block][SI_COUNT] Parseval sums of ep_psi (Kernel.py:635-640); may be null
};

// sums over the full spectrum on the state the NEXT stage starts from:
//   [0] sum wv2^2 Re(qh conj ph)   [1] sum -wv2 Re(qh conj ph)   [2] sum Re(qh conj ph)      (ph Hermitian)
enum { SI_QLAP2PSI = 0, SI_PLAPQ, SI_PQ, SI_COUNT };

__device__ __forceinline__ void pack_uv_general(double k1, double l1, double k2, double l2, cd G1, cd G2,
                                                cd& out1, cd& out2) {
    // HU(K) = 0.5*(-i l1 G1 + conj(-i l2 G2)),  HV(K) = 0.5*(i k1 G1 + conj(i k2 G2))
    // -i l G = (l*G.y, -l*G.x);  conj(-i l G) = (l*G.y, l*G.x)
    const cd HU = make_double2(0.5 * (l1 * G1.y + l2 * G2.y), 0.5 * (-l1 * G1.x + l2 * G2.x));
    //  i k G = (-k*G.y, k*G.x);  conj(i k G) = (-k*G.y, -k*G.x)
    const cd HV = make_double2(0.5 * (-k1 * G1.y - k2 * G2.y), 0.5 * (k1 * G1.x - k2 * G2.x));
    // packed(K) = HU + i HV ; packed(-K) = conj(HU) + i conj(HV)
    out1 = make_double2(HU.x - HV.y, HU.y + HV.x);
    out2 = make_double2(HU.x + HV.y, -HU.y + HV.x);
}

// mcoef: [member][MC_COUNT] (this kernel reads the member's f instead of a.f, which the batch-1 fused inversion uses)
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_spec_invert(InvertArgs a, const double* __restrict__ mcoef) {
    double s[SI_COUNT] = {0.0, 0.0, 0.0};
    const int N = a.g.N, H = N >> 1, NC = a.g.ncl;
    const size_t npts = (size_t)N * NC, mb = (size_t)blockIdx.y * npts;
    const double f = mcoef[(size_t)blockIdx.y * MC_COUNT + MC_F];
    const size_t total = (size_t)(H + 1) * NC;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(t / NC), lc = (int)(t % NC);
        const int kyp = (N - ky) & (N - 1), lcp = grid_partner(a.g, lc);
        if (kyp == ky && lcp < lc) continue;              // each (K, -K) pair once
        const int kx = grid_kx(a.g, lc), kxp = grid_kx(a.g, lcp);
        const size_t i1 = mb + (size_t)ky * NC + lc, i2 = mb + (size_t)kyp * NC + lcp;
        const bool self = (i1 == i2);
        const double k1 = a.g.dk * (double)sidx(kx, N), l1 = a.g.dk * (double)sidx(ky, N);
        const double k2 = a.g.dk * (double)sidx(kxp, N), l2 = a.g.dk * (double)sidx(kyp, N);
        const double wv2 = __dadd_rn(__dmul_rn(k1, k1), __dmul_rn(l1, l1));
        const double wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
        const cd q1 = a.qh[i1], q2 = a.qh[i2];
        if (a.flags & MF_YBJ) {
            const cd G1 = make_double2(-wv2i * q1.x, -wv2i * q1.y), G2 = make_double2(-wv2i * q2.x, -wv2i * q2.y);
            a.ph[i1] = G1;
            if (!self) a.ph[i2] = G2;
            cd o1, o2;
            pack_uv_general(k1, l1, k2, l2, G1, G2, o1, o2);
            a.uvgen[i1] = o1;
            if (!self) a.uvgen[i2] = o2;
            continue;
        }
        const cd Hq = make_double2(0.5 * (q1.x + q2.x), 0.5 * (q1.y - q2.y));   // Herm(qh)(K)
        cd qw = make_double2(0.0, 0.0), qwb = qw;
        double fl1 = 0.0, fl2 = 0.0;
        if (a.flags & MF_WAVE_PV) {
            const cd W1 = a.W[i1], W2 = a.W[i2];
            const cd A = make_double2(0.5 * (W1.x + W2.x), 0.5 * (W1.y - W2.y));     // fft(|phi|^2)(K)
            cd Jc = make_double2(a.inv_jscale * 0.5 * (W1.y + W2.y), a.inv_jscale * -0.5 * (W1.x - W2.x));   // -0.5i (W1 - conj W2)
            if (ky == 0 && kx == 0) Jc = make_double2(0.0, 0.0);
            // qwh = base * filtr per element (CoupledModel.py:86); what enters p and qw is Re ifft(...), i.e. the
            // Hermitian part, whose coefficient is base * (filtr(K) + filtr(-K)) / 2
            fl1 = a.filtr[(size_t)ky * NC + lc];
            fl2 = a.filtr_sym ? fl1 : a.filtr[(size_t)kyp * NC + lcp];
            const double fs = 0.5 * (fl1 + fl2);
            qwb.x = 0.5 * (0.5 * (-wv2 * A.x) + Jc.x) / f;
            qwb.y = 0.5 * (0.5 * (-wv2 * A.y) + Jc.y) / f;
            qw.x = qwb.x * fs;
            qw.y = qwb.y * fs;
        }
        const cd ph1 = make_double2(wv2i * qw.x - wv2i * Hq.x, wv2i * qw.y - wv2i * Hq.y);
        {   // Re(Hq conj ph(K)) + Re(conj(Hq) conj ph(-K)), ph(-K) = conj ph(K)
            const double r = (self ? 1.0 : 2.0) * (Hq.x * ph1.x + Hq.y * ph1.y);
            s[SI_QLAP2PSI] += wv2 * wv2 * r;
            s[SI_PLAPQ] += -wv2 * r;
            s[SI_PQ] += r;
        }
        // qs(K) = Hq + i qw ; qs(-K) = conj(Hq) + i conj(qw)
        a.ph[i1] = ph1;
        a.qs[i1] = make_double2(Hq.x - qw.y, Hq.y + qw.x);
        if (a.qwh) a.qwh[i1] = make_double2(qwb.x * fl1, qwb.y * fl1);
        if (!self) {
            a.ph[i2] = make_double2(ph1.x, -ph1.y);
            a.qs[i2] = make_double2(Hq.x + qw.y, -Hq.y + qw.x);
            if (a.qwh) a.qwh[i2] = make_double2(qwb.x * fl2, -qwb.y * fl2);
        }
    }
    if (a.partials) block_reduce_store<SI_COUNT>(s, a.partials);
}

// QL wave advection velocity (QLModel.py:65-66): packed spectrum of Re ifft(-il ph_q) + i Re ifft(ik ph_q),
// ph_q = -wv2i*qh, from whatever qh is current when jacobian_psi_phi is called.
__global__ void k_spec_uvq(Grid g, const cd* __restrict__ qh, cd* __restrict__ uvq) {
    const int N = g.N, H = N >> 1, NC = g.ncl;
    const size_t npts = (size_t)N * NC, mb = (size_t)blockIdx.y * npts;
    const size_t total = (size_t)(H + 1) * NC;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(t / NC), lc = (int)(t % NC);
        const int kyp = (N - ky) & (N - 1), lcp = grid_partner(g, lc);
        if (kyp == ky && lcp < lc) continue;
        const int kx = grid_kx(g, lc), kxp = grid_kx(g, lcp);
        const size_t i1 = mb + (size_t)ky * NC + lc, i2 = mb + (size_t)kyp * NC + lcp;
        const double k1 = g.dk * (double)sidx(kx, N), l1 = g.dk * (double)sidx(ky, N);
        const double k2 = g.dk * (double)sidx(kxp, N), l2 = g.dk * (double)sidx(kyp, N);
        const double wv2 = __dadd_rn(__dmul_rn(k1, k1), __dmul_rn(l1, l1));
        const double wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
        const cd q1 = qh[i1], q2 = qh[i2];
        const cd G1 = make_double2(-wv2i * q1.x, -wv2i * q1.y), G2 = make_double2(-wv2i * q2.x, -wv2i * q2.y);
        cd o1, o2;
        pack_uv_general(k1, l1, k2, l2, G1, G2, o1, o2);
        uvq[i1] = o1;
        if (i1 != i2) uvq[i2] = o2;
    }
}

// ======================================================================
// [D] physical-space products and budget means of one stage
//  (Kernel.py:664-701 energy conversion, :457-486 Jacobians, :332 refraction,
//   :629-633 ep_phi, :646-652 chi_phi physical parts)
//  sums (per member): see SD_* below.
// ======================================================================
enum {
    SD_G1 = 0,    // sum q_psi * Im(conj(phi) lapphi)
    SD_G2,        // sum Re(conj(lapphi) J)
    SD_X1,        // sum -Im(diss conj(J))
    SD_X2,        // sum 0.5 Re(diss conj(phi)) q_psi
    SD_PHI_R, SD_PHI_I,       // sum phi
    SD_QPC_R, SD_QPC_I,       // sum q_psi conj(phi)
    SD_PHI2,      // sum |phi|^2
    SD_GRAD2,     // sum |phix|^2 + |phiy|^2
    SD_LAP2,      // sum |lapphi|^2
    SD_J_R, SD_J_I,           // sum of the wave-advection product (for the (0,0) fix)
    SD_Q2,        // sum q^2
    SD_QP2,       // sum q_psi^2
    SD_QP3,       // sum q_psi^3
    SD_COUNT
};

struct PhysArgs {
    size_t npts;
    int flags;
    const double* mcoef;      // [member][MC_COUNT]: nu4w, nuw, muw of diss
    const cd *uv, *qs, *phi, *phix, *phiy, *lapphi, *lap2phi, *uvq;
    cd *P1, *P2;
    double* partials;
};

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_phys_rhs(PhysArgs a) {
    const size_t mb = (size_t)blockIdx.y * a.npts;
    double s[SD_COUNT];
#pragma unroll
    for (int k = 0; k < SD_COUNT; ++k) s[k] = 0.0;
    const bool ybj = (a.flags & MF_YBJ) != 0, wr = !(a.flags & MF_NO_WRITE);
    const bool nosums = ybj || (a.flags & MF_SKIP_P1);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd uv = a.uv[mb + i], qs = a.qs[mb + i];
        const cd phi = a.phi[mb + i], px = a.phix[mb + i], py = a.phiy[mb + i];
        const double u = uv.x, v = uv.y, q = qs.x, qpsi = qs.x - qs.y;
        const cd J = make_double2(u * px.x + v * py.x, u * px.y + v * py.y);
        cd Jadv = J;
        if (a.flags & MF_QL_ADV) {
            const cd w = a.uvq[mb + i];
            Jadv = make_double2(w.x * px.x + w.y * py.x, w.x * px.y + w.y * py.y);
        }
        if (wr) {
            if (!ybj && !(a.flags & (MF_SKIP_P1 | MF_P1_BY_LOADER))) a.P1[mb + i] = make_double2(u * q, v * q);
            if (!(a.flags & MF_SKIP_P2))
                a.P2[mb + i] = make_double2(-Jadv.x + 0.5 * phi.y * qpsi, -Jadv.y - 0.5 * phi.x * qpsi);
        }
        if (nosums) continue;
        s[SD_PHI_R] += phi.x; s[SD_PHI_I] += phi.y;
        s[SD_QPC_R] += qpsi * phi.x; s[SD_QPC_I] += -qpsi * phi.y;
        s[SD_PHI2] += phi.x * phi.x + phi.y * phi.y;
        s[SD_GRAD2] += px.x * px.x + px.y * px.y + py.x * py.x + py.y * py.y;
        s[SD_J_R] += Jadv.x; s[SD_J_I] += Jadv.y;
        s[SD_Q2] += q * q;
        s[SD_QP2] += qpsi * qpsi;
        s[SD_QP3] += qpsi * qpsi * qpsi;
        if (a.flags & MF_SPEC_BUDGET) continue;      // the lapphi terms come from k_spec_stage
        const double* mc = a.mcoef + (size_t)blockIdx.y * MC_COUNT;
        const double nuw = mc[MC_NUW], muw = mc[MC_MUW];
        const cd lp = a.lapphi[mb + i];
        cd diss = make_double2(nuw * lp.x - muw * phi.x, nuw * lp.y - muw * phi.y);
        if (a.flags & MF_HAS_LAP2) {
            const double nu4w = mc[MC_NU4W];
            const cd l2 = a.lap2phi[mb + i];
            diss.x += -nu4w * l2.x; diss.y += -nu4w * l2.y;
        }
        s[SD_G1] += qpsi * (phi.x * lp.y - phi.y * lp.x);            // Im(conj(phi) lap)
        s[SD_G2] += lp.x * J.x + lp.y * J.y;                          // Re(conj(lap) J)
        s[SD_X1] += -(diss.y * J.x - diss.x * J.y);                   // -Im(diss conj(J))
        s[SD_X2] += 0.5 * (diss.x * phi.x + diss.y * phi.y) * qpsi;   // 0.5 Re(diss conj(phi)) q_psi
        s[SD_LAP2] += lp.x * lp.x + lp.y * lp.y;
    }
    if (!nosums) block_reduce_store<SD_COUNT>(s, a.partials);
}

// sums over the blocks of one member in a fixed order: out[member][k].  256 threads: thread (part, k) adds the blocks
// part, part + 16, ... of sum k, then thread k adds the 16 parts - always the same order, so results are reproducible.
__global__ void __launch_bounds__(256) k_finalize(const double* __restrict__ partials, int nblk, int K, double* __restrict__ out, int is_max) {
    __shared__ double sh[16][17];
    const int m = blockIdx.x, k = threadIdx.x & 15, part = threadIdx.x >> 4;
    const double* p = partials + (size_t)m * nblk * K;
    double x = is_max ? -1.0e300 : 0.0;
    if (k < K)
        for (int b = part; b < nblk; b += 16) x = is_max ? fmax(x, p[(size_t)b * K + k]) : x + p[(size_t)b * K + k];
    sh[part][k] = x;
    __syncthreads();
    if (threadIdx.x < K) {
        double y = sh[0][threadIdx.x];
        for (int q = 1; q < 16; ++q) y = is_max ? fmax(y, sh[q][threadIdx.x]) : y + sh[q][threadIdx.x];
        out[(size_t)m * K + threadIdx.x] = y;
    }
}

// ======================================================================
// [E] spectral stage update, (K,-K) pairs (Kernel.py:324-334, :346-351, :363-368, :380-387;
//     YBJModel.py:62-84) + the spectral budget sums (Parseval form of Kernel.py:635-640
//     ep_psi and the nu4w term of :646-652 chi_phi), evaluated on the pre-update state.
// ======================================================================
// Spectral budget sums of a stage (MF_SPEC_BUDGET), on the phih the stage starts from and the raw transform P2h of
// P2 = -J(psi,phi) - 0.5i phi q_psi.  With lap = ifft(-wv2 phih), diss = ifft((-nu4w wv4 - nuw wv2 - muw) phih):
//   mean Re(conj(lap) P2)  = -(0.5 G1 + G2)   so  gamma1 + gamma2 = 0.5 hslash Re(T1) / (M^2 f)
//   mean Im(diss conj(P2)) =  X1 + X2         so  xi1 + xi2 = (-nu4w Im T2 - nuw Im T1 - muw Im T0) / (M^2 f)
// where Tn = sum_K wv2^n phih(K) conj(P2h(K))  (Parseval; G1, G2, X1, X2 as in k_phys_rhs, Kernel.py:684-700).
enum { SE_T0R = 0, SE_T0I, SE_T1R, SE_T1I, SE_T2R, SE_T2I, SE_LAP2, SE_WV6PHI, SE_COUNT };

struct StageArgs {
    Grid g;
    int stage;        // 1..4
    int flags;
    int do_q;         // 0 for YBJ (and for the phi half of a split stage)
    int do_phi;       // 0 for the q half of a split stage
    int sums_here;    // this launch evaluates the stage's spectral budget sums (exactly one launch per stage does)
    int hsym;         // q equation: store the element at -K as the conjugate of the one at K (needs filtr(K) == filtr(-K))
    const cd *P1, *P2;
    const cd *y0q, *y0p;      // state at the start of the step
    cd *yq, *yp;              // current stage state (stage 1: output buffers distinct from y0)
    cd *y1q, *y1p, *F0q, *F0p, *Fabq, *Fabp;
    const cd* ph;
    TableSet tq, tp;
    const double* filtr;
    const double* sumsD;      // per member [SD_COUNT] (for the (0,0) fix)
    double* partials;         // [member][block][SE_COUNT]
};

__device__ __forceinline__ cd etd_update(int stage, cd y0, cd y1, cd Fn, cd& F0, cd& Fab, const TableSet& t, size_t ti,
                                         double fl) {
    cd r;
    if (stage == 1 || stage == 2) {
        r = cadd(cmul(t.E2[ti], y0), cmul(Fn, t.Q[ti]));
        if (stage == 1) F0 = Fn; else Fab = Fn;
    } else if (stage == 3) {
        const cd c = make_double2(2.0 * Fn.x - F0.x, 2.0 * Fn.y - F0.y);
        r = cadd(cmul(t.E2[ti], y1), cmul(c, t.Q[ti]));
        Fab = cadd(Fab, Fn);
    } else {
        const cd ab2 = make_double2(2.0 * Fab.x, 2.0 * Fab.y);
        r = cadd(cadd(cadd(cmul(t.E[ti], y0), cmul(F0, t.f0[ti])), cmul(ab2, t.fab[ti])), cmul(Fn, t.fc[ti]));
    }
    return make_double2(r.x * fl, r.y * fl);
}

// ST (stage 1..4), DQ / DP (update the q / phi equation) are compile-time so that every instantiation carries only
// the loads of its stage and equation.  Every launch updates one equation: a body that updated both needed 128 registers
// and ran at ~79 % of the HBM peak, the two halves launched back to back are lighter and faster (they share only the 8 B
// filter value).  PM: the updated equation's tables hold one set per member (a parameter sweep), indexed like the state;
// otherwise one shared set indexed by the wavenumber alone.
template <int ST, bool DQ, bool DP, bool PM>
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_spec_stage(StageArgs a) {
    const int N = a.g.N, H = N >> 1, NC = a.g.ncl;
    const size_t npts = (size_t)N * NC, mb = (size_t)blockIdx.y * npts;
    const size_t total = (size_t)(H + 1) * NC;
    constexpr int st = ST;
    double s[SE_COUNT];
#pragma unroll
    for (int k = 0; k < SE_COUNT; ++k) s[k] = 0.0;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(t / NC), lc = (int)(t % NC);
        const int kyp = (N - ky) & (N - 1), lcp = grid_partner(a.g, lc);
        if (kyp == ky && lcp < lc) continue;
        const int kx = grid_kx(a.g, lc), kxp = grid_kx(a.g, lcp);
        const size_t t1 = (size_t)ky * NC + lc, t2 = (size_t)kyp * NC + lcp;   // table indices
        const bool mode00 = (ky == 0 && kx == 0);
        const size_t i1 = mb + t1, i2 = mb + t2;
        const bool self = (t1 == t2);
        const double fl1 = a.filtr[t1], fl2 = a.hsym ? fl1 : a.filtr[t2];   // hsym implies filtr(K) == filtr(-K)
        const bool specb = (a.flags & MF_SPEC_BUDGET) != 0;
        if (a.sums_here && (specb || (a.flags & MF_HAS_LAP2))) {   // |phih|^2 moments on the pre-update phih (Kernel.py:629-652)
            const cd c1 = (st == 1) ? a.y0p[i1] : a.yp[i1], c2 = (st == 1) ? a.y0p[i2] : a.yp[i2];
            const double k1 = a.g.dk * (double)sidx(kx, N), l1 = a.g.dk * (double)sidx(ky, N);
            const double wv2 = k1 * k1 + l1 * l1, w4 = wv2 * wv2;
            const double m2 = (c1.x * c1.x + c1.y * c1.y) + (self ? 0.0 : (c2.x * c2.x + c2.y * c2.y));
            s[SE_LAP2] += w4 * m2;
            s[SE_WV6PHI] += w4 * wv2 * m2;
            if (specb) {
                const cd F1 = a.P2[i1], F2 = a.P2[i2];   // raw transform, before the (0,0) fix
                double zr = c1.x * F1.x + c1.y * F1.y, zi = c1.y * F1.x - c1.x * F1.y;
                if (!self) { zr += c2.x * F2.x + c2.y * F2.y; zi += c2.y * F2.x - c2.x * F2.y; }
                s[SE_T0R] += zr; s[SE_T0I] += zi;
                s[SE_T1R] += wv2 * zr; s[SE_T1I] += wv2 * zi;
                s[SE_T2R] += w4 * zr; s[SE_T2I] += w4 * zi;
            }
        }
        // ---------------- phi equation
        if constexpr (DP) {
            cd F1 = a.P2[i1], F2 = a.P2[i2];
            if ((a.flags & MF_FIX00) && mode00) {
                const double* sd = a.sumsD + (size_t)blockIdx.y * SD_COUNT;
                F1.x += sd[SD_J_R]; F1.y += sd[SD_J_I];
                F2 = F1;
            }
            const cd cur1 = (st == 1) ? a.y0p[i1] : a.yp[i1];
            const cd cur2 = (st == 1) ? a.y0p[i2] : a.yp[i2];
            cd F0a, F0b, Faba, Fabb, y1a, y1b;
            if (st >= 3) { F0a = a.F0p[i1]; F0b = a.F0p[i2]; }
            if (st >= 3) { Faba = a.Fabp[i1]; Fabb = a.Fabp[i2]; }
            if (st == 3) { y1a = a.y1p[i1]; y1b = a.y1p[i2]; }
            const cd b1 = (st == 1) ? cur1 : a.y0p[i1], b2 = (st == 1) ? cur2 : a.y0p[i2];
            const cd n1 = etd_update(st, b1, y1a, F1, F0a, Faba, a.tp, PM ? i1 : t1, fl1);
            a.yp[i1] = n1;
            if (st == 1) { a.F0p[i1] = F0a; a.y1p[i1] = n1; }
            if (st == 2 || st == 3) a.Fabp[i1] = Faba;
            if (!self) {
                const cd n2 = etd_update(st, b2, y1b, F2, F0b, Fabb, a.tp, PM ? i2 : t2, fl2);
                a.yp[i2] = n2;
                if (st == 1) { a.F0p[i2] = F0b; a.y1p[i2] = n2; }
                if (st == 2 || st == 3) a.Fabp[i2] = Fabb;
            }
        }
        // ---------------- q equation
        if constexpr (DQ) {
            const double k1 = a.g.dk * (double)sidx(kx, N), l1 = a.g.dk * (double)sidx(ky, N);
            const double k2 = a.g.dk * (double)sidx(kxp, N), l2 = a.g.dk * (double)sidx(kyp, N);
            const cd p1 = a.P1[i1], p2 = a.P1[i2];
            // A = fft(u q)(K) = 0.5 (P(K) + conj P(-K)),  B = fft(v q)(K) = -0.5 i (P(K) - conj P(-K))
            const cd A = make_double2(0.5 * (p1.x + p2.x), 0.5 * (p1.y - p2.y));
            const cd B = make_double2(0.5 * (p1.y + p2.y), -0.5 * (p1.x - p2.x));
            // jach(K) = i k A + i l B ; jach(-K) = i k2 conj(A) + i l2 conj(B);  Fn = -jach
            cd F1 = make_double2(k1 * A.y + l1 * B.y, -(k1 * A.x + l1 * B.x));
            cd F2 = make_double2(-(k2 * A.y + l2 * B.y), -(k2 * A.x + l2 * B.x));
            if (mode00) { F1 = make_double2(0.0, 0.0); F2 = F1; }
            // q is real: every array of the q equation, its tables and the (symmetric) filter are Hermitian, so with
            // a.hsym the element at -K is stored as the conjugate of the one at K and none of its operands are read
            // (not on the Nyquist lines: numpy's signed wavenumber there is -N/2 for K and for -K alike, so the reference's
            // Jacobian and tables are not conjugate-symmetric on them)
            const bool hs = a.hsym && !self && kx != H && ky != H;
            cd F0a, F0b, Faba, Fabb, y1a, y1b, b2;
            if (st >= 3) { F0a = a.F0q[i1]; if (!hs) F0b = a.F0q[i2]; }
            if (st >= 3) { Faba = a.Fabq[i1]; if (!hs) Fabb = a.Fabq[i2]; }
            if (st == 3) { y1a = a.y1q[i1]; if (!hs) y1b = a.y1q[i2]; }
            const cd b1 = a.y0q[i1];                       // the ep_psi sums of this state: k_spec_invert
            if (!hs) b2 = a.y0q[i2];
            const cd n1 = etd_update(st, b1, y1a, F1, F0a, Faba, a.tq, PM ? i1 : t1, fl1);
            a.yq[i1] = n1;
            if (st == 1) { a.F0q[i1] = F0a; a.y1q[i1] = n1; }
            if (st == 2 || st == 3) a.Fabq[i1] = Faba;
            if (!self) {
                cd n2;
                if (hs) {
                    n2 = make_double2(n1.x, -n1.y);
                    F0b = make_double2(F0a.x, -F0a.y);
                    Fabb = make_double2(Faba.x, -Faba.y);
                } else n2 = etd_update(st, b2, y1b, F2, F0b, Fabb, a.tq, PM ? i2 : t2, fl2);
                a.yq[i2] = n2;
                if (st == 1) { a.F0q[i2] = F0b; a.y1q[i2] = n2; }
                if (st == 2 || st == 3) a.Fabq[i2] = Fabb;
            }
        }
    }
    if (a.sums_here) block_reduce_store<SE_COUNT>(s, a.partials);
}

template <bool DQ, bool DP, bool PM>
static void launch_spec_stage_pm(const StageArgs& a, dim3 grid, cudaStream_t st) {
    switch (a.stage) {
        case 1: k_spec_stage<1, DQ, DP, PM><<<grid, NIWQG_PW_THREADS, 0, st>>>(a); break;
        case 2: k_spec_stage<2, DQ, DP, PM><<<grid, NIWQG_PW_THREADS, 0, st>>>(a); break;
        case 3: k_spec_stage<3, DQ, DP, PM><<<grid, NIWQG_PW_THREADS, 0, st>>>(a); break;
        default: k_spec_stage<4, DQ, DP, PM><<<grid, NIWQG_PW_THREADS, 0, st>>>(a); break;
    }
}
// pm: the tables of the equation this launch updates are per member
template <bool DQ, bool DP>
static cudaError_t launch_spec_stage(const StageArgs& a, dim3 grid, cudaStream_t st, bool pm) {
    if (pm) launch_spec_stage_pm<DQ, DP, true>(a, grid, st);
    else launch_spec_stage_pm<DQ, DP, false>(a, grid, st);
    return cudaGetLastError();
}

// ======================================================================
// per-stage budget tendencies and their RK4-weighted accumulation
// (Kernel.py:319-322, :390-392, :697-701)
// ======================================================================
struct BudgetArgs {
    int stage;           // 1..4 ; 0 = evaluate only (diagnostics tick)
    double M;            // N*N
    double dt;
    const double* mcoef; // [member][MC_COUNT]: f, hslash, kappa2 and the dissipation coefficients
    const double *sumsD, *sumsE, *sumsI;   // physical (k_phys_rhs), stage-spectral (k_spec_stage), k_spec_invert
    int spec_budget;
    double* scal;        // [member][NIWQG_S_COUNT]
    double* stagev;      // [member][4][3]
};

// ======================================================================
// generic reductions
// ======================================================================
// sum over the full c2c spectrum (mode (0,0) removed) of |X|^2 weighted by wv2^pw, pw in {0,1,2}
// sums: [0] sum wv2*|ph|^2  [1] sum wv2^2*|qh|^2  [2] sum wv2*|wv2i qh|^2  [3] sum wv2*|wv2i qwh|^2
//       [4] sum (k'k + l'l) Re(phq conj(phw))     [5..7] Parseval forms of ep_psi on the current state
//       [8] sum wv2^3 |phih|^2
enum { SS_KE = 0, SS_CHIQ, SS_KEQ, SS_KEW, SS_KEQW, SS_QLAP2PSI, SS_PLAPQ, SS_PQ, SS_WV6PHI, SS_COUNT };

struct SpecSumArgs {
    Grid g;
    const cd *ph, *qh, *qwh, *phih;
};

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_spec_sums(SpecSumArgs a, double* partials) {
    const int N = a.g.N, NC = a.g.ncl;
    const size_t npts = (size_t)N * NC, mb = (size_t)blockIdx.y * npts;
    double s[SS_COUNT];
#pragma unroll
    for (int k = 0; k < SS_COUNT; ++k) s[k] = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / NC), kx = grid_kx(a.g, (int)(i % NC));
        if (ky == 0 && kx == 0) continue;
        const double k = a.g.dk * (double)sidx(kx, N), l = a.g.dk * (double)sidx(ky, N);
        const double wv2 = k * k + l * l, wv2i = 1.0 / wv2;
        const cd ph = a.ph[mb + i], qh = a.qh[mb + i];
        s[SS_KE] += wv2 * (ph.x * ph.x + ph.y * ph.y);
        s[SS_CHIQ] += wv2 * wv2 * (qh.x * qh.x + qh.y * qh.y);
        const cd phq = make_double2(-wv2i * qh.x, -wv2i * qh.y);
        s[SS_KEQ] += wv2 * (phq.x * phq.x + phq.y * phq.y);
        if (a.qwh) {
            const cd qw = a.qwh[mb + i];
            const cd phw = make_double2(wv2i * qw.x, wv2i * qw.y);
            s[SS_KEW] += wv2 * (phw.x * phw.x + phw.y * phw.y);
            const double kk = (kx == (N >> 1)) ? 0.0 : k * k, ll = (ky == (N >> 1)) ? 0.0 : l * l;
            s[SS_KEQW] += (kk + ll) * (phq.x * phw.x + phq.y * phw.y);
        }
        const double r = qh.x * ph.x + qh.y * ph.y;    // Re(qh conj(ph)); ph Hermitian => anti-Hermitian part of qh drops
        s[SS_QLAP2PSI] += wv2 * wv2 * r;
        s[SS_PLAPQ] += -wv2 * r;
        s[SS_PQ] += r;
        if (a.phih) {
            const cd p = a.phih[mb + i];
            s[SS_WV6PHI] += wv2 * wv2 * wv2 * (p.x * p.x + p.y * p.y);
        }
    }
    block_reduce_store<SS_COUNT>(s, partials);
}

// physical sums for the status line / pe_niw / cfl: [0] sum |a|^2+|b|^2 ; max: [0] max(|u|,|v|,|phi|)
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_grad2_sum(const cd* __restrict__ px, const cd* __restrict__ py,
                                                                size_t npts, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd a = px[mb + i], b = py[mb + i];
        s[0] += a.x * a.x + a.y * a.y + b.x * b.x + b.y * b.y;
    }
    block_reduce_store<1>(s, partials);
}

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_cfl_max(const cd* __restrict__ uv, const cd* __restrict__ phi,
                                                              size_t npts, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd w = uv[mb + i];
        double m = fmax(fabs(w.x), fabs(w.y));
        if (phi) { const cd p = phi[mb + i]; m = fmax(m, sqrt(p.x * p.x + p.y * p.y)); }
        s[0] = fmax(s[0], m);
    }
    block_reduce_max_store<1>(s, partials);
}

// second pass of conc_niw (Kernel.py:613-619): centred sums given the means
// [0] sum ups*q_psi  [1] sum ups^2  [2] sum (q_psi - mean)^2,  ups = |phi|^2 - mean|phi|^2
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_conc_sums(const cd* __restrict__ phi, const cd* __restrict__ qs,
                                                                size_t npts, const double* __restrict__ sumsD,
                                                                const double* __restrict__ sumsX, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    const double mphi2 = sumsD[(size_t)blockIdx.y * SD_COUNT + SD_PHI2] / (double)npts;
    const double mqp = sumsX[blockIdx.y] / (double)npts;
    double s[3] = {0.0, 0.0, 0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd p = phi[mb + i], q = qs[mb + i];
        const double ups = (p.x * p.x + p.y * p.y) - mphi2, qp = q.x - q.y;
        s[0] += ups * qp;
        s[1] += ups * ups;
        s[2] += (qp - mqp) * (qp - mqp);
    }
    block_reduce_store<3>(s, partials);
}

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qpsi_sum(const cd* __restrict__ qs, size_t npts, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd q = qs[mb + i];
        s[0] += q.x - q.y;
    }
    block_reduce_store<1>(s, partials);
}

// Physical arrays of a grid whose row pass is split over a cluster of C CTAs (N = 8192: C = 2) are stored with x
// de-interleaved: position p of a row holds x = C*(p % M) + p / M (M = N/C).  All physical-space kernels are
// pointwise, so only uploads (set_q, set_phi, set_c, fft2) and downloads (attribute reads) convert.
template <typename T>
__global__ void k_deint(const T* __restrict__ in, T* __restrict__ out, size_t total, int N, int M, int C, int to_deint) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / N;
        const int p = (int)(i % N), x = C * (p % M) + p / M;
        if (to_deint) out[row * N + p] = in[row * N + x];
        else out[row * N + x] = in[row * N + p];
    }
}

// split / merge helpers for attribute reads and seeding
__global__ void k_extract_real(const cd* __restrict__ in, double* __restrict__ out, size_t n, int which) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const cd x = in[i];
        out[i] = which == 0 ? x.x : which == 1 ? x.y : x.x - x.y;
    }
}
__global__ void k_real_to_cplx(const double* __restrict__ in, cd* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = make_double2(in[i], 0.0);
}
