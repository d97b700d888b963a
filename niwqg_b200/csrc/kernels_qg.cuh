// kernels_qg.cuh -- the stand-alone QG model (niwqg/QGModel.py) on the c2c engine.
//
// State lives in numpy's rfft2 layout (N rows x N/2+1 columns).  irfft2(H) equals
// ifft2 of the "full Hermitian extension" FH(H):
//     FH(H)(ky,kx) = H(ky,kx)                                 0 < kx < N/2
//                  = 0.5*(H(ky,kx) + conj(H(-ky,kx)))           kx in {0, N/2}   (c2r drops the rest)
//                  = conj(H(-ky, N-kx))                         kx > N/2
// so three real fields (u, v, q) ride on two c2c inverse transforms (u + i v packed, q),
// and rfft2 of the two products u*q, v*q on one packed forward transform.
#pragma once
#include "common.cuh"
#include "kernels_family.cuh"

enum { QGX_PLAIN = 0 };

__device__ __forceinline__ double qg_k(int kx, double dk) { return dk * (double)kx; }   // QGModel.py:246 (kx <= N/2)

struct QgExpandArgs {
    int N, nk;
    double dk;
    const cd* qh;     // [B][N][nk]
    cd* ph;           // [B][N][nk]   ph = -wv2i*qh (QGModel.py:501)
    cd* uv;           // [B][N][N]    spectrum of u + i v   (may be null)
    cd* qs;           // [B][N][N]    spectrum of q         (may be null)
};

// derived half-spectrum fields at a source point: -i l ph, i k ph  with ph = -wv2i*h
__device__ __forceinline__ void qg_uv_terms(cd h, double k, double l, cd& du, cd& dv, cd& ph) {
    const double wv2 = k * k + l * l;
    const double wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
    ph = make_double2(-wv2i * h.x, -wv2i * h.y);
    du = make_double2(l * ph.y, -l * ph.x);      // -i l ph
    dv = make_double2(-k * ph.y, k * ph.x);      //  i k ph
}

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_expand(QgExpandArgs a) {
    const int N = a.N, nk = a.nk, H = N >> 1;
    const size_t npts = (size_t)N * N, nspec = (size_t)N * nk;
    const size_t mbf = (size_t)blockIdx.y * npts, mbh = (size_t)blockIdx.y * nspec;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / N), kx = (int)(i % N);
        const int kyp = (N - ky) & (N - 1);
        cd U, V, Q;
        if (kx > H) {
            const int sx = N - kx;
            const cd h = a.qh[mbh + (size_t)kyp * nk + sx];
            cd du, dv, ph;
            qg_uv_terms(h, qg_k(sx, a.dk), a.dk * (double)sidx(kyp, N), du, dv, ph);
            U = cconj(du); V = cconj(dv); Q = cconj(h);
        } else {
            const cd h = a.qh[mbh + (size_t)ky * nk + kx];
            cd du, dv, ph;
            qg_uv_terms(h, qg_k(kx, a.dk), a.dk * (double)sidx(ky, N), du, dv, ph);
            if (a.ph) a.ph[mbh + (size_t)ky * nk + kx] = ph;
            if (kx == 0 || kx == H) {
                const cd h2 = a.qh[mbh + (size_t)kyp * nk + kx];
                cd du2, dv2, ph2;
                qg_uv_terms(h2, qg_k(kx, a.dk), a.dk * (double)sidx(kyp, N), du2, dv2, ph2);
                U = make_double2(0.5 * (du.x + du2.x), 0.5 * (du.y - du2.y));
                V = make_double2(0.5 * (dv.x + dv2.x), 0.5 * (dv.y - dv2.y));
                Q = make_double2(0.5 * (h.x + h2.x), 0.5 * (h.y - h2.y));
            } else {
                U = du; V = dv; Q = h;
            }
        }
        if (a.uv) a.uv[mbf + i] = make_double2(U.x - V.y, U.y + V.x);   // U + i V
        if (a.qs) a.qs[mbf + i] = Q;
    }
}

struct QgExpand1Args {
    int N, nk;
    double dk;
    const cd* in;   // [B][N][nk]
    cd* out;        // [B][N][N]
    int mode;
};

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_expand1(QgExpand1Args a) {
    const int N = a.N, nk = a.nk, H = N >> 1;
    const size_t npts = (size_t)N * N, nspec = (size_t)N * nk;
    const size_t mbf = (size_t)blockIdx.y * npts, mbh = (size_t)blockIdx.y * nspec;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / N), kx = (int)(i % N);
        const int kyp = (N - ky) & (N - 1);
        cd X;
        if (kx > H) {
            X = cconj(a.in[mbh + (size_t)kyp * nk + (N - kx)]);
        } else {
            X = a.in[mbh + (size_t)ky * nk + kx];
            if (kx == 0 || kx == H) {
                const cd X2 = a.in[mbh + (size_t)kyp * nk + kx];
                X = make_double2(0.5 * (X.x + X2.x), 0.5 * (X.y - X2.y));
            }
        }
        a.out[mbf + i] = X;
    }
}

__global__ void k_qg_take_half(const cd* __restrict__ full, cd* __restrict__ half, int N, int nk) {
    const size_t npts = (size_t)N * N, nspec = (size_t)N * nk;
    const size_t mbf = (size_t)blockIdx.y * npts, mbh = (size_t)blockIdx.y * nspec;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nspec; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / nk), kx = (int)(i % nk);
        half[mbh + i] = full[mbf + (size_t)ky * N + kx];
    }
}

__global__ void k_qg_set_q_real(const double* __restrict__ q, cd* __restrict__ qs, size_t npts) {
    const size_t mb = (size_t)blockIdx.y * npts;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x)
        qs[mb + i] = make_double2(q[mb + i], 0.0);
}

// P1 = u q + i v q ;  P2 = u c + i v c  (QGModel.py:479-481, :493-495); c carried in cphys.x
__global__ void k_qg_products(const cd* __restrict__ uv, const cd* __restrict__ qs, const cd* __restrict__ cphys,
                              cd* __restrict__ P1, cd* __restrict__ P2, size_t npts) {
    const size_t mb = (size_t)blockIdx.y * npts;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd w = uv[mb + i];
        const double q = qs[mb + i].x;
        P1[mb + i] = make_double2(w.x * q, w.y * q);
        if (cphys) {
            const double c = cphys[mb + i].x;
            P2[mb + i] = make_double2(w.x * c, w.y * c);
        }
    }
}

// ----------------------------------------------------------------------
// stage update on the half spectrum + budget sums (QGModel.py:338-407, :588-598)
// ----------------------------------------------------------------------
enum { QE_QLAP2PSI = 0, QE_PLAPQ, QE_PQ, QE_C2, QE_GRADC2, QE_LAPC2, QE_COUNT };

struct QgStageArgs {
    int N, nk, stage, ps;
    double dk, nu4c;
    const cd *P1, *P2;              // full N x N packed forward transforms
    const cd* y0q; cd *yq, *y1q, *F0q, *Fabq;
    const cd* y0c; cd *yc, *y1c, *F0c, *Fabc;
    TableSet tq, tc;
    const double* filtr;
    double* partials;
};

// -jacobian at K=(ky,kx) (half spectrum) from the packed transform P
__device__ __forceinline__ cd qg_neg_jac(const cd* __restrict__ P, size_t mbf, int N, int ky, int kx, double k, double l) {
    const int kyp = (N - ky) & (N - 1), kxp = (N - kx) & (N - 1);
    const cd p1 = P[mbf + (size_t)ky * N + kx], p2 = P[mbf + (size_t)kyp * N + kxp];
    const cd A = make_double2(0.5 * (p1.x + p2.x), 0.5 * (p1.y - p2.y));
    const cd B = make_double2(0.5 * (p1.y + p2.y), -0.5 * (p1.x - p2.x));
    return make_double2(k * A.y + l * B.y, -(k * A.x + l * B.x));
}

__device__ __forceinline__ cd qg_update_point(int st, const cd* y0, cd* y, cd* y1, cd* F0, cd* Fab, const TableSet& t,
                                              size_t gi, size_t ti, cd Fn, double fl) {
    cd F0v = make_double2(0, 0), Fabv = F0v, y1v = F0v;
    if (st >= 3) { F0v = F0[gi]; Fabv = Fab[gi]; }
    if (st == 3) y1v = y1[gi];
    const cd n = etd_update(st, y0[gi], y1v, Fn, F0v, Fabv, t, ti, fl);
    y[gi] = n;
    if (st == 1) { F0[gi] = F0v; y1[gi] = n; }
    if (st == 2 || st == 3) Fab[gi] = Fabv;
    return n;
}

// PMQ / PMC: the q / c tables hold one set per member (a parameter sweep), indexed like the state
template <bool PMQ, bool PMC>
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_stage(QgStageArgs a) {
    const int N = a.N, nk = a.nk, H = N >> 1, st = a.stage;
    const size_t npts = (size_t)N * N, nspec = (size_t)N * nk;
    const size_t mbf = (size_t)blockIdx.y * npts, mbh = (size_t)blockIdx.y * nspec;
    double s[QE_COUNT];
#pragma unroll
    for (int k = 0; k < QE_COUNT; ++k) s[k] = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nspec; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / nk), kx = (int)(i % nk);
        const int kyp = (N - ky) & (N - 1);
        const bool edge = (kx == 0 || kx == H);
        if (edge && ky > H) continue;            // handled by the (ky' = N-ky) thread
        const bool pair = edge && (kyp != ky);
        const double k = qg_k(kx, a.dk), l1 = a.dk * (double)sidx(ky, N), l2 = a.dk * (double)sidx(kyp, N);
        const size_t t1 = (size_t)ky * nk + kx, t2 = (size_t)kyp * nk + kx;
        const double wv2 = k * k + l1 * l1;      // same for both members of an edge pair
        const double wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
        // ---- q equation
        const cd qn1 = qg_update_point(st, a.y0q, a.yq, a.y1q, a.F0q, a.Fabq, a.tq, mbh + t1, PMQ ? mbh + t1 : t1,
                                       qg_neg_jac(a.P1, mbf, N, ky, kx, k, l1), a.filtr[t1]);
        cd qn2 = qn1;
        if (pair)
            qn2 = qg_update_point(st, a.y0q, a.yq, a.y1q, a.F0q, a.Fabq, a.tq, mbh + t2, PMQ ? mbh + t2 : t2,
                                  qg_neg_jac(a.P1, mbf, N, kyp, kx, k, l2), a.filtr[t2]);
        // ---- ep_psi on (new qh, new ph, stale q):  stale q is y0 for stages 1-3, the new qh for stage 4
        {
            cd qs1 = (st == 4) ? qn1 : a.y0q[mbh + t1];
            cd X = qn1;   // FH(qh_new) at this point
            double w = 2.0;
            if (edge) {
                const cd qs2 = (st == 4) ? qn2 : a.y0q[mbh + t2];
                qs1 = make_double2(0.5 * (qs1.x + qs2.x), 0.5 * (qs1.y - qs2.y));
                X = make_double2(0.5 * (qn1.x + qn2.x), 0.5 * (qn1.y - qn2.y));
                w = pair ? 2.0 : 1.0;            // the pair thread stands for both rows ky and -ky
            }
            // ph_new = -wv2i X ; lap2psi <-> wv4 ph_new = -wv2 X ; lapq <-> -wv2 X ; p <-> -wv2i X
            const double rq = qs1.x * X.x + qs1.y * X.y;            // Re(qstale conj(X))
            const double xx = X.x * X.x + X.y * X.y;
            s[QE_QLAP2PSI] += w * (-wv2) * rq;                      // Re(qstale conj(-wv2 X))
            s[QE_PLAPQ] += w * ((wv2 != 0.0) ? xx : 0.0);           // Re(-wv2i X conj(-wv2 X))
            s[QE_PQ] += w * (-wv2i) * rq;                           // Re(-wv2i X conj(qstale))
        }
        if (!a.ps) continue;
        // ---- passive scalar
        const cd cn1 = qg_update_point(st, a.y0c, a.yc, a.y1c, a.F0c, a.Fabc, a.tc, mbh + t1, PMC ? mbh + t1 : t1,
                                       qg_neg_jac(a.P2, mbf, N, ky, kx, k, l1), a.filtr[t1]);
        cd cn2 = cn1;
        if (pair)
            cn2 = qg_update_point(st, a.y0c, a.yc, a.y1c, a.F0c, a.Fabc, a.tc, mbh + t2, PMC ? mbh + t2 : t2,
                                  qg_neg_jac(a.P2, mbf, N, kyp, kx, k, l2), a.filtr[t2]);
        {
            // C2 = spec_var(ch), gradC2 = spec_var(wv ch): weights 2 (interior) / 1 (edge columns), no projection (QGModel.py:611-619)
            const double a1 = cn1.x * cn1.x + cn1.y * cn1.y, a2 = cn2.x * cn2.x + cn2.y * cn2.y;
            const double wsv = edge ? 1.0 : 2.0;
            const bool zero = (ky == 0 && kx == 0);
            if (!zero) { s[QE_C2] += wsv * a1; s[QE_GRADC2] += wsv * wv2 * a1; }
            if (pair) { s[QE_C2] += wsv * a2; s[QE_GRADC2] += wsv * wv2 * a2; }
            // mean(lapc^2) = sum |FH(-wv2 ch)|^2
            cd X = cn1;
            double w = 2.0;
            if (edge) { X = make_double2(0.5 * (cn1.x + cn2.x), 0.5 * (cn1.y - cn2.y)); w = pair ? 2.0 : 1.0; }
            s[QE_LAPC2] += w * wv2 * wv2 * (X.x * X.x + X.y * X.y);
        }
    }
    block_reduce_store<QE_COUNT>(s, a.partials);
}

struct QgBudgetArgs {
    int stage, ps;
    double M, dt;
    const double* mcoef;     // [member][MC_COUNT]: nu4, nu, mu, nu4c, muc
    const double* sumsE;
    double *scal, *stagev;
};

__global__ void k_qg_budget(QgBudgetArgs a) {
    const int m = blockIdx.x;
    if (threadIdx.x != 0) return;
    const double* se = a.sumsE + (size_t)m * QE_COUNT;
    const double* mc = a.mcoef + (size_t)m * MC_COUNT;
    double* sc = a.scal + (size_t)m * NIWQG_S_COUNT;
    double* sv = a.stagev + (size_t)m * 12 + (a.stage - 1) * 3;
    const double M2 = a.M * a.M;
    const double nu4 = mc[MC_NU4], nu = mc[MC_NU], mu = mc[MC_MU], nu4c = mc[MC_NU4C], muc = mc[MC_MUC];
    sv[0] = nu4 * (se[QE_QLAP2PSI] / M2) - nu * (se[QE_PLAPQ] / M2) + mu * (se[QE_PQ] / M2);   // QGModel.py:588-593
    // ep_c uses self.nu for the gradient term (QGModel.py:597)
    sv[1] = a.ps ? (-2 * nu4c * (se[QE_LAPC2] / M2) - 2 * nu * (se[QE_GRADC2] / M2) - 2 * muc * (se[QE_C2] / M2)) : 0.0;
    if (a.stage == 4) {
        const double* s0 = a.stagev + (size_t)m * 12;
        sc[NIWQG_S_KE] += a.dt * (s0[0] + 2 * (s0[3] + s0[6]) + s0[9]) / 6.;
        if (a.ps) sc[NIWQG_S_CVAR] += a.dt * (s0[1] + 2 * (s0[4] + s0[7]) + s0[10]) / 6.;
    }
}

// ----------------------------------------------------------------------
// spectral sums on the half spectrum (diagnostics / status / set_q / set_c)
// ----------------------------------------------------------------------
enum { QS_KE = 0, QS_CHIQ, QS_QLAP2PSI, QS_PLAPQ, QS_PQ, QS_C2, QS_GRADC2, QS_LAPC2, QS_LAP2CLAPC, QS_COUNT };

struct QgSumArgs {
    int N, nk;
    double dk;
    const cd *qh, *ch;
    const cd* qs;
};

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_spec_sums(QgSumArgs a, double* partials) {
    const int N = a.N, nk = a.nk, H = N >> 1;
    const size_t nspec = (size_t)N * nk, mbh = (size_t)blockIdx.y * nspec;
    double s[QS_COUNT];
#pragma unroll
    for (int k = 0; k < QS_COUNT; ++k) s[k] = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nspec; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / nk), kx = (int)(i % nk);
        const int kyp = (N - ky) & (N - 1);
        const bool edge = (kx == 0 || kx == H);
        const double k = qg_k(kx, a.dk), l = a.dk * (double)sidx(ky, N);
        const double wv2 = k * k + l * l, wv2i = (wv2 != 0.0) ? 1.0 / wv2 : 0.0;
        const double wsv = edge ? 1.0 : 2.0;
        const bool zero = (ky == 0 && kx == 0);
        const cd q = a.qh[mbh + i];
        const double qq = q.x * q.x + q.y * q.y;
        if (!zero) {
            s[QS_KE] += wsv * wv2 * wv2i * wv2i * qq;      // |wv * (-wv2i qh)|^2
            s[QS_CHIQ] += wsv * wv2 * wv2 * qq;            // |wv2 qh|^2
        }
        // Parseval forms with the irfft2 projection: per half-spectrum point the weight is 2 (interior) or,
        // on the edge columns, 1 with the column-Hermitian part X = 0.5 (q(ky) + conj q(-ky))
        cd X = q;
        if (edge) {
            const cd q2 = a.qh[mbh + (size_t)kyp * nk + kx];
            X = make_double2(0.5 * (q.x + q2.x), 0.5 * (q.y - q2.y));
        }
        const double xx = X.x * X.x + X.y * X.y;
        s[QS_QLAP2PSI] += wsv * (-wv2) * xx;
        s[QS_PLAPQ] += wsv * ((wv2 != 0.0) ? xx : 0.0);
        s[QS_PQ] += wsv * (-wv2i) * xx;
        if (a.ch) {
            const cd c = a.ch[mbh + i];
            const double cc = c.x * c.x + c.y * c.y;
            if (!zero) { s[QS_C2] += wsv * cc; s[QS_GRADC2] += wsv * wv2 * cc; }
            cd Y = c;
            if (edge) {
                const cd c2 = a.ch[mbh + (size_t)kyp * nk + kx];
                Y = make_double2(0.5 * (c.x + c2.x), 0.5 * (c.y - c2.y));
            }
            const double yy = Y.x * Y.x + Y.y * Y.y;
            s[QS_LAPC2] += wsv * wv2 * wv2 * yy;
            s[QS_LAP2CLAPC] += wsv * (-wv2 * wv2 * wv2) * yy;
        }
    }
    block_reduce_store<QS_COUNT>(s, partials);
}

__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_q2_sum(const cd* __restrict__ qs, size_t npts, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const double q = qs[mb + i].x;
        s[0] += q * q;
    }
    block_reduce_store<1>(s, partials);
}

// jacobian_psi_q as a half-spectrum array (QGModel.py:469-481) from the packed transform
__global__ void k_qg_jacobian_out(const cd* __restrict__ P, cd* __restrict__ out, int N, int nk, double dk) {
    const size_t nspec = (size_t)N * nk;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nspec; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / nk), kx = (int)(i % nk);
        const cd nj = qg_neg_jac(P, 0, N, ky, kx, qg_k(kx, dk), dk * (double)sidx(ky, N));
        out[i] = make_double2(-nj.x, -nj.y);
    }
}

// sum over the full spectrum of FH(-wv2 ch) * conj(FH(jach_c)): for Gamma_c (QGModel.py:731)
__global__ void __launch_bounds__(NIWQG_PW_THREADS) k_qg_gamma_sum(const cd* __restrict__ P, const cd* __restrict__ ch, int N,
                                                                   int nk, double dk, double* partials) {
    const int H = N >> 1;
    const size_t npts = (size_t)N * N, nspec = (size_t)N * nk;
    const size_t mbf = (size_t)blockIdx.y * npts, mbh = (size_t)blockIdx.y * nspec;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nspec; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / nk), kx = (int)(i % nk);
        const int kyp = (N - ky) & (N - 1);
        const bool edge = (kx == 0 || kx == H);
        const double k = qg_k(kx, dk), l = dk * (double)sidx(ky, N);
        const double wv2 = k * k + l * l;
        cd nj = qg_neg_jac(P, mbf, N, ky, kx, k, l);
        cd c = ch[mbh + i];
        if (edge) {
            const cd nj2 = qg_neg_jac(P, mbf, N, kyp, kx, k, dk * (double)sidx(kyp, N));
            const cd c2 = ch[mbh + (size_t)kyp * nk + kx];
            nj = make_double2(0.5 * (nj.x + nj2.x), 0.5 * (nj.y - nj2.y));
            c = make_double2(0.5 * (c.x + c2.x), 0.5 * (c.y - c2.y));
        }
        // Re( (-wv2 c) conj(jach) ),  jach = -nj
        s[0] += (edge ? 1.0 : 2.0) * wv2 * (c.x * nj.x + c.y * nj.y);
    }
    block_reduce_store<1>(s, partials);
}

// ----------------------------------------------------------------------
// family helpers used by the attribute-level API (niwqg_jacobian)
// ----------------------------------------------------------------------
// split a packed forward transform W = fft(a + i b) into fft(a) (part 0) or fft(b) (part 1); zero00 clears mode (0,0)
__global__ void k_split_packed(const cd* __restrict__ W, cd* __restrict__ out, int N, int part, int zero00, double scale) {
    const size_t npts = (size_t)N * N;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / N), kx = (int)(i % N);
        const size_t i2 = (size_t)((N - ky) & (N - 1)) * N + ((N - kx) & (N - 1));
        const cd w1 = W[i], w2 = W[i2];
        cd r = part == 0 ? make_double2(0.5 * (w1.x + w2.x), 0.5 * (w1.y - w2.y))
                         : make_double2(0.5 * (w1.y + w2.y), -0.5 * (w1.x - w2.x));
        if (zero00 && i == 0) r = make_double2(0.0, 0.0);
        out[i] = make_double2(scale * r.x, scale * r.y);
    }
}

// jacobian_psi_q (Kernel.py:471-486) from P = fft(u q + i v q)
__global__ void k_jac_psi_q_out(const cd* __restrict__ P, cd* __restrict__ out, int N, double dk) {
    const size_t npts = (size_t)N * N;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const int ky = (int)(i / N), kx = (int)(i % N);
        const size_t i2 = (size_t)((N - ky) & (N - 1)) * N + ((N - kx) & (N - 1));
        const cd p1 = P[i], p2 = P[i2];
        const cd A = make_double2(0.5 * (p1.x + p2.x), 0.5 * (p1.y - p2.y));
        const cd B = make_double2(0.5 * (p1.y + p2.y), -0.5 * (p1.x - p2.x));
        const double k = dk * (double)sidx(kx, N), l = dk * (double)sidx(ky, N);
        cd r = make_double2(-(k * A.y + l * B.y), k * A.x + l * B.x);
        if (i == 0) r = make_double2(0.0, 0.0);
        out[i] = r;
    }
}

__global__ void k_adv_product(const cd* __restrict__ uv, const cd* __restrict__ px, const cd* __restrict__ py,
                              cd* __restrict__ out, size_t npts) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd w = uv[i], a = px[i], b = py[i];
        out[i] = make_double2(w.x * a.x + w.y * b.x, w.x * a.y + w.y * b.y);
    }
}
