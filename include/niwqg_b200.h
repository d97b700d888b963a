/* niwqg_b200.h -- C ABI of the B200-native ETDRK4 hot path of niwqg.
 *
 * Plain pointers and sizes only; no torch / C++ types.  One handle = one model
 * instance (optionally an ensemble of `batch` independent members that share the
 * grid, time step and filter, and either share the physical coefficients or take
 * their own: niwqg_create_ensemble) on one device and one CUDA stream.  All calls
 * are asynchronous on that stream except the ones that return data to the host.
 *
 * Each entry point names the reference interface it replaces (paths relative to
 * the reference tree, cesar-rocha/niwqg).
 *
 * Return value: 0 on success, negative on error; niwqg_last_error() gives text.
 */
#ifndef NIWQG_B200_H
#define NIWQG_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* model variants: the reference's Model subclasses (Seam 2, SURVEY.md section 8b) */
#define NIWQG_MODEL_QG        0  /* niwqg/QGModel.py        */
#define NIWQG_MODEL_COUPLED   1  /* niwqg/CoupledModel.py   */
#define NIWQG_MODEL_UNCOUPLED 2  /* niwqg/UnCoupledModel.py */
#define NIWQG_MODEL_YBJ       3  /* niwqg/YBJModel.py       */
#define NIWQG_MODEL_QL        4  /* niwqg/QLModel.py (repaired, SURVEY.md section 8c) */

/* constructor keywords of niwqg/Kernel.py:70-98 and niwqg/QGModel.py:65-91 that
 * reach the arithmetic */
typedef struct niwqg_params {
    size_t struct_size; /* = sizeof(niwqg_params): a binding built against another layout is rejected, not over-read */
    int model;          /* NIWQG_MODEL_*                                        */
    int nx;             /* grid edge, power of two, 32..8192 (ny==nx, F9)        */
    int batch;          /* ensemble members (>=1)                                */
    int device;         /* CUDA device ordinal                                   */
    double L, dt, U, f, N, m;
    double nu, nu4, mu;         /* q-equation dissipation                        */
    double nuw, nu4w, muw;      /* phi-equation dissipation                      */
    double beta;                /* QGModel only                                  */
    int use_filter, dealias;
    int passive_scalar;         /* QGModel only                                  */
    double nu4c, nuc, muc;      /* QGModel passive scalar                        */
    /* slab decomposition of ONE grid over nranks GPUs (one process per GPU); 0 or 1 = single GPU.
     * Physical arrays passed to set_q / set_phi and returned by get_field are then the rank's rows
     * [rank*nx/nranks, (rank+1)*nx/nranks); spectral arrays are (nx, nx/nranks) column slabs in the
     * conjugate-symmetric ownership described in csrc/common.cuh (struct Grid). */
    int rank, nranks;
    char nccl_id[128];          /* ncclUniqueId from niwqg_nccl_unique_id() on rank 0, shared by the caller */
} niwqg_params;

/* the coefficients of niwqg_params that one member of an ensemble may set for itself (a parameter sweep in one
 * batch); the other fields of niwqg_params - grid, dt, filter, model, slab layout - are common to all members */
typedef struct niwqg_member_params {
    size_t struct_size; /* = sizeof(niwqg_member_params) */
    double U, f, N, m;
    double nu, nu4, mu;         /* q-equation dissipation                        */
    double nuw, nu4w, muw;      /* phi-equation dissipation                      */
    double beta;                /* QGModel only                                  */
    double nu4c, nuc, muc;      /* QGModel passive scalar                        */
} niwqg_member_params;

typedef struct niwqg_handle niwqg_handle;

/* field identifiers for niwqg_get_field (attribute names of the reference model) */
enum niwqg_field {
    NIWQG_F_Q = 0,      /* q      real    (N,N)            */
    NIWQG_F_QH,         /* qh     complex (N,N) | (N,N/2+1) for QG */
    NIWQG_F_PH,         /* ph     complex, as qh           */
    NIWQG_F_P,          /* p      real    (computed on demand) */
    NIWQG_F_PHI,        /* phi    complex                   */
    NIWQG_F_PHIH,       /* phih   complex                   */
    NIWQG_F_PHIX, NIWQG_F_PHIY, NIWQG_F_LAPPHI,             /* complex */
    NIWQG_F_U, NIWQG_F_V,                                    /* real    */
    NIWQG_F_QW,         /* qw     real  (Coupled/QL)        */
    NIWQG_F_QPSI,       /* q_psi  real                      */
    NIWQG_F_QWH,        /* qwh    complex                   */
    NIWQG_F_C, NIWQG_F_CH,                                   /* QG passive scalar */
    /* tables: FILTR is shared by all members (member argument ignored); the ETDRK4 tables of an equation are
     * per member when the members' coefficients of that equation differ (niwqg_create_ensemble), else shared */
    NIWQG_F_FILTR,      /* real                             */
    NIWQG_F_EXPCH, NIWQG_F_EXPCH_H, NIWQG_F_QHCOEF, NIWQG_F_F0, NIWQG_F_FAB, NIWQG_F_FC,
    NIWQG_F_EXPCHW, NIWQG_F_EXPCH_HW, NIWQG_F_QHWCOEF, NIWQG_F_F0W, NIWQG_F_FABW, NIWQG_F_FCW,
    NIWQG_F_EXPCHC, NIWQG_F_EXPCH_HC, NIWQG_F_QHCCOEF, NIWQG_F_F0C, NIWQG_F_FABC, NIWQG_F_FCC,
    /* carried physical buffers as the device holds them (complex (N,N)); Q, QW, QPSI, U, V are views of UV and QS */
    NIWQG_F_UV,         /* u + i v                          */
    NIWQG_F_QS,         /* q + i qw (Coupled/QL), q + i (q - q_psi) otherwise */
    NIWQG_F_LAP2PHI,    /* ifft(wv4 phih) (models with nu4w != 0) */
    NIWQG_F_UVQ,        /* QL: uq + i vq of the vortex flow */
    NIWQG_F_COUNT
};

/* scalar slots returned by niwqg_get_scalars / niwqg_diagnostics, per member */
enum niwqg_scalar {
    NIWQG_S_KE = 0, NIWQG_S_PW, NIWQG_S_KW,                   /* integrated budgets (Kernel.py:390-392) */
    NIWQG_S_GAMMA1, NIWQG_S_GAMMA2, NIWQG_S_XI1, NIWQG_S_XI2, NIWQG_S_PI,   /* Kernel.py:697-701 */
    NIWQG_S_KE_QG, NIWQG_S_ENS, NIWQG_S_KE_NIW, NIWQG_S_CKE_NIW, NIWQG_S_IKE_NIW, NIWQG_S_PE_NIW,
    NIWQG_S_CONC, NIWQG_S_SKEW, NIWQG_S_EP_PHI, NIWQG_S_EP_PSI, NIWQG_S_CHI_Q, NIWQG_S_CHI_PHI,
    NIWQG_S_KE_QG_Q, NIWQG_S_KE_QG_W, NIWQG_S_KE_QG_QW,      /* CoupledModel.py:99-113 */
    NIWQG_S_CFL,
    NIWQG_S_CVAR, NIWQG_S_C2, NIWQG_S_GRADC2, NIWQG_S_GAMMA_C, NIWQG_S_EP_C, NIWQG_S_CHI_C,   /* QGModel.py:595-737 */
    NIWQG_S_COUNT
};

/* kinds for niwqg_fft2 */
#define NIWQG_FFT_C2C_FWD 0   /* numpy.fft.fft2   (Kernel.py:565)  */
#define NIWQG_FFT_C2C_INV 1   /* numpy.fft.ifft2  (Kernel.py:566)  */
#define NIWQG_FFT_R2C     2   /* numpy.fft.rfft2  (QGModel.py:551) */
#define NIWQG_FFT_C2R     3   /* numpy.fft.irfft2 (QGModel.py:552) */
#define NIWQG_FFT_R2C_FULL 4  /* fft2 of a real array, full spectrum out (Kernel.py:531) */

/* Model(**kwargs): Kernel.__init__ (niwqg/Kernel.py:70-152) / QGModel.Model.__init__
 * (niwqg/QGModel.py:65-139): grid, filter (:267-284) and ETDRK4 tables (:400-454)
 * are generated on the device. */
int niwqg_create(const niwqg_params* p, niwqg_handle** out);
/* An ensemble whose members take their own coefficients: members[b] (p->batch entries) replaces the coefficient
 * fields of p for member b; p gives everything else.  An equation (q, phi, passive scalar c) whose coefficients are
 * equal in every member keeps one shared table set, any other gets one set per member (DESIGN.md section 3.3).
 * members == NULL: exactly niwqg_create. */
int niwqg_create_ensemble(const niwqg_params* p, const niwqg_member_params* members, niwqg_handle** out);
int niwqg_destroy(niwqg_handle* h);
const char* niwqg_last_error(const niwqg_handle* h);   /* h may be NULL: last create error */

/* set_q (niwqg/Kernel.py:520-535, niwqg/QGModel.py:507-520): q is batch*N*N doubles on the
 * host (on_device=0) or device (1).  Inverts with whatever phi is current (F5).  q == NULL: use the array queued by
 * niwqg_stage_q. */
int niwqg_set_q(niwqg_handle* h, const double* q, int on_device);
/* set_phi (niwqg/Kernel.py:538-551): phi is batch*N*N interleaved complex doubles (NULL: the array queued by
 * niwqg_stage_phi). */
int niwqg_set_phi(niwqg_handle* h, const double* phi, int on_device);
/* set_c (niwqg/QGModel.py:522-534) */
int niwqg_set_c(niwqg_handle* h, const double* c, int on_device);
/* Input pipeline for a caller that seeds every step from host arrays (bench.py's end-to-end leg): queue the upload of
 * the NEXT niwqg_set_q / niwqg_set_phi input from a (pinned) host array on the handle's copy stream and return at once,
 * so the copy runs while the device is still stepping.  A following niwqg_set_q(h, NULL, 0) / niwqg_set_phi(h, NULL, 0)
 * seeds the model from the staged array exactly as if it had been passed directly.  The host array must stay unchanged
 * until that call returns.  Same layout and size as the set_* argument (this rank's rows in a slab run). */
int niwqg_stage_q(niwqg_handle* h, const double* q);
int niwqg_stage_phi(niwqg_handle* h, const double* phi);

/* Initial conditions generated on the device (niwqg/InitialConditions.py), then seeded exactly like set_q / set_phi:
 * no whole-grid host array is involved (at 8192^2 the reference generators need several 1 GiB arrays, a Python loop
 * over every grid point and four host round trips of the FFT seam).
 *   LAMB_DIPOLE (U, R)            q    InitialConditions.py:77-114
 *   MCWILLIAMS  (k0, E, seed)     q    :4-41   random red spectrum; rand01 = the caller's np.random.rand(N, N) for
 *   DANIOUX     (k0, E, seed)     q    :43-75  parity with the host generator, or NULL: Philox4x32-10(seed)
 *   WAVEPACKET  (k, l, R, x0, y0) phi  :117-145
 *   PLANEWAVE   (k, l, phase)     phi  :147-169 (the phase scales the amplitude, as in the reference)
 *   UNIFORM     (re, im)          phi  uniform near-inertial wave, examples/LambDipole.py:52 */
#define NIWQG_IC_LAMB_DIPOLE 0
#define NIWQG_IC_MCWILLIAMS  1
#define NIWQG_IC_DANIOUX     2
#define NIWQG_IC_WAVEPACKET  3
#define NIWQG_IC_PLANEWAVE   4
#define NIWQG_IC_UNIFORM     5
int niwqg_ic(niwqg_handle* h, int kind, const double* params, int nparams, const double* rand01);

/* nsteps calls of _step_etdrk4 (niwqg/Kernel.py:307-397; YBJModel.py:52-87;
 * QGModel.py:328-407) back to back, asynchronous on the handle's stream. */
int niwqg_step(niwqg_handle* h, int nsteps);

/* the scalar side of increment_diagnostics (niwqg/Diagnostics.py:41-58 ->
 * Kernel._calc_derived_fields, Kernel.py:870-878, registry :718-868): fills
 * out[batch][NIWQG_S_COUNT]; like the reference it refreshes phix/phiy as a side
 * effect of pe_niw (Kernel.py:608-611, F6). */
int niwqg_diagnostics(niwqg_handle* h, double* out);
/* _print_status body (niwqg/Kernel.py:590-594): out[batch][4] = ke_qg, ke_niw,
 * pe_niw (refreshes phix/phiy), cfl. */
int niwqg_status(niwqg_handle* h, double* out);
/* Ke, Pw, Kw and the last stage's conversion terms: out[batch][NIWQG_S_COUNT] (only the
 * first 8 slots are defined).  Coupled/UnCoupled evaluate the stage budgets in spectral space, where only the sums
 * enter: slot GAMMA1 then holds gamma1+gamma2 and XI1 holds xi1+xi2 (GAMMA2 = XI2 = 0); niwqg_diagnostics returns
 * the separate terms. */
int niwqg_get_scalars(niwqg_handle* h, double* out);

/* attribute read (Seam 3, SURVEY.md section 8b): copies one member's field to dst
 * (host if on_device==0).  bytes must equal the field's size. */
int niwqg_get_field(niwqg_handle* h, int field, int member, void* dst, size_t bytes, int on_device);
size_t niwqg_field_bytes(const niwqg_handle* h, int field);
/* The same copy to a (pinned) host buffer, queued on the handle's copy stream behind the work already issued: returns
 * at once, so the caller can start the next uploads while the result is still on its way (full-duplex PCIe).  dst is
 * valid after niwqg_wait_transfers (or niwqg_sync).  One real and one complex field can be in flight at a time; a
 * further request waits for the staging buffer it needs. */
int niwqg_get_field_async(niwqg_handle* h, int field, int member, void* dst, size_t bytes);
int niwqg_wait_transfers(niwqg_handle* h);

/* Checkpoint / exact restart (DESIGN.md section 6b).  The state of a handle is every buffer a step reads before it
 * writes it, plus the scalar carry.  Restoring all of it into a handle of the same model, grid, batch and parameters
 * makes the following steps bit-for-bit those of the handle it was read from.
 *
 * niwqg_state_slots: writes the field ids that make up this handle's state to ids[0..] and returns their number
 * (at most 16; negative if max is too small).  Reading them with niwqg_get_field changes nothing on the device.
 * niwqg_set_field: the inverse of niwqg_get_field for a state slot, same layout and size (natural x order, the rank's
 * rows / column slab in a slab run, the half spectrum for QG).  Writes into the buffers of the current ping-pong
 * parity; setting QH / PHIH marks the model seeded like set_q / set_phi.
 * niwqg_carry_count / niwqg_get_carry / niwqg_set_carry: the per-member scalars a step carries into the next one
 * (budgets Ke, Pw, Kw, cvar ... and the ep_psi sums of the last inversion), niwqg_carry_count(h) doubles.  In a slab
 * run they are grid-wide and equal on every rank. */
int niwqg_state_slots(const niwqg_handle* h, int* ids, int max);
int niwqg_set_field(niwqg_handle* h, int field, int member, const void* src, size_t bytes, int on_device);
int niwqg_carry_count(const niwqg_handle* h);
int niwqg_get_carry(niwqg_handle* h, double* out);
int niwqg_set_carry(niwqg_handle* h, const double* in);

/* the FFT backend seam (niwqg/Kernel.py:553-566, niwqg/QGModel.py:536-552): one N x N
 * transform with numpy conventions, host buffers. */
int niwqg_fft2(niwqg_handle* h, const void* in, void* out, int kind);

/* jacobian_psi_q / jacobian_phic_phi / jacobian_psi_phi (niwqg/Kernel.py:457-486,
 * niwqg/CoupledModel.py:59-73), evaluated on the current state of member 0 and copied to
 * the host as a spectral array; used by the reference's tests/test_advection.py. */
#define NIWQG_JAC_PSI_Q    0
#define NIWQG_JAC_PHIC_PHI 1
#define NIWQG_JAC_PSI_PHI  2
int niwqg_jacobian(niwqg_handle* h, int which, void* out);

/* rank 0: a fresh ncclUniqueId (128 bytes) for niwqg_params.nccl_id; the caller broadcasts it (e.g. with
 * torch.distributed).  NCCL is dlopen()ed from $NIWQG_NCCL_LIB or the default search path. */
int niwqg_nccl_unique_id(char* out128);

/* Fused slab exchange over NVLink peer memory: every rank exports the CUDA-IPC handles of its two receive buffers
 * (out: 4 x 64 bytes - two per lane, see DESIGN.md section 6), the caller all-gathers them, and niwqg_ipc_import() maps the peers' buffers; from then on the
 * first pass of every slab transform stores straight into the owners' buffers instead of going through ncclSend/Recv.
 * Without these calls the NCCL all-to-all path is used. */
int niwqg_ipc_export(niwqg_handle* h, char* out, size_t bytes);
int niwqg_ipc_import(niwqg_handle* h, const char* all_ranks, size_t bytes_per_rank);
/* switch back to the NCCL all-to-all exchange (all ranks must agree, e.g. after one of them failed to import) */
int niwqg_ipc_disable(niwqg_handle* h);

/* Lagrangian particles (drifters, DESIGN.md section 3.4).  A particle is a point (x, y) in metres in the frame of the
 * model's grid (values at the cell centres x_i = (i + 1/2) dx, physical arrays [iy][ix]), stored unwrapped in fp64;
 * velocities are interpolated periodically with the tensor-product 4-point (cubic) Lagrange stencil.  Every step
 * advances the particles by classical RK4 whose four stages read the model's own ETDRK4 stage fields: stage 1 the
 * state at t_n, stages 2 and 3 the states a and b at t_n + dt/2, stage 4 the state c at t_n + dt, each as the model
 * carries it (YBJ: its frozen u, v and the phi of t_n, which stays stale through the stages).  The velocity is
 * U + u_psi (the member's mean flow and the packed uv buffer); with waves, plus the wave velocity at the level where
 * the vertical factor is 1, u_w + i v_w = exp(-i f t) phi (the member's f; inertial loops are clockwise for f > 0).
 * In the Coupled and QL models u_psi is already the Lagrangian-mean flow, so waves=1 gives drifter-like loops but
 * counts the O(a^2) Stokes drift twice.  The wave phase uses a device clock set here and advanced by dt every step.
 * Particles only read the model: fields, scalars and diagnostics are bit for bit those of a run without them.
 * Single-GPU handles only: a slab handle (nranks > 1) returns an error from every call below but the count.
 *
 * niwqg_particles_set: xy = batch x count x 2 doubles (host, or device when on_device), all finite; t = the clock;
 * waves = 1 adds the wave velocity (models with phi only).  count = 0 removes the particles.  Replaces any particles
 * already set.  Seeding or removing drops the captured step graphs, which the next steps capture again.
 * niwqg_particles_count: particles per member (0: none).
 * niwqg_particles_get: xy = the batch x count x 2 positions, *t = the clock (either may be NULL).
 * niwqg_particles_sample: field = NIWQG_F_Q, NIWQG_F_U, NIWQG_F_V (out: batch x count doubles) or NIWQG_F_PHI (out:
 * batch x count complex), interpolated at the current positions with the same stencil, from exactly what
 * niwqg_get_field returns.  Changes no state. */
int niwqg_particles_set(niwqg_handle* h, const double* xy, int count, double t, int waves, int on_device);
int niwqg_particles_count(const niwqg_handle* h);
int niwqg_particles_get(niwqg_handle* h, double* xy, double* t);
int niwqg_particles_sample(niwqg_handle* h, int field, double* out);

int niwqg_sync(niwqg_handle* h);
/* CUDA-event timing on the handle's stream: elapsed ms of `nsteps` steps */
int niwqg_time_steps(niwqg_handle* h, int nsteps, float* ms);
/* per-kernel-kind CUDA-event timing on the handle's stream.  Reads the records accumulated since the
 * last call into ms_out[9] / count_out[9] (kinds: 0 FFT row pass, 1 FFT column pass, 2 physical-space
 * pointwise, 3 spectral pointwise, 4 small reductions, 5 NCCL all-to-all / barriers of slab transforms, 6 stand-alone
 * radix stage of the split transforms, 7 / 8 forward row pass that forms its input from three / two physical fields
 * while loading them), clears them and switches recording on/off.
 * ms_out/count_out may be NULL. */
int niwqg_profile(niwqg_handle* h, int enable, double* ms_out, long long* count_out);
/* number of kernel launches issued by this handle so far */
long long niwqg_launch_count(const niwqg_handle* h);
/* the cudaStream_t the handle launches on (for external event timing) */
void* niwqg_stream(const niwqg_handle* h);

#ifdef __cplusplus
}
#endif
#endif
