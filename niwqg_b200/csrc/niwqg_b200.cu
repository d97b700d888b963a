// niwqg_b200.cu -- C-ABI host side of the B200-native niwqg hot path (see include/niwqg_b200.h).
//
// One handle owns every device buffer of one model instance and issues the whole
// ETDRK4 step as a fixed sequence of kernel launches on one stream; nothing
// crosses the ABI per transform.  No cuFFT, no CPU fallback: every arithmetic
// kernel is in fft2d.cuh / kernels_family.cuh / kernels_qg.cuh.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <dlfcn.h>
#include <nccl.h>
#include "../../include/niwqg_b200.h"
#include "fft2d.cuh"
#include "fft_split.cuh"
#include "kernels_family.cuh"
#include "kernels_fused.cuh"
#include "kernels_qg.cuh"
#include "kernels_ic.cuh"
#include "kernels_particles.cuh"

static std::string g_create_error;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char buf__[512];                                                                       \
            snprintf(buf__, sizeof buf__, "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            h->err = buf__;                                                                        \
            return -2;                                                                             \
        }                                                                                          \
    } while (0)

struct niwqg_handle {
    niwqg_params p;
    int N = 0, B = 1, model = 0, flags = 0;
    bool qg = false;
    int nk = 0;                 // spectral row length: N (c2c) or N/2+1 (QG)
    size_t npts = 0, nspec = 0; // N*N, N*nk
    double dk = 0, dx = 0, jscale = 1.0;
    // per-member coefficients (niwqg_create_ensemble; copies of p otherwise): host rows for the finalisation of
    // diagnostics / status, device rows mcoef[B][MC_COUNT] for the kernels
    std::vector<niwqg_member_params> mp;
    std::vector<double> kappa2m, hslashm;
    double* mcoef = nullptr;
    bool pm_q = false, pm_p = false, pm_c = false;   // per-member tables of the q / phi / c equation
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<void*> allocs;
    std::string err;
    long long launches = 0;
    // tables
    TableSet tq{}, tp{}, tc{};
    double* filtr = nullptr;
    cd *tw_row = nullptr, *tw_col = nullptr, *twc = nullptr;   // stage twiddles of the row / column local length, w_N^t
    // spectral state (c2c family: [B][N][N]; QG: [B][N][nk])
    cd* qh[2] = {nullptr, nullptr};
    cd* phih[2] = {nullptr, nullptr};
    cd* chh[2] = {nullptr, nullptr};
    int cq = 0, cp = 0, cc = 0;
    cd *y1q = nullptr, *y1p = nullptr, *y1c = nullptr;
    cd *F0q = nullptr, *F0p = nullptr, *F0c = nullptr, *Fabq = nullptr, *Fabp = nullptr, *Fabc = nullptr;
    cd *ph = nullptr, *qwh = nullptr;
    // physical carried fields
    cd *phi = nullptr, *phix = nullptr, *phiy = nullptr, *lapphi = nullptr, *lap2phi = nullptr;
    cd *uv = nullptr, *qs = nullptr, *uvq = nullptr;
    // scratch
    cd *W = nullptr, *P1 = nullptr, *P2 = nullptr;
    double* rscratch = nullptr;   // [B][N][N] doubles
    // reductions
    double *part = nullptr, *sumsD = nullptr, *sumsE = nullptr, *sumsX = nullptr, *sumsI = nullptr, *scal = nullptr,
           *stagev = nullptr;
    bool q_set = false, phi_set = false;
    int deintC = 1, deintM = 0;   // physical x order: de-interleaved mod deintC when the row pass is a cluster (k_deint)
    // slab decomposition over nranks GPUs (one process per GPU): physical arrays hold nyl = N/P rows, spectral
    // arrays all N rows of ncl = N/P columns (Grid, common.cuh); each 2-D transform = local pass, NCCL all-to-all,
    // local pass
    int rank = 0, nranks = 1, nyl = 0, ncl = 0;
    Grid g{};
    double Mg = 0;              // N*N of the GLOBAL grid (mean denominators)
    cd *X = nullptr, *Y = nullptr;   // all-to-all send / receive buffers (NCCL path)
    // fused path: passes push straight into the peers' receive buffers (CUDA IPC), double-buffered per transform
    // Two LANES (stream + communicator + receive buffers each): independent transforms of one group (phi/phix/phiy,
    // u+iv / q+iqw, the two RHS products) alternate between them, so one transform's NVLink-bound pushing pass
    // overlaps another's HBM-bound local pass.  Lane 0 is the handle's main stream.
    static constexpr int NLANE = 2;
    cd* Yp[NLANE][2] = {};
    cd* peerY[NLANE][2][8] = {};
    bool p2p = false;
    int ybuf[NLANE] = {0, 0};
    double* bar[NLANE] = {nullptr, nullptr};   // 1-element all-reduce buffers: the cross-GPU barrier between passes
    cudaStream_t lane_stream[NLANE] = {nullptr, nullptr};
    ncclComm_t lane_comm[NLANE] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // CUDA graphs of one whole step, one per ping-pong parity of the state buffers (key = cq*4 + cp*2 + cc): small grids
    // are launch-bound (~100 launches of a few microseconds each per step)
    struct StepGraph { cudaGraphExec_t exec = nullptr; int cq = 0, cp = 0, cc = 0; long long launches = 0; };
    StepGraph graphs[8];
    bool use_graphs = false;
    int direct_steps = 0;       // steps issued without a graph (the first ones set kernel attributes lazily)
    int exchange = 0;           // 0: pushes fused into the first pass; 1: first pass writes the exchange layout locally,
                                // the copy engines move the chunks to the peers (no SM involved, overlaps the other lane)
    cd* Xl[NLANE] = {nullptr, nullptr};   // per-lane send staging of the copy-engine exchange
    ncclComm_t comm = nullptr;
    bool col3 = false;          // 8192^2, one GPU, one member, not split: three-pass column transform (0.714 vs 0.771 ms
                                // for the cluster kernel)
    cd* S3[2] = {nullptr, nullptr};   // its scratch array, one per lane
    cd* tw_c3 = nullptr;              // stage twiddles of its 512-point local transforms
    // split transforms (fft_split.cuh): x = 2 x N/2 on de-interleaved physical rows, y = 16 x N/16, three streaming launches
    // per 2-D transform.  Default for 8192^2 on one GPU (1.09 vs 1.22 ms per transform); NIWQG_SPLIT=1 forces it for every
    // N >= 2048 (tests), NIWQG_SPLIT=0 switches it off.
    int split = 0;
    cd* T[3] = {nullptr, nullptr, nullptr};   // scratch arrays of the split path
    cd *tw_half = nullptr, *tw_m = nullptr;   // stage twiddles of the N/2-point rows and of the N/16-point column transforms
    // host <-> device transfers of whole fields run on their own stream through staging buffers, so an upload overlaps the
    // compute still queued on the main stream (set_phi's copy under set_q's inversion) and a download overlaps whatever
    // the caller does next (niwqg_get_field_async: the next step's uploads)
    cudaStream_t copy_stream = nullptr, copy_out = nullptr;     // uploads / downloads: separate streams, PCIe is full duplex
    cudaEvent_t ev_up_done = nullptr, ev_up_free = nullptr, ev_dn_ready = nullptr, ev_dn_done[2] = {nullptr, nullptr};
    bool up_free_rec = false, dn_done_rec[2] = {false, false};
    void* stage_in = nullptr;                 // B * npts * 16 bytes
    // niwqg_stage_q / niwqg_stage_phi: the next set_* input, uploaded ahead of time ([0] q, [1] phi)
    void* pre_buf[2] = {nullptr, nullptr};
    cudaEvent_t pre_done[2] = {nullptr, nullptr}, pre_free[2] = {nullptr, nullptr};
    bool pre_staged[2] = {false, false}, pre_free_rec[2] = {false, false};
    void* stage_out[2] = {nullptr, nullptr};  // one member: real (npts * 8) / complex (npts * 16)
    double* pin = nullptr;                    // pinned host scratch for the scalars of diagnostics / status
    int slab_panel = 0;         // slab, pushed exchange of inverse transforms: panel receive layout (FftArgs::panel); = cluster
                                // size of the column pass for N >= 1024, else 0 (rows of ncl columns)
    int flag_barrier = 1;       // slab: peer-memory flags instead of the 1-element all-reduce between the two passes
                                // (validated on 2 and 8 GPUs: 13.33 vs 13.47 ms/step at 8; NIWQG_SLAB_BARRIER=nccl switches back)
    unsigned bar_epoch[NLANE] = {0, 0};
    // optional per-kernel-kind CUDA-event timing (bench.py's roofline leg)
    bool prof = false;
    struct ProfRec { int kind; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_recs;
    std::vector<cudaEvent_t> prof_pool;
    size_t prof_used = 0;
    // Lagrangian particles (kernels_particles.cuh): np per member, none when 0.  One allocation: x_n, the stage position
    // and the RK4 accumulator ([B][np] double2 each), then the particle clock (2 doubles)
    int np = 0;
    bool pwaves = false;
    double2* pbuf = nullptr;
};

enum { PK_FFT_ROW = 0, PK_FFT_COL, PK_PHYS, PK_SPEC, PK_SMALL, PK_COMM, PK_FFT_P, PK_FFT_ROWLD, PK_FFT_ROWLD2, PK_COUNT };

static cudaEvent_t prof_event(niwqg_handle* h) {
    if (h->prof_used == h->prof_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->prof_pool.push_back(e);
    }
    return h->prof_pool[h->prof_used++];
}
struct ProfScope {
    niwqg_handle* h; int kind; cudaEvent_t a;
    ProfScope(niwqg_handle* h_, int k) : h(h_), kind(k), a(nullptr) {
        if (h->prof && kind >= 0) { a = prof_event(h); cudaEventRecord(a, h->stream); }
    }
    ~ProfScope() {
        if (h->prof && kind >= 0) { cudaEvent_t b = prof_event(h); cudaEventRecord(b, h->stream); h->prof_recs.push_back({kind, a, b}); }
    }
};
#define PROF(kind) ProfScope prof_scope__(h, kind)
#define PROF_ON(kind, lane) ProfScope prof_scope__(h, (lane) == 0 ? (kind) : -1)

// ---------------------------------------------------------------------------
static int dalloc(niwqg_handle* h, void** p, size_t bytes, bool zero = true) {
    CK(cudaMalloc(p, bytes));
    h->allocs.push_back(*p);
    if (zero) CK(cudaMemsetAsync(*p, 0, bytes, h->stream));
    return 0;
}
#define DA(ptr, bytes)                                              \
    do {                                                            \
        int r__ = dalloc(h, (void**)&(ptr), (bytes));               \
        if (r__) return r__;                                        \
    } while (0)

static dim3 pw_grid(const niwqg_handle* h) { return dim3(NIWQG_PW_BLOCKS, h->B); }

static void build_twiddles(int N, std::vector<cd>& tw) {
    tw.assign(fftc::tw_table_len(N) + 1, make_double2(1.0, 0.0));
    const long double PI = 3.141592653589793238462643383279502884L;
    for (int NS = 16; NS < N; NS *= 16) {
        const int R = (N / NS >= 16) ? 16 : N / NS;
        for (int kk = 0; kk < NS; ++kk) {
            const long double a = -2.0L * PI * (long double)kk / ((long double)NS * R);
            tw[fftc::tw_offset(NS) + kk] = make_double2((double)cosl(a), (double)sinl(a));
        }
    }
}

// ---- NCCL, resolved at run time so that single-GPU use needs no NCCL at all
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t*, ncclConfig_t*) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load(std::string& err) {
    if (g_nccl.lib) return 0;
    const char* path = getenv("NIWQG_NCCL_LIB");
    void* lib = dlopen(path && *path ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { err = std::string("cannot load NCCL: ") + dlerror(); return -4; }
#define NIWQG_SYM(field, name)                                                     \
    *(void**)(&g_nccl.field) = dlsym(lib, name);                                   \
    if (!g_nccl.field) { err = std::string("NCCL symbol missing: ") + name; return -4; }
    NIWQG_SYM(GetUniqueId, "ncclGetUniqueId") NIWQG_SYM(CommInitRank, "ncclCommInitRank")
    NIWQG_SYM(CommDestroy, "ncclCommDestroy") NIWQG_SYM(AllReduce, "ncclAllReduce") NIWQG_SYM(Send, "ncclSend")
    NIWQG_SYM(Recv, "ncclRecv") NIWQG_SYM(GroupStart, "ncclGroupStart") NIWQG_SYM(GroupEnd, "ncclGroupEnd")
    NIWQG_SYM(GetErrorString, "ncclGetErrorString") NIWQG_SYM(CommSplit, "ncclCommSplit")
#undef NIWQG_SYM
    g_nccl.lib = lib;
    return 0;
}
#define NK(call)                                                                                   \
    do {                                                                                           \
        ncclResult_t e__ = (call);                                                                 \
        if (e__ != ncclSuccess) {                                                                  \
            char buf__[512];                                                                       \
            snprintf(buf__, sizeof buf__, "%s:%d: %s: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(e__)); \
            h->err = buf__;                                                                        \
            return -5;                                                                             \
        }                                                                                          \
    } while (0)

// the distributed-FFT transpose: chunk s of `send` goes to rank s, chunk r of `recv` comes from rank r
static int slab_all_to_all(niwqg_handle* h, const cd* send, cd* recv) {
    PROF(PK_COMM);
    const size_t chunk = (size_t)h->nyl * h->ncl;
    NK(g_nccl.GroupStart());
    for (int r = 0; r < h->nranks; ++r) {
        NK(g_nccl.Send(send + (size_t)r * chunk, 2 * chunk, ncclDouble, r, h->comm, h->stream));
        NK(g_nccl.Recv(recv + (size_t)r * chunk, 2 * chunk, ncclDouble, r, h->comm, h->stream));
    }
    NK(g_nccl.GroupEnd());
    return 0;
}

static cudaError_t launch_col_natural(niwqg_handle* h, const FftArgs& a, int batch, int lane);
static int slab_barrier(niwqg_handle* h, int lane, cudaStream_t st);

// ---- cross-GPU barrier between the pushing pass of a slab transform and the pass that reads the receive buffer:
// every rank raises a flag in every peer's memory once its pushes are behind it, and waits until all P flags in its own
// memory have reached the transform's epoch.  Two 1-CTA launches on the lane's stream instead of a 1-element
// ncclAllReduce (NIWQG_SLAB_BARRIER=nccl switches back).  The pushing kernel has completed when k_slab_signal runs (stream
// order), so its peer stores are performed; the fence + system-scope store publish the flag after them.
struct SlabFlags { unsigned* peer[8]; };
__global__ void k_slab_signal(SlabFlags f, int nranks, int rank, unsigned epoch) {
    const int r = threadIdx.x;
    if (r >= nranks) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.peer[r] + rank), "r"(epoch) : "memory");
}
__global__ void k_slab_wait(const unsigned* flags, int nranks, unsigned epoch) {
    const int r = threadIdx.x;
    if (r >= nranks) return;
    unsigned v;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + r) : "memory");
        if (v < epoch) __nanosleep(200);
    } while (v < epoch);
}

// one resident wave of the FFT passes and of the persistent fused kernels: 148 SMs x 2 CTAs
static constexpr int WAVE_CTAS = 296;

static void fft_common_args(niwqg_handle* h, FftArgs& a) {
    a.twc = h->twc;
    a.dk = h->dk;
    a.pf_groups = WAVE_CTAS;    // L2 prefetch distance of the FFT passes in CTAs
    // variant and one_cta_per_sm are constants on the host: column clusters push (DIF, plain remote stores), row clusters
    // pull (DIT), two CTAs per SM (measured best: profiles/r01b_cluster_variants.txt, r01d_async_push.txt)
    a.variant = 6;
    a.one_cta_per_sm = 0;
    a.g = h->g;
    a.xmap_in = a.xmap_out = 0;
    a.deint_in = a.deint_out = 0;
    a.tma_in = 1;               // column passes whose rows are narrower than a 128 B line fetch their tile by TMA
                                // (1024^2: 4345 -> 4983 GB/s)
    a.xchunk = h->nyl * h->ncl;
    a.mstride = h->npts;
    a.pitch = h->ncl;
}

// ---- split path (fft_split.cuh): the three launches of a 2-D transform
static int split_rows(niwqg_handle* h, const void* in, void* out, int pro, int epi, double sc, bool conj_out) {
    FftArgs a{};
    fft_common_args(h, a);
    const int Nh = h->N / 2;
    a.in = in; a.out = out; a.pro = pro; a.epi = epi; a.tw = h->tw_half;
    a.nlines = 2 * h->N; a.pitch = Nh; a.mstride = (size_t)Nh * Nh; a.g = Grid{Nh, h->dk, Nh, Nh / 2, 0, 0};
    a.conj_in = 0; a.conj_out = conj_out ? 1 : 0; a.scale = sc; a.scale_im = conj_out ? -sc : sc;
    a.tma_in = 2;          // row tiles fetched by one bulk copy (cp.async.bulk) instead of 16 LDG.128 per thread
    a.pf_groups = 0;       // measured on 16384 lines of 4096: 0.362 ms without the L2 prefetch, 0.382 ms with it
    { PROF(PK_FFT_ROW); CK(launch_pass<false>(Nh, a, 1, h->stream)); }
    h->launches++;
    return 0;
}
// forward row pass that forms its input while loading the operands: LD_WAVEPV W = |phi|^2 + i jscale i J(phi*,phi) from phi,
// phix, phiy (replaces k_phys_wavepv and the re-read of W), LD_UQVQ P1 = (uq, vq) from uv, qs (k_phys_rhs then skips the P1
// store)
static int split_rows_loader(niwqg_handle* h, int ld, cd* out) {
    FftArgs a{};
    fft_common_args(h, a);
    const int Nh = h->N / 2;
    if (ld == LD_WAVEPV) { a.in = h->phi; a.in2 = h->phix; a.in3 = h->phiy; a.ld_scale = h->jscale; }
    else { a.in = h->uv; a.in2 = h->qs; a.in3 = nullptr; a.ld_scale = 1.0; }
    a.out = out; a.pro = PRO_NONE; a.epi = EPI_NONE; a.tw = h->tw_half;
    a.nlines = 2 * h->N; a.pitch = Nh; a.mstride = (size_t)Nh * Nh; a.g = Grid{Nh, h->dk, Nh, Nh / 2, 0, 0};
    a.conj_in = 0; a.conj_out = 0; a.scale = 1.0; a.scale_im = 1.0;
    cudaError_t e = cudaErrorInvalidValue;
    {
        PROF(ld == LD_WAVEPV ? PK_FFT_ROWLD : PK_FFT_ROWLD2);
#define NIWQG_LD_CASE(NN) case NN: e = (ld == LD_WAVEPV) ? launch_split_rows_loader<NN, LD_WAVEPV>(a, h->stream) \
                                                          : launch_split_rows_loader<NN, LD_UQVQ>(a, h->stream); break;
        switch (h->N) {
            NIWQG_LD_CASE(2048)
            NIWQG_LD_CASE(4096)
            NIWQG_LD_CASE(8192)
        }
#undef NIWQG_LD_CASE
    }
    CK(e);
    h->launches++;
    return 0;
}
static int split_colsub(niwqg_handle* h, const cd* in, cd* out, bool dit) {
    FftArgs a{};
    fft_common_args(h, a);
    a.in = in; a.out = out; a.pro = PRO_NONE; a.epi = EPI_NONE; a.tw = h->tw_m; a.scale = 1.0; a.scale_im = 1.0;
    cudaError_t e = cudaErrorInvalidValue;
    {
        PROF(PK_FFT_COL);
        switch (h->N) {
            case 2048: e = dit ? launch_split_colsub<2048, true>(a, h->stream) : launch_split_colsub<2048, false>(a, h->stream); break;
            case 4096: e = dit ? launch_split_colsub<4096, true>(a, h->stream) : launch_split_colsub<4096, false>(a, h->stream); break;
            case 8192: e = dit ? launch_split_colsub<8192, true>(a, h->stream) : launch_split_colsub<8192, false>(a, h->stream); break;
        }
    }
    CK(e);
    h->launches++;
    return 0;
}
static int split_p(niwqg_handle* h, const cd* in, cd* const* out, const int* pro, int nout, bool dit, bool conj_in) {
    SplitPArgs p{};
    p.in = in; p.nout = nout; p.conj_in = conj_in ? 1 : 0; p.scale = 1.0; p.dk = h->dk; p.twc = h->twc;
    for (int o = 0; o < nout; ++o) { p.out[o] = out[o]; p.pro[o] = pro[o]; }
    cudaError_t e = cudaErrorInvalidValue;
    {
        PROF(PK_FFT_P);
        switch (h->N) {
            case 2048: e = dit ? launch_split_p<2048, true>(p, h->stream) : launch_split_p<2048, false>(p, h->stream); break;
            case 4096: e = dit ? launch_split_p<4096, true>(p, h->stream) : launch_split_p<4096, false>(p, h->stream); break;
            case 8192: e = dit ? launch_split_p<8192, true>(p, h->stream) : launch_split_p<8192, false>(p, h->stream); break;
        }
    }
    CK(e);
    h->launches++;
    return 0;
}
// forward: rows (in -> out), M-point column transforms (out -> T0), radix-16 x radix-2 combine (T0 -> out)
// inverse: prologue + conj + radix stage (in -> T0), M-point column transforms (T0 -> out), rows in place with conj + 1/N^2
static int fft2_split(niwqg_handle* h, const void* in, cd* out, bool inverse, int pro, int epi, void* real_out) {
    int r;
    if (!inverse) {
        if ((r = split_rows(h, in, out, pro == PRO_REAL_IN ? PRO_REAL_IN : PRO_NONE, EPI_NONE, 1.0, false))) return r;
        if ((r = split_colsub(h, out, h->T[0], true))) return r;
        cd* outs[1] = {out};
        const int pros[1] = {PRO_NONE};
        if ((r = split_p(h, h->T[0], outs, pros, 1, true, false))) return r;
        return 0;
    }
    cd* outs[1] = {h->T[0]};
    const int pros[1] = {pro};
    if ((r = split_p(h, (const cd*)in, outs, pros, 1, false, true))) return r;
    if ((r = split_colsub(h, h->T[0], out, false))) return r;
    const double sc = 1.0 / ((double)h->N * (double)h->N);
    return split_rows(h, out, epi == EPI_REAL_OUT ? real_out : (void*)out, PRO_NONE, epi, sc, true);
}

// 2-D c2c transform of `batch` members: in -> out (may alias), forward or inverse.
// One GPU: row pass then column pass.  Slab: forward = row pass (rows are local) -> all-to-all -> column pass
// (columns are local); inverse = column pass -> all-to-all -> row pass.  The spectral prologue multiply and the
// conjugation of an inverse transform ride on whichever pass comes first, conj + 1/N^2 on the last.
static int fft2(niwqg_handle* h, const void* in, cd* out, bool inverse, int pro, int batch, int epi = EPI_NONE,
                void* real_out = nullptr, int lane = 0) {
    FftArgs a{};
    fft_common_args(h, a);
    const double sc = inverse ? 1.0 / ((double)h->N * (double)h->N) : 1.0;
    void* final_out = (epi == EPI_REAL_OUT) ? real_out : (void*)out;
    if (h->split && batch == 1) return fft2_split(h, in, out, inverse, pro, epi, real_out);
    if (h->nranks == 1) {
        // pass 1: rows
        a.in = in; a.out = out; a.pro = pro; a.epi = EPI_NONE; a.tw = h->tw_row; a.nlines = h->N;
        a.conj_in = inverse ? 1 : 0; a.conj_out = 0; a.scale = 1.0; a.scale_im = 1.0;
        { PROF_ON(PK_FFT_ROW, lane); CK(launch_pass<false>(h->N, a, batch, h->lane_stream[lane])); }
        // pass 2: columns
        a.in = out; a.out = final_out; a.pro = PRO_NONE; a.epi = epi; a.tw = h->tw_col; a.nlines = h->N;
        a.conj_in = 0; a.conj_out = inverse ? 1 : 0;
        a.scale = sc; a.scale_im = inverse ? -sc : sc;
        { PROF_ON(PK_FFT_COL, lane); CK(launch_col_natural(h, a, batch, lane)); }
        h->launches += 2;
        return 0;
    }
    if (batch != 1) { h->err = "slab transforms take one member"; return -1; }
    if (h->p2p) {
        cudaStream_t st = h->lane_stream[lane];
        // fused exchange: the first pass stores into the owners' receive buffers over NVLink; one tiny all-reduce is
        // the barrier that says "everybody's pushes have landed"; the second pass reads the local receive buffer.
        const int b = h->ybuf[lane];
        h->ybuf[lane] ^= 1;     // the peers may still be reading the other buffer (previous transform's second pass)
        const bool ce = h->exchange == 1;
        a.push = ce ? 0 : 1;
        for (int r = 0; r < h->nranks; ++r) a.peer[r] = h->peerY[lane][b][r];
        int sh = 0;
        while ((1 << sh) < h->nyl) ++sh;
        a.nyl_shift = sh;
        a.panel = (inverse && !ce) ? h->slab_panel : 0;      // both passes of the transform see the same receive layout
        a.in = in; a.out = ce ? (void*)h->Xl[lane] : nullptr; a.pro = pro; a.epi = EPI_NONE; a.scale = 1.0; a.scale_im = 1.0;
        a.conj_out = 0;
        if (!inverse) {
            a.tw = h->tw_row; a.nlines = h->nyl; a.conj_in = 0; a.xmap_out = ce ? 1 : 0;
            { PROF_ON(PK_FFT_ROW, lane); CK(launch_pass<false>(h->N, a, 1, st)); }
            a.xmap_out = 0;
        } else {
            a.tw = h->tw_col; a.nlines = h->ncl; a.conj_in = 1;
            { PROF_ON(PK_FFT_COL, lane); CK(launch_pass<true>(h->N, a, 1, st)); }
        }
        {
            PROF_ON(PK_COMM, lane);
            if (ce) {
                // chunk r of the send staging -> chunk [my rank] of rank r's receive buffer, by the copy engines
                const size_t chunk = (size_t)h->nyl * h->ncl;
                for (int k = 0; k < h->nranks; ++k) {
                    const int r = (h->rank + k) % h->nranks;          // start with my own chunk, then ring order
                    CK(cudaMemcpyAsync(h->peerY[lane][b][r] + (size_t)h->rank * chunk, h->Xl[lane] + (size_t)r * chunk,
                                       chunk * sizeof(cd), cudaMemcpyDeviceToDevice, st));
                }
            }
            int rb = slab_barrier(h, lane, st);
            if (rb) return rb;
        }
        a.push = 0;
        a.in = h->Yp[lane][b]; a.out = final_out; a.pro = PRO_NONE; a.epi = epi; a.conj_in = 0;
        if (!inverse) {
            a.tw = h->tw_col; a.nlines = h->ncl;
            { PROF_ON(PK_FFT_COL, lane); CK(launch_pass<true>(h->N, a, 1, st)); }
        } else {
            a.tw = h->tw_row; a.nlines = h->nyl; a.xmap_in = 1; a.conj_out = 1; a.scale = sc; a.scale_im = -sc;
            { PROF_ON(PK_FFT_ROW, lane); CK(launch_pass<false>(h->N, a, 1, st)); }
        }
        h->launches += 3;
        return 0;
    }
    if (!inverse) {
        a.in = in; a.out = h->X; a.pro = pro; a.epi = EPI_NONE; a.tw = h->tw_row; a.nlines = h->nyl; a.xmap_out = 1;
        a.conj_in = 0; a.conj_out = 0; a.scale = 1.0; a.scale_im = 1.0;
        { PROF(PK_FFT_ROW); CK(launch_pass<false>(h->N, a, 1, h->stream)); }
        int r = slab_all_to_all(h, h->X, h->Y);
        if (r) return r;
        a.in = h->Y; a.out = final_out; a.pro = PRO_NONE; a.epi = epi; a.tw = h->tw_col; a.nlines = h->ncl; a.xmap_out = 0;
        { PROF(PK_FFT_COL); CK(launch_pass<true>(h->N, a, 1, h->stream)); }
    } else {
        a.in = in; a.out = h->X; a.pro = pro; a.epi = EPI_NONE; a.tw = h->tw_col; a.nlines = h->ncl;
        a.conj_in = 1; a.conj_out = 0; a.scale = 1.0; a.scale_im = 1.0;
        { PROF(PK_FFT_COL); CK(launch_pass<true>(h->N, a, 1, h->stream)); }
        int r = slab_all_to_all(h, h->X, h->Y);
        if (r) return r;
        a.in = h->Y; a.out = final_out; a.pro = PRO_NONE; a.epi = epi; a.tw = h->tw_row; a.nlines = h->nyl; a.xmap_in = 1;
        a.conj_in = 0; a.conj_out = 1; a.scale = sc; a.scale_im = -sc;
        { PROF(PK_FFT_ROW); CK(launch_pass<false>(h->N, a, 1, h->stream)); }
    }
    h->launches += 2;
    return 0;
}
// column pass of the natural layout: the cluster kernel, or - 8192^2, see niwqg_handle::col3 - the three-pass variant
static cudaError_t launch_col_natural(niwqg_handle* h, const FftArgs& a, int batch, int lane) {
    if (h->col3 && a.epi == EPI_NONE) {
        FftArgs b = a;
        b.tw = h->tw_c3;
        h->launches++;      // two kernels for this pass (the caller counts one)
        return launch_col3<8192, 16, 8>(b, h->S3[lane], batch, h->lane_stream[lane]);
    }
    return launch_pass<true>(h->N, a, batch, h->lane_stream[lane]);
}

// One pass of an inverse transform in the natural single-GPU layout (shared row pass of phi / phiy, below).
static int inv_row_pass(niwqg_handle* h, const cd* in, cd* out, int pro, int lane) {
    FftArgs a{};
    fft_common_args(h, a);
    a.in = in; a.out = out; a.pro = pro; a.epi = EPI_NONE; a.tw = h->tw_row; a.nlines = h->N;
    a.conj_in = 1; a.conj_out = 0; a.scale = 1.0; a.scale_im = 1.0;
    { PROF_ON(PK_FFT_ROW, lane); CK(launch_pass<false>(h->N, a, h->B, h->lane_stream[lane])); }
    h->launches++;
    return 0;
}
static int inv_col_pass(niwqg_handle* h, const cd* in, cd* out, int pro, int lane) {
    FftArgs a{};
    fft_common_args(h, a);
    const double sc = 1.0 / ((double)h->N * (double)h->N);
    a.in = in; a.out = out; a.pro = pro; a.epi = EPI_NONE; a.tw = h->tw_col; a.nlines = h->N;
    a.conj_in = 0; a.conj_out = 1; a.scale = sc; a.scale_im = -sc;
    { PROF_ON(PK_FFT_COL, lane); CK(launch_col_natural(h, a, h->B, lane)); }
    h->launches++;
    return 0;
}

// The two halves of an inverse slab transform with the fused exchange, for transforms that share their first half
// (wave_fields): column pass pushing into the peers' receive buffer `b` of `lane` + barrier, and the row pass that
// reads a receive buffer.
static int slab_inv_push(niwqg_handle* h, const cd* in, int pro, int lane, int* bout) {
    FftArgs a{};
    fft_common_args(h, a);
    cudaStream_t st = h->lane_stream[lane];
    const int b = h->ybuf[lane];
    h->ybuf[lane] ^= 1;
    *bout = b;
    a.push = 1;
    for (int r = 0; r < h->nranks; ++r) a.peer[r] = h->peerY[lane][b][r];
    int sh = 0;
    while ((1 << sh) < h->nyl) ++sh;
    a.nyl_shift = sh;
    a.panel = h->slab_panel;
    a.in = in; a.out = nullptr; a.pro = pro; a.epi = EPI_NONE; a.scale = 1.0; a.scale_im = 1.0; a.conj_out = 0;
    a.tw = h->tw_col; a.nlines = h->ncl; a.conj_in = 1;
    { PROF_ON(PK_FFT_COL, lane); CK(launch_pass<true>(h->N, a, 1, st)); }
    { PROF_ON(PK_COMM, lane); int rb = slab_barrier(h, lane, st); if (rb) return rb; }
    h->launches += 2;
    return 0;
}
static int slab_inv_row(niwqg_handle* h, int lane, int b, cd* out, int pro) {
    FftArgs a{};
    fft_common_args(h, a);
    const double sc = 1.0 / ((double)h->N * (double)h->N);
    a.in = h->Yp[lane][b]; a.out = out; a.pro = pro; a.epi = EPI_NONE; a.conj_in = 0;
    int sh = 0;
    while ((1 << sh) < h->nyl) ++sh;
    a.nyl_shift = sh;
    a.panel = h->slab_panel;
    a.tw = h->tw_row; a.nlines = h->nyl; a.xmap_in = 1; a.conj_out = 1; a.scale = sc; a.scale_im = -sc;
    { PROF_ON(PK_FFT_ROW, lane); CK(launch_pass<false>(h->N, a, 1, h->lane_stream[lane])); }
    h->launches++;
    return 0;
}

static int slab_barrier(niwqg_handle* h, int lane, cudaStream_t st) {
    if (!h->flag_barrier) {
        NK(g_nccl.AllReduce(h->bar[lane], h->bar[lane], 1, ncclDouble, ncclSum, h->lane_comm[lane], st));
        return 0;
    }
    SlabFlags f{};
    for (int r = 0; r < h->nranks; ++r) f.peer[r] = (unsigned*)(h->peerY[lane][0][r] + h->npts);   // behind the receive buffer
    const unsigned epoch = ++h->bar_epoch[lane];
    k_slab_signal<<<1, 32, 0, st>>>(f, h->nranks, h->rank, epoch);
    k_slab_wait<<<1, 32, 0, st>>>((const unsigned*)(h->Yp[lane][0] + h->npts), h->nranks, epoch);
    CK(cudaGetLastError());
    return 0;
}

#define FFT(...)                          \
    do {                                  \
        int r__ = fft2(h, __VA_ARGS__);   \
        if (r__) return r__;              \
    } while (0)

// A group of mutually independent transforms (same or different inputs, distinct outputs).  Slab runs with the fused
// exchange alternate them between the two lanes; everything else runs them back to back on the main stream.
struct FftJob { const void* in; cd* out; bool inverse; int pro; };
static int fft2_group(niwqg_handle* h, const FftJob* jobs, int n) {
    // (one GPU: the column pass of one transform, bound by the DSMEM exchange, runs next to the row pass of the other)
    const bool par = (h->p2p || h->nranks == 1) && !h->prof && n > 1 && !h->split;
    if (!par) {
        for (int i = 0; i < n; ++i) FFT(jobs[i].in, jobs[i].out, jobs[i].inverse, jobs[i].pro, h->B);
        return 0;
    }
    CK(cudaEventRecord(h->ev_fork, h->lane_stream[0]));
    CK(cudaStreamWaitEvent(h->lane_stream[1], h->ev_fork, 0));
    for (int i = 0; i < n; ++i) FFT(jobs[i].in, jobs[i].out, jobs[i].inverse, jobs[i].pro, h->B, EPI_NONE, nullptr, i & 1);
    CK(cudaEventRecord(h->ev_join, h->lane_stream[1]));
    CK(cudaStreamWaitEvent(h->lane_stream[0], h->ev_join, 0));
    return 0;
}

static int finalize(niwqg_handle* h, int K, double* out, int is_max = 0, int nblk = NIWQG_PW_BLOCKS) {
    PROF(PK_SMALL);
    k_finalize<<<h->B, 256, 0, h->stream>>>(h->part, nblk, K, out, is_max);
    CK(cudaGetLastError());
    h->launches += 1;
    if (h->nranks > 1)   // every rank reduced its slab; the grid-wide sum / max is the same on all ranks afterwards
        NK(g_nccl.AllReduce(out, out, (size_t)h->B * K, ncclDouble, is_max ? ncclMax : ncclSum, h->comm, h->stream));
    return 0;
}
#define FIN(...)                              \
    do {                                      \
        int r__ = finalize(h, __VA_ARGS__);   \
        if (r__) return r__;                  \
    } while (0)

__global__ void k_budget(BudgetArgs a) {
    const int m = blockIdx.x;
    if (threadIdx.x != 0) return;
    const double* sd = a.sumsD + (size_t)m * SD_COUNT;
    const double* se = a.sumsE + (size_t)m * SE_COUNT;
    const double* si = a.sumsI + (size_t)m * SI_COUNT;
    const double* mc = a.mcoef + (size_t)m * MC_COUNT;
    double* sc = a.scal + (size_t)m * NIWQG_S_COUNT;
    const double M = a.M, M2 = M * M;
    const double f = mc[MC_F], hslash = mc[MC_HSLASH], kappa2 = mc[MC_KAPPA2];
    const double nu4 = mc[MC_NU4], nu = mc[MC_NU], mu = mc[MC_MU], nu4w = mc[MC_NU4W], nuw = mc[MC_NUW], muw = mc[MC_MUW];
    double g1, g2, x1, x2, lap2m;
    if (a.spec_budget) {
        // only the sums gamma1+gamma2 and xi1+xi2 enter the stage tendencies (Kernel.py:320-321); Parseval forms
        g1 = 0.5 * hslash * (se[SE_T1R] / M2) / f;
        g2 = 0.0;
        x1 = ((-nu4w * se[SE_T2I] - nuw * se[SE_T1I] - muw * se[SE_T0I]) / M2) / f;
        x2 = 0.0;
        lap2m = se[SE_LAP2] / M2;
    } else {
        g1 = 0.5 * 0.5 * hslash * (sd[SD_G1] / M) / f;
        g2 = 0.5 * hslash * (sd[SD_G2] / M) / f;
        x1 = (sd[SD_X1] / M) / f; x2 = (sd[SD_X2] / M) / f;
        lap2m = sd[SD_LAP2] / M;
    }
    const double ar = sd[SD_PHI_R] / M, ai = sd[SD_PHI_I] / M, br = sd[SD_QPC_R] / M, bi = sd[SD_QPC_I] / M;
    const double pi = 0.5 * (ar * bi + ai * br);
    const double ep_psi = nu4 * (si[SI_QLAP2PSI] / M2) - nu * (si[SI_PLAPQ] / M2) + mu * (si[SI_PQ] / M2);
    const double chi_phi = -0.5 * nu4w * (se[SE_WV6PHI] / M2) / kappa2 - 0.5 * nuw * lap2m / kappa2 -
                           0.5 * muw * (sd[SD_GRAD2] / M) / kappa2;
    const double ep_phi = -nu4w * lap2m - nuw * (sd[SD_GRAD2] / M) - muw * (sd[SD_PHI2] / M);
    sc[NIWQG_S_GAMMA1] = g1; sc[NIWQG_S_GAMMA2] = g2; sc[NIWQG_S_XI1] = x1; sc[NIWQG_S_XI2] = x2; sc[NIWQG_S_PI] = pi;
    if (a.stage == 0) {
        sc[NIWQG_S_EP_PSI] = ep_psi; sc[NIWQG_S_CHI_PHI] = chi_phi; sc[NIWQG_S_EP_PHI] = ep_phi;
        return;
    }
    double* sv = a.stagev + (size_t)m * 12 + (a.stage - 1) * 3;
    sv[0] = -(g1 + g2) + (x1 + x2) + ep_psi;
    sv[1] = g1 + g2 + chi_phi;
    sv[2] = ep_phi;
    if (a.stage == 4) {
        const double* s0 = a.stagev + (size_t)m * 12;
        sc[NIWQG_S_KE] += a.dt * (s0[0] + 2 * (s0[3] + s0[6]) + s0[9]) / 6.;
        sc[NIWQG_S_PW] += a.dt * (s0[1] + 2 * (s0[4] + s0[7]) + s0[10]) / 6.;
        sc[NIWQG_S_KW] += a.dt * (s0[2] + 2 * (s0[5] + s0[8]) + s0[11]) / 6.;
    }
}

static BudgetArgs budget_args(niwqg_handle* h, int stage) {
    BudgetArgs b{};
    b.stage = stage; b.M = h->Mg; b.dt = h->p.dt; b.mcoef = h->mcoef;
    b.sumsD = h->sumsD; b.sumsE = h->sumsE; b.sumsI = h->sumsI; b.scal = h->scal; b.stagev = h->stagev;
    b.spec_budget = (h->flags & MF_SPEC_BUDGET) ? 1 : 0;
    return b;
}

// ---------------------------------------------------------------------------
// family building blocks
// ---------------------------------------------------------------------------
// phi-derived physical fields from the current phih: phi, lapphi (+lap2phi) always; phix, phiy when `grad`
static int wave_fields(niwqg_handle* h, bool want_phi, bool grad, bool lap) {
    const cd* ph = h->phih[h->cp];
    if (h->split && want_phi && grad && !lap) {
        // phi, phix, phiy: the streaming radix stage reads phih once and writes the three intermediates
        const int pros[3] = {PRO_NONE, PRO_IK, PRO_IL};
        cd* dst[3] = {h->phi, h->phix, h->phiy};
        int r = split_p(h, ph, h->T, pros, 3, false, true);
        const double sc = 1.0 / ((double)h->N * (double)h->N);
        for (int o = 0; o < 3 && !r; ++o) {
            r = split_colsub(h, h->T[o], dst[o], false);
            if (!r) r = split_rows(h, dst[o], dst[o], PRO_NONE, EPI_NONE, sc, true);
        }
        return r;
    }
    if (h->nranks == 1 && !h->split && want_phi && grad && !lap) {
        // phi = ifft(phih), phix = ifft(ik phih), phiy = ifft(il phih) in 2 row passes + 3 column passes instead of 3 + 3:
        // the i l factor depends on the column-pass direction only, so phiy shares the row pass of phi and gets its
        // factor (conjugated: the intermediate is in the conjugated domain) in the prologue of its column pass.
        const bool par = !h->prof;
        const int l1 = par ? 1 : 0;
        if (par) {
            CK(cudaEventRecord(h->ev_fork, h->lane_stream[0]));
            CK(cudaStreamWaitEvent(h->lane_stream[1], h->ev_fork, 0));
        }
        int r = inv_row_pass(h, ph, h->phi, PRO_NONE, 0);
        if (!r) r = inv_row_pass(h, ph, h->phix, PRO_IK, l1);
        if (!r) r = inv_col_pass(h, h->phix, h->phix, PRO_NONE, l1);
        if (!r) r = inv_col_pass(h, h->phi, h->phiy, PRO_IL_CONJ, 0);     // reads the shared row pass ...
        if (!r) r = inv_col_pass(h, h->phi, h->phi, PRO_NONE, 0);         // ... before it is transformed in place
        if (r) return r;
        if (par) {
            CK(cudaEventRecord(h->ev_join, h->lane_stream[1]));
            CK(cudaStreamWaitEvent(h->lane_stream[0], h->ev_join, 0));
        }
        return 0;
    }
    if (h->nranks > 1 && h->p2p && h->exchange == 0 && want_phi && grad && !lap) {
        // slab: the column pass comes first, so phi and phix share it (one exchange less): phix gets its conj(i k) in the
        // prologue of its row pass, phiy = ifft(il phih) has its own column pass
        const bool par = !h->prof;
        const int l1 = par ? 1 : 0;
        if (par) {
            CK(cudaEventRecord(h->ev_fork, h->lane_stream[0]));
            CK(cudaStreamWaitEvent(h->lane_stream[1], h->ev_fork, 0));
        }
        int b0 = 0, b1 = 0;
        int r = slab_inv_push(h, ph, PRO_NONE, 0, &b0);
        if (!r) r = slab_inv_push(h, ph, PRO_IL, l1, &b1);
        if (!r) r = slab_inv_row(h, l1, b1, h->phiy, PRO_NONE);
        if (!r) r = slab_inv_row(h, 0, b0, h->phi, PRO_NONE);
        if (!r) r = slab_inv_row(h, 0, b0, h->phix, PRO_IK_CONJ);
        if (r) return r;
        if (par) {
            CK(cudaEventRecord(h->ev_join, h->lane_stream[1]));
            CK(cudaStreamWaitEvent(h->lane_stream[0], h->ev_join, 0));
        }
        return 0;
    }
    FftJob jobs[5];
    int n = 0;
    if (want_phi) jobs[n++] = FftJob{ph, h->phi, true, PRO_NONE};
    if (grad) {
        jobs[n++] = FftJob{ph, h->phix, true, PRO_IK};
        jobs[n++] = FftJob{ph, h->phiy, true, PRO_IL};
    }
    if (lap) {
        jobs[n++] = FftJob{ph, h->lapphi, true, PRO_NEG_WV2};
        if (h->flags & MF_HAS_LAP2) jobs[n++] = FftJob{ph, h->lap2phi, true, PRO_WV4};
    }
    return fft2_group(h, jobs, n);
}

// _invert + _calc_rel_vorticity + (u,v) for the current (qh, phi, phix, phiy)
// keep_qwh: store the wave-PV spectrum qwh (only diagnostics and attribute reads use it: the step itself carries it
// inside the packed q + i qw spectrum), so the stages that are overwritten before anyone can look skip the write
static int invert_family(niwqg_handle* h, bool keep_qwh = true) {
    InvertArgs ia{};
    ia.g = h->g;
    ia.flags = h->flags; ia.qh = h->qh[h->cq]; ia.filtr = h->filtr;
    ia.filtr_sym = (h->p.use_filter || !h->p.dealias) ? 1 : 0;
    ia.ph = h->ph; ia.qs = h->qs;
    if (h->flags & MF_WAVE_PV) {
        { PROF(PK_PHYS); k_phys_wavepv<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phi, h->phix, h->phiy, h->W, h->npts, h->jscale); }
        CK(cudaGetLastError());
        h->launches++;
        FFT(h->W, h->W, false, PRO_NONE, h->B);
        ia.W = h->W; ia.qwh = keep_qwh ? h->qwh : nullptr; ia.inv_jscale = 1.0 / h->jscale;
    }
    if (h->flags & MF_YBJ) ia.uvgen = h->uv;
    ia.partials = (h->flags & MF_YBJ) ? nullptr : h->part;
    { PROF(PK_SPEC); k_spec_invert<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(ia, h->mcoef); }
    CK(cudaGetLastError());
    h->launches++;
    if (ia.partials) FIN(SI_COUNT, h->sumsI);   // ep_psi sums of the state the next stage starts from
    if (h->flags & MF_YBJ) {
        FFT(h->uv, h->uv, true, PRO_NONE, h->B);
    } else {
        const FftJob jobs[2] = {FftJob{h->ph, h->uv, true, PRO_UV}, FftJob{h->qs, h->qs, true, PRO_NONE}};
        int r = fft2_group(h, jobs, 2);
        if (r) return r;
    }
    return 0;
}

static PhysArgs phys_args(niwqg_handle* h, int extra_flags) {
    PhysArgs pa{};
    pa.npts = h->npts; pa.flags = h->flags | extra_flags;
    pa.mcoef = h->mcoef;
    pa.uv = h->uv; pa.qs = h->qs; pa.phi = h->phi; pa.phix = h->phix; pa.phiy = h->phiy;
    pa.lapphi = h->lapphi; pa.lap2phi = h->lap2phi; pa.uvq = h->uvq;
    pa.P1 = h->P1; pa.P2 = h->P2; pa.partials = h->part;
    return pa;
}

static int ql_wave_velocity(niwqg_handle* h) {   // uq, vq from the current qh (QLModel.py:65-66)
    { PROF(PK_SPEC); k_spec_uvq<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->g, h->qh[h->cq], h->uvq); }
    CK(cudaGetLastError());
    h->launches++;
    FFT(h->uvq, h->uvq, true, PRO_NONE, h->B);
    return 0;
}

// ---------------------------------------------------------------------------
// Lagrangian particles: one RK4 stage wherever the model's uv (and phi) hold the fields of ETDRK4 stage `st`
// ---------------------------------------------------------------------------
static PartArgs particle_args(const niwqg_handle* h) {
    PartArgs a{};
    a.xn = h->pbuf; a.xs = h->pbuf + (size_t)h->B * h->np; a.acc = h->pbuf + 2 * (size_t)h->B * h->np;
    a.clk = (double*)(h->pbuf + 3 * (size_t)h->B * h->np);
    a.mcoef = h->mcoef; a.npts = h->npts; a.P = h->np; a.N = h->N;
    a.dshift = h->deintC > 1 ? 1 : 0;               // deintC is 1 or 2 (split path)
    a.dM = h->deintC > 1 ? h->deintM : h->N;
    a.L = h->p.L; a.dx = h->dx; a.dt = h->p.dt;
    return a;
}
static dim3 particle_grid(const niwqg_handle* h) { return dim3((unsigned)((h->np + 127) / 128), h->B); }

static int particles_stage(niwqg_handle* h, int st) {
    if (!h->np) return 0;
    PartArgs a = particle_args(h);
    a.uv = h->uv; a.phi = h->pwaves ? h->phi : nullptr;
    const dim3 g = particle_grid(h);
    cudaStream_t s = h->stream;
#define NIWQG_PSTAGE(S)                                                        \
    case S:                                                                    \
        if (h->pwaves) k_particles<S, true><<<g, 128, 0, s>>>(a);              \
        else k_particles<S, false><<<g, 128, 0, s>>>(a);                       \
        break;
    switch (st) { NIWQG_PSTAGE(1) NIWQG_PSTAGE(2) NIWQG_PSTAGE(3) NIWQG_PSTAGE(4) }
#undef NIWQG_PSTAGE
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

// Coupled / UnCoupled step on the split transform path with the fused spectral kernels (kernels_fused.cuh): the
// forward transforms stop after their M-point column transforms, the kernel that consumes the spectrum does the radix
// combine itself; the kernels that produce a spectrum emit the radix stage of its inverse transforms.
template <int N>
static int step_family_fused_n(niwqg_handle* h) {
    const int oq = h->cq, op = h->cp, nq = 1 - oq, np = 1 - op;
    const bool wave = (h->flags & MF_WAVE_PV) != 0;
    const double sc = 1.0 / ((double)N * (double)N);
    const int grid = WAVE_CTAS;     // persistent grid of the fused kernels
    int r;
    for (int st = 1; st <= 4; ++st) {
        if ((r = particles_stage(h, st))) return r;
        PhysArgs pa = phys_args(h, MF_P1_BY_LOADER);
        { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
        CK(cudaGetLastError());
        h->launches++;
        FIN(SD_COUNT, h->sumsD);
        if ((r = split_rows_loader(h, LD_UQVQ, h->P1))) return r;   // P1 = (uq, vq) formed while loading uv, qs
        if ((r = split_colsub(h, h->P1, h->T[0], true))) return r;
        if ((r = split_rows(h, h->P2, h->P2, PRO_NONE, EPI_NONE, 1.0, false))) return r;
        if ((r = split_colsub(h, h->P2, h->T[1], true))) return r;
        FStageArgs fa{};
        StageArgs& sa = fa.s;
        sa.g = h->g; sa.stage = st; sa.flags = h->flags; sa.do_q = 1; sa.do_phi = 1; sa.sums_here = 1;
        sa.P1 = h->P1; sa.P2 = h->P2;
        sa.y0q = h->qh[oq]; sa.y0p = h->phih[op]; sa.yq = h->qh[nq]; sa.yp = h->phih[np];
        sa.y1q = h->y1q; sa.y1p = h->y1p; sa.F0q = h->F0q; sa.F0p = h->F0p; sa.Fabq = h->Fabq; sa.Fabp = h->Fabp;
        if (st == 1) { sa.yq = h->y1q; sa.yp = h->y1p; }     // the stage-1 state is written once, as y1 (read again at stage 3)
        sa.ph = h->ph; sa.tq = h->tq; sa.tp = h->tp; sa.filtr = h->filtr; sa.sumsD = h->sumsD; sa.partials = h->part;
        fa.twc = h->twc; fa.dk = h->dk;
        sa.hsym = (h->p.use_filter || !h->p.dealias) ? 1 : 0;
        fa.T = h->T[0];
        { PROF(PK_SPEC); CK((launch_fstage<N>(fa, false, grid, h->stream))); }
        fa.T = h->T[1];
        fa.out[0] = h->T[1]; fa.out[1] = h->T[2]; fa.out[2] = h->T[0];   // in place over its own input; T0 is free again
        fa.nout = wave ? 3 : 1;
        { PROF(PK_SPEC); CK((launch_fstage<N>(fa, true, grid, h->stream))); }
        h->launches += 2;
        if (st == 1) { h->cq = nq; h->cp = np; }
        FIN(SE_COUNT, h->sumsE, 0, grid);
        { PROF(PK_SMALL); k_budget<<<h->B, 32, 0, h->stream>>>(budget_args(h, st)); }
        CK(cudaGetLastError());
        h->launches++;
        // self.phi = ifft(phih); phix, phiy (jacobian_phic_phi): the remaining two launches of each inverse transform
        if ((r = split_colsub(h, h->T[1], h->phi, false))) return r;
        if ((r = split_rows(h, h->phi, h->phi, PRO_NONE, EPI_NONE, sc, true))) return r;
        if (wave) {
            if ((r = split_colsub(h, h->T[2], h->phix, false))) return r;
            if ((r = split_rows(h, h->phix, h->phix, PRO_NONE, EPI_NONE, sc, true))) return r;
            if ((r = split_colsub(h, h->T[0], h->phiy, false))) return r;
            if ((r = split_rows(h, h->phiy, h->phiy, PRO_NONE, EPI_NONE, sc, true))) return r;
            if ((r = split_rows_loader(h, LD_WAVEPV, h->W))) return r;
            if ((r = split_colsub(h, h->W, h->T[0], true))) return r;
        }
        // _invert(); _calc_rel_vorticity(); u, v
        FInvertArgs ia{};
        ia.i.g = h->g; ia.i.flags = h->flags; ia.i.f = h->p.f; ia.i.qh = (st == 1) ? h->y1q : h->qh[h->cq]; ia.i.filtr = h->filtr;
        ia.i.filtr_sym = (h->p.use_filter || !h->p.dealias) ? 1 : 0;
        ia.i.ph = h->ph; ia.i.qs = h->qs; ia.i.W = h->T[0]; ia.i.qwh = (wave && st == 4) ? h->qwh : nullptr;
        ia.i.inv_jscale = 1.0 / h->jscale; ia.i.partials = h->part;
        ia.T = h->T[0]; ia.out_uv = h->T[1]; ia.out_qs = h->T[2]; ia.twc = h->twc; ia.dk = h->dk;
        { PROF(PK_SPEC); CK((launch_finvert<N>(ia, wave, grid, h->stream))); }
        h->launches++;
        FIN(SI_COUNT, h->sumsI, 0, grid);
        if ((r = split_colsub(h, h->T[1], h->uv, false))) return r;
        if ((r = split_rows(h, h->uv, h->uv, PRO_NONE, EPI_NONE, sc, true))) return r;
        if ((r = split_colsub(h, h->T[2], h->qs, false))) return r;
        if ((r = split_rows(h, h->qs, h->qs, PRO_NONE, EPI_NONE, sc, true))) return r;
    }
    return 0;
}
static int step_family_fused(niwqg_handle* h) {
    switch (h->N) {
        case 2048: return step_family_fused_n<2048>(h);
        case 4096: return step_family_fused_n<4096>(h);
        case 8192: return step_family_fused_n<8192>(h);
    }
    h->err = "fused step: unsupported grid";
    return -1;
}

static int step_family(niwqg_handle* h) {
    if (h->split && (h->flags & MF_SPEC_BUDGET)) return step_family_fused(h);   // Coupled / UnCoupled
    const bool ybj = (h->flags & MF_YBJ) != 0, ql = (h->flags & MF_QL_ADV) != 0;
    const int oq = h->cq, op = h->cp;          // y0 buffers
    const int nq = ybj ? oq : 1 - oq, np = 1 - op;
    for (int st = 1; st <= 4; ++st) {
        if (int rp = particles_stage(h, st)) return rp;
        if (ybj) {   // _calc_grad_phi from the stage's phih (YBJModel.py:135-139); phi stays stale (F7)
            const cd* cur = (st == 1) ? h->phih[op] : h->phih[np];
            const FftJob jobs[2] = {FftJob{cur, h->phix, true, PRO_IK}, FftJob{cur, h->phiy, true, PRO_IL}};
            int r = fft2_group(h, jobs, 2);
            if (r) return r;
        }
        StageArgs sa{};
        sa.g = h->g;
        sa.stage = st; sa.flags = h->flags; sa.do_q = ybj ? 0 : 1; sa.do_phi = 1;
        sa.hsym = (h->p.use_filter || !h->p.dealias) ? 1 : 0;
        sa.P1 = h->P1; sa.P2 = h->P2;
        sa.y0q = h->qh[oq]; sa.y0p = h->phih[op]; sa.yq = h->qh[nq]; sa.yp = h->phih[np];
        sa.y1q = h->y1q; sa.y1p = h->y1p; sa.F0q = h->F0q; sa.F0p = h->F0p; sa.Fabq = h->Fabq; sa.Fabp = h->Fabp;
        sa.ph = h->ph; sa.tq = h->tq; sa.tp = h->tp; sa.filtr = h->filtr; sa.sumsD = h->sumsD; sa.partials = h->part;
        if (!ql) {
            PhysArgs pa = phys_args(h, 0);
            { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
            CK(cudaGetLastError());
            h->launches++;
            if (!ybj) {
                FIN(SD_COUNT, h->sumsD);
                const FftJob jobs[2] = {FftJob{h->P1, h->P1, false, PRO_NONE}, FftJob{h->P2, h->P2, false, PRO_NONE}};
                int r = fft2_group(h, jobs, 2);
                if (r) return r;
            } else {
                FFT(h->P2, h->P2, false, PRO_NONE, h->B);
            }
            if (ybj) {
                sa.sums_here = 0;
                { PROF(PK_SPEC); CK((launch_spec_stage<false, true>(sa, pw_grid(h), h->stream, h->pm_p))); }
                h->launches++;
            } else {
                // two lighter kernels: q equation, then phi equation + the stage's spectral budget sums
                sa.do_q = 1; sa.do_phi = 0; sa.sums_here = 0;
                { PROF(PK_SPEC); CK((launch_spec_stage<true, false>(sa, pw_grid(h), h->stream, h->pm_q))); }
                sa.do_q = 0; sa.do_phi = 1; sa.sums_here = 1;
                { PROF(PK_SPEC); CK((launch_spec_stage<false, true>(sa, pw_grid(h), h->stream, h->pm_p))); }
                h->launches += 2;
            }
            if (st == 1) { h->cq = nq; h->cp = np; }
        } else {
            // repaired QL: jacobian_psi_phi reads qh AFTER the stage's q update (Kernel.py:326-332 order),
            // so the stage is split: q half, wave velocity from the new qh, phi half.
            PhysArgs pa = phys_args(h, MF_SKIP_P2);
            { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
            CK(cudaGetLastError());
            FIN(SD_COUNT, h->sumsD);
            FFT(h->P1, h->P1, false, PRO_NONE, h->B);
            sa.do_phi = 0; sa.sums_here = 1;
            { PROF(PK_SPEC); CK((launch_spec_stage<true, false>(sa, pw_grid(h), h->stream, h->pm_q))); }
            if (st == 1) h->cq = nq;
            int r = ql_wave_velocity(h);
            if (r) return r;
            pa = phys_args(h, MF_SKIP_P1);
            { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
            CK(cudaGetLastError());
            FFT(h->P2, h->P2, false, PRO_NONE, h->B);
            sa.do_q = 0; sa.do_phi = 1; sa.sums_here = 0;
            { PROF(PK_SPEC); CK((launch_spec_stage<false, true>(sa, pw_grid(h), h->stream, h->pm_p))); }
            h->launches += 4;
            if (st == 1) h->cp = np;
        }
        if (!ybj) {
            FIN(SE_COUNT, h->sumsE);
            { PROF(PK_SMALL); k_budget<<<h->B, 32, 0, h->stream>>>(budget_args(h, st)); }
            CK(cudaGetLastError());
            h->launches++;
            // self.phi = ifft(phih); _invert(); _calc_rel_vorticity()  (Kernel.py:337-339 / :395-397)
            const bool grad = (h->flags & MF_WAVE_PV) != 0;   // only jacobian_phic_phi refreshes phix, phiy (F6)
            int r = wave_fields(h, true, grad, !(h->flags & MF_SPEC_BUDGET));
            if (r) return r;
            r = invert_family(h, st == 4);
            if (r) return r;
        }
    }
    if (ybj) FFT(h->phih[h->cp], h->phi, true, PRO_NONE, h->B);   // YBJModel.py:87
    return 0;
}

// ---------------------------------------------------------------------------
// QG model (half spectrum)  -- see kernels_qg.cuh
// ---------------------------------------------------------------------------
static int qg_expand_and_invert(niwqg_handle* h, const cd* qh_cur, bool want_uv = true) {
    QgExpandArgs ea{};
    ea.N = h->N; ea.nk = h->nk; ea.dk = h->dk; ea.qh = qh_cur; ea.ph = h->ph; ea.uv = want_uv ? h->uv : nullptr; ea.qs = h->qs;
    { PROF(PK_SPEC); k_qg_expand<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(ea); }
    CK(cudaGetLastError());
    h->launches++;
    if (want_uv) FFT(h->uv, h->uv, true, PRO_NONE, h->B);
    FFT(h->qs, h->qs, true, PRO_NONE, h->B);
    return 0;
}

static int qg_scalar_physical(niwqg_handle* h, const cd* ch_cur) {
    QgExpand1Args ea{};
    ea.N = h->N; ea.nk = h->nk; ea.dk = h->dk; ea.in = ch_cur; ea.out = h->W; ea.mode = QGX_PLAIN;
    { PROF(PK_SPEC); k_qg_expand1<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(ea); }
    CK(cudaGetLastError());
    h->launches++;
    FFT(h->W, h->W, true, PRO_NONE, h->B);
    return 0;
}

static int step_qg(niwqg_handle* h) {
    const bool ps = h->p.passive_scalar != 0;
    const int oq = h->cq, nq = 1 - oq, oc = h->cc, nc = 1 - oc;
    for (int st = 1; st <= 4; ++st) {
        // jacobian_psi_q (QGModel.py:469-481): u, v, q from the current (qh, ph)
        const cd* cur = (st == 1) ? h->qh[oq] : h->qh[nq];
        int r = qg_expand_and_invert(h, cur);
        if (r) return r;
        if ((r = particles_stage(h, st))) return r;
        const cd* ccur = nullptr;
        if (ps) {
            ccur = (st == 1) ? h->chh[oc] : h->chh[nc];
            r = qg_scalar_physical(h, ccur);       // c = irfft2(ch) -> W.x   (QGModel.py:493)
            if (r) return r;
        }
        { PROF(PK_PHYS); k_qg_products<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->uv, h->qs, ps ? h->W : nullptr, h->P1, h->P2,
                                                                       h->npts); }
        CK(cudaGetLastError());
        h->launches++;
        FFT(h->P1, h->P1, false, PRO_NONE, h->B);
        if (ps) FFT(h->P2, h->P2, false, PRO_NONE, h->B);
        QgStageArgs sa{};
        sa.N = h->N; sa.nk = h->nk; sa.dk = h->dk; sa.stage = st; sa.ps = ps ? 1 : 0;
        sa.P1 = h->P1; sa.P2 = h->P2;
        sa.y0q = h->qh[oq]; sa.yq = h->qh[nq]; sa.y1q = h->y1q; sa.F0q = h->F0q; sa.Fabq = h->Fabq;
        sa.y0c = h->chh[oc]; sa.yc = h->chh[nc]; sa.y1c = h->y1c; sa.F0c = h->F0c; sa.Fabc = h->Fabc;
        sa.tq = h->tq; sa.tc = h->tc; sa.filtr = h->filtr; sa.partials = h->part;
        sa.nu4c = h->p.nu4c;
        {
            PROF(PK_SPEC);
            const dim3 g = pw_grid(h);
            if (h->pm_q && h->pm_c) k_qg_stage<true, true><<<g, NIWQG_PW_THREADS, 0, h->stream>>>(sa);
            else if (h->pm_q) k_qg_stage<true, false><<<g, NIWQG_PW_THREADS, 0, h->stream>>>(sa);
            else if (h->pm_c) k_qg_stage<false, true><<<g, NIWQG_PW_THREADS, 0, h->stream>>>(sa);
            else k_qg_stage<false, false><<<g, NIWQG_PW_THREADS, 0, h->stream>>>(sa);
        }
        CK(cudaGetLastError());
        h->launches++;
        if (st == 1) { h->cq = nq; h->cc = nc; }
        FIN(QE_COUNT, h->sumsE);
        QgBudgetArgs ba{};
        ba.stage = st; ba.M = h->Mg; ba.dt = h->p.dt; ba.mcoef = h->mcoef; ba.ps = ps ? 1 : 0;
        ba.sumsE = h->sumsE; ba.scal = h->scal; ba.stagev = h->stagev;
        { PROF(PK_SMALL); k_qg_budget<<<h->B, 32, 0, h->stream>>>(ba); }
        CK(cudaGetLastError());
        h->launches++;
    }
    // final _invert + physical q (and c) (QGModel.py:397-404); u, v stay those of the stage-4 Jacobian,
    // which is what Gamma_c reads at the diagnostics tick (QGModel.py:731 -> :494)
    int r = qg_expand_and_invert(h, h->qh[h->cq], false);
    if (r) return r;
    if (ps) { r = qg_scalar_physical(h, h->chh[h->cc]); if (r) return r; }
    return 0;
}

// Gamma_c sum (QGModel.py:731): sum FH(lapc-hat) conj(FH(jacobian_psi_c-hat)) -> sumsD[member]
static int qg_gamma_c(niwqg_handle* h) {
    int r = qg_scalar_physical(h, h->chh[h->cc]);      // jacobian_psi_c refreshes c = irfft2(ch) (QGModel.py:493)
    if (r) return r;
    { PROF(PK_PHYS); k_qg_products<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->uv, h->qs, h->W, h->P1, h->P2, h->npts); }
    CK(cudaGetLastError());
    FFT(h->P2, h->P2, false, PRO_NONE, h->B);
    k_qg_gamma_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->P2, h->chh[h->cc], h->N, h->nk, h->dk, h->part);
    CK(cudaGetLastError());
    h->launches += 2;
    FIN(1, h->sumsD);
    return 0;
}

// ---------------------------------------------------------------------------
// physical arrays cross the ABI in natural x order; on the device they may be de-interleaved (k_deint)
// ---------------------------------------------------------------------------
static const size_t STAGED_BYTES = 32u << 20;      // transfers at least this large go through the copy stream

template <typename T>
static int upload_phys(niwqg_handle* h, const void* src, T* dst, size_t nelem, int on_device) {
    const size_t bytes = nelem * sizeof(T);
    if (on_device || bytes < STAGED_BYTES || !h->stage_in) {
        const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        T* to = (h->deintC <= 1) ? dst : (T*)h->P2;
        CK(cudaMemcpyAsync(to, src, bytes, kind, h->stream));
        if (!on_device) {                       // the caller may reuse its buffer when we return
            CK(cudaEventRecord(h->ev_up_done, h->stream));
            CK(cudaEventSynchronize(h->ev_up_done));
        }
        if (h->deintC > 1) {
            k_deint<T><<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>((const T*)h->P2, dst, nelem, h->N, h->deintM, h->deintC, 1);
            CK(cudaGetLastError());
            h->launches++;
        }
        return 0;
    }
    // host -> staging on the copy stream (as soon as the previous upload has been consumed), staging -> field on the
    // main stream behind whatever is already queued there
    if (h->up_free_rec) CK(cudaStreamWaitEvent(h->copy_stream, h->ev_up_free, 0));
    CK(cudaMemcpyAsync(h->stage_in, src, bytes, cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->ev_up_done, h->copy_stream));
    CK(cudaStreamWaitEvent(h->stream, h->ev_up_done, 0));
    if (h->deintC > 1) {
        k_deint<T><<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>((const T*)h->stage_in, dst, nelem, h->N, h->deintM, h->deintC, 1);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        CK(cudaMemcpyAsync(dst, h->stage_in, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    CK(cudaEventRecord(h->ev_up_free, h->stream));
    h->up_free_rec = true;
    CK(cudaEventSynchronize(h->ev_up_done));    // the caller may reuse its buffer when we return
    return 0;
}
// niwqg_stage_*: host -> pre_buf[w] on the copy stream, no wait
static int stage_upload(niwqg_handle* h, int w, const void* src, size_t bytes) {
    if (!src) { h->err = "stage: null host array"; return -1; }
    if (!h->pre_buf[w]) {
        CK(cudaMalloc(&h->pre_buf[w], bytes));
        CK(cudaEventCreateWithFlags(&h->pre_done[w], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->pre_free[w], cudaEventDisableTiming));
    }
    if (h->pre_free_rec[w]) CK(cudaStreamWaitEvent(h->copy_stream, h->pre_free[w], 0));   // the previous consumer has read it
    CK(cudaMemcpyAsync(h->pre_buf[w], src, bytes, cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->pre_done[w], h->copy_stream));
    h->pre_staged[w] = true;
    return 0;
}
// set_*(NULL): pre_buf[w] -> field (device layout) on the main stream
template <typename T>
static int upload_staged(niwqg_handle* h, int w, T* dst, size_t nelem) {
    if (!h->pre_staged[w]) { h->err = "set_q / set_phi without an array: nothing was staged (niwqg_stage_q / niwqg_stage_phi)"; return -1; }
    CK(cudaStreamWaitEvent(h->stream, h->pre_done[w], 0));
    if (h->deintC > 1) {
        k_deint<T><<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>((const T*)h->pre_buf[w], dst, nelem, h->N, h->deintM, h->deintC, 1);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        CK(cudaMemcpyAsync(dst, h->pre_buf[w], nelem * sizeof(T), cudaMemcpyDeviceToDevice, h->stream));
    }
    CK(cudaEventRecord(h->pre_free[w], h->stream));
    h->pre_free_rec[w] = true;
    h->pre_staged[w] = false;
    CK(cudaEventSynchronize(h->pre_done[w]));   // the caller may reuse its buffer when we return
    return 0;
}
// field (device layout) -> caller.  async: returns once the copy is queued (niwqg_wait_transfers completes it)
template <typename T>
static int download_phys(niwqg_handle* h, const T* src, void* dst, size_t nelem, int on_device, T* stage, bool async = false) {
    const size_t bytes = nelem * sizeof(T);
    const int k = sizeof(T) == sizeof(cd) ? 1 : 0;
    if (on_device || bytes < STAGED_BYTES || !h->stage_out[k]) {
        const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        if (h->deintC > 1) {
            k_deint<T><<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>(src, stage, nelem, h->N, h->deintM, h->deintC, 0);
            CK(cudaGetLastError());
            h->launches++;
            src = stage;
        }
        CK(cudaMemcpyAsync(dst, src, bytes, kind, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    T* so = (T*)h->stage_out[k];
    if (h->dn_done_rec[k]) CK(cudaStreamWaitEvent(h->stream, h->ev_dn_done[k], 0));    // staging free again
    if (h->deintC > 1) {
        k_deint<T><<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>(src, so, nelem, h->N, h->deintM, h->deintC, 0);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        CK(cudaMemcpyAsync(so, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
    }
    CK(cudaEventRecord(h->ev_dn_ready, h->stream));
    CK(cudaStreamWaitEvent(h->copy_out, h->ev_dn_ready, 0));
    CK(cudaMemcpyAsync(dst, so, bytes, cudaMemcpyDeviceToHost, h->copy_out));
    CK(cudaEventRecord(h->ev_dn_done[k], h->copy_out));
    h->dn_done_rec[k] = true;
    if (!async) CK(cudaEventSynchronize(h->ev_dn_done[k]));
    return 0;
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" {

const char* niwqg_last_error(const niwqg_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int niwqg_destroy(niwqg_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->p.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& g : h->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    if (h->lane_stream[1]) cudaStreamSynchronize(h->lane_stream[1]);
    if (h->p2p)
        for (int r = 0; r < h->nranks; ++r)
            for (int l = 0; l < niwqg_handle::NLANE; ++l)
                for (int b = 0; b < 2; ++b)
                    if (r != h->rank && h->peerY[l][b][r]) cudaIpcCloseMemHandle(h->peerY[l][b][r]);
    if (h->lane_comm[1] && g_nccl.CommDestroy) g_nccl.CommDestroy(h->lane_comm[1]);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    if (h->lane_stream[1]) cudaStreamDestroy(h->lane_stream[1]);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (void* p : h->allocs) cudaFree(p);
    for (cudaEvent_t e : h->prof_pool) cudaEventDestroy(e);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->copy_out) { cudaStreamSynchronize(h->copy_out); cudaStreamDestroy(h->copy_out); }
    for (cudaEvent_t e : {h->ev_up_done, h->ev_up_free, h->ev_dn_ready, h->ev_dn_done[0], h->ev_dn_done[1]}) if (e) cudaEventDestroy(e);
    for (int w = 0; w < 2; ++w) {
        if (h->pre_buf[w]) cudaFree(h->pre_buf[w]);
        if (h->pre_done[w]) cudaEventDestroy(h->pre_done[w]);
        if (h->pre_free[w]) cudaEventDestroy(h->pre_free[w]);
    }
    if (h->pin) cudaFreeHost(h->pin);
    if (h->pbuf) cudaFree(h->pbuf);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return 0;
}

static int create_impl(niwqg_handle* h) {
    const niwqg_params& p = h->p;
    const int N = p.nx;
    CK(cudaSetDevice(p.device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&h->ev0));
    CK(cudaEventCreate(&h->ev1));
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_up_done, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_up_free, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_dn_ready, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_dn_done[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_dn_done[1], cudaEventDisableTiming));
    h->N = N; h->B = p.batch; h->model = p.model; h->qg = (p.model == NIWQG_MODEL_QG);
    CK(cudaMallocHost((void**)&h->pin, ((size_t)p.batch * (NIWQG_S_COUNT + 64) + 64) * sizeof(double)));
    h->nranks = p.nranks > 1 ? p.nranks : 1;
    h->rank = h->nranks > 1 ? p.rank : 0;
    h->nyl = N / h->nranks; h->ncl = N / h->nranks;
    h->nk = h->qg ? N / 2 + 1 : h->ncl;
    h->npts = (size_t)h->nyl * N; h->nspec = (size_t)N * h->nk;
    h->Mg = (double)N * (double)N;
    // the physical x order is de-interleaved on the split path only: for the cluster row pass (a push kernel with
    // contiguous stores on that layout) it measured slower than the natural layout (0.578 vs 0.535 ms per 8192^2 row pass)
    if (h->nranks == 1 && h->B == 1 && !h->qg && N >= 2048) {
        const char* e = getenv("NIWQG_SPLIT");
        h->split = e ? (atoi(e) != 0) : (N == 8192);
        if (h->split) { h->deintM = N / 2; h->deintC = 2; }
    }
    h->col3 = h->nranks == 1 && N == 8192 && h->B == 1 && !h->split;
    h->g = Grid{N, 2.0 * M_PI / p.L, h->ncl, h->ncl / 2, h->rank, h->nranks > 1 ? 1 : 0};
    if (h->nranks > 1) {
        int r = nccl_load(h->err);
        if (r) return r;
        ncclUniqueId id;
        memcpy(&id, p.nccl_id, sizeof id);
        NK(g_nccl.CommInitRank(&h->comm, h->nranks, id, h->rank));
    }
    h->dk = 2.0 * M_PI / p.L; h->dx = p.L / N;
    {   // power of two nearest 1/k_mid^2, k_mid = dk*N/8 (scaling of the packed wave-PV transform)
        const double kmid = h->dk * N / 8.0;
        h->jscale = exp2(rint(log2(1.0 / (kmid * kmid))));
    }
    h->kappa2m.assign(h->B, 0.0);
    h->hslashm.assign(h->B, 0.0);
    if (!h->qg) {
        for (int b = 0; b < h->B; ++b) {
            const niwqg_member_params& c = h->mp[b];
            const double kappa = c.m * c.f / c.N;     // Kernel.py:121-125
            h->kappa2m[b] = kappa * kappa;
            h->hslashm[b] = c.f / h->kappa2m[b];
        }
    }
    switch (p.model) {
        case NIWQG_MODEL_COUPLED: h->flags = MF_WAVE_PV | MF_FIX00 | MF_SPEC_BUDGET; break;
        case NIWQG_MODEL_UNCOUPLED: h->flags = MF_FIX00 | MF_SPEC_BUDGET; break;
        case NIWQG_MODEL_YBJ: h->flags = MF_YBJ; break;
        case NIWQG_MODEL_QL: h->flags = MF_WAVE_PV | MF_QL_ADV; break;
        default: h->flags = 0;
    }
    for (int b = 0; b < h->B; ++b)
        if (!h->qg && h->mp[b].nu4w != 0.0) h->flags |= MF_HAS_LAP2;
    const size_t B = h->B, cb = sizeof(cd);
    const size_t fsz = B * h->npts * cb, ssz = B * h->nspec * cb, tsz = h->nspec * cb;
    // twiddles
    {
        std::vector<cd> tw;
        build_twiddles(pass_local_len(N, false), tw);
        DA(h->tw_row, tw.size() * cb);
        CK(cudaMemcpyAsync(h->tw_row, tw.data(), tw.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        build_twiddles(pass_local_len(N, true), tw);
        DA(h->tw_col, tw.size() * cb);
        CK(cudaMemcpyAsync(h->tw_col, tw.data(), tw.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        tw.resize(N);
        const long double PI = 3.141592653589793238462643383279502884L;
        for (int t = 0; t < N; ++t) {
            const long double a = -2.0L * PI * (long double)t / (long double)N;
            tw[t] = make_double2((double)cosl(a), (double)sinl(a));
        }
        DA(h->twc, tw.size() * cb);
        CK(cudaMemcpyAsync(h->twc, tw.data(), tw.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    {   // per-member coefficients of the kernels (k_spec_invert, k_phys_rhs, k_budget, k_qg_budget, set_phi's Pw)
        std::vector<double> mc((size_t)B * MC_COUNT);
        for (size_t b = 0; b < B; ++b) {
            const niwqg_member_params& c = h->mp[b];
            double* r = &mc[b * MC_COUNT];
            r[MC_F] = c.f; r[MC_HSLASH] = h->hslashm[b]; r[MC_KAPPA2] = h->kappa2m[b];
            r[MC_NU4] = c.nu4; r[MC_NU] = c.nu; r[MC_MU] = c.mu; r[MC_NU4W] = c.nu4w; r[MC_NUW] = c.nuw; r[MC_MUW] = c.muw;
            r[MC_NU4C] = c.nu4c; r[MC_MUC] = c.muc;
            r[MC_PW_SEED] = h->qg ? 0.0 : 0.25 / h->Mg / h->kappa2m[b];
            r[MC_U] = c.U;
        }
        DA(h->mcoef, mc.size() * sizeof(double));
        CK(cudaMemcpyAsync(h->mcoef, mc.data(), mc.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    // tables: one set per equation, or one per member when the members' coefficients of that equation differ
    DA(h->filtr, h->nspec * sizeof(double));
    InitArgs ia{};
    ia.g = h->g; ia.N = N; ia.nk = h->nk; ia.half = h->qg ? 1 : 0; ia.dk = h->dk; ia.dt = p.dt; ia.dx = h->dx;
    ia.use_filter = p.use_filter; ia.dealias = p.dealias;
    bool filtr_done = false;
    // row[IC_*] of member b for one equation (eq 0: q, 1: phi, 2: passive scalar c)
    auto eq_row = [&](int eq, int b, double* r) {
        const niwqg_member_params& c = h->mp[b];
        if (eq == 0) { r[IC_RE_A4] = c.nu4; r[IC_RE_A2] = c.nu; r[IC_RE_A0] = c.mu; r[IC_IM_WV2] = 0.0; r[IC_BETA] = h->qg ? c.beta : 0.0; r[IC_U] = c.U; }
        else if (eq == 1) { r[IC_RE_A4] = c.nu4w; r[IC_RE_A2] = c.nuw; r[IC_RE_A0] = c.muw; r[IC_IM_WV2] = 0.5 * c.f / h->kappa2m[b]; r[IC_BETA] = 0.0; r[IC_U] = c.U; }
        else { r[IC_RE_A4] = c.nu4c; r[IC_RE_A2] = c.nuc; r[IC_RE_A0] = c.muc; r[IC_IM_WV2] = 0.0; r[IC_BETA] = 0.0; r[IC_U] = 0.0; }   // QGModel.py:452
    };
    // equal in every member: the keywords of the equation (niwqg_member_params), not the derived rows
    auto eq_shared = [&](int eq) {
        for (int b = 1; b < h->B; ++b) {
            const niwqg_member_params &c = h->mp[b], &c0 = h->mp[0];
            const bool same = eq == 0 ? (c.U == c0.U && c.nu4 == c0.nu4 && c.nu == c0.nu && c.mu == c0.mu && (!h->qg || c.beta == c0.beta))
                            : eq == 1 ? (c.U == c0.U && c.f == c0.f && c.N == c0.N && c.m == c0.m && c.nu4w == c0.nu4w &&
                                         c.nuw == c0.nuw && c.muw == c0.muw)
                                      : (c.nu4c == c0.nu4c && c.nuc == c0.nuc && c.muc == c0.muc);
            if (!same) return false;
        }
        return true;
    };
    auto init_eq = [&](int eq, TableSet& t, bool& pm) -> int {
        pm = !eq_shared(eq);
        const size_t tb = (pm ? B : 1) * tsz;
        DA(t.E, tb); DA(t.E2, tb); DA(t.Q, tb); DA(t.f0, tb); DA(t.fab, tb); DA(t.fc, tb);
        ia.t = t;
        ia.filtr = filtr_done ? nullptr : h->filtr;
        filtr_done = true;
        double r[IC_COUNT];
        eq_row(eq, 0, r);
        ia.re_a4 = r[IC_RE_A4]; ia.re_a2 = r[IC_RE_A2]; ia.re_a0 = r[IC_RE_A0]; ia.im_wv2 = r[IC_IM_WV2];
        ia.beta = r[IC_BETA]; ia.U = r[IC_U];
        ia.mc = nullptr;
        if (pm) {   // every member's row, filled in one launch (member = blockIdx.y)
            std::vector<double> rows(B * IC_COUNT);
            for (size_t b = 0; b < B; ++b) eq_row(eq, (int)b, &rows[b * IC_COUNT]);
            double* d = nullptr;
            DA(d, rows.size() * sizeof(double));
            CK(cudaMemcpyAsync(d, rows.data(), rows.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            ia.mc = d;
        }
        k_init_tables<<<dim3(NIWQG_PW_BLOCKS, pm ? h->B : 1), NIWQG_PW_THREADS, 0, h->stream>>>(ia);
        CK(cudaGetLastError());
        return 0;
    };
    {
        int r = 0;
        if (p.model != NIWQG_MODEL_YBJ) r = init_eq(0, h->tq, h->pm_q);
        if (!r && !h->qg) r = init_eq(1, h->tp, h->pm_p);
        else if (!r && p.passive_scalar) r = init_eq(2, h->tc, h->pm_c);
        if (r) return r;
    }
    // state
    DA(h->qh[0], ssz); DA(h->ph, ssz); DA(h->uv, fsz); DA(h->qs, fsz);
    DA(h->P1, fsz); DA(h->P2, fsz); DA(h->W, fsz);
    DA(h->rscratch, B * h->npts * sizeof(double));
    h->lane_stream[0] = h->stream;
    h->lane_comm[0] = h->comm;
    // measured: 7% at 512^2, nothing at 2048^2, slightly negative at 8192^2 (the step is a chain of dependent kernels,
    // ~5 us each whatever launches them; larger grids: kernels of 0.4-2 ms, the launch gaps a graph removes are noise)
    // -> small grids only
    h->use_graphs = (h->nranks == 1) && N <= 1024;
    if (h->split) {
        for (int o = 0; o < 3; ++o) DA(h->T[o], fsz);
        std::vector<cd> tw;
        build_twiddles(N / 2, tw);
        DA(h->tw_half, tw.size() * cb);
        CK(cudaMemcpyAsync(h->tw_half, tw.data(), tw.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        build_twiddles(N / 16, tw);
        DA(h->tw_m, tw.size() * cb);
        CK(cudaMemcpyAsync(h->tw_m, tw.data(), tw.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    if (h->col3) {
        DA(h->S3[0], fsz); DA(h->S3[1], fsz);
        std::vector<cd> tw3;
        build_twiddles(512, tw3);
        DA(h->tw_c3, tw3.size() * cb);
        CK(cudaMemcpyAsync(h->tw_c3, tw3.data(), tw3.size() * cb, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    CK(cudaStreamCreateWithFlags(&h->lane_stream[1], cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    if (h->nranks > 1) {
        DA(h->X, fsz); DA(h->Y, fsz);
        h->slab_panel = (N >= NIWQG_COL_M && h->nyl >= N / NIWQG_COL_M && h->ncl % 4 == 0) ? N / NIWQG_COL_M : 0;
        // (+4 KB behind the first receive buffer of a lane: the barrier flags, mapped by the peers with the buffer)
        for (int l = 0; l < niwqg_handle::NLANE; ++l) { DA(h->Yp[l][0], fsz + 4096); DA(h->Yp[l][1], fsz); DA(h->bar[l], 64); DA(h->Xl[l], fsz); }
        if (const char* e = getenv("NIWQG_SLAB_BARRIER")) h->flag_barrier = strcmp(e, "nccl") != 0;
        if (const char* e = getenv("NIWQG_SLAB_EXCHANGE")) h->exchange = (strcmp(e, "ce") == 0) ? 1 : 0;
        NK(g_nccl.CommSplit(h->comm, 0, h->rank, &h->lane_comm[1], nullptr));
    }
    if (p.model != NIWQG_MODEL_YBJ) { DA(h->qh[1], ssz); DA(h->y1q, ssz); DA(h->F0q, ssz); DA(h->Fabq, ssz); }
    if (!h->qg) {
        DA(h->phih[0], ssz); DA(h->phih[1], ssz); DA(h->y1p, ssz); DA(h->F0p, ssz); DA(h->Fabp, ssz);
        DA(h->phi, fsz); DA(h->phix, fsz); DA(h->phiy, fsz); DA(h->lapphi, fsz);
        if (h->flags & MF_HAS_LAP2) DA(h->lap2phi, fsz);
        if (h->flags & MF_WAVE_PV) DA(h->qwh, ssz);
        if (h->flags & MF_QL_ADV) DA(h->uvq, fsz);
    } else if (p.passive_scalar) {
        DA(h->chh[0], ssz); DA(h->chh[1], ssz); DA(h->y1c, ssz); DA(h->F0c, ssz); DA(h->Fabc, ssz);
    }
    if (B * h->npts * sizeof(cd) >= STAGED_BYTES) {
        DA(h->stage_in, B * h->npts * sizeof(cd));
        DA(h->stage_out[0], h->npts * sizeof(double));
        DA(h->stage_out[1], h->npts * sizeof(cd));
    }
    DA(h->part, B * NIWQG_PW_BLOCKS * 16 * sizeof(double));
    DA(h->sumsD, B * 16 * sizeof(double)); DA(h->sumsE, B * 16 * sizeof(double)); DA(h->sumsX, B * 16 * sizeof(double));
    DA(h->sumsI, B * 16 * sizeof(double));
    DA(h->scal, B * NIWQG_S_COUNT * sizeof(double)); DA(h->stagev, B * 24 * sizeof(double));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// the coefficient fields of p, as member parameters
static niwqg_member_params member_of(const niwqg_params& p) {
    niwqg_member_params c{};
    c.struct_size = sizeof(niwqg_member_params);
    c.U = p.U; c.f = p.f; c.N = p.N; c.m = p.m; c.nu = p.nu; c.nu4 = p.nu4; c.mu = p.mu;
    c.nuw = p.nuw; c.nu4w = p.nu4w; c.muw = p.muw; c.beta = p.beta; c.nu4c = p.nu4c; c.nuc = p.nuc; c.muc = p.muc;
    return c;
}

int niwqg_create(const niwqg_params* p, niwqg_handle** out) { return niwqg_create_ensemble(p, nullptr, out); }

int niwqg_create_ensemble(const niwqg_params* p, const niwqg_member_params* members, niwqg_handle** out) {
    if (!p || !out) { g_create_error = "null argument"; return -1; }
    *out = nullptr;
    if (p->struct_size != sizeof(niwqg_params)) {
        g_create_error = "niwqg_params.struct_size does not match this library (binding built against another header)";
        return -1;
    }
    const int N = p->nx;
    if (N < 32 || N > 8192 || (N & (N - 1))) { g_create_error = "nx must be a power of two in [32, 8192]"; return -1; }
    if (p->batch < 1) { g_create_error = "batch must be >= 1"; return -1; }
    if (p->model < NIWQG_MODEL_QG || p->model > NIWQG_MODEL_QL) { g_create_error = "unknown model"; return -1; }
    if (p->nranks > 1) {
        const int P = p->nranks;
        if ((P & (P - 1)) || N / P < 16 || p->rank < 0 || p->rank >= P) { g_create_error = "slab: nranks must be a power of two with nx/nranks >= 16, 0 <= rank < nranks"; return -1; }
        if (p->model == NIWQG_MODEL_QG) { g_create_error = "slab: QGModel (half spectrum) is single-GPU only"; return -1; }
        if (p->batch != 1) { g_create_error = "slab: batch must be 1 (ensembles shard whole members per GPU instead)"; return -1; }
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_create_error = "no CUDA device: niwqg_b200 has no CPU fallback";
        return -3;
    }
    if (members)
        for (int b = 0; b < p->batch; ++b)
            if (members[b].struct_size != sizeof(niwqg_member_params)) {
                g_create_error = "niwqg_member_params.struct_size does not match this library (binding built against another header)";
                return -1;
            }
    niwqg_handle* h = new niwqg_handle();
    h->p = *p;
    h->mp.assign(p->batch, member_of(*p));
    if (members) {
        for (int b = 0; b < p->batch; ++b) h->mp[b] = members[b];
        // the batch-1 paths (split / fused step, jacobians) and everything shared read p: member 0's coefficients
        const niwqg_member_params& c = members[0];
        h->p.U = c.U; h->p.f = c.f; h->p.N = c.N; h->p.m = c.m; h->p.nu = c.nu; h->p.nu4 = c.nu4; h->p.mu = c.mu;
        h->p.nuw = c.nuw; h->p.nu4w = c.nu4w; h->p.muw = c.muw; h->p.beta = c.beta;
        h->p.nu4c = c.nu4c; h->p.nuc = c.nuc; h->p.muc = c.muc;
    }
    int r = create_impl(h);
    if (r) { g_create_error = h->err; niwqg_destroy(h); return r; }
    *out = h;
    return 0;
}

int niwqg_nccl_unique_id(char* out128) {
    std::string err;
    int r = nccl_load(err);
    if (r) { g_create_error = err; return r; }
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return -5; }
    memcpy(out128, &id, sizeof id);
    return 0;
}

int niwqg_ipc_export(niwqg_handle* h, char* out, size_t bytes) {
    const int nb = niwqg_handle::NLANE * 2;
    if (bytes < nb * sizeof(cudaIpcMemHandle_t)) { h->err = "ipc_export: buffer too small"; return -1; }
    if (h->nranks <= 1) { h->err = "ipc_export: not a slab handle"; return -1; }
    CK(cudaSetDevice(h->p.device));
    memset(out, 0, bytes);
    for (int l = 0; l < niwqg_handle::NLANE; ++l)
        for (int b = 0; b < 2; ++b) {
            if (!h->Yp[l][b]) continue;
            cudaIpcMemHandle_t mh;
            CK(cudaIpcGetMemHandle(&mh, h->Yp[l][b]));
            memcpy(out + (l * 2 + b) * sizeof mh, &mh, sizeof mh);
        }
    return 0;
}

int niwqg_ipc_import(niwqg_handle* h, const char* all, size_t bytes_per_rank) {
    if (h->nranks <= 1 || h->nranks > 8) { h->err = "ipc_import: 2..8 ranks"; return -1; }
    CK(cudaSetDevice(h->p.device));
    for (int r = 0; r < h->nranks; ++r)
        for (int l = 0; l < niwqg_handle::NLANE; ++l)
            for (int b = 0; b < 2; ++b) {
                if (!h->Yp[l][b]) continue;
                if (r == h->rank) { h->peerY[l][b][r] = h->Yp[l][b]; continue; }
                cudaIpcMemHandle_t mh;
                memcpy(&mh, all + (size_t)r * bytes_per_rank + (l * 2 + b) * sizeof mh, sizeof mh);
                void* ptr = nullptr;
                CK(cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess));
                h->peerY[l][b][r] = (cd*)ptr;
            }
    h->p2p = true;
    return 0;
}

int niwqg_ipc_disable(niwqg_handle* h) {   // back to the NCCL all-to-all exchange (e.g. when a peer could not map the buffers)
    CK(cudaSetDevice(h->p.device));
    CK(cudaStreamSynchronize(h->stream));
    h->p2p = false;
    return 0;
}

int niwqg_sync(niwqg_handle* h) {
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->copy_stream));
    CK(cudaStreamSynchronize(h->copy_out));
    return 0;
}

long long niwqg_launch_count(const niwqg_handle* h) { return h->launches; }
void* niwqg_stream(const niwqg_handle* h) { return (void*)h->stream; }

static int ke_qg_family(niwqg_handle* h) {   // 0.5*spec_var(wv*ph) (Kernel.py:600-602) -> sumsX via k_spec_sums
    SpecSumArgs sa{};
    sa.g = h->g; sa.ph = h->ph; sa.qh = h->qh[h->cq]; sa.qwh = h->qwh;
    sa.phih = (h->flags & MF_HAS_LAP2) ? h->phih[h->cp] : nullptr;
    k_spec_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(sa, h->part);
    CK(cudaGetLastError());
    h->launches++;
    FIN(SS_COUNT, h->sumsX);
    return 0;
}

// scal[m][slot] = factor * sums[m][idx]; mfactor != null: the member's factor mfactor[m * MC_COUNT] instead
__global__ void k_set_scalar_from_sum(double* scal, int slot, const double* sums, int K, int idx, double factor,
                                      const double* mfactor = nullptr) {
    const int m = blockIdx.x;
    if (mfactor) factor = mfactor[(size_t)m * MC_COUNT];
    if (threadIdx.x == 0) scal[(size_t)m * NIWQG_S_COUNT + slot] = factor * sums[(size_t)m * K + idx];
}

// set_q once the physical q sits in h->rscratch in the device layout
static int seed_q(niwqg_handle* h) {
    const size_t n = (size_t)h->B * h->npts;
    const double M2 = h->Mg * h->Mg;
    if (h->qg) {
        // qh = rfft2(q): full c2c of the real field, keep columns 0..N/2 (QGModel.py:516-518)
        FFT(h->rscratch, h->W, false, PRO_REAL_IN, h->B);
        k_qg_take_half<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->W, h->qh[h->cq], h->N, h->nk);
        CK(cudaGetLastError());
        h->launches++;
        int r = qg_expand_and_invert(h, h->qh[h->cq]);
        if (r) return r;
        // physical q carried for ep_psi (stale-q semantics) is the user's array: qs.x <- q
        k_qg_set_q_real<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->rscratch, h->qs, h->npts);
        CK(cudaGetLastError());
        h->launches++;
        QgSumArgs sa{};
        sa.N = h->N; sa.nk = h->nk; sa.dk = h->dk; sa.qh = h->qh[h->cq]; sa.ch = nullptr;
        k_qg_spec_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(sa, h->part);
        CK(cudaGetLastError());
        h->launches++;
        FIN(QS_COUNT, h->sumsX);
        k_set_scalar_from_sum<<<h->B, 32, 0, h->stream>>>(h->scal, NIWQG_S_KE, h->sumsX, QS_COUNT, QS_KE, 0.5 / M2);
        CK(cudaGetLastError());
        h->launches += 1;
        h->q_set = true;
        return 0;
    }
    FFT(h->rscratch, h->qh[h->cq], false, PRO_REAL_IN, h->B);
    if (h->flags & MF_WAVE_PV) {   // jacobian_phic_phi refreshes phix, phiy from the current phih (CoupledModel.py:70)
        int r = wave_fields(h, false, true, false);
        if (r) return r;
    }
    int r = invert_family(h);
    if (r) return r;
    if (h->flags & MF_YBJ) {
        // YBJ._invert does not touch q: q (and q_psi) stay the user's array (YBJModel.py:141-146, Kernel.py:530)
        k_real_to_cplx<<<pw_grid(h).x, NIWQG_PW_THREADS, 0, h->stream>>>(h->rscratch, h->qs, n);
        CK(cudaGetLastError());
        h->launches++;
    }
    r = ke_qg_family(h);
    if (r) return r;
    k_set_scalar_from_sum<<<h->B, 32, 0, h->stream>>>(h->scal, NIWQG_S_KE, h->sumsX, SS_COUNT, SS_KE, 0.5 / M2);
    CK(cudaGetLastError());
    h->launches++;
    h->q_set = true;
    return 0;
}

static int pe_niw_refresh(niwqg_handle* h, double* sums_out) {   // Kernel.py:608-611
    int r = wave_fields(h, false, true, false);
    if (r) return r;
    k_grad2_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phix, h->phiy, h->npts, h->part);
    CK(cudaGetLastError());
    h->launches++;
    FIN(1, sums_out);
    return 0;
}

__global__ void k_phi2_sum(const cd* __restrict__ phi, size_t npts, double* partials) {
    const size_t mb = (size_t)blockIdx.y * npts;
    double s[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
        const cd p = phi[mb + i];
        s[0] += p.x * p.x + p.y * p.y;
    }
    block_reduce_store<1>(s, partials);
}

int niwqg_set_q(niwqg_handle* h, const double* q, int on_device) {
    CK(cudaSetDevice(h->p.device));
    const size_t n = (size_t)h->B * h->npts;
    { int r0 = q ? upload_phys<double>(h, q, h->rscratch, n, on_device) : upload_staged<double>(h, 0, h->rscratch, n); if (r0) return r0; }
    return seed_q(h);
}

int niwqg_stage_q(niwqg_handle* h, const double* q) {
    CK(cudaSetDevice(h->p.device));
    return stage_upload(h, 0, q, (size_t)h->B * h->npts * sizeof(double));
}

// set_phi once the physical phi sits in h->phi in the device layout
static int seed_phi(niwqg_handle* h) {
    FFT(h->phi, h->phih[h->cp], false, PRO_NONE, h->B);
    int r = pe_niw_refresh(h, h->sumsX);
    if (r) return r;
    const double M = h->Mg;
    k_set_scalar_from_sum<<<h->B, 32, 0, h->stream>>>(h->scal, NIWQG_S_PW, h->sumsX, 1, 0, 0.0, h->mcoef + MC_PW_SEED);
    CK(cudaGetLastError());
    k_phi2_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phi, h->npts, h->part);
    CK(cudaGetLastError());
    FIN(1, h->sumsX);
    k_set_scalar_from_sum<<<h->B, 32, 0, h->stream>>>(h->scal, NIWQG_S_KW, h->sumsX, 1, 0, 0.5 / M);
    CK(cudaGetLastError());
    h->launches += 3;
    // lapphi follows phih (the reference recomputes it at every _calc_energy_conversion, Kernel.py:685)
    if (!(h->flags & MF_SPEC_BUDGET)) {
        r = wave_fields(h, false, false, true);
        if (r) return r;
    }
    h->phi_set = true;
    return 0;
}

int niwqg_set_phi(niwqg_handle* h, const double* phi, int on_device) {
    if (h->qg) { h->err = "set_phi: QGModel has no wave field"; return -1; }
    CK(cudaSetDevice(h->p.device));
    const size_t n = (size_t)h->B * h->npts;
    { int r0 = phi ? upload_phys<cd>(h, phi, h->phi, n, on_device) : upload_staged<cd>(h, 1, h->phi, n); if (r0) return r0; }
    return seed_phi(h);
}

int niwqg_stage_phi(niwqg_handle* h, const double* phi) {
    if (h->qg) { h->err = "stage_phi: QGModel has no wave field"; return -1; }
    CK(cudaSetDevice(h->p.device));
    return stage_upload(h, 1, phi, (size_t)h->B * h->npts * sizeof(cd));
}

int niwqg_ic(niwqg_handle* h, int kind, const double* prm, int nprm, const double* rand01) {
    CK(cudaSetDevice(h->p.device));
    const IcGeom g{h->N, h->nyl, h->rank * h->nyl, h->deintC, h->deintM, h->p.L};
    const dim3 grid = pw_grid(h);
    auto need = [&](int n) { if (nprm < n) { h->err = "ic: too few parameters"; return false; } return true; };
    switch (kind) {
        case NIWQG_IC_LAMB_DIPOLE: {
            if (!need(2)) return -1;
            k_ic_lamb<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(g, prm[0], prm[1], h->rscratch);
            CK(cudaGetLastError());
            h->launches++;
            return seed_q(h);
        }
        case NIWQG_IC_WAVEPACKET: case NIWQG_IC_PLANEWAVE: case NIWQG_IC_UNIFORM: {
            if (h->qg) { h->err = "ic: QGModel has no wave field"; return -1; }
            double k = 0, l = 0, R = 1, x0 = 0, y0 = 0, phase = 0;
            if (kind == NIWQG_IC_WAVEPACKET) { if (!need(5)) return -1; k = prm[0]; l = prm[1]; R = prm[2]; x0 = prm[3]; y0 = prm[4]; }
            else if (kind == NIWQG_IC_PLANEWAVE) { if (!need(3)) return -1; k = prm[0]; l = prm[1]; phase = prm[2]; }
            else { if (!need(2)) return -1; k = prm[0]; l = prm[1]; }
            k_ic_phi<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(g, kind - NIWQG_IC_WAVEPACKET, k, l, R, x0, y0, phase, h->phi);
            CK(cudaGetLastError());
            h->launches++;
            return seed_phi(h);
        }
        case NIWQG_IC_MCWILLIAMS: case NIWQG_IC_DANIOUX: {
            // random red spectrum (InitialConditions.py:4-41, :43-75) through the model's own transforms
            if (!need(3)) return -1;
            if (h->qg || h->nranks > 1 || h->B != 1) { h->err = "ic: random spectra need a single-GPU, single-member c2c model"; return -1; }
            const int N = h->N;
            const double M2 = h->Mg * h->Mg;
            const double* rnd = nullptr;
            if (rand01) {       // the caller's uniform numbers (np.random.rand(N, N)): parity with the host generator
                CK(cudaMemcpyAsync(h->P2, rand01, h->npts * sizeof(double), cudaMemcpyHostToDevice, h->stream));
                rnd = (const double*)h->P2;
            }
            k_ic_spectrum<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(N, h->dk, kind == NIWQG_IC_MCWILLIAMS ? 0 : 1, prm[0], rnd,
                                                                    (unsigned long long)prm[2], h->P1);
            CK(cudaGetLastError());
            FFT(h->P1, h->P1, true, PRO_NONE, 1);                 // ph = fft(ifft(ph).real)
            k_ic_real<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(h->P1, h->npts);
            CK(cudaGetLastError());
            FFT(h->P1, h->P1, false, PRO_NONE, 1);
            k_ic_energy<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(N, h->dk, h->P1, h->part);
            CK(cudaGetLastError());
            FIN(1, h->sumsX);
            k_ic_scale<<<grid, NIWQG_PW_THREADS, 0, h->stream>>>(N, h->dk, prm[1], M2, h->sumsX, h->P1);
            CK(cudaGetLastError());
            FFT(h->P1, h->P1, true, PRO_NONE, 1, EPI_REAL_OUT, h->rscratch);    // q = ifft(-wv2 pih).real, device layout
            h->launches += 4;
            return seed_q(h);
        }
    }
    h->err = "ic: unknown kind";
    return -1;
}

int niwqg_set_c(niwqg_handle* h, const double* c, int on_device) {
    if (!h->qg || !h->p.passive_scalar) { h->err = "set_c: needs QGModel(passive_scalar=True)"; return -1; }
    CK(cudaSetDevice(h->p.device));
    const size_t n = (size_t)h->B * h->npts;
    { int r0 = upload_phys<double>(h, c, h->rscratch, n, on_device); if (r0) return r0; }
    FFT(h->rscratch, h->W, false, PRO_REAL_IN, h->B);
    k_qg_take_half<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->W, h->chh[h->cc], h->N, h->nk);
    CK(cudaGetLastError());
    QgSumArgs sa{};
    sa.N = h->N; sa.nk = h->nk; sa.dk = h->dk; sa.qh = h->qh[h->cq]; sa.ch = h->chh[h->cc];
    k_qg_spec_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(sa, h->part);
    CK(cudaGetLastError());
    FIN(QS_COUNT, h->sumsX);
    const double M2 = h->Mg * h->Mg;
    k_set_scalar_from_sum<<<h->B, 32, 0, h->stream>>>(h->scal, NIWQG_S_CVAR, h->sumsX, QS_COUNT, QS_C2, 1.0 / M2);
    CK(cudaGetLastError());
    h->launches += 3;
    // physical c carried in W.x is the user's array
    k_real_to_cplx<<<pw_grid(h).x, NIWQG_PW_THREADS, 0, h->stream>>>(h->rscratch, h->W, n);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

int niwqg_step(niwqg_handle* h, int nsteps) {
    CK(cudaSetDevice(h->p.device));
    if (!h->q_set || (!h->qg && !h->phi_set)) {
        // the reference raises AttributeError (u, v, phix... undefined) when stepping an unseeded model
        h->err = "step: set_q" + std::string(h->qg ? "" : " and set_phi") + " must be called first";
        return -1;
    }
    for (int s = 0; s < nsteps; ++s) {
        if (h->use_graphs && !h->prof && h->direct_steps >= 2) {
            niwqg_handle::StepGraph& g = h->graphs[h->cq * 4 + h->cp * 2 + h->cc];
            if (!g.exec) {
                // capture one step issued from this buffer parity (host-side bookkeeping runs, kernels are recorded)
                const long long l0 = h->launches;
                cudaGraph_t graph = nullptr;
                CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
                int r = h->qg ? step_qg(h) : step_family(h);
                cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
                if (r) { if (graph) cudaGraphDestroy(graph); return r; }
                CK(ce);
                CK(cudaGraphInstantiate(&g.exec, graph, 0));
                CK(cudaGraphDestroy(graph));
                g.cq = h->cq; g.cp = h->cp; g.cc = h->cc; g.launches = h->launches - l0;
            } else {
                h->cq = g.cq; h->cp = g.cp; h->cc = g.cc; h->launches += g.launches;
            }
            CK(cudaGraphLaunch(g.exec, h->stream));
            continue;
        }
        int r = h->qg ? step_qg(h) : step_family(h);
        if (r) return r;
        h->direct_steps++;
    }
    return 0;
}

int niwqg_time_steps(niwqg_handle* h, int nsteps, float* ms) {
    CK(cudaSetDevice(h->p.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaEventRecord(h->ev0, h->stream));
    int r = niwqg_step(h, nsteps);
    if (r) return r;
    CK(cudaEventRecord(h->ev1, h->stream));
    CK(cudaEventSynchronize(h->ev1));
    CK(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return 0;
}

int niwqg_profile(niwqg_handle* h, int enable, double* ms_out, long long* count_out) {
    CK(cudaSetDevice(h->p.device));
    CK(cudaStreamSynchronize(h->stream));
    if (ms_out && count_out) {
        for (int k = 0; k < PK_COUNT; ++k) { ms_out[k] = 0.0; count_out[k] = 0; }
        for (auto& r : h->prof_recs) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, r.a, r.b));
            ms_out[r.kind] += ms;
            count_out[r.kind] += 1;
        }
    }
    h->prof_recs.clear();
    h->prof_used = 0;
    h->prof = enable != 0;
    return 0;
}

int niwqg_get_scalars(niwqg_handle* h, double* out) {
    CK(cudaSetDevice(h->p.device));
    CK(cudaMemcpyAsync(out, h->scal, (size_t)h->B * NIWQG_S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_status(niwqg_handle* h, double* out) {
    CK(cudaSetDevice(h->p.device));
    std::vector<double> sx((size_t)h->B * 16), tmp((size_t)h->B * 16);
    const double M = h->Mg, M2 = M * M;
    if (h->qg) {
        // ke_qg and cfl from the current (qh, ph): u, v are refreshed from ph (QGModel.py:571-629)
        int r = qg_expand_and_invert(h, h->qh[h->cq]);
        if (r) return r;
        QgSumArgs sa{};
        sa.N = h->N; sa.nk = h->nk; sa.dk = h->dk; sa.qh = h->qh[h->cq]; sa.ch = nullptr;
        k_qg_spec_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(sa, h->part);
        CK(cudaGetLastError());
        FIN(QS_COUNT, h->sumsX);
        CK(cudaMemcpyAsync(sx.data(), h->sumsX, (size_t)h->B * QS_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        k_cfl_max<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->uv, nullptr, h->npts, h->part);
        CK(cudaGetLastError());
        FIN(1, h->sumsD, 1);
        CK(cudaMemcpyAsync(tmp.data(), h->sumsD, (size_t)h->B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->launches += 2;
        for (int m = 0; m < h->B; ++m) {
            out[m * 4 + 0] = 0.5 * sx[(size_t)m * QS_COUNT + QS_KE] / M2;
            out[m * 4 + 1] = 0.0; out[m * 4 + 2] = 0.0;
            out[m * 4 + 3] = tmp[m] * h->p.dt / h->dx;
        }
        return 0;
    }
    // every result is copied into pinned host scratch in stream order (the next kernel may reuse sumsX): ONE sync
    const int B = h->B;
    double *p_ke = h->pin, *p_kw = p_ke + (size_t)B * SS_COUNT, *p_pw = p_kw + B, *p_cfl = p_pw + B;
    int r = ke_qg_family(h);
    if (r) return r;
    CK(cudaMemcpyAsync(p_ke, h->sumsX, (size_t)B * SS_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    k_phi2_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phi, h->npts, h->part);
    CK(cudaGetLastError());
    FIN(1, h->sumsX);
    CK(cudaMemcpyAsync(p_kw, h->sumsX, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    r = pe_niw_refresh(h, h->sumsX);
    if (r) return r;
    CK(cudaMemcpyAsync(p_pw, h->sumsX, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    k_cfl_max<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->uv, h->phi, h->npts, h->part);
    CK(cudaGetLastError());
    FIN(1, h->sumsX, 1);
    CK(cudaMemcpyAsync(p_cfl, h->sumsX, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->launches += 2;
    for (int m = 0; m < B; ++m) {
        out[m * 4 + 0] = 0.5 * p_ke[(size_t)m * SS_COUNT + SS_KE] / M2;
        out[m * 4 + 1] = 0.5 * p_kw[m] / M;
        out[m * 4 + 2] = 0.25 * p_pw[m] / M / h->kappa2m[m];
        out[m * 4 + 3] = p_cfl[m] * h->p.dt / h->dx;
    }
    return 0;
}

int niwqg_diagnostics(niwqg_handle* h, double* out) {
    CK(cudaSetDevice(h->p.device));
    const int B = h->B;
    const double M = h->Mg, M2 = M * M;
    std::vector<double> sc((size_t)B * NIWQG_S_COUNT), sd((size_t)B * 16), ss((size_t)B * 16), sg((size_t)B), s3((size_t)B * 3),
        sq((size_t)B);
    if (h->qg) {
        // _calc_derived_fields + registry of QGModel.py:632-737
        const bool ps = h->p.passive_scalar != 0;
        QgSumArgs sa{};
        sa.N = h->N; sa.nk = h->nk; sa.dk = h->dk; sa.qh = h->qh[h->cq]; sa.ch = ps ? h->chh[h->cc] : nullptr;
        sa.qs = h->qs;
        k_qg_spec_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(sa, h->part);
        CK(cudaGetLastError());
        FIN(QS_COUNT, h->sumsX);
        k_qg_q2_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->qs, h->npts, h->part);
        CK(cudaGetLastError());
        FIN(1, h->sumsD);
        h->launches += 2;
        CK(cudaMemcpyAsync(ss.data(), h->sumsX, (size_t)B * QS_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(sq.data(), h->sumsD, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(sc.data(), h->scal, sc.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        std::vector<double> gam((size_t)B, 0.0);
        if (ps) {
            // Gamma_c = 2*mean(lapc * irfft2(jacobian_psi_c))  (QGModel.py:731)
            int r = qg_gamma_c(h);
            if (r) return r;
            CK(cudaMemcpyAsync(sg.data(), h->sumsD, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            for (int m = 0; m < B; ++m) gam[m] = 2.0 * sg[m] / M2;
        }
        for (int m = 0; m < B; ++m) {
            double* o = out + (size_t)m * NIWQG_S_COUNT;
            const double* s = &ss[(size_t)m * QS_COUNT];
            for (int k = 0; k < NIWQG_S_COUNT; ++k) o[k] = 0.0;
            o[NIWQG_S_KE] = sc[(size_t)m * NIWQG_S_COUNT + NIWQG_S_KE];
            o[NIWQG_S_CVAR] = ps ? sc[(size_t)m * NIWQG_S_COUNT + NIWQG_S_CVAR] : 0.0;
            o[NIWQG_S_KE_QG] = 0.5 * s[QS_KE] / M2;
            o[NIWQG_S_ENS] = 0.5 * sq[m] / M;
            const niwqg_member_params& p = h->mp[m];
            o[NIWQG_S_EP_PSI] = p.nu4 * s[QS_QLAP2PSI] / M2 - p.nu * s[QS_PLAPQ] / M2 + p.mu * s[QS_PQ] / M2;
            o[NIWQG_S_CHI_Q] = -p.nu4 * s[QS_CHIQ] / M2;
            if (ps) {
                const double C2 = s[QS_C2] / M2, gradC2 = s[QS_GRADC2] / M2, lapc2 = s[QS_LAPC2] / M2, lap2clapc = s[QS_LAP2CLAPC] / M2;
                o[NIWQG_S_C2] = C2; o[NIWQG_S_GRADC2] = gradC2; o[NIWQG_S_GAMMA_C] = gam[m];
                o[NIWQG_S_EP_C] = -2 * p.nu4c * lapc2 - 2 * p.nu * gradC2 - 2 * p.muc * C2;          // QGModel.py:595-598
                o[NIWQG_S_CHI_C] = 2 * p.nu4c * lap2clapc - 2 * p.nu * lapc2 - 2 * p.muc * gradC2;  // QGModel.py:600-604
            }
        }
        return 0;
    }
    // ---- kernel family: _calc_energy_conversion on the current state (stale phix/phiy for UnCoupled, F6)
    // results land in pinned host scratch in stream order: one synchronisation for the whole tick
    double* p_ss = h->pin;                                    // [B][SS_COUNT]
    double* p_sd = p_ss + (size_t)B * 16;                     // [B][SD_COUNT]
    double* p_sc = p_sd + (size_t)B * 16;                     // [B][NIWQG_S_COUNT]
    double* p_s3 = p_sc + (size_t)B * NIWQG_S_COUNT;          // [B][3]
    double* p_sg = p_s3 + (size_t)B * 3;                      // [B]
    const bool ybj = (h->flags & MF_YBJ) != 0;
    if (ybj || (h->flags & MF_SPEC_BUDGET)) {
        // lapphi = ifft(-wv2*phih) is recomputed by every _calc_energy_conversion (Kernel.py:685); during a step the
        // spectral-budget models never transform it, so the tick does
        int r0 = wave_fields(h, false, false, true);
        if (r0) return r0;
    }
    PhysArgs pa = phys_args(h, MF_NO_WRITE);
    pa.flags &= ~(MF_YBJ | MF_SPEC_BUDGET);   // the tick evaluates every budget term separately, in physical space
    { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
    CK(cudaGetLastError());
    FIN(SD_COUNT, h->sumsD);
    int r = ke_qg_family(h);      // spectral sums -> sumsX
    if (r) return r;
    // budget terms of the tick use Parseval sums from k_spec_sums: copy into the SE layout
    CK(cudaMemcpyAsync(p_ss, h->sumsX, (size_t)B * SS_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(p_sd, h->sumsD, (size_t)B * SD_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(p_sc, h->scal, (size_t)B * NIWQG_S_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    // conc_niw second pass (centred sums)
    k_qpsi_sum<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->qs, h->npts, h->part);
    CK(cudaGetLastError());
    FIN(1, h->sumsE);
    k_conc_sums<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phi, h->qs, h->npts, h->sumsD, h->sumsE, h->part);
    CK(cudaGetLastError());
    FIN(3, h->sumsE);
    CK(cudaMemcpyAsync(p_s3, h->sumsE, (size_t)B * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    h->launches += 3;
    // pe_niw: refreshes phix, phiy (Kernel.py:608-611) -- after the conversion terms, as in the registry order
    r = pe_niw_refresh(h, h->sumsE);
    if (r) return r;
    CK(cudaMemcpyAsync(p_sg, h->sumsE, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int m = 0; m < B; ++m) {
        const niwqg_member_params& p = h->mp[m];
        const double hslash = h->hslashm[m], kappa2 = h->kappa2m[m];
        double* o = out + (size_t)m * NIWQG_S_COUNT;
        const double* D = &p_sd[(size_t)m * SD_COUNT];
        const double* S = &p_ss[(size_t)m * SS_COUNT];
        for (int k = 0; k < NIWQG_S_COUNT; ++k) o[k] = 0.0;
        o[NIWQG_S_KE] = p_sc[(size_t)m * NIWQG_S_COUNT + NIWQG_S_KE];
        o[NIWQG_S_PW] = p_sc[(size_t)m * NIWQG_S_COUNT + NIWQG_S_PW];
        o[NIWQG_S_KW] = p_sc[(size_t)m * NIWQG_S_COUNT + NIWQG_S_KW];
        o[NIWQG_S_GAMMA1] = 0.5 * 0.5 * hslash * (D[SD_G1] / M) / p.f;
        o[NIWQG_S_GAMMA2] = 0.5 * hslash * (D[SD_G2] / M) / p.f;
        o[NIWQG_S_XI1] = (D[SD_X1] / M) / p.f;
        o[NIWQG_S_XI2] = (D[SD_X2] / M) / p.f;
        const double ar = D[SD_PHI_R] / M, ai = D[SD_PHI_I] / M, br = D[SD_QPC_R] / M, bi = D[SD_QPC_I] / M;
        o[NIWQG_S_PI] = 0.5 * (ar * bi + ai * br);
        o[NIWQG_S_KE_QG] = 0.5 * S[SS_KE] / M2;
        o[NIWQG_S_ENS] = 0.5 * D[SD_Q2] / M;
        o[NIWQG_S_KE_NIW] = 0.5 * D[SD_PHI2] / M;
        o[NIWQG_S_CKE_NIW] = 0.5 * (ar * ar + ai * ai);
        o[NIWQG_S_IKE_NIW] = o[NIWQG_S_KE_NIW] - o[NIWQG_S_CKE_NIW];
        const double grad2 = p_sg[m] / M;     // refreshed phix, phiy
        o[NIWQG_S_PE_NIW] = 0.25 * grad2 / kappa2;
        const double* c3 = &p_s3[(size_t)m * 3];
        o[NIWQG_S_CONC] = (c3[0] / M) / sqrt(c3[1] / M) / sqrt(c3[2] / M);
        o[NIWQG_S_SKEW] = (D[SD_QP3] / M) / pow(D[SD_QP2] / M, 1.5);
        const double lap2m = D[SD_LAP2] / M, phi2m = D[SD_PHI2] / M;
        o[NIWQG_S_EP_PHI] = -p.nu4w * lap2m - p.nuw * grad2 - p.muw * phi2m;
        if (ybj)   // YBJ never defines p (zeros, YBJModel.py:44): only the q*lap2psi term survives
            o[NIWQG_S_EP_PSI] = p.nu4 * S[SS_QLAP2PSI] / M2;
        else
            o[NIWQG_S_EP_PSI] = p.nu4 * S[SS_QLAP2PSI] / M2 - p.nu * S[SS_PLAPQ] / M2 + p.mu * S[SS_PQ] / M2;
        o[NIWQG_S_CHI_Q] = -p.nu4 * S[SS_CHIQ] / M2;
        o[NIWQG_S_CHI_PHI] = -0.5 * p.nu4w * (S[SS_WV6PHI] / M2) / kappa2 - 0.5 * p.nuw * lap2m / kappa2 -
                             0.5 * p.muw * grad2 / kappa2;
        if (h->flags & MF_WAVE_PV) {
            o[NIWQG_S_KE_QG_Q] = 0.5 * S[SS_KEQ] / M2;
            o[NIWQG_S_KE_QG_W] = 0.5 * S[SS_KEW] / M2;
            o[NIWQG_S_KE_QG_QW] = S[SS_KEQW] / M2;
        }
    }
    return 0;
}

size_t niwqg_field_bytes(const niwqg_handle* h, int field) {
    const size_t r = h->npts * sizeof(double), c = h->npts * sizeof(cd), s = h->nspec * sizeof(cd);
    switch (field) {
        case NIWQG_F_Q: case NIWQG_F_P: case NIWQG_F_U: case NIWQG_F_V: case NIWQG_F_QW: case NIWQG_F_QPSI: case NIWQG_F_C:
            return r;
        case NIWQG_F_PHI: case NIWQG_F_PHIX: case NIWQG_F_PHIY: case NIWQG_F_LAPPHI:
        case NIWQG_F_UV: case NIWQG_F_QS: case NIWQG_F_LAP2PHI: case NIWQG_F_UVQ: return c;
        case NIWQG_F_FILTR: return h->nspec * sizeof(double);
        default: return s;
    }
}

static int get_field_impl(niwqg_handle* h, int field, int member, void* dst, size_t bytes, int on_device, bool async) {
    CK(cudaSetDevice(h->p.device));
    if (member < 0 || member >= h->B) { h->err = "get_field: bad member"; return -1; }
    if (bytes != niwqg_field_bytes(h, field)) { h->err = "get_field: size mismatch"; return -1; }
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t mo = (size_t)member * h->npts, so = (size_t)member * h->nspec;
    const void* src = nullptr;
    auto real_of = [&](const cd* f, int which) -> int {
        if (!f) { h->err = "get_field: field not defined for this model"; return -1; }
        k_extract_real<<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>(f + mo, h->rscratch, h->npts, which);
        CK(cudaGetLastError());
        h->launches++;
        src = h->rscratch;
        return 0;
    };
    int r = 0;
    switch (field) {
        case NIWQG_F_Q: r = real_of(h->qs, 0); break;
        case NIWQG_F_QW: r = real_of(h->qs, 1); break;
        case NIWQG_F_QPSI: r = real_of(h->qs, 2); break;
        case NIWQG_F_U: r = real_of(h->uv, 0); break;
        case NIWQG_F_V: r = real_of(h->uv, 1); break;
        case NIWQG_F_C: r = real_of(h->p.passive_scalar ? h->W : nullptr, 0); break;
        case NIWQG_F_P: {
            // p = Re ifft(ph): on demand, one member, through scratch P1
            if (h->qg) {
                QgExpand1Args ea{};
                ea.N = h->N; ea.nk = h->nk; ea.dk = h->dk; ea.in = h->ph + so; ea.out = h->P1; ea.mode = QGX_PLAIN;
                { PROF(PK_SPEC); k_qg_expand1<<<dim3(NIWQG_PW_BLOCKS, 1), NIWQG_PW_THREADS, 0, h->stream>>>(ea); }
                CK(cudaGetLastError());
                h->launches++;
                FFT(h->P1, h->P1, true, PRO_NONE, 1, EPI_REAL_OUT, h->rscratch);
            } else {
                FFT(h->ph + so, h->P1, true, PRO_NONE, 1, EPI_REAL_OUT, h->rscratch);
            }
            src = h->rscratch;
        } break;
        case NIWQG_F_QH: src = h->qh[h->cq] + so; break;
        case NIWQG_F_PH: src = h->ph + so; break;
        case NIWQG_F_PHI: src = h->phi ? h->phi + mo : nullptr; break;
        case NIWQG_F_PHIH: src = h->phih[h->cp] ? h->phih[h->cp] + so : nullptr; break;
        case NIWQG_F_PHIX: src = h->phix ? h->phix + mo : nullptr; break;
        case NIWQG_F_PHIY: src = h->phiy ? h->phiy + mo : nullptr; break;
        case NIWQG_F_LAPPHI:
            if (h->lapphi && (h->flags & MF_SPEC_BUDGET)) {   // not carried during steps: evaluate from the current phih
                int r0 = wave_fields(h, false, false, true);
                if (r0) return r0;
            }
            src = h->lapphi ? h->lapphi + mo : nullptr;
            break;
        case NIWQG_F_UV: src = h->uv + mo; break;
        case NIWQG_F_QS: src = h->qs + mo; break;
        case NIWQG_F_LAP2PHI: src = h->lap2phi ? h->lap2phi + mo : nullptr; break;
        case NIWQG_F_UVQ: src = h->uvq ? h->uvq + mo : nullptr; break;
        case NIWQG_F_QWH: src = h->qwh ? h->qwh + so : nullptr; break;
        case NIWQG_F_CH: src = h->chh[h->cc] ? h->chh[h->cc] + so : nullptr; break;
        case NIWQG_F_FILTR: src = h->filtr; break;
        case NIWQG_F_EXPCH: src = h->tq.E + (h->pm_q ? so : 0); break;
        case NIWQG_F_EXPCH_H: src = h->tq.E2 + (h->pm_q ? so : 0); break;
        case NIWQG_F_QHCOEF: src = h->tq.Q + (h->pm_q ? so : 0); break;
        case NIWQG_F_F0: src = h->tq.f0 + (h->pm_q ? so : 0); break;
        case NIWQG_F_FAB: src = h->tq.fab + (h->pm_q ? so : 0); break;
        case NIWQG_F_FC: src = h->tq.fc + (h->pm_q ? so : 0); break;
        case NIWQG_F_EXPCHW: src = h->tp.E + (h->pm_p ? so : 0); break;
        case NIWQG_F_EXPCH_HW: src = h->tp.E2 + (h->pm_p ? so : 0); break;
        case NIWQG_F_QHWCOEF: src = h->tp.Q + (h->pm_p ? so : 0); break;
        case NIWQG_F_F0W: src = h->tp.f0 + (h->pm_p ? so : 0); break;
        case NIWQG_F_FABW: src = h->tp.fab + (h->pm_p ? so : 0); break;
        case NIWQG_F_FCW: src = h->tp.fc + (h->pm_p ? so : 0); break;
        case NIWQG_F_EXPCHC: src = h->tc.E + (h->pm_c ? so : 0); break;
        case NIWQG_F_EXPCH_HC: src = h->tc.E2 + (h->pm_c ? so : 0); break;
        case NIWQG_F_QHCCOEF: src = h->tc.Q + (h->pm_c ? so : 0); break;
        case NIWQG_F_F0C: src = h->tc.f0 + (h->pm_c ? so : 0); break;
        case NIWQG_F_FABC: src = h->tc.fab + (h->pm_c ? so : 0); break;
        case NIWQG_F_FCC: src = h->tc.fc + (h->pm_c ? so : 0); break;
        default: h->err = "get_field: unknown field"; return -1;
    }
    if (r) return r;
    if (!src) { h->err = "get_field: field not defined for this model"; return -1; }
    switch (field) {   // physical fields leave in natural x order
        case NIWQG_F_Q: case NIWQG_F_QW: case NIWQG_F_QPSI: case NIWQG_F_U: case NIWQG_F_V: case NIWQG_F_C: case NIWQG_F_P:
            r = download_phys<double>(h, (const double*)src, dst, h->npts, on_device, (double*)h->P2, async);
            break;
        case NIWQG_F_PHI: case NIWQG_F_PHIX: case NIWQG_F_PHIY: case NIWQG_F_LAPPHI:
        case NIWQG_F_UV: case NIWQG_F_QS: case NIWQG_F_LAP2PHI: case NIWQG_F_UVQ:
            r = download_phys<cd>(h, (const cd*)src, dst, h->npts, on_device, h->P2, async);
            break;
        default:
            CK(cudaMemcpyAsync(dst, src, bytes, kind, h->stream));
            CK(cudaStreamSynchronize(h->stream));
    }
    return r;
}

int niwqg_get_field(niwqg_handle* h, int field, int member, void* dst, size_t bytes, int on_device) {
    return get_field_impl(h, field, member, dst, bytes, on_device, false);
}

int niwqg_get_field_async(niwqg_handle* h, int field, int member, void* dst, size_t bytes) {
    return get_field_impl(h, field, member, dst, bytes, 0, true);
}

int niwqg_wait_transfers(niwqg_handle* h) {
    CK(cudaSetDevice(h->p.device));
    CK(cudaStreamSynchronize(h->copy_stream));
    CK(cudaStreamSynchronize(h->copy_out));
    return 0;
}

// ---- checkpoint / exact restart: the state is every buffer a step (or the attribute and diagnostics reads that follow
// it) reads before writing it.  Not state: y1/F0/Fab and the sums other than sumsI (written within a stage before they
// are read), P1/P2/W/T/rscratch (scratch), lapphi of the spectral-budget models (recomputed wherever it is read).
static const int MAX_SLOTS = 16;
static int state_slots(const niwqg_handle* h, int* ids) {
    int n = 0;
    ids[n++] = NIWQG_F_QH;
    ids[n++] = NIWQG_F_PH;
    ids[n++] = NIWQG_F_UV;      // YBJ: u, v of set_q; QG: the stage-4 velocity that Gamma_c reads
    ids[n++] = NIWQG_F_QS;      // physical q is the user's array after set_q (QG, YBJ) until it is next inverted
    if (h->qg) {
        if (h->p.passive_scalar) { ids[n++] = NIWQG_F_CH; ids[n++] = NIWQG_F_C; }   // C: W.x, the user's array after set_c
        return n;
    }
    ids[n++] = NIWQG_F_PHIH;
    ids[n++] = NIWQG_F_PHI;     // YBJ: refreshed at the end of a step only
    ids[n++] = NIWQG_F_PHIX;    // UnCoupled / YBJ: refreshed at status and diagnostics ticks only (F6)
    ids[n++] = NIWQG_F_PHIY;
    if (h->flags & MF_WAVE_PV) ids[n++] = NIWQG_F_QWH;
    if (!(h->flags & MF_SPEC_BUDGET)) {      // k_phys_rhs reads them; YBJ refreshes them at diagnostics ticks only
        ids[n++] = NIWQG_F_LAPPHI;
        if (h->flags & MF_HAS_LAP2) ids[n++] = NIWQG_F_LAP2PHI;
    }
    if (h->flags & MF_QL_ADV) ids[n++] = NIWQG_F_UVQ;   // read by the diagnostics pass
    return n;
}

int niwqg_state_slots(const niwqg_handle* h, int* ids, int max) {
    int all[MAX_SLOTS];
    const int n = state_slots(h, all);
    if (max < n) return -1;
    for (int i = 0; i < n; ++i) ids[i] = all[i];
    return n;
}

int niwqg_set_field(niwqg_handle* h, int field, int member, const void* src, size_t bytes, int on_device) {
    CK(cudaSetDevice(h->p.device));
    if (member < 0 || member >= h->B) { h->err = "set_field: bad member"; return -1; }
    int ids[MAX_SLOTS];
    const int n = state_slots(h, ids);
    bool slot = false;
    for (int i = 0; i < n; ++i) slot = slot || ids[i] == field;
    if (!slot) { h->err = "set_field: not a state slot of this model"; return -1; }
    if (bytes != niwqg_field_bytes(h, field)) { h->err = "set_field: size mismatch"; return -1; }
    const size_t mo = (size_t)member * h->npts, so = (size_t)member * h->nspec;
    cd* spec = nullptr;
    cd* phys = nullptr;
    switch (field) {
        case NIWQG_F_QH: spec = h->qh[h->cq]; break;
        case NIWQG_F_PHIH: spec = h->phih[h->cp]; break;
        case NIWQG_F_CH: spec = h->chh[h->cc]; break;
        case NIWQG_F_PH: spec = h->ph; break;
        case NIWQG_F_QWH: spec = h->qwh; break;
        case NIWQG_F_PHI: phys = h->phi; break;
        case NIWQG_F_PHIX: phys = h->phix; break;
        case NIWQG_F_PHIY: phys = h->phiy; break;
        case NIWQG_F_LAPPHI: phys = h->lapphi; break;
        case NIWQG_F_LAP2PHI: phys = h->lap2phi; break;
        case NIWQG_F_UV: phys = h->uv; break;
        case NIWQG_F_QS: phys = h->qs; break;
        case NIWQG_F_UVQ: phys = h->uvq; break;
        case NIWQG_F_C: {
            int r = upload_phys<double>(h, src, h->rscratch + mo, h->npts, on_device);
            if (r) return r;
            k_real_to_cplx<<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>(h->rscratch + mo, h->W + mo, h->npts);
            CK(cudaGetLastError());
            h->launches++;
        } break;
    }
    if (spec) {
        CK(cudaMemcpyAsync(spec + so, src, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));       // the caller may reuse its buffer when we return
    }
    if (phys) {
        int r = upload_phys<cd>(h, src, phys + mo, h->npts, on_device);
        if (r) return r;
    }
    if (field == NIWQG_F_QH) h->q_set = true;
    if (field == NIWQG_F_PHIH) h->phi_set = true;
    return 0;
}

// carry layout: scal [B][NIWQG_S_COUNT], then sumsI [B][SI_COUNT] (k_budget reads the sums of the previous step's last
// inversion at stage 1)
int niwqg_carry_count(const niwqg_handle* h) { return h->B * (NIWQG_S_COUNT + SI_COUNT); }

int niwqg_get_carry(niwqg_handle* h, double* out) {
    CK(cudaSetDevice(h->p.device));
    const size_t ns = (size_t)h->B * NIWQG_S_COUNT;
    CK(cudaMemcpyAsync(out, h->scal, ns * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(out + ns, h->sumsI, (size_t)h->B * SI_COUNT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_set_carry(niwqg_handle* h, const double* in) {
    CK(cudaSetDevice(h->p.device));
    const size_t ns = (size_t)h->B * NIWQG_S_COUNT;
    CK(cudaMemcpyAsync(h->scal, in, ns * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->sumsI, in + ns, (size_t)h->B * SI_COUNT * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_fft2(niwqg_handle* h, const void* in, void* out, int kind) {
    CK(cudaSetDevice(h->p.device));
    const size_t c = h->npts * sizeof(cd);
    const int N = h->N, nh = N / 2 + 1;
    if (h->nranks > 1 && (kind == NIWQG_FFT_R2C || kind == NIWQG_FFT_C2R)) { h->err = "fft2: half-spectrum kinds are single-GPU only"; return -1; }
    switch (kind) {
        case NIWQG_FFT_C2C_FWD:
            { int r0 = upload_phys<cd>(h, in, h->P1, h->npts, 0); if (r0) return r0; }
            FFT(h->P1, h->P1, false, PRO_NONE, 1);
            CK(cudaMemcpyAsync(out, h->P1, c, cudaMemcpyDeviceToHost, h->stream));
            break;
        case NIWQG_FFT_C2C_INV:
            CK(cudaMemcpyAsync(h->P1, in, c, cudaMemcpyHostToDevice, h->stream));
            FFT(h->P1, h->P1, true, PRO_NONE, 1);
            { int r0 = download_phys<cd>(h, h->P1, out, h->npts, 0, h->P2); if (r0) return r0; }
            break;
        case NIWQG_FFT_R2C_FULL:
        case NIWQG_FFT_R2C:
            { int r0 = upload_phys<double>(h, in, h->rscratch, h->npts, 0); if (r0) return r0; }
            FFT(h->rscratch, h->P1, false, PRO_REAL_IN, 1);
            if (kind == NIWQG_FFT_R2C_FULL)
                CK(cudaMemcpyAsync(out, h->P1, c, cudaMemcpyDeviceToHost, h->stream));
            else
                CK(cudaMemcpy2DAsync(out, nh * sizeof(cd), h->P1, N * sizeof(cd), nh * sizeof(cd), N, cudaMemcpyDeviceToHost,
                                     h->stream));
            break;
        case NIWQG_FFT_C2R: {
            CK(cudaMemcpyAsync(h->P2, in, (size_t)N * nh * sizeof(cd), cudaMemcpyHostToDevice, h->stream));
            QgExpand1Args ea{};
            ea.N = N; ea.nk = nh; ea.dk = h->dk; ea.in = h->P2; ea.out = h->P1; ea.mode = QGX_PLAIN;
            { PROF(PK_SPEC); k_qg_expand1<<<dim3(NIWQG_PW_BLOCKS, 1), NIWQG_PW_THREADS, 0, h->stream>>>(ea); }
            CK(cudaGetLastError());
            h->launches++;
            FFT(h->P1, h->P1, true, PRO_NONE, 1, EPI_REAL_OUT, h->rscratch);
            { int r0 = download_phys<double>(h, h->rscratch, out, h->npts, 0, (double*)h->P2); if (r0) return r0; }
        } break;
        default: h->err = "fft2: unknown kind"; return -1;
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_jacobian(niwqg_handle* h, int which, void* out) {
    CK(cudaSetDevice(h->p.device));
    if (h->B != 1) { h->err = "jacobian: batch==1 only"; return -1; }
    if (h->nranks > 1) { h->err = "jacobian: single-GPU layout only"; return -1; }
    if (h->qg) {
        if (which != NIWQG_JAC_PSI_Q) { h->err = "jacobian: QGModel has J(psi,q) only"; return -1; }
        int r = qg_expand_and_invert(h, h->qh[h->cq]);
        if (r) return r;
        { PROF(PK_PHYS); k_qg_products<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->uv, h->qs, nullptr, h->P1, h->P2, h->npts); }
        CK(cudaGetLastError());
        FFT(h->P1, h->P1, false, PRO_NONE, 1);
        k_qg_jacobian_out<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->P1, h->P2, h->N, h->nk, h->dk);
        CK(cudaGetLastError());
        h->launches += 2;
        CK(cudaMemcpyAsync(out, h->P2, h->nspec * sizeof(cd), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    const size_t c = h->npts * sizeof(cd);
    if (which == NIWQG_JAC_PHIC_PHI) {
        if (!(h->flags & MF_WAVE_PV)) { h->err = "jacobian_phic_phi: Coupled/QL only"; return -1; }
        int r = wave_fields(h, false, true, false);     // refreshes phix, phiy (CoupledModel.py:70)
        if (r) return r;
        { PROF(PK_PHYS); k_phys_wavepv<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->phi, h->phix, h->phiy, h->W, h->npts, h->jscale); }
        CK(cudaGetLastError());
        FFT(h->W, h->W, false, PRO_NONE, 1);
        k_split_packed<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->W, h->P1, h->N, 1, 1, 1.0 / h->jscale);
        CK(cudaGetLastError());
        h->launches += 2;
        CK(cudaMemcpyAsync(out, h->P1, c, cudaMemcpyDeviceToHost, h->stream));
    } else {
        // both need the [D] products of the current carried state
        PhysArgs pa = phys_args(h, 0);
        pa.flags &= ~MF_YBJ;
        { PROF(PK_PHYS); k_phys_rhs<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(pa); }
        CK(cudaGetLastError());
        h->launches++;
        if (which == NIWQG_JAC_PSI_Q) {
            FFT(h->P1, h->P1, false, PRO_NONE, 1);
            k_jac_psi_q_out<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(h->P1, h->P2, h->N, h->dk);
            CK(cudaGetLastError());
            h->launches++;
            CK(cudaMemcpyAsync(out, h->P2, c, cudaMemcpyDeviceToHost, h->stream));
        } else {
            // fft(u phix + v phiy): reuse P1 as scratch for the plain product
            if (h->flags & MF_QL_ADV) { int r = ql_wave_velocity(h); if (r) return r; }
            k_adv_product<<<pw_grid(h), NIWQG_PW_THREADS, 0, h->stream>>>(
                (h->flags & MF_QL_ADV) ? h->uvq : h->uv, h->phix, h->phiy, h->P1, h->npts);
            CK(cudaGetLastError());
            FFT(h->P1, h->P1, false, PRO_NONE, 1);
            if (h->flags & MF_FIX00) CK(cudaMemsetAsync(h->P1, 0, sizeof(cd), h->stream));
            h->launches++;
            CK(cudaMemcpyAsync(out, h->P1, c, cudaMemcpyDeviceToHost, h->stream));
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}


// ---- Lagrangian particles (kernels_particles.cuh, DESIGN.md section 3.4)
static const char* const PARTICLES_SLAB =
    "particles: not available on a slab handle (nranks > 1): particles would have to migrate between ranks";

int niwqg_particles_set(niwqg_handle* h, const double* xy, int count, double t, int waves, int on_device) {
    if (h->nranks > 1) { h->err = PARTICLES_SLAB; return -1; }
    if (count < 0) { h->err = "particles_set: count must be >= 0"; return -1; }
    if (count > 0 && !xy) { h->err = "particles_set: null positions"; return -1; }
    if (waves && !h->phi) { h->err = "particles_set: waves=1 needs a model with a wave field phi (not QGModel)"; return -1; }
    if (!std::isfinite(t)) { h->err = "particles_set: the clock t must be finite"; return -1; }
    CK(cudaSetDevice(h->p.device));
    const size_t n = (size_t)h->B * count;           // particles over all members
    std::vector<double> host;
    if (on_device && count > 0) {                    // checked on the host like any other input
        host.resize(2 * n);
        CK(cudaMemcpy(host.data(), xy, 2 * n * sizeof(double), cudaMemcpyDeviceToHost));
        xy = host.data();
    }
    for (size_t i = 0; i < 2 * n; ++i)
        if (!std::isfinite(xy[i])) { h->err = "particles_set: positions must be finite"; return -1; }
    const size_t bytes = 3 * n * sizeof(double2) + 2 * sizeof(double);
    if (count > 0) {
        size_t fr = 0, tot = 0;
        CK(cudaMemGetInfo(&fr, &tot));
        if (bytes > fr) {
            char buf[256];
            snprintf(buf, sizeof buf, "particles_set: %zu particles need %zu bytes of device memory, %zu are free", n, bytes, fr);
            h->err = buf;
            return -1;
        }
    }
    // the step graphs captured the particle launches (or their absence): drop them, the next steps capture anew
    CK(cudaStreamSynchronize(h->stream));
    for (auto& g : h->graphs)
        if (g.exec) { CK(cudaGraphExecDestroy(g.exec)); g = niwqg_handle::StepGraph{}; }
    if (h->pbuf) { CK(cudaFree(h->pbuf)); h->pbuf = nullptr; }
    h->np = 0;
    h->pwaves = false;
    if (count == 0) return 0;
    CK(cudaMalloc((void**)&h->pbuf, bytes));
    h->np = count;
    h->pwaves = waves != 0;
    const double clk[2] = {t, t};
    CK(cudaMemcpyAsync(h->pbuf, xy, n * sizeof(double2), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync((double*)(h->pbuf + 3 * n), clk, sizeof clk, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_particles_count(const niwqg_handle* h) { return h->np; }

int niwqg_particles_get(niwqg_handle* h, double* xy, double* t) {
    if (h->nranks > 1) { h->err = PARTICLES_SLAB; return -1; }
    if (!h->np) { h->err = "particles_get: the model has no particles"; return -1; }
    CK(cudaSetDevice(h->p.device));
    const size_t n = (size_t)h->B * h->np;
    if (xy) CK(cudaMemcpyAsync(xy, h->pbuf, n * sizeof(double2), cudaMemcpyDeviceToHost, h->stream));
    if (t) CK(cudaMemcpyAsync(t, (const double*)(h->pbuf + 3 * n), sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int niwqg_particles_sample(niwqg_handle* h, int field, double* out) {
    if (h->nranks > 1) { h->err = PARTICLES_SLAB; return -1; }
    if (!h->np) { h->err = "particles_sample: the model has no particles"; return -1; }
    CK(cudaSetDevice(h->p.device));
    PartArgs a = particle_args(h);
    const size_t n = (size_t)h->B * h->np;
    // the result goes to the stage-position and accumulator arrays: every step writes them before it reads them
    double2* dout = a.xs;
    const dim3 g = particle_grid(h);
    if (field == NIWQG_F_PHI) {
        if (!h->phi) { h->err = "particles_sample: the model has no wave field phi"; return -1; }
        k_particles_sample<cd><<<g, 128, 0, h->stream>>>(a, h->phi, dout);
    } else {
        const cd* src = nullptr;
        int which = 0;
        switch (field) {   // what niwqg_get_field returns: the same extraction into scratch, for every member
            case NIWQG_F_Q: src = h->qs; which = 0; break;
            case NIWQG_F_U: src = h->uv; which = 0; break;
            case NIWQG_F_V: src = h->uv; which = 1; break;
            default: h->err = "particles_sample: field must be Q, U, V or PHI"; return -1;
        }
        k_extract_real<<<NIWQG_PW_BLOCKS, NIWQG_PW_THREADS, 0, h->stream>>>(src, h->rscratch, (size_t)h->B * h->npts, which);
        CK(cudaGetLastError());
        h->launches++;
        k_particles_sample<double><<<g, 128, 0, h->stream>>>(a, h->rscratch, (double*)dout);
    }
    CK(cudaGetLastError());
    h->launches++;
    const size_t w = (field == NIWQG_F_PHI) ? 2 : 1;
    CK(cudaMemcpyAsync(out, dout, n * w * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

}  // extern "C"
