// bilevel-gait-gen_b200 -- the C ABI (include/bgg.h) over the CUDA kernels.  No torch types, no exceptions across
// the boundary.  There is no CPU fallback: without a CUDA device bgg_create fails with BGG_ECUDA.
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bgg.h"
#include "bgg_kernels.cuh"

using namespace bgg;

static_assert(BGG_MAX_CONTACTS == kMaxContacts, "include/bgg.h and csrc/bgg_ws.cuh disagree");
static_assert(sizeof(WsHeader) == 256, "per-instance result record (header) is 256 bytes");

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail(BGG_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

struct bgg_handle {
    Params P{};
    WsLayout L{};
    RobotKin kin{};
    bool kin_set = false;
    int device = 0;
    int batch = 0;
    cudaStream_t stream = nullptr;
    Instance* d_inst = nullptr;
    char* d_ws = nullptr;
    double *d_state = nullptr, *d_t0 = nullptr, *d_ee = nullptr;
    // pinned staging
    double *h_state = nullptr, *h_t0 = nullptr, *h_ee = nullptr;
    WsHeader* h_hdr = nullptr;   // pinned [batch]
    WsHeader* d_hdr = nullptr;   // compact copy of the headers [batch]
    double* d_zout = nullptr;    // compact copy of the decision vectors [batch][zcap], allocated on first use
    double* h_zout = nullptr;    // pinned
    int zcap = 0;
    // Shared-memory sizing without a host round trip inside a solve: every solve measures its batch maxima (nu, n_samples) on the
    // device and ships them to pinned memory behind an event; the NEXT solve's first pass is launched with the latest maxima that
    // have arrived (worst case until the first ones do), instances that outgrew them are caught by a second pass.  One record
    // for the main batch, one for the line-search children (their contact schedules differ from the parents').
    struct Caps {
        int* d_max = nullptr;        // device: maxima of the solve in flight
        int* h_max = nullptr;        // pinned
        cudaEvent_t ev = nullptr;
        bool pending = false;
        int nu = 0, ns = 0;          // 0: unknown (launch with the worst case)
    };
    Caps caps_main, caps_ls;
    int last_nu_max = 0, last_ns_max = 0;   // caps the main batch's last solve was launched with (sizing of k_gradient)
    int max_smem = 0, sm_count = 0;
    bool profiling = false;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    float last_ms[4] = {0, 0, 0, 0};
    int64_t launches = 0;
    cudaEvent_t user_ev[8] = {};
    bool costs_set = false;
    // controller tick (bgg_controller_tick_batch): the gait optimiser's step lives on the device between the tick that computes it
    // and the tick that searches along it; allocated on the first tick
    double* d_tick = nullptr;        // step | xk | new_times, each [batch][4][kMaxContacts]
    int32_t* d_tick_i = nullptr;     // LP status [batch][4] | deriv_ready [batch] | ls_best [batch]
    double* d_tick_ls = nullptr;     // line-search costs [batch * K]
    int32_t* d_tick_lsq = nullptr;   // line-search quality [batch * K]
    int tick_ls_cap = 0;
    double* h_tick = nullptr;        // pinned: dH/dtheta [batch][4][kMaxContacts]
    int32_t* h_tick_i = nullptr;     // pinned: deriv_ready [batch] | ls_best [batch]
    // line-search children (batch x K copies), allocated on first use
    int ls_cap = 0;
    Instance* d_ls_inst = nullptr;
    char* d_ls_ws = nullptr;
    double *d_ls_state = nullptr, *d_ls_t0 = nullptr, *d_ls_ee = nullptr;
};

// decision vectors after the line-search update, compacted to [B][stride] (entries n .. stride-1 of a row are zero)
__global__ void k_gather_z(WsLayout L, const char* __restrict__ ws, double* __restrict__ out, int stride) {
    const int b = blockIdx.x;
    const char* w = ws + static_cast<size_t>(b) * L.stride;
    const int n = reinterpret_cast<const WsHeader*>(w + L.hdr)->n;
    const double* z = reinterpret_cast<const double*>(w + L.zprev);
    for (int i = threadIdx.x; i < stride; i += blockDim.x) out[static_cast<size_t>(b) * stride + i] = (i < n) ? z[i] : 0.0;
}

// controller tick helpers
__global__ void k_deriv_ready(WsLayout L, const char* __restrict__ ws, int B, int32_t* __restrict__ ready, double* __restrict__ dH) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const char* w = ws + static_cast<size_t>(b) * L.stride;
    ready[b] = reinterpret_cast<const GradInfo*>(w + L.ginfo)->status == 0 ? 1 : 0;   // GaitOpt returns false unless the solve was Solved
    const double* g = reinterpret_cast<const double*>(w + L.gdH);
    for (int i = 0; i < kNumEE * kMaxContacts; ++i) dH[static_cast<size_t>(b) * kNumEE * kMaxContacts + i] = g[i];
}
__global__ void k_mask_step(double* __restrict__ step, const int32_t* __restrict__ ready, int B) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B * kNumEE * kMaxContacts && !ready[i / (kNumEE * kMaxContacts)]) step[i] = 0.0;   // no derivative: every candidate is the unchanged schedule
}

__global__ void k_gather_headers(WsLayout L, const char* __restrict__ ws, WsHeader* __restrict__ out, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) out[b] = *reinterpret_cast<const WsHeader*>(ws + static_cast<size_t>(b) * L.stride + L.hdr);
}

__global__ void k_reset(Params P, Instance* inst, int B, const double* __restrict__ ct, int nct) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    Instance& I = inst[b];
    for (int k = 0; k <= kMaxNodes; ++k)
        for (int c = 0; c < kNxMan; ++c) I.states[k][c] = 0.0;
    const double def[5] = {0.0, 0.3, 0.6, 0.9, 1.2};
    for (int e = 0; e < kNumEE; ++e) {
        double t[16];
        const int n = ct ? nct : 5;
        for (int i = 0; i < n; ++i) t[i] = ct ? ct[e * nct + i] : def[i];
        init_foot(I.foot[e], t, n, e == 1 || e == 2);            // trajectory.cpp:25-28
        set_swing_pos_z(I.foot[e], P.swing_height, P.foot_offset);
    }
    I.ee_box[0] = P.ee_box_nominal[0];
    I.ee_box[1] = P.ee_box_nominal[1];
    I.init_time = 0.0;
    I.run_count = 0;
    I.pad_ = 0;
}

__global__ void k_warm_states(Instance* inst, int B, int N, const double* __restrict__ states, int per_node) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * (N + 1)) return;
    const int b = i / (N + 1), k = i % (N + 1);
    const double* src = per_node ? states + static_cast<size_t>(i) * kNxMan : states + static_cast<size_t>(b) * kNxMan;
    for (int c = 0; c < kNxMan; ++c) inst[b].states[k][c] = src[c];
}

// bad[0] counts the feet that were refused: the reference asserts size == GetNumContacts and throws on a negative time
// (end_effector_splines.cpp:860-892); a foot whose knot list holds another number of contacts than the caller passes would
// read its neighbour's times
__global__ void k_set_contact_times(Instance* inst, int first, int count, const double* __restrict__ times, int nct, int* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count * kNumEE) return;
    const int b = first + i / kNumEE, e = i % kNumEE;
    const double* t = times + static_cast<size_t>(i) * nct;
    bool ok = num_contacts(inst[b].foot[e]) == nct;
    for (int k = 0; ok && k < nct; ++k) ok = t[k] >= 0.0 && (k == 0 || t[k] >= t[k - 1]);
    if (!ok) {
        atomicAdd(bad, 1);
        return;
    }
    set_contact_times(inst[b].foot[e], t, nct);
}

__global__ void k_eval_splines(const Instance* inst, int b, const double* __restrict__ times, int T, double* __restrict__ force,
                               double* __restrict__ pos) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * kNumEE) return;
    const int e = i % kNumEE;
    const double t = times[i / kNumEE];
    for (int c = 0; c < 3; ++c) {
        force[i * 3 + c] = value_at(inst[b].foot[e], true, c, t);
        pos[i * 3 + c] = value_at(inst[b].foot[e], false, c, t);
    }
}

// Synthetic plant of the closed-loop sweeps (SURVEY 8d, config #5): the next measured state is node 1 of the solved
// trajectory (apps/mpc_demo.cpp:185, test/gait_opt_playground.cpp:128), time advances by dt and the measured feet are the
// trajectory's own feet at the new time.  Writes the next solve's inputs in place on the device.
__global__ void k_plant_step(const Instance* __restrict__ inst, int B, double dt, double* __restrict__ state, double* __restrict__ t0,
                             double* __restrict__ ee) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * kNumEE) return;
    const int b = i / kNumEE, e = i % kNumEE;
    const double tn = inst[b].init_time + dt;
    for (int c = 0; c < 3; ++c) ee[(b * kNumEE + e) * 3 + c] = value_at(inst[b].foot[e], false, c, tn);
    if (e == 0) {
        for (int c = 0; c < kNxMan; ++c) state[b * kNxMan + c] = inst[b].states[1][c];
        t0[b] = tn;
    }
}

// register-resident FP64 FMA chains: the ceiling the solver kernels are measured against (bench.py, "fp64" entry)
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// Scratch device allocations of one call, released on every exit path.  Stream-ordered (cudaMallocAsync on the handle's stream, from
// the device's default pool with its release threshold lifted in bgg_create): after the first calls no allocation reaches the
// driver.  Plain cudaMalloc / cudaFree per call cost 0.3 - 1 ms each next to the multi-GB line-search workspace, with outliers of
// hundreds of milliseconds (tools/time_gait_steps.py).
struct DevPool {
    cudaStream_t stream;
    std::vector<void*> p;
    explicit DevPool(cudaStream_t s) : stream(s) {}
    ~DevPool() { for (void* q_ : p) cudaFreeAsync(q_, stream); }
    template <typename T> T* get(size_t nelem) {
        void* d = nullptr;
        if (cudaMallocAsync(&d, sizeof(T) * (nelem ? nelem : 1), stream) != cudaSuccess) return nullptr;
        p.push_back(d);
        return static_cast<T*>(d);
    }
};

namespace bgg {
constexpr int kQpMaxN_capi = 128;
size_t qp_ws_doubles(int n, int mi, int me);
int launch_qp_generic(int count, int n, int m, int mi, int me, int nnzP, int nnzA, const int* Pcol, const int* Prow, const double* Pval,
                      const int* Acol, const int* Arow, const double* Aval, const double* q, const double* b, const int* in_rows,
                      const int* eq_rows, const int* row_slot, double* ws, double* x, double* y, double* s, int32_t* status, int32_t* iters,
                      double tol_feas, double tol_gap, double tol_inf, double eps, double delta, int max_iter, int max_smem, cudaStream_t stream);
constexpr int kQpAdjMaxDim_capi = 160;
size_t qp_adj_ws_doubles(int n, int mi, int me);
int launch_qp_adjoint(int count, int n, int m, int mi, int me, int nnzP, int nnzA, const int* Pcol, const int* Prow, const double* Pval,
                      const int* Acol, const int* Arow, const double* Aval, const int* in_rows, const int* eq_rows, const int* row_slot,
                      const double* x, const double* y, const double* s, const double* dx, double* ws, double* dz, double* dy, double* db,
                      double* dA, int32_t* status, int max_smem, cudaStream_t stream);
}  // namespace bgg

// Row classification shared by bgg_qp_solve_batch and bgg_qp_adjoint_batch (csrc/bgg_qp_common.cuh): equality rows, and inequality
// rows with at least one stored entry (an empty row reads 0 + s = b and is reported s = b, y = 0).  Returns an error message or null.
struct QpRows {
    std::vector<int> row_slot, in_rows, eq_rows;
};
static const char* qp_classify_rows(int m, int nnzA, const int32_t* A_rowidx, const uint8_t* is_eq, QpRows& R) {
    std::vector<int> cnt(m, 0);
    R.row_slot.assign(m, -1);
    R.in_rows.clear();
    R.eq_rows.clear();
    for (int k = 0; k < nnzA; ++k) {
        if (A_rowidx[k] < 0 || A_rowidx[k] >= m) return "row index out of range";
        cnt[A_rowidx[k]]++;
    }
    for (int r = 0; r < m; ++r) {
        if (is_eq[r]) { R.row_slot[r] = -(static_cast<int>(R.eq_rows.size()) + 2); R.eq_rows.push_back(r); }
        else if (cnt[r] > 0) { R.row_slot[r] = static_cast<int>(R.in_rows.size()); R.in_rows.push_back(r); }
    }
    return nullptr;
}

extern "C" {

int bgg_measure_fp64_peak(int device, double* tflops) {
    if (!tflops) return fail(BGG_EINVAL, "null argument");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, iters = 1 << 16;
    double* d = nullptr;
    CU(cudaMalloc(&d, 8 * static_cast<size_t>(blocks) * 256));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    k_fp64_peak<<<blocks, 256>>>(d, iters);   // warm-up
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        k_fp64_peak<<<blocks, 256>>>(d, iters);
        cudaEventRecord(e1);
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double tf = 2.0 * 8.0 * iters * static_cast<double>(blocks) * 256 / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *tflops = best;
    return BGG_OK;
}

const char* bgg_last_error(void) { return g_err.c_str(); }

int bgg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int bgg_create(const bgg_config* cfg, const bgg_robot* robot, bgg_handle** out) {
    if (!cfg || !robot || !out) return fail(BGG_EINVAL, "null argument");
    if (cfg->num_nodes <= kEENodeStart || cfg->num_nodes > kMaxNodes) return fail(BGG_EINVAL, "num_nodes must be in (4, 64]");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(BGG_ECUDA, "no CUDA device: this library has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(BGG_EINVAL, "bad device ordinal");
    CU(cudaSetDevice(cfg->device));
    bgg_handle* h = new bgg_handle;
    h->device = cfg->device;
    Params& P = h->P;
    P.N = cfg->num_nodes;
    P.max_nu = cfg->max_spline_vars > 0 ? cfg->max_spline_vars : kMaxSplineVars;
    if (P.max_nu < P.N + 1 || P.max_nu % 8) {
        delete h;
        return fail(BGG_EINVAL, "max_spline_vars must be a multiple of 8 and >= num_nodes + 1");
    }
    if (P.max_nu > kMaxSplineVars) {
        delete h;
        return fail(BGG_EINVAL, "max_spline_vars must not exceed 160: the condensing and KKT kernels are sized for at most 160 spline variables");
    }
    P.dt = cfg->integrator_dt;
    P.mass = robot->mass;
    std::memcpy(P.Ir, robot->Ir, sizeof P.Ir);
    std::memcpy(P.Ir_inv, robot->Ir_inv, sizeof P.Ir_inv);
    std::memcpy(P.gravity, robot->gravity, sizeof P.gravity);
    std::memcpy(P.hip_xy, robot->hip_xy, sizeof P.hip_xy);
    P.friction_coef = cfg->friction_coef;
    P.force_bound = cfg->force_bound;
    P.swing_height = cfg->swing_height;
    P.foot_offset = cfg->foot_offset;
    P.force_cost = cfg->force_cost;
    P.ee_box_nominal[0] = cfg->ee_box_size[0];
    P.ee_box_nominal[1] = cfg->ee_box_size[1];
    for (int i = 0; i < kNx; ++i) P.Q[i] = P.w[i] = P.Phi[i] = P.Phi_w[i] = 0.0;
    P.merit_mu = 5000.0;      // mpc.cpp:65
    P.td_fraction = 0.75;     // mpc.cpp:73
    P.ipm_tol_feas = cfg->ipm_tol_feas > 0 ? cfg->ipm_tol_feas : 1e-8;
    P.ipm_tol_gap = cfg->ipm_tol_gap > 0 ? cfg->ipm_tol_gap : 1e-8;
    P.ipm_eq_delta = cfg->ipm_eq_delta > 0 ? cfg->ipm_eq_delta : 1e-10;
    P.ipm_reg_eps = cfg->ipm_reg_eps > 0 ? cfg->ipm_reg_eps : 1e-10;
    P.ipm_tol_infeas = cfg->ipm_tol_infeas > 0 ? cfg->ipm_tol_infeas : 1e-8;
    P.ipm_max_iter = cfg->ipm_max_iter > 0 ? cfg->ipm_max_iter : 50;
    P.ipm_refine = cfg->ipm_refine < 0 ? 0 : (cfg->ipm_refine == 0 ? 1 : cfg->ipm_refine);
    P.ipm_refine_mu_frac = cfg->ipm_refine_after < 0 ? 1e300 : pow(10.0, -static_cast<double>(cfg->ipm_refine_after == 0 ? 12 : cfg->ipm_refine_after));
    P.ipm_refine_from_iter = 20;
    h->L = make_layout(P.N, P.max_nu);
    int max_smem = 0;
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device);
    h->max_smem = max_smem;
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, h->device);
    if (ipm_smem_bytes(h->L) > static_cast<size_t>(max_smem) || condense_smem_bytes(h->L) > static_cast<size_t>(max_smem) ||
        finish_smem_bytes(h->L) > static_cast<size_t>(max_smem)) {
        delete h;
        return fail(BGG_EINVAL, "num_nodes / max_spline_vars need more shared memory than the device offers");
    }
    {   // scratch allocations are stream-ordered (DevPool): keep what the pool has grown to instead of returning it at every synchronise
        cudaMemPool_t mp = nullptr;
        if (cudaDeviceGetDefaultMemPool(&mp, h->device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return fail(BGG_ECUDA, "cudaStreamCreate failed");
    }
    for (auto& e : h->ev) cudaEventCreate(&e);
    for (auto& e : h->user_ev) cudaEventCreate(&e);
    for (bgg_handle::Caps* c : {&h->caps_main, &h->caps_ls}) {
        cudaMalloc(&c->d_max, 3 * sizeof(int));
        cudaMallocHost(&c->h_max, 3 * sizeof(int));
        cudaEventCreateWithFlags(&c->ev, cudaEventDisableTiming);
    }
    *out = h;
    return BGG_OK;
}

static void free_batch(bgg_handle* h) {
    cudaFree(h->d_inst);
    cudaFree(h->d_ws);
    cudaFree(h->d_state);
    cudaFree(h->d_t0);
    cudaFree(h->d_ee);
    cudaFree(h->d_hdr);
    cudaFree(h->d_tick); cudaFree(h->d_tick_i); cudaFree(h->d_tick_ls); cudaFree(h->d_tick_lsq);
    cudaFreeHost(h->h_tick); cudaFreeHost(h->h_tick_i);
    h->d_tick = h->d_tick_ls = h->h_tick = nullptr;
    h->d_tick_i = h->d_tick_lsq = h->h_tick_i = nullptr;
    h->tick_ls_cap = 0;
    cudaFree(h->d_zout);
    cudaFreeHost(h->h_zout);
    h->d_zout = h->h_zout = nullptr;
    h->zcap = 0;
    cudaFreeHost(h->h_state);
    cudaFreeHost(h->h_t0);
    cudaFreeHost(h->h_ee);
    cudaFreeHost(h->h_hdr);
    cudaFree(h->d_ls_inst);
    cudaFree(h->d_ls_ws);
    cudaFree(h->d_ls_state);
    cudaFree(h->d_ls_t0);
    cudaFree(h->d_ls_ee);
    h->d_ls_inst = nullptr;
    h->d_ls_ws = nullptr;
    h->d_ls_state = h->d_ls_t0 = h->d_ls_ee = nullptr;
    h->ls_cap = 0;
    h->d_inst = nullptr;
    h->d_ws = nullptr;
    h->d_state = h->d_t0 = h->d_ee = nullptr;
    h->h_state = h->h_t0 = h->h_ee = nullptr;
    h->d_hdr = nullptr;
    h->h_hdr = nullptr;
    h->batch = 0;
    for (bgg_handle::Caps* c : {&h->caps_main, &h->caps_ls}) {   // sizes of another batch say nothing about the next one
        c->pending = false;
        c->nu = c->ns = 0;
    }
    h->last_nu_max = h->last_ns_max = 0;
}

void bgg_destroy(bgg_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    free_batch(h);
    for (auto& e : h->ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : h->user_ev)
        if (e) cudaEventDestroy(e);
    for (bgg_handle::Caps* c : {&h->caps_main, &h->caps_ls}) {
        cudaFree(c->d_max);
        cudaFreeHost(c->h_max);
        if (c->ev) cudaEventDestroy(c->ev);
    }
    cudaStreamDestroy(h->stream);
    delete h;
}

int bgg_set_costs(bgg_handle* h, const double Q[BGG_NX], const double x_des[BGG_NX], const double Phi[BGG_NX],
                  const double Phi_w[BGG_NX]) {
    if (!h || !Q || !x_des) return fail(BGG_EINVAL, "null argument");
    for (int i = 0; i < kNx; ++i) {
        h->P.Q[i] = Q[i];
        h->P.w[i] = (-1 * Q[i]) * x_des[i];             // w_ = -1*Q*state_des, mpc.cpp:539
        h->P.Phi[i] = Phi ? Phi[i] : Q[i];
        h->P.Phi_w[i] = Phi_w ? Phi_w[i] : h->P.w[i];
    }
    h->costs_set = true;
    return BGG_OK;
}

int bgg_batch_reset(bgg_handle* h, int batch, const double* contact_times, int num_contacts) {
    if (!h || batch <= 0) return fail(BGG_EINVAL, "bad batch");
    if (contact_times && (num_contacts < 2 || num_contacts > 8)) return fail(BGG_EINVAL, "num_contacts must be in [2, 8]");
    CU(cudaSetDevice(h->device));
    if (batch != h->batch) {
        cudaStreamSynchronize(h->stream);
        free_batch(h);
        CU(cudaMalloc(&h->d_inst, sizeof(Instance) * static_cast<size_t>(batch)));
        CU(cudaMalloc(&h->d_ws, h->L.stride * static_cast<size_t>(batch)));
        CU(cudaMalloc(&h->d_state, 8 * kNxMan * static_cast<size_t>(batch)));
        CU(cudaMalloc(&h->d_t0, 8 * static_cast<size_t>(batch)));
        CU(cudaMalloc(&h->d_ee, 8 * 12 * static_cast<size_t>(batch)));
        CU(cudaMalloc(&h->d_hdr, sizeof(WsHeader) * static_cast<size_t>(batch)));
        CU(cudaMallocHost(&h->h_state, 8 * kNxMan * static_cast<size_t>(batch)));
        CU(cudaMallocHost(&h->h_t0, 8 * static_cast<size_t>(batch)));
        CU(cudaMallocHost(&h->h_ee, 8 * 12 * static_cast<size_t>(batch)));
        CU(cudaMallocHost(&h->h_hdr, sizeof(WsHeader) * static_cast<size_t>(batch)));
        CU(cudaMemsetAsync(h->d_ws, 0, h->L.stride * static_cast<size_t>(batch), h->stream));
        h->batch = batch;
    }
    double* d_ct = nullptr;
    if (contact_times) {
        CU(cudaMalloc(&d_ct, 8 * kNumEE * num_contacts));
        CU(cudaMemcpyAsync(d_ct, contact_times, 8 * kNumEE * num_contacts, cudaMemcpyHostToDevice, h->stream));
    }
    k_reset<<<(batch + 127) / 128, 128, 0, h->stream>>>(h->P, h->d_inst, batch, d_ct, num_contacts);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    if (d_ct) cudaFree(d_ct);
    return BGG_OK;
}

int bgg_set_warm_states(bgg_handle* h, const double* states, int per_node) {
    if (!h || !states || !h->batch) return fail(BGG_EINVAL, "no batch");
    CU(cudaSetDevice(h->device));
    const size_t cnt = static_cast<size_t>(h->batch) * (per_node ? (h->P.N + 1) : 1) * kNxMan;
    double* d = nullptr;
    CU(cudaMalloc(&d, 8 * cnt));
    CU(cudaMemcpyAsync(d, states, 8 * cnt, cudaMemcpyHostToDevice, h->stream));
    const int tot = h->batch * (h->P.N + 1);
    k_warm_states<<<(tot + 127) / 128, 128, 0, h->stream>>>(h->d_inst, h->batch, h->P.N, d, per_node);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    return BGG_OK;
}

int bgg_set_contact_times(bgg_handle* h, int first, int count, const double* times, int nct) {
    if (!h || !times || first < 0 || count <= 0 || first + count > h->batch) return fail(BGG_EINVAL, "bad range");
    if (nct < 2 || nct > BGG_MAX_CONTACTS) return fail(BGG_EINVAL, "num_contacts must be in [2, BGG_MAX_CONTACTS]");
    CU(cudaSetDevice(h->device));
    const size_t cnt = static_cast<size_t>(count) * kNumEE * nct;
    double* d = nullptr;
    CU(cudaMalloc(&d, 8 * cnt));
    CU(cudaMemcpyAsync(d, times, 8 * cnt, cudaMemcpyHostToDevice, h->stream));
    int* d_bad = nullptr;
    CU(cudaMalloc(&d_bad, sizeof(int)));
    CU(cudaMemsetAsync(d_bad, 0, sizeof(int), h->stream));
    k_set_contact_times<<<(count * kNumEE + 127) / 128, 128, 0, h->stream>>>(h->d_inst, first, count, d, nct, d_bad);
    CU(cudaGetLastError());
    int bad = 0;
    CU(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    cudaFree(d_bad);
    if (bad) return fail(BGG_EINVAL, "contact times refused for " + std::to_string(bad) + " feet: wrong count for the foot's schedule, negative or decreasing times");
    return BGG_OK;
}

int bgg_upload_inputs(bgg_handle* h, const double* state, const double* t0, const double* ee_start) {
    if (!h || !state || !t0 || !ee_start || !h->batch) return fail(BGG_EINVAL, "null argument / no batch");
    CU(cudaSetDevice(h->device));
    const size_t B = h->batch;
    std::memcpy(h->h_state, state, 8 * kNxMan * B);
    std::memcpy(h->h_t0, t0, 8 * B);
    std::memcpy(h->h_ee, ee_start, 8 * 12 * B);
    CU(cudaMemcpyAsync(h->d_state, h->h_state, 8 * kNxMan * B, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_t0, h->h_t0, 8 * B, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_ee, h->h_ee, 8 * 12 * B, cudaMemcpyHostToDevice, h->stream));
    return BGG_OK;
}

// Kept for the callers that size something from the main batch's maxima: solve_pipeline now takes delivery itself.
static void refresh_caps(bgg_handle::Caps& caps) { (void)caps; }

// steps 1-11 of MPCSingleRigidBody::Solve for `B` instances living in (inst, ws) with inputs (state, t0, ee) on the device.
//
// Shared memory (one or two CTAs per SM) is sized from the batch maxima of (spline variables, force samples), which only
// k_prepare knows.  The solve kernels are enqueued at once with the previous solve's maxima -- the usual case: nothing changed --
// and while the device works on them the host waits for the event right behind k_prepare / k_batch_max (about a millisecond into
// the step; the queue behind it is full, the device never idles).  Instances that outgrew the sizes were marked by k_batch_max;
// if there are any, a second pass is launched for them with the exact new maxima.  (Round 2 first launched that second pass
// unconditionally with worst-case sizes, one CTA per SM: in a closed-loop sweep every scenario's horizon grows at the same tick,
// and those ticks took twice as long.)
static int solve_pipeline(bgg_handle* h, bgg_handle::Caps& caps, Instance* inst, char* ws, const double* state, const double* t0, const double* ee,
                          int B, bool profile) {
    // Speculate only while the previous sizes are worth having: two CTAs per SM.  Beyond that (K alone fills the SM's shared memory) a
    // horizon that has shrunk again would run a whole pass at half the occupancy it could have; there the pass waits for the exact
    // sizes (the device idles for one host round trip, tens of microseconds in a step of a second).
    const bool have = caps.nu > 0 && ipm_two_per_sm(h->L, caps.nu, caps.ns);
    auto run_pass = [&](int nu_cap, int ns_cap, int want, bool timed) {
        if (timed) cudaEventRecord(h->ev[1], h->stream);
        launch_condense(h->P, h->L, ws, B, nu_cap, want, h->stream);
        if (timed) cudaEventRecord(h->ev[2], h->stream);
        launch_ipm(h->P, h->L, ws, B, nu_cap, ns_cap, want, h->stream, h->sm_count);
        if (timed) cudaEventRecord(h->ev[3], h->stream);
        launch_finish(h->P, inst, h->L, ws, B, want, h->stream);
        if (timed) cudaEventRecord(h->ev[4], h->stream);
        h->launches += 3;
    };
    if (profile) cudaEventRecord(h->ev[0], h->stream);
    launch_prepare(h->P, inst, state, t0, ee, h->L, ws, B, h->stream);
    launch_batch_max(h->L, ws, B, caps.d_max, have ? (caps.nu + 7) / 8 * 8 : 0, have ? caps.ns : -1, h->stream);   // nothing known: everything is marked
    CU(cudaMemcpyAsync(caps.h_max, caps.d_max, 3 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(caps.ev, h->stream));
    h->launches += 2;
    if (have) run_pass(caps.nu, caps.ns, 0, profile);
    CU(cudaEventSynchronize(caps.ev));
    const int nu_now = caps.h_max[0] > 0 ? caps.h_max[0] : 8, ns_now = caps.h_max[1];
    if (caps.h_max[2] > 0) run_pass(nu_now, ns_now, 2, profile && !have);
    caps.nu = nu_now;
    caps.ns = ns_now;
    if (&caps == &h->caps_main) {
        h->last_nu_max = nu_now;
        h->last_ns_max = ns_now;
    }
    CU(cudaGetLastError());
    return BGG_OK;
}

int bgg_solve_resident(bgg_handle* h) {
    if (!h || !h->batch) return fail(BGG_EINVAL, "no batch");
    if (!h->costs_set) return fail(BGG_ESTATE, "bgg_set_costs has not been called");
    CU(cudaSetDevice(h->device));
    return solve_pipeline(h, h->caps_main, h->d_inst, h->d_ws, h->d_state, h->d_t0, h->d_ee, h->batch, h->profiling);
}

int bgg_advance_plant(bgg_handle* h, double dt) {
    if (!h || !h->batch) return fail(BGG_EINVAL, "no batch");
    CU(cudaSetDevice(h->device));
    const int tot = h->batch * kNumEE;
    k_plant_step<<<(tot + 127) / 128, 128, 0, h->stream>>>(h->d_inst, h->batch, dt, h->d_state, h->d_t0, h->d_ee);
    h->launches += 1;
    CU(cudaGetLastError());
    return BGG_OK;
}

int bgg_set_kinematics(bgg_handle* h, const bgg_kinematics* kin) {
    if (!h || !kin) return fail(BGG_EINVAL, "null argument");
    static_assert(sizeof(bgg_kinematics) == sizeof(RobotKin), "bgg_kinematics and RobotKin share one layout");
    std::memcpy(&h->kin, kin, sizeof h->kin);
    for (int e = 0; e < kNumEE; ++e)
        for (int j = 0; j < 3; ++j) {
            const double* a = h->kin.leg[e].axis[j];
            const double n = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
            if (!(std::fabs(n - 1.0) < 1e-9)) return fail(BGG_EINVAL, "joint axes must be unit vectors");
        }
    h->kin_set = true;
    return BGG_OK;
}

int bgg_ik_batch(bgg_handle* h, int count, const double* state, const double* ee_des, const double* joint_guess, double* q, int32_t* status,
                 int32_t* iters) {
    if (!h || count <= 0 || !state || !ee_des || !joint_guess || !q || !status) return fail(BGG_EINVAL, "bad argument");
    if (!h->kin_set) return fail(BGG_ESTATE, "bgg_set_kinematics has not been called");
    CU(cudaSetDevice(h->device));
    DevPool pool(h->stream);
    const size_t n = static_cast<size_t>(count);
    double *ds = pool.get<double>(13 * n), *de = pool.get<double>(12 * n), *dg = pool.get<double>(12 * n), *dq = pool.get<double>(19 * n);
    int *dst = pool.get<int>(n), *dit = pool.get<int>(4 * n);
    if (!ds || !de || !dg || !dq || !dst || !dit) return fail(BGG_ECUDA, "out of device memory");
    CU(cudaMemcpyAsync(ds, state, 8 * 13 * n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(de, ee_des, 8 * 12 * n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dg, joint_guess, 8 * 12 * n, cudaMemcpyHostToDevice, h->stream));
    launch_ik(h->kin, count, ds, de, dg, dq, dst, dit, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(q, dq, 8 * 19 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(status, dst, 4 * n, cudaMemcpyDeviceToHost, h->stream));
    if (iters) CU(cudaMemcpyAsync(iters, dit, 4 * 4 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BGG_OK;
}

int bgg_targets_from_traj_batch(bgg_handle* h, const double* time, double* q_des, double* v_des, double* force_des, int32_t* status) {
    if (!h || !h->batch) return fail(BGG_EINVAL, "no batch");
    if (!time || !q_des || !v_des || !force_des || !status) return fail(BGG_EINVAL, "null argument");
    if (!h->kin_set) return fail(BGG_ESTATE, "bgg_set_kinematics has not been called");
    CU(cudaSetDevice(h->device));
    DevPool pool(h->stream);
    const size_t n = static_cast<size_t>(h->batch);
    double *dt = pool.get<double>(n), *dq = pool.get<double>(19 * n), *dv = pool.get<double>(18 * n), *df = pool.get<double>(12 * n);
    int* dst = pool.get<int>(n);
    if (!dt || !dq || !dv || !df || !dst) return fail(BGG_ECUDA, "out of device memory");
    CU(cudaMemcpyAsync(dt, time, 8 * n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dq, q_des, 8 * 19 * n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemsetAsync(dv, 0, 8 * 18 * n, h->stream));
    CU(cudaMemsetAsync(df, 0, 8 * 12 * n, h->stream));
    launch_targets_from_traj(h->P, h->kin, h->d_inst, h->batch, dt, dq, dv, df, dst, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(q_des, dq, 8 * 19 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(v_des, dv, 8 * 18 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(force_des, df, 8 * 12 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(status, dst, 4 * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BGG_OK;
}

int bgg_download_results(bgg_handle* h, int32_t* status, int32_t* iters, double* alpha, double* cost, double* z, int z_stride) {
    if (!h || !h->batch) return fail(BGG_EINVAL, "no batch");
    if (z && z_stride < kNx * (h->P.N + 1)) return fail(BGG_EINVAL, "z_stride is smaller than the state part of the decision vector");
    CU(cudaSetDevice(h->device));
    const int B = h->batch;
    k_gather_headers<<<(B + 127) / 128, 128, 0, h->stream>>>(h->L, h->d_ws, h->d_hdr, B);
    h->launches += 1;
    CU(cudaMemcpyAsync(h->h_hdr, h->d_hdr, sizeof(WsHeader) * static_cast<size_t>(B), cudaMemcpyDeviceToHost, h->stream));
    // A caller's buffer that is page-locked (cudaHostAlloc / cudaHostRegister) and has the gathered row length takes the DMA
    // directly; anything else goes through the handle's own pinned staging buffer and one host copy.
    bool direct = false;
    if (z) {
        const int n_max = kNx * (h->P.N + 1) + h->P.max_nu;
        const int stride = z_stride < n_max ? z_stride : n_max;
        cudaPointerAttributes attr{};
        if (stride == z_stride && cudaPointerGetAttributes(&attr, z) == cudaSuccess && attr.type == cudaMemoryTypeHost) direct = true;
        cudaGetLastError();   // an unregistered pointer is not an error here
        if (h->zcap < stride) {
            cudaFree(h->d_zout);
            cudaFreeHost(h->h_zout);
            h->d_zout = h->h_zout = nullptr;
            h->zcap = 0;
            CU(cudaMalloc(&h->d_zout, 8 * static_cast<size_t>(B) * n_max));
            CU(cudaMallocHost(&h->h_zout, 8 * static_cast<size_t>(B) * n_max));
            h->zcap = n_max;
        }
        k_gather_z<<<B, 128, 0, h->stream>>>(h->L, h->d_ws, h->d_zout, stride);
        h->launches += 1;
        CU(cudaMemcpyAsync(direct ? z : h->h_zout, h->d_zout, 8 * static_cast<size_t>(B) * stride, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    if (z) {
        const int n_max = kNx * (h->P.N + 1) + h->P.max_nu;
        const int stride = z_stride < n_max ? z_stride : n_max;
        for (int b = 0; b < B; ++b) {
            if (!h->h_hdr[b].error && h->h_hdr[b].n > z_stride) return fail(BGG_EINVAL, "an instance has more decision variables than z_stride");
            if (!direct) std::memcpy(z + static_cast<size_t>(b) * z_stride, h->h_zout + static_cast<size_t>(b) * stride, 8 * static_cast<size_t>(stride));
        }
    }
    for (int b = 0; b < B; ++b) {
        const WsHeader& w = h->h_hdr[b];
        if (status) status[b] = w.error ? BGG_OTHER : w.status;
        if (iters) iters[b] = w.iters;
        if (alpha) alpha[b] = w.alpha;
        if (cost) cost[b] = w.cost;
    }
    if (h->profiling)
        for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&h->last_ms[i], h->ev[i], h->ev[i + 1]);
    return BGG_OK;
}

int bgg_solve_batch(bgg_handle* h, const double* state, const double* t0, const double* ee_start, int32_t* status,
                    int32_t* iters, double* alpha, double* cost, double* z, int z_stride) {
    int rc = bgg_upload_inputs(h, state, t0, ee_start);
    if (rc) return rc;
    rc = bgg_solve_resident(h);
    if (rc) return rc;
    return bgg_download_results(h, status, iters, alpha, cost, z, z_stride);
}

int bgg_qp_solve_batch(bgg_handle* h, int count, int n, int m, const int32_t* P_colptr, const int32_t* P_rowidx, const double* P_val,
                       const int32_t* A_colptr, const int32_t* A_rowidx, const double* A_val, const double* q, const double* b,
                       const uint8_t* is_eq, double* x, double* y, double* s, int32_t* status, int32_t* iters) {
    if (!h || count <= 0 || n <= 0 || m < 0 || !P_colptr || !P_rowidx || !P_val || !A_colptr || !A_rowidx || !A_val || !q || !b || !is_eq || !x)
        return fail(BGG_EINVAL, "null argument");
    if (n > kQpMaxN_capi) return fail(BGG_EINVAL, "bgg_qp_solve_batch handles at most 128 variables (the MPC QP goes through bgg_solve_batch)");
    CU(cudaSetDevice(h->device));
    const int nnzP = P_colptr[n], nnzA = A_colptr[n];
    QpRows R;
    if (const char* err = qp_classify_rows(m, nnzA, A_rowidx, is_eq, R)) return fail(BGG_EINVAL, err);
    const std::vector<int> &row_slot = R.row_slot, &in_rows = R.in_rows, &eq_rows = R.eq_rows;
    const int mi = static_cast<int>(in_rows.size()), me = static_cast<int>(eq_rows.size());
    const size_t wsd = qp_ws_doubles(n, mi, me);
    DevPool dev(h->stream);
    int *dPc = dev.get<int>(n + 1), *dPr = dev.get<int>(nnzP), *dAc = dev.get<int>(n + 1), *dAr = dev.get<int>(nnzA), *dIn = dev.get<int>(mi), *dEq = dev.get<int>(me),
        *dSlot = dev.get<int>(m);
    double *dPv = dev.get<double>(static_cast<size_t>(count) * nnzP), *dAv = dev.get<double>(static_cast<size_t>(count) * nnzA), *dq = dev.get<double>(static_cast<size_t>(count) * n),
           *db = dev.get<double>(static_cast<size_t>(count) * m), *dws = dev.get<double>(static_cast<size_t>(count) * wsd), *dx = dev.get<double>(static_cast<size_t>(count) * n),
           *dy = dev.get<double>(static_cast<size_t>(count) * m), *dsl = dev.get<double>(static_cast<size_t>(count) * m);
    int32_t *dst = dev.get<int32_t>(count), *dit = dev.get<int32_t>(count);
    if (!dPc || !dPr || !dAc || !dAr || !dIn || !dEq || !dSlot || !dPv || !dAv || !dq || !db || !dws || !dx || !dy || !dsl || !dst || !dit)
        return fail(BGG_ENOMEM, "device allocation failed");
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(dPc, P_colptr, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dPr, P_rowidx, 4 * static_cast<size_t>(nnzP), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAc, A_colptr, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAr, A_rowidx, 4 * static_cast<size_t>(nnzA), cudaMemcpyHostToDevice, st));
    if (mi) CU(cudaMemcpyAsync(dIn, in_rows.data(), 4 * static_cast<size_t>(mi), cudaMemcpyHostToDevice, st));
    if (me) CU(cudaMemcpyAsync(dEq, eq_rows.data(), 4 * static_cast<size_t>(me), cudaMemcpyHostToDevice, st));
    if (m) CU(cudaMemcpyAsync(dSlot, row_slot.data(), 4 * static_cast<size_t>(m), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dPv, P_val, 8 * static_cast<size_t>(count) * nnzP, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAv, A_val, 8 * static_cast<size_t>(count) * nnzA, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dq, q, 8 * static_cast<size_t>(count) * n, cudaMemcpyHostToDevice, st));
    if (m) CU(cudaMemcpyAsync(db, b, 8 * static_cast<size_t>(count) * m, cudaMemcpyHostToDevice, st));
    if (launch_qp_generic(count, n, m, mi, me, nnzP, nnzA, dPc, dPr, dPv, dAc, dAr, dAv, dq, db, dIn, dEq, dSlot, dws, dx, dy, dsl, dst, dit, h->P.ipm_tol_feas,
                          h->P.ipm_tol_gap, h->P.ipm_tol_infeas, h->P.ipm_reg_eps, h->P.ipm_eq_delta, h->P.ipm_max_iter, h->max_smem, st))
        return fail(BGG_EINVAL, "the QP needs more shared memory than the device offers");
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(x, dx, 8 * static_cast<size_t>(count) * n, cudaMemcpyDeviceToHost, st));
    if (y && m) CU(cudaMemcpyAsync(y, dy, 8 * static_cast<size_t>(count) * m, cudaMemcpyDeviceToHost, st));
    if (s && m) CU(cudaMemcpyAsync(s, dsl, 8 * static_cast<size_t>(count) * m, cudaMemcpyDeviceToHost, st));
    if (status) CU(cudaMemcpyAsync(status, dst, 4 * static_cast<size_t>(count), cudaMemcpyDeviceToHost, st));
    if (iters) CU(cudaMemcpyAsync(iters, dit, 4 * static_cast<size_t>(count), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return BGG_OK;
}

int bgg_qp_adjoint_batch(bgg_handle* h, int count, int n, int m, const int32_t* P_colptr, const int32_t* P_rowidx, const double* P_val,
                         const int32_t* A_colptr, const int32_t* A_rowidx, const double* A_val, const uint8_t* is_eq, const double* x,
                         const double* y, const double* s, const double* dx, double* dz, double* dy, double* db, double* dA, int32_t* status) {
    if (!h || count <= 0 || n <= 0 || m < 0 || !P_colptr || !P_rowidx || !P_val || !A_colptr || !A_rowidx || !A_val || !is_eq || !x || !dx ||
        (m > 0 && (!y || !s)))
        return fail(BGG_EINVAL, "null argument");
    if (n > kQpMaxN_capi) return fail(BGG_EINVAL, "bgg_qp_adjoint_batch handles at most 128 variables, as bgg_qp_solve_batch");
    CU(cudaSetDevice(h->device));
    const int nnzP = P_colptr[n], nnzA = A_colptr[n];
    QpRows R;
    if (const char* err = qp_classify_rows(m, nnzA, A_rowidx, is_eq, R)) return fail(BGG_EINVAL, err);
    const int mi = static_cast<int>(R.in_rows.size()), me = static_cast<int>(R.eq_rows.size());
    if (n + me > kQpAdjMaxDim_capi)
        return fail(BGG_EINVAL, "bgg_qp_adjoint_batch handles n + me <= 160 (variables plus equality rows; here " + std::to_string(n + me) +
                                    "): the bordered system is factored in shared memory");
    const size_t C = static_cast<size_t>(count), wsd = qp_adj_ws_doubles(n, mi, me);
    DevPool dev(h->stream);
    int *dPc = dev.get<int>(n + 1), *dPr = dev.get<int>(nnzP), *dAc = dev.get<int>(n + 1), *dAr = dev.get<int>(nnzA), *dIn = dev.get<int>(mi),
        *dEq = dev.get<int>(me), *dSlot = dev.get<int>(m);
    double *dPv = dev.get<double>(C * nnzP), *dAv = dev.get<double>(C * nnzA), *dxx = dev.get<double>(C * n), *dyy = dev.get<double>(C * m),
           *dss = dev.get<double>(C * m), *ddx = dev.get<double>(C * n), *dws = dev.get<double>(C * wsd);
    double *odz = dz ? dev.get<double>(C * n) : nullptr, *ody = (dy && m) ? dev.get<double>(C * m) : nullptr,
           *odb = (db && m) ? dev.get<double>(C * m) : nullptr, *odA = (dA && nnzA) ? dev.get<double>(C * nnzA) : nullptr;
    int32_t* dst = dev.get<int32_t>(C);
    if (!dPc || !dPr || !dAc || !dAr || !dIn || !dEq || !dSlot || !dPv || !dAv || !dxx || !dyy || !dss || !ddx || !dws || !dst ||
        (dz && !odz) || (dy && m && !ody) || (db && m && !odb) || (dA && nnzA && !odA))
        return fail(BGG_ENOMEM, "device allocation failed");
    cudaStream_t st = h->stream;
    CU(cudaMemcpyAsync(dPc, P_colptr, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dPr, P_rowidx, 4 * static_cast<size_t>(nnzP), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAc, A_colptr, 4 * (n + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAr, A_rowidx, 4 * static_cast<size_t>(nnzA), cudaMemcpyHostToDevice, st));
    if (mi) CU(cudaMemcpyAsync(dIn, R.in_rows.data(), 4 * static_cast<size_t>(mi), cudaMemcpyHostToDevice, st));
    if (me) CU(cudaMemcpyAsync(dEq, R.eq_rows.data(), 4 * static_cast<size_t>(me), cudaMemcpyHostToDevice, st));
    if (m) CU(cudaMemcpyAsync(dSlot, R.row_slot.data(), 4 * static_cast<size_t>(m), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dPv, P_val, 8 * C * nnzP, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dAv, A_val, 8 * C * nnzA, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dxx, x, 8 * C * n, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ddx, dx, 8 * C * n, cudaMemcpyHostToDevice, st));
    if (m) CU(cudaMemcpyAsync(dyy, y, 8 * C * m, cudaMemcpyHostToDevice, st));
    if (m) CU(cudaMemcpyAsync(dss, s, 8 * C * m, cudaMemcpyHostToDevice, st));
    if (launch_qp_adjoint(count, n, m, mi, me, nnzP, nnzA, dPc, dPr, dPv, dAc, dAr, dAv, dIn, dEq, dSlot, dxx, dyy, dss, ddx, dws, odz, ody, odb,
                          odA, dst, h->max_smem, st))
        return fail(BGG_EINVAL, "the adjoint system needs more shared memory than the device offers");
    h->launches += 1;
    CU(cudaGetLastError());
    if (dz) CU(cudaMemcpyAsync(dz, odz, 8 * C * n, cudaMemcpyDeviceToHost, st));
    if (dy && m) CU(cudaMemcpyAsync(dy, ody, 8 * C * m, cudaMemcpyDeviceToHost, st));
    if (db && m) CU(cudaMemcpyAsync(db, odb, 8 * C * m, cudaMemcpyDeviceToHost, st));
    if (dA && nnzA) CU(cudaMemcpyAsync(dA, odA, 8 * C * nnzA, cudaMemcpyDeviceToHost, st));
    if (status) CU(cudaMemcpyAsync(status, dst, 4 * C, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return BGG_OK;
}

static int ensure_ls_children(bgg_handle* h, size_t C) {
    if (static_cast<int>(C) <= h->ls_cap) return BGG_OK;
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->d_ls_inst); cudaFree(h->d_ls_ws); cudaFree(h->d_ls_state); cudaFree(h->d_ls_t0); cudaFree(h->d_ls_ee);
    h->ls_cap = 0;
    CU(cudaMalloc(&h->d_ls_inst, sizeof(Instance) * C));
    CU(cudaMalloc(&h->d_ls_ws, h->L.stride * C));
    CU(cudaMalloc(&h->d_ls_state, 8 * kNxMan * C));
    CU(cudaMalloc(&h->d_ls_t0, 8 * C));
    CU(cudaMalloc(&h->d_ls_ee, 8 * 12 * C));
    CU(cudaMemsetAsync(h->d_ls_ws, 0, h->L.stride * C, h->stream));
    h->ls_cap = static_cast<int>(C);
    return BGG_OK;
}

int bgg_controller_tick_batch(bgg_handle* h, int mode, int K, const double* state, const double* t0, const double* ee_start, int32_t* status,
                              int32_t* iters, double* alpha, double* cost, double* z, int z_stride, int32_t* deriv_ready, double* dHdtheta,
                              int32_t* ls_best, double* ls_costs, int32_t* ls_quality) {
    if (!h || !h->batch || !state || !t0 || !ee_start) return fail(BGG_EINVAL, "null argument / no batch");
    if (mode < BGG_TICK_SOLVE || mode > BGG_TICK_LINE_SEARCH) return fail(BGG_EINVAL, "mode must be BGG_TICK_SOLVE, BGG_TICK_SOLVE_GAIT_OPT or BGG_TICK_LINE_SEARCH");
    if (mode == BGG_TICK_LINE_SEARCH && K <= 0) return fail(BGG_EINVAL, "the line search needs K > 0 candidates");
    if (!h->costs_set) return fail(BGG_ESTATE, "bgg_set_costs has not been called");
    CU(cudaSetDevice(h->device));
    const size_t B = h->batch, nv = B * kNumEE * kMaxContacts;
    if (!h->d_tick) {   // first tick of this batch
        CU(cudaMalloc(&h->d_tick, 8 * 4 * nv));
        CU(cudaMalloc(&h->d_tick_i, 4 * (B * kNumEE + 2 * B)));
        CU(cudaMallocHost(&h->h_tick, 8 * nv));
        CU(cudaMallocHost(&h->h_tick_i, 4 * 2 * B));
        CU(cudaMemsetAsync(h->d_tick, 0, 8 * 4 * nv, h->stream));
        CU(cudaMemsetAsync(h->d_tick_i, 0, 4 * (B * kNumEE + 2 * B), h->stream));
    }
    double *d_step = h->d_tick, *d_xk = h->d_tick + nv, *d_times = h->d_tick + 2 * nv, *d_dH = h->d_tick + 3 * nv;
    int32_t *d_lpst = h->d_tick_i, *d_ready = h->d_tick_i + B * kNumEE, *d_best = d_ready + B;
    int rc = bgg_upload_inputs(h, state, t0, ee_start);
    if (rc) return rc;
    if (mode == BGG_TICK_LINE_SEARCH) {
        // GaitOptimizer::LineSearch (gait_optimizer.cpp:671-753) from the step of the last GaitOpt tick: K copies, one RTI solve each,
        // arg-min, SetWarmStartTrajectory(best); instances without a derivative search along a zero step (a plain update)
        const size_t C = B * K;
        if ((rc = ensure_ls_children(h, C))) return rc;
        if (static_cast<int>(C) > h->tick_ls_cap) {
            CU(cudaStreamSynchronize(h->stream));
            cudaFree(h->d_tick_ls); cudaFree(h->d_tick_lsq);
            h->tick_ls_cap = 0;
            CU(cudaMalloc(&h->d_tick_ls, 8 * C));
            CU(cudaMalloc(&h->d_tick_lsq, 4 * C));
            h->tick_ls_cap = static_cast<int>(C);
        }
        k_mask_step<<<static_cast<unsigned>((nv + 255) / 256), 256, 0, h->stream>>>(d_step, d_ready, h->batch);
        launch_ls_expand(h->d_inst, h->d_ls_inst, h->batch, K, d_xk, d_step, h->d_state, h->d_t0, h->d_ee, h->d_ls_state, h->d_ls_t0, h->d_ls_ee, h->stream);
        if ((rc = solve_pipeline(h, h->caps_ls, h->d_ls_inst, h->d_ls_ws, h->d_ls_state, h->d_ls_t0, h->d_ls_ee, static_cast<int>(C), false))) return rc;
        launch_ls_select(h->d_inst, h->d_ls_inst, h->L, h->d_ls_ws, h->batch, K, d_best, h->d_tick_ls, h->d_tick_lsq, h->stream);
        CU(cudaMemsetAsync(d_ready, 0, 4 * B, h->stream));   // deriv_ready_ = false (mpc_controller.cpp:335)
        h->launches += 3;
    } else {
        if ((rc = solve_pipeline(h, h->caps_main, h->d_inst, h->d_ws, h->d_state, h->d_t0, h->d_ee, h->batch, h->profiling))) return rc;
        if (mode == BGG_TICK_SOLVE_GAIT_OPT) {
            // MPCController::GaitOpt (:518-573): derivative terms and dH/dtheta, then the contact-time LP; the step stays on the device.
            // The gradient kernel's dense system is sized exactly: this solve's own maxima (its k_prepare is done by now or in a few
            // microseconds; the solve kernels are queued behind it, so the device stays busy while the host looks).
            refresh_caps(h->caps_main);
            h->last_nu_max = h->caps_main.nu;
            h->last_ns_max = h->caps_main.ns;
            if (launch_gradient(h->P, h->d_inst, h->L, h->d_ws, h->batch, h->last_nu_max, h->last_ns_max, h->max_smem - 14 * 1024, h->stream))
                return fail(BGG_EINVAL, "the gait-gradient kernel needs more shared memory than the device offers for this many spline variables");
            k_deriv_ready<<<(h->batch + 127) / 128, 128, 0, h->stream>>>(h->L, h->d_ws, h->batch, d_ready, d_dH);
            launch_gait_lp(h->d_inst, h->L, h->d_ws, h->batch, nullptr, h->d_t0, 1.0, 1.0, d_step, d_xk, d_times, d_lpst, h->stream);
            h->launches += 3;
        } else {
            CU(cudaMemsetAsync(d_ready, 0, 4 * B, h->stream));   // :344
        }
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h->h_tick_i, d_ready, 4 * 2 * B, cudaMemcpyDeviceToHost, h->stream));
    if (mode == BGG_TICK_SOLVE_GAIT_OPT && dHdtheta) CU(cudaMemcpyAsync(h->h_tick, d_dH, 8 * nv, cudaMemcpyDeviceToHost, h->stream));
    rc = bgg_download_results(h, status, iters, alpha, cost, z, z_stride);   // the tick's only wait for the device
    if (rc) return rc;
    if (deriv_ready) std::memcpy(deriv_ready, h->h_tick_i, 4 * B);
    if (ls_best) {
        if (mode == BGG_TICK_LINE_SEARCH) std::memcpy(ls_best, h->h_tick_i + B, 4 * B);
        else for (size_t b = 0; b < B; ++b) ls_best[b] = -1;
    }
    if (mode == BGG_TICK_SOLVE_GAIT_OPT && dHdtheta) std::memcpy(dHdtheta, h->h_tick, 8 * nv);
    if (mode == BGG_TICK_LINE_SEARCH) {   // per-candidate record (diagnostics; the stream is idle here)
        if (ls_costs) CU(cudaMemcpy(ls_costs, h->d_tick_ls, 8 * B * K, cudaMemcpyDeviceToHost));
        if (ls_quality) CU(cudaMemcpy(ls_quality, h->d_tick_lsq, 4 * B * K, cudaMemcpyDeviceToHost));
    }
    return BGG_OK;
}

int bgg_controller_get_step(bgg_handle* h, double* step, double* xk, double* new_times) {
    if (!h || !h->batch || !h->d_tick) return fail(BGG_ESTATE, "no controller tick has run");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    const size_t nv = static_cast<size_t>(h->batch) * kNumEE * kMaxContacts;
    if (step) CU(cudaMemcpy(step, h->d_tick, 8 * nv, cudaMemcpyDeviceToHost));
    if (xk) CU(cudaMemcpy(xk, h->d_tick + nv, 8 * nv, cudaMemcpyDeviceToHost));
    if (new_times) CU(cudaMemcpy(new_times, h->d_tick + 2 * nv, 8 * nv, cudaMemcpyDeviceToHost));
    return BGG_OK;
}

int bgg_synchronize(bgg_handle* h) {
    if (!h) return fail(BGG_EINVAL, "null handle");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    return BGG_OK;
}

int bgg_set_profiling(bgg_handle* h, int enable) {
    if (!h) return fail(BGG_EINVAL, "null handle");
    h->profiling = enable != 0;
    return BGG_OK;
}

int bgg_last_kernel_ms(bgg_handle* h, float ms[4]) {
    if (!h || !ms) return fail(BGG_EINVAL, "null argument");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    if (h->profiling)
        for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&h->last_ms[i], h->ev[i], h->ev[i + 1]);
    for (int i = 0; i < 4; ++i) ms[i] = h->last_ms[i];
    return BGG_OK;
}

int bgg_kernel_launch_count(bgg_handle* h, int64_t* launches) {
    if (!h || !launches) return fail(BGG_EINVAL, "null argument");
    *launches = h->launches;
    return BGG_OK;
}

int bgg_event_record(bgg_handle* h, int slot) {
    if (!h || slot < 0 || slot >= 8) return fail(BGG_EINVAL, "bad event slot");
    CU(cudaSetDevice(h->device));
    CU(cudaEventRecord(h->user_ev[slot], h->stream));
    return BGG_OK;
}

int bgg_event_elapsed_ms(bgg_handle* h, int a, int b, float* ms) {
    if (!h || !ms || a < 0 || a >= 8 || b < 0 || b >= 8) return fail(BGG_EINVAL, "bad event slot");
    CU(cudaSetDevice(h->device));
    CU(cudaEventSynchronize(h->user_ev[b]));
    CU(cudaEventElapsedTime(ms, h->user_ev[a], h->user_ev[b]));
    return BGG_OK;
}

static int fetch(bgg_handle* h, void* dst, const void* dsrc, size_t bytes) {
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(dst, dsrc, bytes, cudaMemcpyDeviceToHost));
    return BGG_OK;
}

int bgg_get_sizes(bgg_handle* h, int b, bgg_sizes* out) {
    if (!h || !out || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    WsHeader w;
    const int rc = fetch(h, &w, h->d_ws + static_cast<size_t>(b) * h->L.stride + h->L.hdr, sizeof w);
    if (rc) return rc;
    out->n = w.n; out->nu = w.nu; out->nf = w.nf; out->np = w.np; out->n_samples = w.n_samples; out->n_eebox = w.n_eebox;
    out->n_eq = w.n_eq; out->n_td = w.n_td; out->m_ineq = w.m_ineq; out->status = w.status; out->iters = w.iters;
    out->ls_iters = w.ls_iters; out->error = w.error;
    for (int e = 0; e < kNumEE; ++e) {
        out->nfv[e] = w.nfv[e]; out->npv[e] = w.npv[e]; out->fbase[e] = w.fbase[e]; out->pbase[e] = w.pbase[e];
    }
    out->t0 = w.t0; out->alpha = w.alpha; out->cost = w.cost; out->prim_res = w.prim_res; out->dual_res = w.dual_res;
    out->gap = w.gap; out->eq_violation = w.eq_violation; out->step_norm = w.step_norm; out->merit = w.merit;
    out->merit_dd = w.merit_dd; out->ee_box[0] = w.ee_box[0]; out->ee_box[1] = w.ee_box[1];
    out->qp_cost = w.qp_cost;
    out->refined_iters = w.refined_iters;
    out->no_iterate = w.no_iterate;
    return BGG_OK;
}

int bgg_param_partials(bgg_handle* h, int b, int ee, int contact_idx, int cap, int32_t* counts, int32_t* Ar, int32_t* Ac, double* Av, int32_t* Gr,
                       int32_t* Gc, double* Gv, double* db) {
    if (!h || b < 0 || b >= h->batch || ee < 0 || ee >= kNumEE || contact_idx < 0 || cap <= 0 || !counts || !Ar || !Ac || !Av || !Gr || !Gc || !Gv || !db)
        return fail(BGG_EINVAL, "bad argument");
    bgg_sizes sz;
    int rc = bgg_get_sizes(h, b, &sz);
    if (rc) return rc;
    if (sz.error) return fail(BGG_ESTATE, "the instance has no QP (k_prepare refused it)");
    if (sz.status != kSolved) return 1;   // the reference returns false (mpc_single_rigid_body.cpp:644-647)
    {
        std::vector<double> t(kNumEE * kMaxContacts);
        std::vector<int32_t> ty(kNumEE * kMaxContacts), n(kNumEE);
        rc = bgg_get_contact_times(h, b, 1, t.data(), ty.data(), n.data());
        if (rc) return rc;
        if (contact_idx >= n[ee]) return fail(BGG_EINVAL, "contact_idx is beyond the foot's contact times");
    }
    CU(cudaSetDevice(h->device));
    const int N = h->P.N, nu_cap = h->L.max_nu;
    const size_t nd = param_partials_doubles(N, nu_cap);
    DevPool pool(h->stream);
    double* d_out = pool.get<double>(nd);
    double* d_ut = pool.get<double>(nu_cap);
    if (!d_out || !d_ut) return fail(BGG_ECUDA, "out of device memory");
    launch_param_partials(h->P, h->d_inst, h->L, h->d_ws, b, ee, contact_idx, nu_cap, d_out, d_ut, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    std::vector<double> o(nd);
    CU(cudaMemcpyAsync(o.data(), d_out, 8 * nd, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    // ---- blocks -> triplets in the reference's numbering: columns [states 12 (N + 1) | force variables | position variables]; equality
    // rows [dynamics | touch-down | foot start]; inequality rows [force box + / - | friction pyramid | foot box + / -]
    const double dt = h->P.dt, mu = h->P.friction_coef;
    const int nf = static_cast<int>(o[1]), ns = static_cast<int>(o[22]), ntd = static_cast<int>(o[23]);
    const int fsi = kNx * (N + 1), psi = fsi + nf;
    const int num_dyn = kNx * (N + 1), num_loc = 16 * (N - 3), num_start = 2 * kNumEE;
    const int eq_td = num_dyn, eq_start = num_dyn + ntd, in_cone = 2 * ns, in_loc = 6 * ns;
    const int num_eq = num_dyn + ntd + num_start, num_in = 6 * ns + num_loc;
    int na = 0, ng = 0;
    bool overflow = false;
    auto putA = [&](int r, int c, double v) {
        if (v == 0.0) return;
        if (na < cap) { Ar[na] = r; Ac[na] = c; Av[na] = v; }
        else overflow = true;
        ++na;
    };
    auto putG = [&](int r, int c, double v) {
        if (v == 0.0) return;
        if (ng < cap) { Gr[ng] = r; Gc[ng] = c; Gv[ng] = v; }
        else overflow = true;
        ++ng;
    };
    for (int i = 0; i < num_eq; ++i) db[i] = 0.0;
    const double* dyn = o.data() + kPartHdr;
    const size_t dyn_stride = 9 + 6 * static_cast<size_t>(nu_cap) + 6;
    const int rowmap[6] = {3, 4, 5, 9, 10, 11};
    for (int k = 0; k < N; ++k) {   // :651-668: dt * dA, dt * dB, db = -dt * dC
        const double* dA = dyn + k * dyn_stride;
        const double* dB = dA + 9;
        const double* dC = dB + 6 * static_cast<size_t>(nu_cap);
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) putA((k + 1) * kNx + 9 + r, k * kNx + c, dt * dA[3 * r + c]);
        for (int r = 0; r < 6; ++r) {
            for (int j = 0; j < sz.nu; ++j) putA((k + 1) * kNx + rowmap[r], fsi + j, dt * dB[static_cast<size_t>(r) * nu_cap + j]);
            db[(k + 1) * kNx + rowmap[r]] = -(dt * dC[r]);
        }
    }
    const double* frc = dyn + N * dyn_stride;
    const double* loc = frc + 10 * 3 * 6;
    const double* start = loc + static_cast<size_t>(N + 1) * 2 * 4;
    const double* tdp = start + 2 * 4;
    if (o[18] != 0.0) {   // mpc.cpp:416-531 (force box on z, + rows then - rows) and :240-350 (friction pyramid)
        const int row0 = static_cast<int>(o[19]);
        const double pyr[4][3] = {{1, 0, -mu}, {-1, 0, -mu}, {0, 1, -mu}, {0, -1, -mu}};
        for (int j = 0; j < 2; ++j)
            for (int i = 0; i < kSamplesPerStance; ++i) {
                const double* p = frc + (static_cast<size_t>(i) * 3 + 2) * 6;
                for (int a = 0; a < static_cast<int>(p[1]); ++a) putG(j * ns + row0 + i, fsi + static_cast<int>(p[0]) + a, (j == 0 ? 1.0 : -1.0) * p[2 + a]);
            }
        for (int i = 0; i < kSamplesPerStance; ++i)
            for (int c = 0; c < 3; ++c) {
                const double* p = frc + (static_cast<size_t>(i) * 3 + c) * 6;
                for (int fc = 0; fc < 4; ++fc)
                    for (int a = 0; a < static_cast<int>(p[1]); ++a)
                        putG(in_cone + 4 * (row0 + i) + fc, fsi + static_cast<int>(p[0]) + a, pyr[fc][c] * p[2 + a]);
            }
    }
    {   // :705-733 foot box of this foot at nodes 4 .. N, + rows then - rows
        int idx = 2 * ee;
        for (int node = kEENodeStart; node <= N; ++node) {
            for (int c = 0; c < 2; ++c) {
                const double* p = loc + (static_cast<size_t>(node) * 2 + c) * 4;
                for (int a = 0; a < static_cast<int>(p[1]); ++a) {
                    putG(in_loc + idx, psi + static_cast<int>(p[0]) + a, p[2 + a]);
                    putG(in_loc + idx + num_loc / 2, psi + static_cast<int>(p[0]) + a, -p[2 + a]);
                }
                idx++;
            }
            idx += 2 * (kNumEE - 1);
        }
    }
    if (o[20] != 0.0) {   // :889-927 touch-down rows
        const int trow = static_cast<int>(o[21]);
        for (int c = 0; c < 2; ++c) {
            const double* p = tdp + 5 * c;
            if (trow + c < ntd) db[eq_td + trow + c] = p[4];
            for (int a = 0; a < static_cast<int>(p[1]); ++a) putA(eq_td + trow + c, psi + static_cast<int>(p[0]) + a, p[2 + a]);
        }
    }
    for (int c = 0; c < 2; ++c) {   // :733-752: every foot's start-row partial lands on rows 0-1 of the block (kept)
        const double* p = start + 4 * c;
        for (int a = 0; a < static_cast<int>(p[1]); ++a) putA(eq_start + c, psi + static_cast<int>(p[0]) + a, p[2 + a]);
    }
    counts[0] = na; counts[1] = ng; counts[2] = num_eq; counts[3] = num_in;
    if (overflow) return fail(BGG_EINVAL, "cap is smaller than the number of non-zeros");
    return BGG_OK;
}

int bgg_get_dynamics(bgg_handle* h, int first, int count, double* Ad, double* Bd, double* cd, int nu_stride) {
    if (!h || !Ad || !Bd || !cd || first < 0 || count <= 0 || first + count > h->batch) return fail(BGG_EINVAL, "bad range");
    for (int b = first; b < first + count; ++b) {
        bgg_sizes sz;
        const int rc = bgg_get_sizes(h, b, &sz);
        if (rc) return rc;
        if (sz.nu > nu_stride) return fail(BGG_EINVAL, "nu_stride is smaller than an instance's number of spline variables");
    }
    CU(cudaSetDevice(h->device));
    const size_t N = h->P.N;
    double *dA, *dB, *dc;
    CU(cudaMalloc(&dA, 8 * count * N * 144));
    CU(cudaMalloc(&dB, 8 * count * N * kNx * nu_stride));
    CU(cudaMalloc(&dc, 8 * count * N * kNx));
    launch_export_dynamics(h->P, h->L, h->d_ws + static_cast<size_t>(first) * h->L.stride, count, dA, dB, dc, nu_stride, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(Ad, dA, 8 * count * N * 144, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(Bd, dB, 8 * count * N * kNx * nu_stride, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cd, dc, 8 * count * N * kNx, cudaMemcpyDeviceToHost));
    cudaFree(dA);
    cudaFree(dB);
    cudaFree(dc);
    return BGG_OK;
}

int bgg_get_condensed(bgg_handle* h, int b, double* H, double* g, double* phipos, double* xoff) {
    if (!h || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    bgg_sizes sz;
    int rc = bgg_get_sizes(h, b, &sz);
    if (rc) return rc;
    const char* ws = h->d_ws + static_cast<size_t>(b) * h->L.stride;
    const int nu = sz.nu, N = h->P.N;
    if (H && (rc = fetch(h, H, ws + h->L.H, 8 * static_cast<size_t>(nu) * nu))) return rc;
    if (g && (rc = fetch(h, g, ws + h->L.g, 8 * static_cast<size_t>(nu)))) return rc;
    if (phipos) {
        std::vector<double> tmp(static_cast<size_t>(2 * (N - 3)) * h->L.max_nu);
        if ((rc = fetch(h, tmp.data(), ws + h->L.phipos, 8 * tmp.size()))) return rc;
        for (int r = 0; r < 2 * (N - 3); ++r)
            for (int i = 0; i < nu; ++i) phipos[static_cast<size_t>(r) * nu + i] = tmp[static_cast<size_t>(r) * h->L.max_nu + i];
    }
    if (xoff && (rc = fetch(h, xoff, ws + h->L.xoff, 8 * static_cast<size_t>(kNx) * (N + 1)))) return rc;
    return BGG_OK;
}

int bgg_export_qp_csc(bgg_handle* h, int first, int count, int32_t* dims, int32_t* colptr, int32_t* rowidx, double* val,
                      int nnz_cap, double* p_diag, double* q, double* ub, int n_stride, int m_stride) {
    if (!h || !dims || !colptr || !rowidx || !val || !p_diag || !q || !ub || first < 0 || count <= 0 || first + count > h->batch)
        return fail(BGG_EINVAL, "bad argument");
    const int n_max = kNx * (h->P.N + 1) + h->P.max_nu;
    const int m_max = kNx * (h->P.N + 1) + h->L.max_rows + kMaxEq;
    if (n_stride < n_max || m_stride < m_max || nnz_cap <= 0)
        return fail(BGG_EINVAL, "strides must cover 12(N+1)+max_spline_vars columns and every constraint row");
    CU(cudaSetDevice(h->device));
    const size_t c = count;
    int32_t *d_dims, *d_cp, *d_ri;
    double *d_val, *d_pd, *d_q, *d_ub;
    CU(cudaMalloc(&d_dims, 4 * 6 * c));
    CU(cudaMalloc(&d_cp, 4 * c * (n_stride + 1)));
    CU(cudaMalloc(&d_ri, 4 * c * nnz_cap));
    CU(cudaMalloc(&d_val, 8 * c * nnz_cap));
    CU(cudaMalloc(&d_pd, 8 * c * n_stride));
    CU(cudaMalloc(&d_q, 8 * c * n_stride));
    CU(cudaMalloc(&d_ub, 8 * c * m_stride));
    CU(cudaMemsetAsync(d_cp, 0, 4 * c * (n_stride + 1), h->stream));
    CU(cudaMemsetAsync(d_ri, 0, 4 * c * nnz_cap, h->stream));
    CU(cudaMemsetAsync(d_val, 0, 8 * c * nnz_cap, h->stream));
    CU(cudaMemsetAsync(d_pd, 0, 8 * c * n_stride, h->stream));
    CU(cudaMemsetAsync(d_q, 0, 8 * c * n_stride, h->stream));
    CU(cudaMemsetAsync(d_ub, 0, 8 * c * m_stride, h->stream));
    launch_export_csc(h->P, h->L, h->d_ws + static_cast<size_t>(first) * h->L.stride, count, d_cp, d_ri, d_val, d_pd, d_q, d_ub,
                      d_dims, n_stride, m_stride, nnz_cap, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(dims, d_dims, 4 * 6 * c, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(colptr, d_cp, 4 * c * (n_stride + 1), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(rowidx, d_ri, 4 * c * nnz_cap, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(val, d_val, 8 * c * nnz_cap, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(p_diag, d_pd, 8 * c * n_stride, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(q, d_q, 8 * c * n_stride, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ub, d_ub, 8 * c * m_stride, cudaMemcpyDeviceToHost));
    cudaFree(d_dims); cudaFree(d_cp); cudaFree(d_ri); cudaFree(d_val); cudaFree(d_pd); cudaFree(d_q); cudaFree(d_ub);
    return BGG_OK;
}

int bgg_get_solution(bgg_handle* h, int b, double* qp_sol, double* z, double* lam, double* slack, double* nu_eq) {
    if (!h || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    bgg_sizes sz;
    int rc = bgg_get_sizes(h, b, &sz);
    if (rc) return rc;
    const char* ws = h->d_ws + static_cast<size_t>(b) * h->L.stride;
    if (qp_sol && (rc = fetch(h, qp_sol, ws + h->L.zqp, 8 * static_cast<size_t>(sz.n)))) return rc;
    if (z && (rc = fetch(h, z, ws + h->L.zprev, 8 * static_cast<size_t>(sz.n)))) return rc;
    if (lam && (rc = fetch(h, lam, ws + h->L.lam, 8 * static_cast<size_t>(sz.m_ineq)))) return rc;
    if (slack && (rc = fetch(h, slack, ws + h->L.slack, 8 * static_cast<size_t>(sz.m_ineq)))) return rc;
    if (nu_eq && (rc = fetch(h, nu_eq, ws + h->L.nueq, 8 * static_cast<size_t>(sz.n_eq)))) return rc;
    return BGG_OK;
}

int bgg_gait_gradient_batch(bgg_handle* h, int32_t* status, int32_t* n_contacts, double* dHdtheta) {
    if (!h || !h->batch) return fail(BGG_EINVAL, "no batch");
    if (!h->last_nu_max) return fail(BGG_ESTATE, "bgg_gait_gradient_batch needs a solve first");
    CU(cudaSetDevice(h->device));
    const int B = h->batch;
    refresh_caps(h->caps_main);   // the main batch's own maxima of its last solve (not the line-search children's)
    if (h->caps_main.nu > 0) {
        h->last_nu_max = h->caps_main.nu;
        h->last_ns_max = h->caps_main.ns;
    }
    // 14 KB of the opt-in shared memory are taken by the kernel's static arrays (the four staged foot splines)
    if (launch_gradient(h->P, h->d_inst, h->L, h->d_ws, B, h->last_nu_max, h->last_ns_max, h->max_smem - 14 * 1024, h->stream))
        return fail(BGG_EINVAL, "the gait-gradient kernel needs more shared memory than the device offers for this many spline variables");
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    std::vector<GradInfo> gi(B);
    std::vector<double> dh(static_cast<size_t>(B) * kNumEE * kMaxContacts);
    CU(cudaMemcpy2D(gi.data(), sizeof(GradInfo), h->d_ws + h->L.ginfo, h->L.stride, sizeof(GradInfo), B, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy2D(dh.data(), 8 * kNumEE * kMaxContacts, h->d_ws + h->L.gdH, h->L.stride, 8 * kNumEE * kMaxContacts, B,
                    cudaMemcpyDeviceToHost));
    for (int b = 0; b < B; ++b) {
        if (status) status[b] = gi[b].status;
        if (n_contacts)
            for (int e = 0; e < kNumEE; ++e) n_contacts[b * kNumEE + e] = gi[b].nct[e];
    }
    if (dHdtheta) std::memcpy(dHdtheta, dh.data(), 8 * dh.size());
    return BGG_OK;
}

int bgg_optimize_contact_times_batch(bgg_handle* h, const double* time, double trust, double alpha, const double* dHdtheta,
                                     double* step, double* xk, double* new_times, int32_t* status) {
    if (!h || !h->batch || !time || !step || !xk || !new_times) return fail(BGG_EINVAL, "null argument / no batch");
    CU(cudaSetDevice(h->device));
    const size_t B = h->batch, nv = B * kNumEE * kMaxContacts;
    DevPool pool(h->stream);
    double *d_time = pool.get<double>(B), *d_grad = nullptr, *d_out = pool.get<double>(3 * nv);
    int32_t* d_st = pool.get<int32_t>(B * kNumEE);
    if (!d_time || !d_out || !d_st) return fail(BGG_ECUDA, "out of device memory");
    CU(cudaMemcpyAsync(d_time, time, 8 * B, cudaMemcpyHostToDevice, h->stream));
    if (dHdtheta) {
        d_grad = pool.get<double>(nv);
        if (!d_grad) return fail(BGG_ECUDA, "out of device memory");
        CU(cudaMemcpyAsync(d_grad, dHdtheta, 8 * nv, cudaMemcpyHostToDevice, h->stream));
    }
    launch_gait_lp(h->d_inst, h->L, h->d_ws, h->batch, d_grad, d_time, trust, alpha, d_out, d_out + nv, d_out + 2 * nv, d_st, h->stream);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(step, d_out, 8 * nv, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(xk, d_out + nv, 8 * nv, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(new_times, d_out + 2 * nv, 8 * nv, cudaMemcpyDeviceToHost, h->stream));
    if (status) CU(cudaMemcpyAsync(status, d_st, 4 * B * kNumEE, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BGG_OK;
}

int bgg_line_search_batch(bgg_handle* h, int K, const double* xk, const double* step, const double* state, const double* t0,
                          const double* ee_start, int32_t* best, double* costs, int32_t* quality) {
    if (!h || !h->batch || K <= 0 || !xk || !step || !state || !t0 || !ee_start) return fail(BGG_EINVAL, "null argument / no batch");
    if (!h->costs_set) return fail(BGG_ESTATE, "bgg_set_costs has not been called");
    CU(cudaSetDevice(h->device));
    const size_t B = h->batch, C = B * K, nv = B * kNumEE * kMaxContacts;
    {
        const int rc0 = ensure_ls_children(h, C);
        if (rc0) return rc0;
    }
    int rc = bgg_upload_inputs(h, state, t0, ee_start);
    if (rc) return rc;
    DevPool pool(h->stream);
    double* d_vec = pool.get<double>(2 * nv);
    int32_t *d_best = pool.get<int32_t>(B), *d_q = pool.get<int32_t>(C);
    double* d_costs = pool.get<double>(C);
    if (!d_vec || !d_best || !d_q || !d_costs) return fail(BGG_ECUDA, "out of device memory");
    CU(cudaMemcpyAsync(d_vec, xk, 8 * nv, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d_vec + nv, step, 8 * nv, cudaMemcpyHostToDevice, h->stream));
    launch_ls_expand(h->d_inst, h->d_ls_inst, h->batch, K, d_vec, d_vec + nv, h->d_state, h->d_t0, h->d_ee, h->d_ls_state, h->d_ls_t0,
                     h->d_ls_ee, h->stream);
    rc = solve_pipeline(h, h->caps_ls, h->d_ls_inst, h->d_ls_ws, h->d_ls_state, h->d_ls_t0, h->d_ls_ee, static_cast<int>(C), false);
    if (rc) return rc;
    launch_ls_select(h->d_inst, h->d_ls_inst, h->L, h->d_ls_ws, h->batch, K, d_best, d_costs, d_q, h->stream);
    h->launches += 2;
    CU(cudaGetLastError());
    if (best) CU(cudaMemcpyAsync(best, d_best, 4 * B, cudaMemcpyDeviceToHost, h->stream));
    if (costs) CU(cudaMemcpyAsync(costs, d_costs, 8 * C, cudaMemcpyDeviceToHost, h->stream));
    if (quality) CU(cudaMemcpyAsync(quality, d_q, 4 * C, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return BGG_OK;
}

int bgg_get_adjoint(bgg_handle* h, int b, double* dz, double* dlam, double* dnu_dyn, double* dnu_eq, double* nu_dyn) {
    if (!h || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    bgg_sizes sz;
    int rc = bgg_get_sizes(h, b, &sz);
    if (rc) return rc;
    const char* ws = h->d_ws + static_cast<size_t>(b) * h->L.stride;
    const size_t nd = 8 * static_cast<size_t>(kNx) * (h->P.N + 1);
    if (dz && (rc = fetch(h, dz, ws + h->L.gdz, 8 * static_cast<size_t>(sz.n)))) return rc;
    if (dlam && (rc = fetch(h, dlam, ws + h->L.gdlam, 8 * static_cast<size_t>(sz.m_ineq)))) return rc;
    if (dnu_dyn && (rc = fetch(h, dnu_dyn, ws + h->L.gdnu, nd))) return rc;
    if (dnu_eq && (rc = fetch(h, dnu_eq, ws + h->L.gdnue, 8 * static_cast<size_t>(sz.n_eq)))) return rc;
    if (nu_dyn && (rc = fetch(h, nu_dyn, ws + h->L.dualx, nd))) return rc;
    return BGG_OK;
}

int bgg_get_contact_times(bgg_handle* h, int first, int count, double* times, int32_t* types, int32_t* counts) {
    if (!h || !times || !types || !counts || first < 0 || count <= 0 || first + count > h->batch) return fail(BGG_EINVAL, "bad range");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    std::vector<Instance> tmp(count);
    CU(cudaMemcpy(tmp.data(), h->d_inst + first, sizeof(Instance) * static_cast<size_t>(count), cudaMemcpyDeviceToHost));
    for (int b = 0; b < count; ++b)
        for (int e = 0; e < kNumEE; ++e) {
            const FootSpline& s = tmp[b].foot[e];
            int c = 0;
            for (int i = 0; i < BGG_MAX_CONTACTS; ++i) {
                times[(b * kNumEE + e) * BGG_MAX_CONTACTS + i] = 0.0;
                types[(b * kNumEE + e) * BGG_MAX_CONTACTS + i] = 0;
            }
            for (int i = 0; i < s.n && c < BGG_MAX_CONTACTS; ++i)
                if (s.ttype[i] != kInter) {
                    times[(b * kNumEE + e) * BGG_MAX_CONTACTS + c] = s.t[i];
                    types[(b * kNumEE + e) * BGG_MAX_CONTACTS + c] = s.ttype[i];
                    c++;
                }
            counts[b * kNumEE + e] = c;
        }
    return BGG_OK;
}

int bgg_set_solution(bgg_handle* h, int b, const double* qp_sol, const double* z, const double* lam, const double* slack,
                     const double* nu_eq) {
    if (!h || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    bgg_sizes sz;
    int rc = bgg_get_sizes(h, b, &sz);
    if (rc) return rc;
    char* ws = h->d_ws + static_cast<size_t>(b) * h->L.stride;
    const size_t ustart = static_cast<size_t>(kNx) * (h->P.N + 1);
    if (qp_sol) {
        CU(cudaMemcpy(ws + h->L.zqp, qp_sol, 8 * static_cast<size_t>(sz.n), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(ws + h->L.u, qp_sol + ustart, 8 * static_cast<size_t>(sz.nu), cudaMemcpyHostToDevice));
    }
    if (z) CU(cudaMemcpy(ws + h->L.zprev, z, 8 * static_cast<size_t>(sz.n), cudaMemcpyHostToDevice));
    if (lam) CU(cudaMemcpy(ws + h->L.lam, lam, 8 * static_cast<size_t>(sz.m_ineq), cudaMemcpyHostToDevice));
    if (slack) CU(cudaMemcpy(ws + h->L.slack, slack, 8 * static_cast<size_t>(sz.m_ineq), cudaMemcpyHostToDevice));
    if (nu_eq) CU(cudaMemcpy(ws + h->L.nueq, nu_eq, 8 * static_cast<size_t>(sz.n_eq), cudaMemcpyHostToDevice));
    const int32_t st = kSolved;
    CU(cudaMemcpy(ws + h->L.hdr + offsetof(WsHeader, status), &st, sizeof st, cudaMemcpyHostToDevice));
    return BGG_OK;
}

size_t bgg_instance_bytes(void) { return sizeof(Instance); }

int bgg_get_instance(bgg_handle* h, int b, void* out) {
    if (!h || !out || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    return fetch(h, out, h->d_inst + b, sizeof(Instance));
}

int bgg_set_instance(bgg_handle* h, int b, const void* in) {
    if (!h || !in || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(h->d_inst + b, in, sizeof(Instance), cudaMemcpyHostToDevice));
    return BGG_OK;
}

int bgg_get_states(bgg_handle* h, int b, double* states) {
    if (!h || !states || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad instance");
    return fetch(h, states, reinterpret_cast<const char*>(h->d_inst + b) + offsetof(Instance, states),
                 8 * static_cast<size_t>(kNxMan) * (h->P.N + 1));
}

int bgg_eval_splines(bgg_handle* h, int b, const double* times, int T, double* force, double* position) {
    if (!h || !times || !force || !position || T <= 0 || b < 0 || b >= h->batch) return fail(BGG_EINVAL, "bad argument");
    CU(cudaSetDevice(h->device));
    double *dt, *df, *dp;
    CU(cudaMalloc(&dt, 8 * T));
    CU(cudaMalloc(&df, 8 * T * 12));
    CU(cudaMalloc(&dp, 8 * T * 12));
    CU(cudaMemcpyAsync(dt, times, 8 * T, cudaMemcpyHostToDevice, h->stream));
    k_eval_splines<<<(T * kNumEE + 127) / 128, 128, 0, h->stream>>>(h->d_inst, b, dt, T, df, dp);
    h->launches += 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(force, df, 8 * T * 12, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(position, dp, 8 * T * 12, cudaMemcpyDeviceToHost));
    cudaFree(dt);
    cudaFree(df);
    cudaFree(dp);
    return BGG_OK;
}

}  // extern "C"
