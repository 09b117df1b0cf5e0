// Host runtime of the federation engine (C ABI, loaded with ctypes — no torch/pybind
// headers, so the whole library compiles in seconds and carries no ABI coupling).
//
// An Engine owns, for ONE GPU ("node"):
//   * the comm block (theta mailbox, epoch flag, slot array, slot flags) — allocated here
//     with cudaMalloc (exportable through CUDA IPC) or supplied from outside (torch
//     symmetric memory, which can also supply an NVSwitch multicast alias);
//   * host-mapped pinned memory for theta (root: written by the client thread, read by the
//     kernel over PCIe), for the result and for the completion flag (written by the kernel,
//     polled by the client thread — no cudaStreamSynchronize on the evaluation path);
//   * the model descriptor and the launch configuration.
//
// Root:  b200_engine_eval()  = memcpy theta -> launch -> spin on host flag -> copy result.
// Peers: b200_engine_serve() = keep `ahead` kernels enqueued; each one waits ON THE DEVICE
//        for the root's epoch flag, so a peer's host never sits on the critical path.
//
// The reference's counterpart of this file is its asyncio/gRPC client+server pair
// (/root/reference/pytensor_federated/service.py:75-158, :326-423).
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "fed_comm.cuh"
#include "models.h"

// A/B switch for the early TMA loads of the tensor-core GLM kernels (GlmParams::early_loads)
static bool early_loads_enabled() {
    const char* v = getenv("B200FED_NO_EARLY_LOADS");
    return !(v && *v && *v != '0');
}

extern "C" {
int b200_launch_linreg(const FedComm*, const LinregShard*, int, int, int, cudaStream_t);
int b200_launch_glm_simt(const FedComm*, const GlmSegment*, const GlmParams*, int, cudaStream_t);
size_t b200_glm_simt_smem(int, int, int);
int b200_launch_glm_tc(const FedComm*, const GlmSegment*, const GlmParams*, const void* tmaps, const void* chunks,
                       int n_chunks, unsigned int* work_counter, int grid, cudaStream_t);
int b200_glm_tc_prepare(const GlmSegment* segs_host, int n_segments, const GlmParams* prm, int sm_count, void** tmaps_dev,
                        void** chunks_dev, int* n_chunks);
size_t b200_glm_tc_partial_row_doubles(int n_vals, int n_chains, int n_out, int n_groups, int n_family_params);
int b200_launch_ode(const FedComm*, const OdeShard*, int, int, cudaStream_t);
int b200_launch_glm_fp8(const FedComm*, const GlmSegment*, const GlmParams*, const void* tmaps, const void* chunks,
                        int n_chunks, unsigned int* work_counter, int grid, cudaStream_t stream);
int b200_glm_fp8_prepare(const GlmSegment* segs_host, int n_segments, const GlmParams* prm, int sm_count, void** tmaps_dev,
                         void** chunks_dev, int* n_chunks);
size_t b200_glm_fp8_partial_row_doubles(int n_vals, int n_chains, int n_out, int n_groups);
int b200_launch_glm_generic(const FedComm*, const GlmSegment*, const GlmParams*, int elem_bytes, int grid, cudaStream_t);
}

namespace {

enum ModelKind { MODEL_NONE = 0, MODEL_LINREG = 1, MODEL_GLM_SIMT = 2, MODEL_GLM_TC = 3, MODEL_ODE = 4, MODEL_GLM_FP8 = 5, MODEL_GLM_GENERIC = 6 };

thread_local std::string g_last_error;

int fail(const char* what, cudaError_t err) {
    g_last_error = std::string(what) + ": " + cudaGetErrorString(err);
    return (int)err ? (int)err : -1;
}
#define CK(expr)                                  \
    do {                                          \
        cudaError_t _e = (expr);                  \
        if (_e != cudaSuccess) return fail(#expr, _e); \
    } while (0)

struct CommLayout {
    size_t off_flag, off_theta, off_slots, off_slot_flags, off_ll_theta, off_ll_slots, bytes;
};
CommLayout comm_layout(int world, int n_theta, int n_vals) {
    CommLayout L;
    auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
    L.off_flag = 0;
    L.off_theta = 256;
    L.off_slots = up(L.off_theta + (size_t)n_theta * 4);
    L.off_slot_flags = up(L.off_slots + (size_t)world * n_vals * 8);
    // low-latency mode (flag-in-data): 8 bytes per theta word, 16 bytes per result value
    L.off_ll_theta = up(L.off_slot_flags + (size_t)world * 8);
    L.off_ll_slots = up(L.off_ll_theta + (size_t)n_theta * 8);
    L.bytes = up(L.off_ll_slots + (size_t)world * n_vals * 16);
    return L;
}

struct Engine {
    int device = 0, rank = 0, world = 1, n_theta = 0, n_vals = 0;
    int grid = 1, sm_count = 148;
    cudaStream_t stream = nullptr;
    bool owns_comm = false;
    unsigned char* comm_local = nullptr;
    unsigned char* comm_peer[B200FED_MAX_WORLD] = {};
    unsigned char* comm_mc = nullptr;
    CommLayout layout{};
    // host-mapped
    unsigned char* host_block = nullptr;      // [theta | result | flag | done | trace]
    unsigned char* host_block_dev = nullptr;  // device alias
    size_t h_off_theta = 0, h_off_result = 0, h_off_flag = 0, h_off_done = 0, h_off_ll = 0;
    bool ll_mode = false;  // small results: tagged words instead of fences + flags (fed_comm.cuh)
    bool ll_theta = false; // theta as tagged words (no fence, no flag round trip)
    // device-local
    double* cta_partials = nullptr;
    unsigned int* ticket = nullptr;
    unsigned long long* epoch_counter = nullptr;
    unsigned long long* trace = nullptr;
    unsigned long long* cta_trace = nullptr;   // [max_blocks][8] phase stamps of the last launch (opt-in)
    bool cta_trace_on = false;
    unsigned long long epoch = 0;  // last launched epoch (root)
    unsigned long long timeout_ns = 20ull * 1000 * 1000 * 1000;
    unsigned long long launches = 0;
    float* theta_dev = nullptr;   // optional device-resident theta source (device-timed benchmarking)
    bool theta_from_device = false;
    // model
    ModelKind kind = MODEL_NONE;
    std::vector<LinregShard> linreg;
    LinregShard* linreg_dev = nullptr;
    int linreg_f64 = 1;
    std::vector<GlmSegment> glm_segs;
    GlmSegment* glm_segs_dev = nullptr;
    GlmParams glm{};
    void* glm_tmaps_dev = nullptr;
    void* glm_chunks_dev = nullptr;      // tensor-core kernel: chunk table of the dynamic scheduler
    int glm_n_chunks = 0;
    unsigned int* work_counter = nullptr;
    double* tc_partials = nullptr;       // its partial array: rows of (hi, lo) pairs, then the group partials
    size_t tc_row_doubles = 0;
    int glm_elem_bytes = 2;
    // launcher of a user-compiled likelihood (models/custom.py); null = built-in families
    int (*custom_launcher)(const FedComm*, const GlmSegment*, const GlmParams*, int, int, cudaStream_t) = nullptr;
    std::vector<OdeShard> ode;
    OdeShard* ode_dev = nullptr;
    // launcher of a user-supplied ODE system (models/ode.py: OdeSystem); null = the built-in Lotka-Volterra kernel
    int (*ode_launcher)(const FedComm*, const OdeShard*, int, int, cudaStream_t) = nullptr;
    std::atomic<int> stop_serving{0};

    float* h_theta() { return reinterpret_cast<float*>(host_block + h_off_theta); }
    double* h_result() { return reinterpret_cast<double*>(host_block + h_off_result); }
    volatile unsigned long long* h_flag() { return reinterpret_cast<volatile unsigned long long*>(host_block + h_off_flag); }
    volatile unsigned long long* h_done() { return reinterpret_cast<volatile unsigned long long*>(host_block + h_off_done); }
    volatile unsigned long long* h_idle() { return reinterpret_cast<volatile unsigned long long*>(host_block + h_off_done + 64); }
    double idle_timeout_s = 0.0;   // peers: give up after this long without an evaluation (0 = keep waiting)

    // speculative root launches (b200_engine_set_speculative): kernels are kept enqueued AHEAD of the client's
    // next theta, which they pick up as tagged words from host memory; epochs live on the device (like a peer's)
    bool spec_enabled = false;
    unsigned long long spec_timeout_ns = 0;
    size_t h_off_spec = 0;                       // host-mapped tagged theta words [n_theta]
    unsigned long long* spec_abort = nullptr;    // device word (fed_comm.cuh)
    unsigned long long spec_launched = 0;        // root launches since speculation was switched on ...
    unsigned long long spec_base_done = 0, spec_base_idle = 0;   // ... and the counters at that moment
    volatile unsigned long long* h_spec() { return reinterpret_cast<volatile unsigned long long*>(host_block + h_off_spec); }
    // launches still in the stream: launched - (completed epochs + launches that gave up waiting)
    unsigned long long spec_in_flight() {
        const unsigned long long done = *h_done() & B200FED_EPOCH_MASK;
        const unsigned long long finished = (done - spec_base_done) + (*h_idle() - spec_base_idle);
        return spec_launched > finished ? spec_launched - finished : 0;
    }
};

void fill_comm(Engine* e, FedComm* c, bool root_uses_explicit_epoch) {
    memset(c, 0, sizeof(*c));
    c->rank = e->rank;
    c->world = e->world;
    c->n_theta = e->n_theta;
    c->n_vals = e->n_vals;
    c->timeout_ns = e->timeout_ns;
    const CommLayout& L = e->layout;
    c->theta_local = reinterpret_cast<float*>(e->comm_local + L.off_theta);
    c->flag_local = reinterpret_cast<unsigned long long*>(e->comm_local + L.off_flag);
    unsigned char* root_block = e->comm_peer[0];
    c->root_slots = reinterpret_cast<double*>(root_block + L.off_slots);
    c->root_slot_flags = reinterpret_cast<unsigned long long*>(root_block + L.off_slot_flags);
    c->cta_partials = e->cta_partials;
    c->group_partials = e->cta_partials + (size_t)e->sm_count * 8 * e->n_vals;   // behind the max_blocks rows
    c->ticket = e->ticket;
    c->trace = e->trace;
    c->cta_trace = e->cta_trace_on ? e->cta_trace : nullptr;
    c->done_flag = reinterpret_cast<unsigned long long*>(e->host_block_dev + e->h_off_done);
    c->idle_ticks = reinterpret_cast<unsigned long long*>(e->host_block_dev + e->h_off_done + 64);
    c->ll_mode = e->ll_mode ? 1 : 0;
    c->ll_theta = e->ll_theta ? 1 : 0;
    c->ll_theta_local = reinterpret_cast<unsigned long long*>(e->comm_local + L.off_ll_theta);
    c->ll_root_slots = reinterpret_cast<unsigned long long*>(root_block + L.off_ll_slots);
    if (e->rank == 0) {
        for (int p = 0; p < e->world; ++p)
            c->ll_peer_theta[p] = reinterpret_cast<unsigned long long*>(e->comm_peer[p] + L.off_ll_theta);
        if (e->comm_mc) c->ll_mc_theta = reinterpret_cast<unsigned long long*>(e->comm_mc + L.off_ll_theta);
        c->ll_host_result = reinterpret_cast<unsigned long long*>(e->host_block_dev + e->h_off_ll);
    }
    if (e->rank == 0) {
        c->theta_src = e->theta_from_device ? e->theta_dev
                                            : reinterpret_cast<const float*>(e->host_block_dev + e->h_off_theta);
        for (int p = 0; p < e->world; ++p) {
            c->peer_theta[p] = reinterpret_cast<float*>(e->comm_peer[p] + L.off_theta);
            c->peer_flag[p] = reinterpret_cast<unsigned long long*>(e->comm_peer[p] + L.off_flag);
        }
        if (e->comm_mc) {
            c->mc_theta = reinterpret_cast<float*>(e->comm_mc + L.off_theta);
            c->mc_flag = reinterpret_cast<unsigned long long*>(e->comm_mc + L.off_flag);
        }
        c->host_result = reinterpret_cast<double*>(e->host_block_dev + e->h_off_result);
        c->host_flag = reinterpret_cast<unsigned long long*>(e->host_block_dev + e->h_off_flag);
        // with speculation on, the root counts epochs on the device as the peers do: a launch that gave up
        // waiting for theta leaves the counter alone and the next launch in the stream takes the epoch over
        c->epoch_counter = (root_uses_explicit_epoch && !e->spec_enabled) ? nullptr : e->epoch_counter;
        c->spec_abort = e->spec_abort;
    } else {
        c->epoch_counter = e->epoch_counter;  // peers count epochs on the device
    }
}

int launch_model(Engine* e, const FedComm* c) {
    int rc = -1;
    switch (e->kind) {
        case MODEL_LINREG:
            rc = b200_launch_linreg(c, e->linreg_dev, (int)e->linreg.size(), e->linreg_f64, e->grid, e->stream);
            break;
        case MODEL_GLM_SIMT:
            rc = b200_launch_glm_simt(c, e->glm_segs_dev, &e->glm, e->grid, e->stream);
            break;
        case MODEL_GLM_TC: {
            FedComm ct = *c;   // double-double rows + group partials of the dynamically scheduled kernel
            ct.cta_partials = e->tc_partials;
            ct.group_partials = e->tc_partials + (size_t)e->sm_count * e->tc_row_doubles;
            rc = b200_launch_glm_tc(&ct, e->glm_segs_dev, &e->glm, e->glm_tmaps_dev, e->glm_chunks_dev, e->glm_n_chunks,
                                    e->work_counter, e->grid, e->stream);
            break;
        }
        case MODEL_ODE:
            rc = (e->ode_launcher ? e->ode_launcher : b200_launch_ode)(c, e->ode_dev, (int)e->ode.size(), e->grid, e->stream);
            break;
        case MODEL_GLM_FP8: {
            FedComm ct = *c;   // same partial layout as the bf16 tensor-core kernel
            ct.cta_partials = e->tc_partials;
            ct.group_partials = e->tc_partials + (size_t)e->sm_count * e->tc_row_doubles;
            rc = b200_launch_glm_fp8(&ct, e->glm_segs_dev, &e->glm, e->glm_tmaps_dev, e->glm_chunks_dev, e->glm_n_chunks,
                                     e->work_counter, e->grid, e->stream);
            break;
        }
        case MODEL_GLM_GENERIC:
            rc = (e->custom_launcher ? e->custom_launcher : b200_launch_glm_generic)(c, e->glm_segs_dev, &e->glm,
                                                                                      e->glm_elem_bytes, e->grid, e->stream);
            break;
        default:
            g_last_error = "no model attached to the engine";
            return -2;
    }
    if (rc != 0) {
        g_last_error = std::string("kernel launch failed: ") + (rc > 0 ? cudaGetErrorString((cudaError_t)rc) : "unsupported shape");
        return rc;
    }
    e->launches++;
    return 0;
}

// Releases everything an Engine owns (also the partially constructed one of a failed create).
void release_engine(Engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->owns_comm && e->comm_local) cudaFree(e->comm_local);
    if (e->host_block) cudaFreeHost(e->host_block);
    void* device_ptrs[] = {e->cta_partials, e->ticket,       e->epoch_counter, e->trace,  e->theta_dev, e->cta_trace, e->spec_abort,
                           e->glm_chunks_dev, e->work_counter, e->tc_partials,
                           e->linreg_dev,   e->glm_segs_dev, e->glm_tmaps_dev, e->ode_dev};
    for (void* p : device_ptrs)
        if (p) cudaFree(p);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

__global__ void fed_stop_kernel(FedComm comm) {
    // root asks every node to drain its pre-enqueued kernels
    if (threadIdx.x < comm.world) fed::st_release_sys(comm.peer_flag[threadIdx.x], B200FED_STOP_EPOCH);
}

__global__ void fed_reset_kernel(unsigned long long* flag, unsigned long long* slot_flags, int world,
                                 unsigned int* ticket, unsigned long long* epoch_counter, unsigned int* work_counter) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) ticket[i] = 0;
    if (threadIdx.x == 0) {
        *flag = 0;
        *epoch_counter = 0;
        *work_counter = 0;
    }
    if (threadIdx.x < world) slot_flags[threadIdx.x] = 0;
}

}  // namespace

extern "C" {

const char* b200_last_error() { return g_last_error.c_str(); }

int b200_device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// ---- raw memory helpers (IPC bootstrap without torch) ----------------------------------
int b200_malloc(int device, size_t bytes, void** out) {
    CK(cudaSetDevice(device));
    CK(cudaMalloc(out, bytes));
    CK(cudaMemset(*out, 0, bytes));
    return 0;
}
int b200_free(int device, void* p) {
    CK(cudaSetDevice(device));
    CK(cudaFree(p));
    return 0;
}
int b200_ipc_get_handle(void* dptr, unsigned char* out64) {
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, dptr));
    memcpy(out64, &h, sizeof(h));
    return 0;
}
int b200_ipc_open_handle(int device, const unsigned char* in64, void** out) {
    cudaIpcMemHandle_t h;
    memcpy(&h, in64, sizeof(h));
    CK(cudaSetDevice(device));
    CK(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
int b200_ipc_close_handle(void* p) {
    CK(cudaIpcCloseMemHandle(p));
    return 0;
}
int b200_enable_peer_access(int device, int peer) {
    CK(cudaSetDevice(device));
    int can = 0;
    CK(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) {
        g_last_error = "peer access not supported between these devices";
        return -3;
    }
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail("cudaDeviceEnablePeerAccess", e);
    cudaGetLastError();
    return 0;
}

// ---- engine ------------------------------------------------------------------------------
size_t b200_comm_block_bytes(int world, int n_theta, int n_vals) { return comm_layout(world, n_theta, n_vals).bytes; }

void* b200_engine_create(int device, int rank, int world, int n_theta, int n_vals, int max_grid) {
    if (world < 1 || world > B200FED_MAX_WORLD || rank < 0 || rank >= world) {
        g_last_error = "invalid rank/world";
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        g_last_error = "cudaSetDevice failed";
        return nullptr;
    }
    Engine* e = new Engine();
    e->device = device;
    e->rank = rank;
    e->world = world;
    e->n_theta = n_theta;
    e->n_vals = n_vals;
    e->layout = comm_layout(world, n_theta, n_vals);
    cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, device);
    e->grid = max_grid > 0 ? max_grid : e->sm_count;
    bool ok = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) == cudaSuccess;
    // host-mapped block
    auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
    e->h_off_theta = 0;
    e->h_off_result = up((size_t)n_theta * 4);
    e->h_off_flag = up(e->h_off_result + (size_t)n_vals * 8);
    e->h_off_done = e->h_off_flag + 256;
    e->h_off_ll = e->h_off_done + 256;
    e->h_off_spec = e->h_off_ll + up((size_t)n_vals * 16);
    const size_t hbytes = e->h_off_spec + up((size_t)n_theta * 8);
    // LL mode for small messages (latency-bound models); B200FED_NO_LL=1 forces the fence+flag protocol
    // (thresholds tunable with B200FED_LL_MAX_VALS / B200FED_LL_MAX_THETA)
    auto env_int = [](const char* name, int dflt) {
        const char* v = getenv(name);
        return v && *v ? atoi(v) : dflt;
    };
    e->ll_theta = n_theta <= env_int("B200FED_LL_MAX_THETA", 4096) && !getenv("B200FED_NO_LL");
    e->ll_mode = e->ll_theta && n_vals <= env_int("B200FED_LL_MAX_VALS", 2048);
    ok = ok && cudaHostAlloc((void**)&e->host_block, hbytes, cudaHostAllocMapped | cudaHostAllocPortable) == cudaSuccess;
    if (ok) memset(e->host_block, 0, hbytes);
    ok = ok && cudaHostGetDevicePointer((void**)&e->host_block_dev, e->host_block, 0) == cudaSuccess;
    const int max_blocks = e->sm_count * 8;
    // per-CTA partial rows, then the group partials of the two-level reduction (fed::epilogue_t)
    const size_t partial_rows = (size_t)max_blocks + max_blocks / 16 + 2;
    ok = ok && cudaMalloc((void**)&e->cta_partials, partial_rows * n_vals * 8) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->ticket, 1024) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->work_counter, 256) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->epoch_counter, 256) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->trace, 256 * 4 * 8) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->cta_trace, (size_t)max_blocks * 8 * 8) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->theta_dev, (size_t)(n_theta > 0 ? n_theta : 1) * 4) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&e->spec_abort, 256) == cudaSuccess;
    if (ok) {
        cudaMemset(e->spec_abort, 0, 256);
        cudaMemset(e->ticket, 0, 1024);
        cudaMemset(e->work_counter, 0, 256);
        cudaMemset(e->epoch_counter, 0, 256);
        cudaMemset(e->trace, 0, 256 * 4 * 8);
        cudaMemset(e->cta_trace, 0, (size_t)max_blocks * 8 * 8);
        cudaMemset(e->theta_dev, 0, (size_t)(n_theta > 0 ? n_theta : 1) * 4);
        cudaDeviceSynchronize();
    }
    if (!ok) {
        g_last_error = std::string("engine allocation failed: ") + cudaGetErrorString(cudaGetLastError());
        release_engine(e);
        return nullptr;
    }
    return e;
}

int b200_engine_max_blocks(void* h) { return static_cast<Engine*>(h)->sm_count * 8; }
int b200_engine_sm_count(void* h) { return static_cast<Engine*>(h)->sm_count; }

// Allocate the comm block here (cudaMalloc => CUDA-IPC exportable).
int b200_engine_alloc_comm(void* h, void** out_ptr) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    CK(cudaMalloc((void**)&e->comm_local, e->layout.bytes));
    CK(cudaMemset(e->comm_local, 0, e->layout.bytes));
    CK(cudaDeviceSynchronize());
    e->owns_comm = true;
    e->comm_peer[e->rank] = e->comm_local;
    *out_ptr = e->comm_local;
    return 0;
}

// Bind comm blocks: `peers[world]` are this process's views of every node's block
// (own entry included); `mc` is the multicast alias or null.
int b200_engine_bind_comm(void* h, void* local, void** peers, void* mc) {
    Engine* e = static_cast<Engine*>(h);
    e->comm_local = static_cast<unsigned char*>(local);
    for (int p = 0; p < e->world; ++p) e->comm_peer[p] = static_cast<unsigned char*>(peers[p]);
    e->comm_peer[e->rank] = e->comm_local;
    e->comm_mc = static_cast<unsigned char*>(mc);
    return 0;
}

int b200_engine_reset(void* h) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    const CommLayout& L = e->layout;
    fed_reset_kernel<<<1, 32, 0, e->stream>>>(reinterpret_cast<unsigned long long*>(e->comm_local + L.off_flag),
                                              reinterpret_cast<unsigned long long*>(e->comm_local + L.off_slot_flags),
                                              e->world, e->ticket, e->epoch_counter, e->work_counter);
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemset(e->comm_local + L.off_ll_theta, 0, L.bytes - L.off_ll_theta));
    CK(cudaDeviceSynchronize());
    memset(e->host_block + e->h_off_ll, 0, (size_t)e->n_vals * 16);
    memset(e->host_block + e->h_off_spec, 0, (size_t)e->n_theta * 8);
    CK(cudaMemset(e->spec_abort, 0, 256));
    e->epoch = 0;
    *e->h_flag() = 0;
    *e->h_done() = 0;
    *e->h_idle() = 0;
    e->spec_launched = e->spec_base_done = e->spec_base_idle = 0;
    e->stop_serving = 0;
    return 0;
}

// Speculation: waits until no launch is left in the stream (kernels that are still waiting for a theta nobody
// will write give up after spec_timeout_ns each).  Everything that needs a quiet stream or explicit control over
// what runs next (device-timed launches, STOP, reset) calls this first.
static int spec_settle(Engine* e) {
    if (!e->spec_enabled) return 0;
    const auto t0 = std::chrono::steady_clock::now();
    unsigned spins = 0;
    while (e->spec_in_flight() != 0) {
        if ((++spins & 0xFFF) == 0) {
            const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (dt > 10.0 + 4e-9 * (double)e->spec_timeout_ns) {
                g_last_error = "speculative launches did not drain";
                return -8;
            }
        }
    }
    return 0;
}

// Root: keep kernels enqueued ahead of the client's next theta (timeout_us > 0), or go back to one launch per
// evaluation (0).  Needs theta as tagged words (n_theta <= 1024 here).  Returns 1 if speculation is on.
int b200_engine_set_speculative(void* h, double timeout_us) {
    Engine* e = static_cast<Engine*>(h);
    if (e->rank != 0) return 0;
    CK(cudaSetDevice(e->device));
    if (spec_settle(e) != 0) return -8;
    CK(cudaStreamSynchronize(e->stream));
    const bool on = timeout_us > 0.0 && e->ll_theta && e->n_theta <= 1024;
    e->spec_enabled = on;
    e->spec_timeout_ns = on ? (unsigned long long)(timeout_us * 1e3) : 0ull;
    // device-resident epochs take over from the host's count (and hand it back)
    CK(cudaMemcpy(e->epoch_counter, &e->epoch, 8, cudaMemcpyHostToDevice));
    e->spec_launched = 0;
    e->spec_base_done = e->epoch;
    e->spec_base_idle = *e->h_idle();
    return on ? 1 : 0;
}

void b200_engine_set_timeout(void* h, double seconds) {
    static_cast<Engine*>(h)->timeout_ns = (unsigned long long)(seconds * 1e9);
}
// Peers: how long serve() keeps re-arming kernels without seeing an evaluation (0 = for ever).  The per-launch
// wait for theta stays the evaluation timeout; a launch that expires counts an idle tick and is replaced.
void b200_engine_set_idle_timeout(void* h, double seconds) { static_cast<Engine*>(h)->idle_timeout_s = seconds; }
void b200_engine_set_grid(void* h, int grid) {
    // the per-CTA partial array holds sm_count * 8 rows; negative values select single-CTA modes
    Engine* e = static_cast<Engine*>(h);
    const int max_blocks = (e->kind == MODEL_GLM_TC || e->kind == MODEL_GLM_FP8) ? e->sm_count : e->sm_count * 8;   // partial rows
    e->grid = grid > max_blocks ? max_blocks : (grid == 0 ? 1 : grid);
}
int b200_engine_grid(void* h) { return static_cast<Engine*>(h)->grid; }
unsigned long long b200_engine_launches(void* h) { return static_cast<Engine*>(h)->launches; }
unsigned long long b200_engine_epoch(void* h) { return static_cast<Engine*>(h)->epoch; }
void* b200_engine_stream(void* h) { return static_cast<Engine*>(h)->stream; }
void* b200_engine_host_theta(void* h) { return static_cast<Engine*>(h)->h_theta(); }
void* b200_engine_host_result(void* h) { return static_cast<Engine*>(h)->h_result(); }

int b200_engine_set_linreg(void* h, int n_shards, const void** x, const void** y, const long long* n,
                           const double* sigma, const int* theta_offset, int is_f64) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    e->linreg.resize(n_shards);
    long long total = 0;
    for (int s = 0; s < n_shards; ++s) {
        e->linreg[s] = LinregShard{x[s], y[s], n[s], sigma[s], theta_offset[s], 0};
        total += n[s];
    }
    if (e->linreg_dev) cudaFree(e->linreg_dev);
    CK(cudaMalloc((void**)&e->linreg_dev, sizeof(LinregShard) * (n_shards > 0 ? n_shards : 1)));
    CK(cudaMemcpy(e->linreg_dev, e->linreg.data(), sizeof(LinregShard) * n_shards, cudaMemcpyHostToDevice));
    e->linreg_f64 = is_f64;
    e->kind = MODEL_LINREG;
    // tiny data => one CTA is the lowest-latency configuration; grow with the data
    long long want = (total + 256 * 64 - 1) / (256 * 64);
    if (want < 1) want = 1;
    if (want > e->sm_count * 4) want = e->sm_count * 4;
    e->grid = (int)want;
    long long max_n = 0;
    for (int s = 0; s < n_shards; ++s) max_n = n[s] > max_n ? n[s] : max_n;
    if (want == 1 && max_n <= 4096) e->grid = -1;  // small mode: one CTA, one warp per shard
    return 0;
}

int b200_engine_set_glm(void* h, int n_segments, const void** X, const float** y, const void** scales,
                        const long long* n_rows, const int* groups, int n_features, int ld, int n_groups,
                        int n_chains, int family, int use_tensor_cores, const int* out_groups, int n_out,
                        int n_family_params) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    if (n_family_params < 0 || (n_family_params > 0 && use_tensor_cores != 1)) {
        g_last_error = "families with fitted parameters run on the tensor-core kernel only";
        return -34;
    }
    const int tile_rows = (use_tensor_cores == 1 || use_tensor_cores == 2) ? 128 : 8;
    e->glm_segs.resize(n_segments);
    long long tiles = 0;
    for (int s = 0; s < n_segments; ++s) {
        GlmSegment g{};
        g.X = X[s];
        g.y = y[s];
        g.scales = scales ? scales[s] : nullptr;
        g.n_rows = n_rows[s];
        g.first_tile = tiles;
        g.group = groups[s];
        g.out_group = out_groups ? out_groups[s] : 0;
        if (g.out_group < 0 || g.out_group >= (n_out > 0 ? n_out : 1)) {
            g_last_error = "segment output block out of range";
            return -31;
        }
        e->glm_segs[s] = g;
        tiles += (n_rows[s] + tile_rows - 1) / tile_rows;
    }
    e->glm = GlmParams{n_segments, n_features, ld, n_groups, n_chains, family, tiles, n_out > 0 ? n_out : 1,
                       early_loads_enabled() ? 1 : 0, n_family_params};
    if ((long long)e->glm.n_out * n_chains * (1 + n_groups + n_features + n_family_params) != e->n_vals) {
        g_last_error = "n_vals does not match n_out x n_chains x (1 + n_groups + n_features + n_family_params)";
        return -33;
    }
    if (e->glm_segs_dev) cudaFree(e->glm_segs_dev);
    CK(cudaMalloc((void**)&e->glm_segs_dev, sizeof(GlmSegment) * (n_segments > 0 ? n_segments : 1)));
    CK(cudaMemcpy(e->glm_segs_dev, e->glm_segs.data(), sizeof(GlmSegment) * n_segments, cudaMemcpyHostToDevice));
    if (use_tensor_cores == 3 || use_tensor_cores == 4) {  // general-shape fallback
        e->glm_elem_bytes = use_tensor_cores == 3 ? 2 : 4;
        e->kind = MODEL_GLM_GENERIC;
        e->grid = e->sm_count * 2;
    } else if (use_tensor_cores == 2) {  // block-scaled fp8
        int rc = b200_glm_fp8_prepare(e->glm_segs.data(), n_segments, &e->glm, e->sm_count, &e->glm_tmaps_dev,
                                      &e->glm_chunks_dev, &e->glm_n_chunks);
        if (rc != 0) {
            g_last_error = "fp8 GLM path rejected this shape (rc=" + std::to_string(rc) + ")";
            return rc;
        }
        e->tc_row_doubles = b200_glm_fp8_partial_row_doubles(e->n_vals, n_chains, e->glm.n_out, n_groups);
        if (e->tc_partials) cudaFree(e->tc_partials);
        const size_t fp8_doubles = (size_t)e->sm_count * e->tc_row_doubles + ((size_t)e->sm_count / 16 + 2) * e->n_vals * 2;
        CK(cudaMalloc((void**)&e->tc_partials, fp8_doubles * 8));
        CK(cudaMemset(e->tc_partials, 0, fp8_doubles * 8));
        e->kind = MODEL_GLM_FP8;
        e->grid = e->sm_count;
        if (e->glm_n_chunks > 0 && e->grid > e->glm_n_chunks) e->grid = e->glm_n_chunks;
    } else if (use_tensor_cores) {
        int rc = b200_glm_tc_prepare(e->glm_segs.data(), n_segments, &e->glm, e->sm_count, &e->glm_tmaps_dev,
                                     &e->glm_chunks_dev, &e->glm_n_chunks);
        if (rc != 0) {
            g_last_error = "tensor-core GLM path rejected this shape (rc=" + std::to_string(rc) + ")";
            return rc;
        }
        e->tc_row_doubles = b200_glm_tc_partial_row_doubles(e->n_vals, n_chains, e->glm.n_out, n_groups, n_family_params);
        if (e->tc_partials) cudaFree(e->tc_partials);
        const size_t tc_doubles = (size_t)e->sm_count * e->tc_row_doubles + ((size_t)e->sm_count / 16 + 2) * e->n_vals * 2;
        CK(cudaMalloc((void**)&e->tc_partials, tc_doubles * 8));
        CK(cudaMemset(e->tc_partials, 0, tc_doubles * 8));
        e->kind = MODEL_GLM_TC;
        e->grid = e->sm_count;
        if (e->glm_n_chunks > 0 && e->grid > e->glm_n_chunks) e->grid = e->glm_n_chunks;
    } else {
        e->kind = MODEL_GLM_SIMT;
        e->grid = e->sm_count * 2;
    }
    if ((long long)e->grid > tiles && tiles > 0) e->grid = (int)tiles;
    return 0;
}

// Installs the launcher of a separately compiled likelihood (same signature as b200_launch_glm_generic).
void b200_engine_set_custom_launcher(void* h, void* fn) {
    static_cast<Engine*>(h)->custom_launcher =
        reinterpret_cast<int (*)(const FedComm*, const GlmSegment*, const GlmParams*, int, int, cudaStream_t)>(fn);
}

// Installs the launcher of a separately compiled ODE system (same signature as b200_launch_ode).
void b200_engine_set_ode_launcher(void* h, void* fn) {
    static_cast<Engine*>(h)->ode_launcher =
        reinterpret_cast<int (*)(const FedComm*, const OdeShard*, int, int, cudaStream_t)>(fn);
}

int b200_engine_set_ode(void* h, int n_shards, const float** t, const float** y0, const float** y_obs, const int* n_series,
                        const int* n_t, const float* sigma, const int* substeps, const int* theta_offset,
                        const int* out_offset) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    e->ode.resize(n_shards);
    long long series = 0;
    for (int s = 0; s < n_shards; ++s) {
        e->ode[s] = OdeShard{t[s], y0[s], y_obs[s], n_series[s], n_t[s], sigma[s], substeps[s],
                             theta_offset ? theta_offset[s] : 0, out_offset ? out_offset[s] : 0};
        series += n_series[s];
    }
    if (e->ode_dev) cudaFree(e->ode_dev);
    CK(cudaMalloc((void**)&e->ode_dev, sizeof(OdeShard) * (n_shards > 0 ? n_shards : 1)));
    CK(cudaMemcpy(e->ode_dev, e->ode.data(), sizeof(OdeShard) * n_shards, cudaMemcpyHostToDevice));
    e->kind = MODEL_ODE;
    long long want = (series + 127) / 128;
    if (want < 1) want = 1;
    if (want > e->sm_count * 4) want = e->sm_count * 4;
    e->grid = (int)want;
    return 0;
}

// Enqueue one evaluation without waiting (device-timed loops).  Root only.  theta is taken
// from the device-resident copy when `theta_on_device` (set by b200_engine_set_device_theta).
int b200_engine_launch(void* h) {
    Engine* e = static_cast<Engine*>(h);
    if (e->rank != 0) {
        g_last_error = "only the root launches explicit epochs";
        return -4;
    }
    if (spec_settle(e) != 0) return -8;
    FedComm c;
    fill_comm(e, &c, true);
    c.epoch = ++e->epoch;
    const int rc = launch_model(e, &c);
    if (rc == 0 && e->spec_enabled) e->spec_launched++;
    return rc;
}

// One launch that takes its theta from the tagged host words and its epoch from the device counter.
static int spec_launch(Engine* e) {
    FedComm c;
    fill_comm(e, &c, false);
    c.spec_theta = reinterpret_cast<const unsigned long long*>(e->host_block_dev + e->h_off_spec);
    c.spec_timeout_ns = e->spec_timeout_ns;
    const int rc = launch_model(e, &c);
    if (rc == 0) e->spec_launched++;
    return rc;
}

int b200_engine_set_device_theta(void* h, const float* theta_host, int n, int enable) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    if (spec_settle(e) != 0) return -8;
    if (theta_host && n > 0) CK(cudaMemcpy(e->theta_dev, theta_host, (size_t)n * 4, cudaMemcpyHostToDevice));
    e->theta_from_device = enable != 0;
    return 0;
}

// Wait (host spin on the mapped completion flag) for epoch `epoch`; copies the result.
// Returns 0, or 1 = theta timeout, 2 = peer timeout (bit-or), -5 = host-side timeout.
int b200_engine_wait(void* h, unsigned long long epoch, double* out, double timeout_s) {
    Engine* e = static_cast<Engine*>(h);
    volatile unsigned long long* flag = e->h_flag();
    const auto t0 = std::chrono::steady_clock::now();
    unsigned long long v;
    unsigned spins = 0;
    if (e->ll_mode) {
        // flag-in-data: the result is complete when every word carries this epoch's tag; errors (and
        // STOP / theta timeouts) still arrive on the legacy flag
        volatile unsigned long long* words = reinterpret_cast<volatile unsigned long long*>(e->host_block + e->h_off_ll);
        const unsigned long long want = epoch & 0xFFFFFFFFull;
        const int n_words = e->n_vals * 2;
        int next = 0;
        while (true) {
            // a word tagged with this epoch OR A LATER ONE is complete for our purposes (like the epoch flag: with
            // several launches in flight an older epoch can still be waited for); signed 32-bit tag distance
            while (next < n_words && (int32_t)((uint32_t)(words[next] >> 32) - (uint32_t)want) >= 0) ++next;
            if (next == n_words) break;
            v = *flag;
            if ((v & B200FED_EPOCH_MASK) >= epoch && (v >> B200FED_STATUS_SHIFT) != 0) return (int)(v >> B200FED_STATUS_SHIFT);
            if ((++spins & 0xFFF) == 0) {
                if (e->spec_enabled && !e->theta_from_device && e->spec_in_flight() == 0 && spec_launch(e) != 0) return -8;
                const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
                if (dt > timeout_s) {
                    cudaError_t err = cudaStreamQuery(e->stream);
                    g_last_error = std::string("timed out waiting for the tagged result words; stream state: ") +
                                   cudaGetErrorString(err);
                    return -5;
                }
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        if (out) {
            for (int i = 0; i < e->n_vals; ++i) {
                const unsigned long long bits = (words[2 * i] & 0xFFFFFFFFull) | ((words[2 * i + 1] & 0xFFFFFFFFull) << 32);
                memcpy(out + i, &bits, 8);
            }
        }
        return 0;
    }
    while (true) {
        v = *flag;
        if ((v & B200FED_EPOCH_MASK) >= epoch) break;
        if ((++spins & 0xFFF) == 0) {
            if (e->spec_enabled && !e->theta_from_device && e->spec_in_flight() == 0 && spec_launch(e) != 0) return -8;
            const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (dt > timeout_s) {
                cudaError_t err = cudaStreamQuery(e->stream);
                g_last_error = std::string("timed out waiting for the completion flag; stream state: ") +
                               cudaGetErrorString(err);
                return -5;
            }
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (out) memcpy(out, e->h_result(), (size_t)e->n_vals * 8);
    return (int)(v >> B200FED_STATUS_SHIFT);
}

// The client call: theta (raw 32-bit words) -> [n_vals] doubles.
int b200_engine_eval(void* h, const void* theta, int n_words, double* out, double timeout_s) {
    Engine* e = static_cast<Engine*>(h);
    if (n_words != e->n_theta) {
        g_last_error = "theta has the wrong number of 32-bit words";
        return -6;
    }
    memcpy(e->h_theta(), theta, (size_t)n_words * 4);
    if (e->spec_enabled && !e->theta_from_device) {
        // speculative path: a kernel enqueued by the previous call is already resident and polling; publish theta
        // as tagged words, top the stream up to two launches (this epoch's + the next one's, which overlaps its
        // launch latency, set-up and first loads with this evaluation) and wait for the result
        const unsigned long long epoch = ++e->epoch;
        const uint32_t* w = static_cast<const uint32_t*>(theta);
        volatile unsigned long long* words = e->h_spec();
        const unsigned long long tag = (epoch & 0xFFFFFFFFull) << 32;
        for (int i = 0; i < n_words; ++i) words[i] = (unsigned long long)w[i] | tag;
        std::atomic_thread_fence(std::memory_order_seq_cst);
        while (e->spec_in_flight() < 2) {
            const int rc = spec_launch(e);
            if (rc != 0) return rc;
        }
        return b200_engine_wait(h, epoch, out, timeout_s);
    }
    std::atomic_thread_fence(std::memory_order_release);
    int rc = b200_engine_launch(h);
    if (rc != 0) return rc;
    return b200_engine_wait(h, e->epoch, out, timeout_s);
}

// Peer loop: keep up to `ahead` kernels enqueued until the root broadcasts STOP, the idle
// timeout fires inside a kernel, or b200_engine_stop_serving() is called from another thread.
// Returns the number of evaluated epochs (>= 0) or a negative error.
long long b200_engine_serve(void* h, int ahead, long long max_epochs) {
    Engine* e = static_cast<Engine*>(h);
    if (cudaSetDevice(e->device) != cudaSuccess) return -1;
    if (ahead < 1) ahead = 1;
    FedComm c;
    fill_comm(e, &c, false);
    // epochs are absolute (device-resident counter); this call serves [base+1, base+max_epochs]
    const unsigned long long base = *e->h_done() & B200FED_EPOCH_MASK;
    if (base == B200FED_STOP_EPOCH) return 0;
    const unsigned long long idle_base = *e->h_idle();
    unsigned long long enqueued = 0;      // kernels launched by this call
    unsigned long long idle_seen = 0;     // ... of which gave up waiting for theta (re-armed below)
    double idle_s = 0.0;                  // time spent idle since the last served evaluation
    unsigned long long last_done = base;
    long long served = 0;
    while (!e->stop_serving.load()) {
        const unsigned long long word = *e->h_done();
        const unsigned long long done = word & B200FED_EPOCH_MASK;
        if (done == B200FED_STOP_EPOCH) break;
        const unsigned long long idle_now = *e->h_idle() - idle_base;
        if (done != last_done) {
            last_done = done;
            idle_s = 0.0;
        }
        if (idle_now != idle_seen) {
            idle_s += (double)(idle_now - idle_seen) * (double)e->timeout_ns * 1e-9;
            idle_seen = idle_now;
            if (e->idle_timeout_s > 0.0 && idle_s > e->idle_timeout_s) {
                g_last_error = "idle timeout: no theta arrived from the root";
                cudaStreamSynchronize(e->stream);
                return -7;
            }
        }
        served = (long long)(done - base);
        const unsigned long long finished = (done - base) + idle_seen;
        const unsigned long long in_flight = enqueued - finished;
        if (max_epochs > 0 && served >= max_epochs) {
            if (in_flight == 0) break;
            std::this_thread::yield();   // surplus kernels cannot exist: in_flight <= max_epochs - served below
            continue;
        }
        const bool room = in_flight < (unsigned long long)ahead &&
                          (max_epochs <= 0 || (long long)(served + in_flight) < max_epochs);
        if (room) {
            int rc = launch_model(e, &c);
            if (rc != 0) return -8;
            enqueued++;
        } else {
            std::this_thread::yield();
        }
    }
    cudaError_t err = cudaStreamSynchronize(e->stream);
    if (err != cudaSuccess) {
        g_last_error = std::string("serve loop: ") + cudaGetErrorString(err);
        return -9;
    }
    const unsigned long long word = *e->h_done();
    if ((word & B200FED_EPOCH_MASK) != B200FED_STOP_EPOCH) served = (long long)((word & B200FED_EPOCH_MASK) - base);
    return served;
}

void b200_engine_stop_serving(void* h) { static_cast<Engine*>(h)->stop_serving = 1; }

// Root: tell every node to drain (STOP epoch is sticky and larger than any real epoch).
int b200_engine_stop_peers(void* h) {
    Engine* e = static_cast<Engine*>(h);
    if (e->rank != 0) return 0;
    CK(cudaSetDevice(e->device));
    spec_settle(e);
    FedComm c;
    fill_comm(e, &c, true);
    fed_stop_kernel<<<1, 32, 0, e->stream>>>(c);
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

int b200_engine_sync(void* h) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// Device-timer trace of epoch `epoch`: [theta released, node partial released, result released] (ns)
int b200_engine_trace(void* h, unsigned long long epoch, unsigned long long* out4) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaMemcpy(out4, e->trace + (epoch & 255) * 4, 32, cudaMemcpyDeviceToHost));
    return 0;
}

// Per-CTA phase stamps (fed::stamp) of the most recent launch: out[grid][8] ns on the %globaltimer clock.
void b200_engine_enable_cta_trace(void* h, int on) { static_cast<Engine*>(h)->cta_trace_on = on != 0; }
int b200_engine_cta_trace(void* h, unsigned long long* out, int max_rows) {
    Engine* e = static_cast<Engine*>(h);
    CK(cudaSetDevice(e->device));
    int rows = e->grid > 0 ? e->grid : 1;
    if (rows > max_rows) rows = max_rows;
    CK(cudaMemcpy(out, e->cta_trace, (size_t)rows * 64, cudaMemcpyDeviceToHost));
    return rows;
}

void b200_engine_destroy(void* h) { release_engine(static_cast<Engine*>(h)); }

}  // extern "C"
