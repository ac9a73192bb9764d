// d2d_internal.h - what the translation units of libd2d_b200.so share: the handle, the error plumbing, the launch helpers
// and the per-kernel-family entry points.  The library is built from several .cu files compiled in parallel
// (gym_d2d_b200/build.py): d2d_abi.cu (the C ABI, host folding, the small kernels of d2d_aux.cuh), d2d_tu_warp.cu (compiled
// three times, once per warps-per-block shape of the warp kernel), d2d_tu_dense.cu and d2d_tu_block.cu.
#pragma once

#include "../../include/d2d_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <string>

#include "d2d_common.cuh"

int d2d_fail(int code, const std::string &msg);      // records the calling thread's last error (d2d_abi.cu)

#define D2D_CUDA(call)                                                                               \
    do {                                                                                             \
        cudaError_t err__ = (call);                                                                  \
        if (err__ != cudaSuccess)                                                                    \
            return d2d_fail(D2D_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(err__));    \
    } while (0)

#define D2D_NUM_IO_BUFFERS 10     // actions + the nine outputs of d2d_step_io_t (actions_out is d2d_episode's)
struct d2d_host_slot {
    // packed form (d2d_host_slot_buffers): one pinned host allocation and its device twin, [actions | outputs]
    void *dev = nullptr, *host = nullptr;
    size_t bytes = 0, out_offset = 0, out_bytes = 0;
    uint32_t mask = 0;
    d2d_step_io_t host_io{}, dev_io{};
    // caller-owned host buffers: per-buffer device staging, allocated on first use
    void *stage[D2D_NUM_IO_BUFFERS] = {};
    void *stage16 = nullptr;       // D2D_STEP_ACTIONS_I16: the int16 actions as uploaded, widened into the int32 action staging
    cudaEvent_t ev_in = nullptr, ev_kernel = nullptr, ev_out = nullptr;
    bool used = false;
};

struct d2d_handle {
    d2d_config_t cfg{};
    int N = 0, V = 0;
    int num_sms = 0;
    bool ple2 = true;
    bool use_warp = true;
    bool spec = false;         // warp kernel instantiated for the reference's default EnvConfig shape
    bool uniform = false;      // every CUE link has the same constants, and every DUE link (no per-device overrides)
    D2DLinkA u_cue{}, u_due{};
    D2DLinkD ud_cue{}, ud_due{};
    float us_cue[2] = {0, 0}, us_due[2] = {0, 0};
    const struct D2DWarpShape *warp = nullptr;   // warp kernel: the shape of the step geometry (nullptr: another kernel family)
    int dense_bt = 0;          // dense kernel (d2d_step_dense.cuh): threads per block, 0 = not used
    int bin_cap = 0;           // dense kernel: record slots per RB bin
    int lpt = 0;               // block / dense kernel: links per thread held in registers (0 = the generic shared-memory kernel)
    int64_t chunk_override = 0;  // D2D_B200_CHUNK: force small launch chunks (tests of the > 2^31-element path)
    bool pdl = true;           // programmatic dependent launch (D2D_B200_PDL=0 disables)
    int grid = 0, block = 0, smem = 0, envs_per_block = 0;
    // second geometry of the warp kernel for the fused multi-step launches (d2d_step_many / d2d_episode / d2d_rollout) of large
    // batches: their warps run for hundreds of microseconds and never hand over per step, and there 8-warp blocks measured
    // better than the 4-warp shape the single steps use (episode at E = 131 072: 785 vs 830 us); warp = nullptr: same geometry as the steps
    struct { const D2DWarpShape *warp = nullptr; int grid = 0, envs_per_block = 0; } many;
    double K_dB = 0.0, ple = 2.0;
    D2DLinkA *dA = nullptr;
    D2DLinkB *dB = nullptr;
    D2DLinkD *dD = nullptr;
    int32_t *dMeta = nullptr;  // [N] power levels | SIDELINK << 16 (general-topology kernel, fp64 helpers)
    float *dPwr = nullptr;
    double *dPwrD = nullptr;
    uint64_t *dRngStep = nullptr;  // ShadowingPathLoss: number of step calls so far, on the device (advanced on the stream, so
                                   // that a replayed CUDA graph draws fresh values at every replay)
    // bound state (caller-owned)
    float *pos = nullptr;
    double *pos64 = nullptr;
    uint8_t *step_count = nullptr;
    double *stats = nullptr;
    uint32_t *episode_index = nullptr;   // d2d_bind_autoreset
    uint64_t ar_base = 0;
    // host-buffer steps (d2d_step_host*): the pipeline slots
    d2d_host_slot slot[D2D_HOST_SLOTS];
    cudaStream_t s_in = nullptr, s_out = nullptr;
    bool pipe_ready = false;
    double *stage_pos = nullptr;
    int64_t stage_pos_envs = 0;
    int64_t launches = 0;
    // programmatic dependent launch bookkeeping (include/d2d_b200.h, "Ordering rule"; kept by d2d_plan_step, d2d_launch_plan.h):
    // the stream of the last kernel this handle enqueued and whether that kernel was one of its own step kernels (anything
    // else - reset, set_positions - wrote state a step kernel reads ahead of griddepcontrol.wait)
    void *last_stream = nullptr;
    int last_kind = 0;             // D2D_LAST_*
    // the per-link output buffers of the last single-kernel plain step ([begin, end) byte ranges; obs, obs_dyn, capacity, rate, rb,
    // Tx power): a d2d_step right behind it that touches none of them stores its own ahead of griddepcontrol.wait (D2D_PF_LATE_WAIT)
    uintptr_t prev_out[6][2] = {};
    bool prev_out_valid = false;
    bool late_wait_on = true;      // D2D_B200_LATE_WAIT=0 switches the late wait off (tests, A/B)
    int grid_late = 0;             // warp kernel: blocks of a late-wait step (0 = the full grid).  Under the late wait consecutive steps overlap
                                   // for as long as the SMs have room for both: a launch that leaves the larger part of the block slots free
                                   // lets its successor's blocks start while its own are still running (d2d_abi.cu, DESIGN.md 4.7)
    void *dDenseOvf = nullptr;     // dense kernel: the blocks' overflow lists (d2d_step_dense.cuh)
    // per-warp tickets (d2d_common.cuh: d2d_ticket_wait): one word per warp slot of the step geometry, and the chain bookkeeping
    uint64_t *dTickets = nullptr;
    uint64_t chain_id = 0;         // id of the current chain of single-launch steps
    uint32_t chain_seq = 0;        // tokens published so far in this chain (0: the previous launch was not a signing step)
    int chain_grid = 0;            // grid of the chain's launches
    bool tickets_on = true;        // D2D_B200_TICKET=0 disables (A/B, tests)
    // d2d_episode: handle-owned scratch for drawn actions when the caller does not ask for them but a later pass needs them
    int32_t *act_scratch = nullptr;
    size_t act_scratch_elems = 0;
};
enum { D2D_LAST_OTHER = 0, D2D_LAST_STEP = 1, D2D_LAST_EPISODE = 2 };

// Save / restore the calling thread's current CUDA device around an entry point: a handle is bound to one device, the
// caller's current device is none of the library's business (a VecD2DEnv on cuda:1 while torch's current device is cuda:0).
struct D2DDeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit D2DDeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) {
            err = cudaSetDevice(device);
            switched = err == cudaSuccess;
        }
    }
    ~D2DDeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
    D2DDeviceGuard(const D2DDeviceGuard &) = delete;
    D2DDeviceGuard &operator=(const D2DDeviceGuard &) = delete;
};
#define D2D_GUARD(h)                                                                                                   \
    D2DDeviceGuard guard__((h)->cfg.cuda_device);                                                                       \
    if (guard__.err != cudaSuccess) return d2d_fail(D2D_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(guard__.err))

// Launch a step kernel, optionally with programmatic stream serialisation (PDL): it may then begin launching while the
// previous kernel in the stream drains; the kernel itself orders its memory accesses with griddepcontrol.wait.
template <typename K>
cudaError_t d2d_launch_step(K kernel, int grid, int block, size_t smem, cudaStream_t st, const D2DParams &P, bool pdl) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, P);
}

template <typename K>
int d2d_allow_smem(K kernel, size_t smem) {
    if (smem > 48 * 1024) D2D_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return D2D_OK;
}

template <typename K>
int d2d_plan_geometry(d2d_handle *h, K kernel, int block, size_t smem, int envs_per_block) {
    int rc = d2d_allow_smem(kernel, smem);
    if (rc) return rc;
    int occ = 0;
    D2D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, smem));
    if (occ < 1) return d2d_fail(D2D_ERR_UNSUPPORTED, "step kernel does not fit on an SM for this configuration");
    const int64_t need = (h->cfg.num_envs + envs_per_block - 1) / envs_per_block;
    const int64_t resident = (int64_t)h->num_sms * occ;
    h->grid = (int)std::max<int64_t>(1, std::min<int64_t>(need, resident));
    h->block = block;
    h->smem = (int)smem;
    h->envs_per_block = envs_per_block;
    return D2D_OK;
}

// ---- per-family entry points (one translation unit each) ------------------------------------------------------------------
// What a step launch asks of a kernel family beyond the parameters
struct D2DLaunchSel {
    bool many = false;       // d2d_step_many: P.T steps per env in this launch
    bool full = false;       // exactly the core outputs (obs, capacity, reward, done) + a bound step counter
    bool exact = false;      // an fp64 position shadow is bound
    bool episode = false;    // d2d_episode / d2d_rollout: P.T slices per env; positions and / or actions are drawn inside the kernel
    bool fast = false;       // ... with drawn actions, no action record and no fp64 shadow: the compiled-in variants
    bool no_reset = false;   // ... d2d_rollout
    bool autoreset = false;  // d2d_step with D2D_STEP_AUTORESET (warp kernel only)
};

// warp kernel (d2d_step_warp.cuh): one TU, and one table of its entry points, per warps-per-block shape (d2d_tu_warp.cu)
#ifndef D2D_LATENCY_ENVS
#define D2D_LATENCY_ENVS 2048      // batches up to this size take the 2-warp latency shape (d2d_step_warp.cuh)
#endif
struct D2DWarpShape {
    int wpb;                                                   // warps per block
    size_t (*smem)(int R);                                     // dynamic shared memory per block for R RBs
    int (*plan)(d2d_handle *h, size_t smem);                   // shared-memory opt-in of every instantiation, h->grid / block / smem / envs_per_block
    cudaError_t (*launch)(const d2d_handle *h, const D2DParams &P, int grid, const D2DLaunchSel &sel, cudaStream_t st, bool pdl);
    cudaError_t (*tables)(const double *pwr_lin_d);            // 10^(p/10) into the TU's constant bank (per device: at every create)
    cudaError_t (*timeline)(void *host_out, size_t bytes);     // the TU's stamp table (-DD2D_TIMELINE builds; nullptr otherwise)
};
extern const D2DWarpShape d2d_warp_shape_2, d2d_warp_shape_4, d2d_warp_shape_8;
inline const D2DWarpShape *d2d_warp_shape(int wpb) { return wpb == 8 ? &d2d_warp_shape_8 : wpb == 2 ? &d2d_warp_shape_2 : &d2d_warp_shape_4; }

// dense kernel (d2d_step_dense.cuh)
size_t d2d_dense_smem(int N, int R, int bin_cap, int bt, int V);
int d2d_dense_bin_cap_host(int N, int R);
int d2d_dense_plan(d2d_handle *h, size_t smem);
cudaError_t d2d_dense_launch(const d2d_handle *h, const D2DParams &P, int grid, const D2DLaunchSel &sel, cudaStream_t st, bool pdl);

// sorting block kernel and the general-topology kernel (d2d_step_block.cuh)
#define D2D_BLOCK_THREADS 256
#define D2D_BLOCK_MAX_LPT 4
size_t d2d_block_smem(int N, int R, int lpt);
int d2d_block_plan(d2d_handle *h, size_t smem);
cudaError_t d2d_block_launch(const d2d_handle *h, const D2DParams &P, int grid, cudaStream_t st, bool pdl);
