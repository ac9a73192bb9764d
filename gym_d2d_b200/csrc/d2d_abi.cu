// d2d_abi.cu - the C ABI of libd2d_b200.so (include/d2d_b200.h): handle management, host-side folding of
// the link-budget constants, and the kernel launches.  sm_100a only; there is no CPU path.  The step kernels live in
// their own translation units (d2d_internal.h).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "d2d_internal.h"
#include "d2d_aux.cuh"
#include "d2d_launch_plan.h"

static_assert(D2D_STATS_REPLICAS * 8 * sizeof(double) == 65536, "stats layout");

namespace {
thread_local std::string g_last_error;
constexpr double kSpeedOfLight = 299792458.0;   // path_loss.py:9
}  // namespace

int d2d_fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
static int fail(int code, const std::string &msg) { return d2d_fail(code, msg); }

namespace {

D2DParams make_params(const d2d_handle *h, const d2d_step_io_t *io) {
    D2DParams P{};
    P.num_envs = h->cfg.num_envs;
    P.N = h->N; P.V = h->V; P.C = h->cfg.num_cues; P.R = h->cfg.num_rbs;
    P.n_pwr_cue = h->cfg.n_pwr_cue; P.n_pwr_due = h->cfg.n_pwr_due;
    P.episode_length = h->cfg.episode_length;
    P.nbins = h->cfg.num_rbs;
    P.bin_cap = h->bin_cap;
    P.magic_cue = d2d_div_magic(h->cfg.n_pwr_cue);
    P.magic_due = d2d_div_magic(h->cfg.n_pwr_due);
    P.npw1_cue = h->cfg.n_pwr_cue == 1 ? 0xffffffffu : 0u;
    P.npw1_due = h->cfg.n_pwr_due == 1 ? 0xffffffffu : 0u;
    P.align4 = (h->V % 2 == 0) && ((1 + h->cfg.num_cues) % 2 == 0) && ((uintptr_t)h->pos % 16 == 0);
    P.ple = (float)h->ple;
    P.neg_half_ple = (float)(-0.5 * h->ple);
    P.snr_slope = (float)(5.0 * h->ple * std::log10(2.0));
    P.min_cap = (float)h->cfg.min_capacity_mbps;
    // worst-case fp32 error of SINR_dB is ~6e-6 dB for ple = 2 (d2d_common.cuh); x 1e4 for a 1e-4 relative bound
    const bool shadowing = h->cfg.path_loss_model == D2D_PL_SHADOWING;
    P.rescue_band_dB = (h->ple2 && !shadowing) ? 0.0625f : 0.5f;
    P.shadow_chi_dB = shadowing ? (float)h->cfg.shadow_chi_dB : 0.0f;
    P.shadow_d0sq = (float)(h->cfg.shadow_d0_m * h->cfg.shadow_d0_m);
    P.shadow_chi_d = shadowing ? h->cfg.shadow_chi_dB : 0.0;
    P.shadow_d0sq_d = h->cfg.shadow_d0_m * h->cfg.shadow_d0_m;
    P.rng_seed = h->cfg.rng_seed; P.first_global_env = h->cfg.first_global_env; P.rng_step = 0;
    if (h->pos64) {
        // positions were rounded to fp32: each coordinate is off by <= ulp(R)/2, a distance by <= ~sqrt(2) ulp(R),
        // i.e. 10 ple log10(e) * sqrt(2) ulp(R) / d dB per term; recompute whatever that could push past 1e-4 relative
        const double ulp = std::ldexp(1.0, std::ilogb(std::max(h->cfg.cell_radius_m, 1.0)) - 23);
        P.rescue_c = (float)(2.0 * 1e4 * 4.3429448190325 * h->ple * std::sqrt(2.0) * ulp);
        P.rescue_dmin2 = (float)std::pow(2.0 * 1e4 * 0.5 * h->ple * std::sqrt(2.0) * ulp, 2.0);   // capacity: d(ln r) = ple * dd/d
    }
    P.u_cue = make_float4(h->u_cue.tx_lin0, h->u_cue.a_lin, h->u_cue.inv_noise, h->u_cue.snr0_dB);
    P.u_due = make_float4(h->u_due.tx_lin0, h->u_due.a_lin, h->u_due.inv_noise, h->u_due.snr0_dB);
    P.us_cue = make_float2(h->us_cue[0], h->us_cue[1]);
    P.us_due = make_float2(h->us_due[0], h->us_due[1]);
    P.uniform = h->uniform ? 1 : 0;
    P.dense_ovf = h->dDenseOvf;
    P.ud_cue = h->ud_cue; P.ud_due = h->ud_due;
    P.reward_fn = h->cfg.reward_fn;
    if (h->cfg.reward_fn != D2D_REWARD_SYSTEM_CAPACITY) {
        // the hard SINR threshold of the per-agent reward functions: links this close to it are decided in fp64
        P.thr_dB = (float)h->cfg.reward_param; P.thr_d = h->cfg.reward_param;
        P.thr_band = (h->ple2 && !shadowing) ? 2e-3f : 1.6e-2f;
    }
    P.ple_d = h->ple;
    P.linkA = h->dA; P.linkB = h->dB; P.linkD = h->dD; P.link_meta = h->dMeta; P.pwr_lin = h->dPwr; P.pwr_lin_d = h->dPwrD;
    P.pos = h->pos; P.pos64 = h->pos64; P.step_count = h->step_count; P.stats = h->stats;
    P.episode_index = h->episode_index; P.ar_base = h->ar_base;
    P.rng_step_dev = h->dRngStep;
    P.cell_radius = (float)h->cfg.cell_radius_m; P.d2d_radius = (float)h->cfg.d2d_radius_m;
    P.pos_out = h->pos;
    P.obs_dyn = reinterpret_cast<float2 *>(io->obs_dyn); P.actions_out = io->actions_out;
    P.actions = io->actions; P.obs = io->obs; P.cap = io->capacity_mbps; P.reward = io->reward;
    P.done = io->done; P.rate = io->rate_bps; P.rb_out = io->rb; P.pwr_out = io->tx_pwr_dBm;
    return P;
}

}  // namespace

D2D_API int d2d_abi_version(void) { return D2D_ABI_VERSION; }

D2D_API const char *d2d_last_error(void) { return g_last_error.c_str(); }

D2D_API int d2d_create(const d2d_config_t *cfg, const d2d_link_t *links, d2d_handle_t **out) {
    if (!cfg || !links || !out) return fail(D2D_ERR_INVALID_ARG, "d2d_create: null argument");
    *out = nullptr;
    if (cfg->abi_version != D2D_ABI_VERSION) return fail(D2D_ERR_INVALID_ARG, "d2d_create: abi_version mismatch");
    if (cfg->num_envs < 1) return fail(D2D_ERR_INVALID_ARG, "d2d_create: num_envs must be >= 1");
    if (cfg->num_rbs < 1 || cfg->num_cues < 0 || cfg->num_due_pairs < 0 || cfg->num_cues + cfg->num_due_pairs < 1)
        return fail(D2D_ERR_INVALID_ARG, "d2d_create: need num_rbs >= 1 and at least one link");
    if (cfg->num_downlinks != 0 && cfg->num_downlinks != cfg->num_cues)
        return fail(D2D_ERR_INVALID_ARG, "d2d_create: num_downlinks must be 0 or num_cues (one 'mbs:cueXX' link per CUE)");
    if (cfg->num_downlinks && (cfg->n_pwr_mbs < 1 || cfg->n_pwr_mbs > D2D_MAX_PWR_LEVELS))
        return fail(D2D_ERR_UNSUPPORTED, "d2d_create: n_pwr_mbs must be in [1, 128]");
    if (cfg->n_pwr_cue < 1 || cfg->n_pwr_due < 1 || cfg->n_pwr_cue > D2D_MAX_PWR_LEVELS || cfg->n_pwr_due > D2D_MAX_PWR_LEVELS)
        return fail(D2D_ERR_UNSUPPORTED, "d2d_create: power levels per link must be in [1, 128]");
    if (cfg->num_rbs > 32767) return fail(D2D_ERR_UNSUPPORTED, "d2d_create: num_rbs must be <= 32767");
    if (cfg->path_loss_model != D2D_PL_LOG_DISTANCE && cfg->path_loss_model != D2D_PL_FREE_SPACE &&
        cfg->path_loss_model != D2D_PL_COST_HATA && cfg->path_loss_model != D2D_PL_SHADOWING)
        return fail(D2D_ERR_UNSUPPORTED, "d2d_create: unsupported path_loss_model (LogDistance / FreeSpace / CostHata / Shadowing only)");
    if (cfg->path_loss_model == D2D_PL_SHADOWING && (!(cfg->shadow_chi_dB >= 0.0) || !(cfg->shadow_d0_m >= 0.0)))
        return fail(D2D_ERR_INVALID_ARG, "d2d_create: shadow_chi_dB and shadow_d0_m must be >= 0");
    if (cfg->obs_fn != D2D_OBS_LINEAR) return fail(D2D_ERR_UNSUPPORTED, "d2d_create: unsupported obs_fn (LinearObsFunction only)");
    if (cfg->reward_fn != D2D_REWARD_SYSTEM_CAPACITY && cfg->reward_fn != D2D_REWARD_SHANNON &&
        cfg->reward_fn != D2D_REWARD_CUE_SINR_SHANNON)
        return fail(D2D_ERR_UNSUPPORTED, "d2d_create: unsupported reward_fn (SystemCapacity / Shannon / CueSinrShannon only)");
    if (!(cfg->carrier_freq_GHz > 0.0)) return fail(D2D_ERR_INVALID_ARG, "d2d_create: carrier_freq_GHz must be > 0");
    const double ple = cfg->path_loss_model == D2D_PL_FREE_SPACE ? 2.0 : cfg->ple;
    if (!(ple > 0.0) || ple > 8.0) return fail(D2D_ERR_INVALID_ARG, "d2d_create: ple must be in (0, 8]");
    if (cfg->episode_length < 1 || cfg->episode_length > 255)
        return fail(D2D_ERR_UNSUPPORTED, "d2d_create: episode_length must be in [1, 255]");

    d2d_handle *h = new (std::nothrow) d2d_handle();
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_create: out of host memory");
    h->cfg = *cfg;
    h->N = cfg->num_cues + cfg->num_due_pairs + cfg->num_downlinks;
    h->V = 1 + cfg->num_cues + 2 * cfg->num_due_pairs;
    h->ple = ple;
    h->ple2 = ple == 2.0;
    if (h->N > 65535) { delete h; return fail(D2D_ERR_UNSUPPORTED, "d2d_create: at most 65535 links per env"); }
    // path_loss.py:28-39
    h->K_dB = 10.0 * ple * std::log10(cfg->carrier_freq_GHz * 1e9) + 10.0 * ple * std::log10((4.0 * M_PI) / kSpeedOfLight);

    auto bail = [&](int code) { d2d_destroy(h); return code; };
    D2DDeviceGuard guard(cfg->cuda_device);        // restores the caller's current device on every return path
    if (guard.err != cudaSuccess) return bail(fail(D2D_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(guard.err)));
    cudaDeviceProp prop{};
    cudaError_t e = cudaGetDeviceProperties(&prop, cfg->cuda_device);
    if (e != cudaSuccess) return bail(fail(D2D_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e)));
    if (prop.major != 10)
        return bail(fail(D2D_ERR_UNSUPPORTED, "libd2d_b200 is built for sm_100a (Blackwell B200) only; device is sm_" +
                                                  std::to_string(prop.major) + std::to_string(prop.minor)));
    h->num_sms = prop.multiProcessorCount;

    // fold the link-budget constants (SURVEY Appendix A) in fp64, store fp32 + fp64 copies
    std::vector<D2DLinkA> A(h->N);
    std::vector<D2DLinkB> B(h->N);
    std::vector<D2DLinkD> Dv(h->N);
    std::vector<int32_t> meta(h->N);
    for (int j = 0; j < h->N; ++j) {
        const d2d_link_t &L = links[j];
        const bool cue = j < cfg->num_cues, down = j >= cfg->num_cues + cfg->num_due_pairs;
        const int expect = cue ? D2D_LINK_UPLINK : down ? D2D_LINK_DOWNLINK : D2D_LINK_SIDELINK;
        if (L.link_type != expect)
            return bail(fail(D2D_ERR_UNSUPPORTED, "d2d_create: link " + std::to_string(j) +
                                                      " has an unsupported link_type (CUE uplinks, DUE sidelinks, then MBS downlinks)"));
        // the path-loss constant K belongs to the RECEIVER (CostHata: A(h_tx, h_rx) - 3 B; log-distance: one K for all), so it
        // is folded into the victim's constants and the radiated weights w carry none: I_true = 10^(-K_rx/10) sum w_k g_k
        const double Kj = cfg->path_loss_model == D2D_PL_COST_HATA ? L.path_loss_const_dB : h->K_dB;
        A[j].tx_lin0 = (float)std::pow(10.0, L.tx_eirp_offset_dB / 10.0);
        const double snr0 = L.tx_eirp_offset_dB + L.rx_offset_dB - Kj - L.rx_noise_dBm;
        A[j].a_lin = (float)std::pow(10.0, snr0 / 10.0);
        A[j].inv_noise = (float)std::pow(10.0, -(Kj + L.rx_noise_dBm) / 10.0);
        A[j].snr0_dB = (float)snr0;
        B[j].sens_dBm = (float)L.rx_sensitivity_dBm;
        B[j].bw_MHz = (float)(1e-6 * (L.tx_rb_bandwidth_kHz * 1000.0));
        // envs/d2d_env.py:80-91: uplink cue j -> mbs; sidelink due pair; downlink mbs -> cue (j - C - D)
        B[j].tx_dev = cue ? 1 + j : down ? 0 : 1 + cfg->num_cues + 2 * (j - cfg->num_cues);
        B[j].rx_dev = cue ? 0 : down ? 1 + (j - cfg->num_cues - cfg->num_due_pairs) : B[j].tx_dev + 1;
        meta[j] = (cue ? cfg->n_pwr_cue : down ? cfg->n_pwr_mbs : cfg->n_pwr_due) | ((!cue && !down) ? 1 << 16 : 0);
        Dv[j].a_lin = std::pow(10.0, snr0 / 10.0);
        Dv[j].t_lin = std::pow(10.0, L.tx_eirp_offset_dB / 10.0);
        Dv[j].inv_noise = std::pow(10.0, -(Kj + L.rx_noise_dBm) / 10.0);
        Dv[j].bw_MHz = 1e-6 * (L.tx_rb_bandwidth_kHz * 1000.0);
    }
    // one set of constants per link type (no per-device overrides)?  Then the default-shape kernel reads them from
    // the constant bank instead of a shared-memory table
    h->uniform = cfg->num_downlinks == 0;
    for (int j = 0; j < h->N && !cfg->num_downlinks; ++j) {
        const int j0 = j < cfg->num_cues ? 0 : cfg->num_cues;
        if (std::memcmp(&A[j], &A[j0], sizeof(D2DLinkA)) != 0 || std::memcmp(&Dv[j], &Dv[j0], sizeof(D2DLinkD)) != 0 ||
            B[j].sens_dBm != B[j0].sens_dBm || B[j].bw_MHz != B[j0].bw_MHz)
            h->uniform = false;
    }
    if (cfg->num_cues > 0) h->ud_cue = Dv[0];
    if (cfg->num_due_pairs > 0) h->ud_due = Dv[cfg->num_cues];
    if (cfg->num_cues > 0) { h->u_cue = A[0]; h->us_cue[0] = B[0].sens_dBm; h->us_cue[1] = B[0].bw_MHz; }
    if (cfg->num_due_pairs > 0) {
        h->u_due = A[cfg->num_cues]; h->us_due[0] = B[cfg->num_cues].sens_dBm; h->us_due[1] = B[cfg->num_cues].bw_MHz;
    }
    float pwr[D2D_MAX_PWR_LEVELS];
    double pwr_d[D2D_MAX_PWR_LEVELS];
    for (int p = 0; p < D2D_MAX_PWR_LEVELS; ++p) {   // conversion.py:4-13
        pwr_d[p] = std::pow(10.0, p / 10.0);
        pwr[p] = (float)pwr_d[p];
    }

#define D2D_CUDA_BAIL(call)                                                                              \
    do {                                                                                                 \
        cudaError_t err__ = (call);                                                                      \
        if (err__ != cudaSuccess)                                                                        \
            return bail(fail(D2D_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(err__)));       \
    } while (0)
    D2D_CUDA_BAIL(cudaMalloc(&h->dA, sizeof(D2DLinkA) * h->N));
    D2D_CUDA_BAIL(cudaMalloc(&h->dB, sizeof(D2DLinkB) * h->N));
    D2D_CUDA_BAIL(cudaMalloc(&h->dD, sizeof(D2DLinkD) * h->N));
    D2D_CUDA_BAIL(cudaMalloc(&h->dMeta, sizeof(int32_t) * h->N));
    D2D_CUDA_BAIL(cudaMemcpy(h->dMeta, meta.data(), sizeof(int32_t) * h->N, cudaMemcpyHostToDevice));
    D2D_CUDA_BAIL(cudaMalloc(&h->dPwr, sizeof(pwr)));
    D2D_CUDA_BAIL(cudaMalloc(&h->dPwrD, sizeof(pwr_d)));
    D2D_CUDA_BAIL(cudaMemcpy(h->dPwrD, pwr_d, sizeof(pwr_d), cudaMemcpyHostToDevice));
    D2D_CUDA_BAIL(cudaMemcpy(h->dA, A.data(), sizeof(D2DLinkA) * h->N, cudaMemcpyHostToDevice));
    D2D_CUDA_BAIL(cudaMemcpy(h->dB, B.data(), sizeof(D2DLinkB) * h->N, cudaMemcpyHostToDevice));
    D2D_CUDA_BAIL(cudaMemcpy(h->dD, Dv.data(), sizeof(D2DLinkD) * h->N, cudaMemcpyHostToDevice));
    D2D_CUDA_BAIL(cudaMemcpy(h->dPwr, pwr, sizeof(pwr), cudaMemcpyHostToDevice));
    if (cfg->path_loss_model == D2D_PL_SHADOWING) {
        D2D_CUDA_BAIL(cudaMalloc(&h->dRngStep, sizeof(uint64_t)));
        D2D_CUDA_BAIL(cudaMemset(h->dRngStep, 0, sizeof(uint64_t)));
    }
#undef D2D_CUDA_BAIL

    // warp kernel: one lane slot per CUE and per DUE pair, one shared-memory bin per RB
    // downlink links and ShadowingPathLoss run on the general-topology kernel
    const bool general = cfg->num_downlinks != 0 || cfg->path_loss_model == D2D_PL_SHADOWING;
    h->use_warp = cfg->num_cues <= 32 && cfg->num_due_pairs <= 32 && cfg->num_rbs <= 64 && !general;
    if (const char *c = std::getenv("D2D_B200_CHUNK")) h->chunk_override = std::atoll(c);
    if (const char *c = std::getenv("D2D_B200_TICKET")) h->tickets_on = std::atoi(c) != 0;
    if (const char *c = std::getenv("D2D_B200_LATE_WAIT")) h->late_wait_on = std::atoi(c) != 0;      // tests / A-B
    const char *pdl = std::getenv("D2D_B200_PDL");
    h->pdl = !(pdl && std::strcmp(pdl, "0") == 0);
    const char *sp = std::getenv("D2D_B200_SPEC");
    const bool spec_ok = !sp || std::atoi(sp) != 0;       // tests: D2D_B200_SPEC=0 forces the generic shapes
    int rc;
    if (h->use_warp) {
        // launch shape by batch size (d2d_step_warp.cuh): well under one wave of envs -> 2-warp blocks, everything else 4-warp blocks
        // (8-warp blocks were the large-batch shape until chains of steps stopped waiting for whole grids: with per-warp tickets
        // the 4-warp shape's 28 resident warps per SM win at every size - E = 131 072: 63.5 vs 65.9 us; D2D_B200_WPB=8 still selects it)
        const char *w = std::getenv("D2D_B200_WPB");
        h->warp = d2d_warp_shape(w ? std::atoi(w) : cfg->num_envs <= D2D_LATENCY_ENVS ? 2 : 4);
        if (h->warp->wpb == 4 && cfg->num_envs >= 65536 && !w) h->many.warp = &d2d_warp_shape_8;     // the fused launches' own shape
        h->spec = spec_ok && h->ple2 && h->uniform && cfg->path_loss_model != D2D_PL_COST_HATA && cfg->num_rbs == 25 && cfg->num_cues == 25 &&
                  cfg->num_due_pairs == 25 && cfg->n_pwr_cue == 24 && cfg->n_pwr_due == 21;
        // per shape this handle launches: the fp64 pass reads 10^(p/10) from the constant bank of the translation unit that holds
        // the shape's kernels (per device: set at every create); then the geometry, in h->grid / block / smem / envs_per_block
        auto setup = [&](const D2DWarpShape *ws) {
            const cudaError_t et = ws->tables(pwr_d);
            if (et != cudaSuccess) return fail(D2D_ERR_CUDA, std::string("cudaMemcpyToSymbol(d2d_pwr_lin_c): ") + cudaGetErrorString(et));
            return ws->plan(h, ws->smem(cfg->num_rbs));
        };
        if (h->many.warp) {
            rc = setup(h->many.warp);
            if (rc != D2D_OK) return bail(rc);
            h->many.grid = h->grid; h->many.envs_per_block = h->envs_per_block;
        }
        rc = setup(h->warp);
    } else {
        // <= 1024 links: the binned one-barrier kernel (d2d_step_dense.cuh), LPT links per thread; when its double-buffered
        // bins do not fit (many RBs) the sorting block kernel; beyond 1024 links / other topologies: everything staged in shared memory
        h->lpt = (h->N <= D2D_BLOCK_THREADS * D2D_BLOCK_MAX_LPT && !general)
                     ? (h->N + D2D_BLOCK_THREADS - 1) / D2D_BLOCK_THREADS : 0;      // downlinks: the general-topology kernel
        h->bin_cap = d2d_dense_bin_cap_host(h->N, cfg->num_rbs);
        const char *dn = std::getenv("D2D_B200_DENSE");
        // threads per block / links per thread: the shape with the fewest (warp, slot) bodies per env - every warp runs the
        // straight-line code of each of its slots whether or not all 32 lanes hold a link (N = 600: 10 warps x 2 slots,
        // all but one full, instead of 8 warps x 3 with the third slot three-quarters empty)
        const int bt = ((h->N + 319) / 320) * 10 < ((h->N + 255) / 256) * 8 && (h->N + 319) / 320 <= 3 ? 320 : 256;
        const bool dense = h->lpt > 0 && cfg->num_rbs <= 512 /* 9 bits of the packed link state */ &&
                           d2d_dense_smem(h->N, cfg->num_rbs, h->bin_cap, bt, h->V) <= 75 * 1024 /* three blocks per SM */ && !(dn && std::atoi(dn) == 0);
        if (dense) {
            h->dense_bt = bt;
            h->lpt = (h->N + bt - 1) / bt;
            // BASELINE config #3's shape has its own instantiation (d2d_step_dense.cuh: SPEC)
            h->spec = spec_ok && h->ple2 && bt == 320 && h->N == 600 && cfg->num_cues == 100 && cfg->num_rbs == 100 && h->bin_cap == 16 &&
                      cfg->n_pwr_cue == 24 && cfg->n_pwr_due == 21;
        }
        const size_t smem = dense ? d2d_dense_smem(h->N, cfg->num_rbs, h->bin_cap, bt, h->V) : d2d_block_smem(h->N, cfg->num_rbs, h->lpt);
        if (smem > 227 * 1024) return bail(fail(D2D_ERR_UNSUPPORTED, "d2d_create: too many links / RBs for one SM's shared memory"));
        rc = dense ? d2d_dense_plan(h, smem) : d2d_block_plan(h, smem);
    }
    if (rc != D2D_OK) return bail(rc);
    if (h->dense_bt) {      // the blocks' overflow lists: [grid][N] records + [grid][N] RBs
        cudaError_t eo = cudaMalloc(&h->dDenseOvf, (size_t)h->grid * h->N * (sizeof(float4) + sizeof(uint16_t)) + 16);
        if (eo != cudaSuccess) return bail(fail(D2D_ERR_CUDA, std::string("dense overflow scratch: ") + cudaGetErrorString(eo)));
    }
    // CueSinrShannonRewardFunction's post-pass keeps one weak-link counter per RB and team in shared memory
    if (cfg->reward_fn == D2D_REWARD_CUE_SINR_SHANNON) {
        const size_t smem = (size_t)(h->N <= 64 ? 8 : 1) * cfg->num_rbs * sizeof(uint32_t);
        if (smem > 200 * 1024) return bail(fail(D2D_ERR_UNSUPPORTED, "d2d_create: CueSinrShannonRewardFunction supports at most " +
                                                                         std::to_string(200 * 1024 / 4 / (h->N <= 64 ? 8 : 1)) + " RBs for this link count"));
        rc = h->N <= 64 ? d2d_allow_smem(d2d_agent_reward_kernel<32>, smem) : d2d_allow_smem(d2d_agent_reward_kernel<256>, smem);
        if (rc != D2D_OK) return bail(rc);
    }
    // Late-wait steps (DESIGN.md 4.7) of small and medium batches run on a FRACTION of the block slots: a launch that fills the machine
    // keeps its successor's blocks out until its own retire, so consecutive steps overlap only in their tails (E = 4096, one env per
    // warp on 1024 of 1036 slots: 4.95 us per step in a long chain).  On three of an SM's seven slots - every warp a software-pipelined
    // loop over 2-3 envs - two launches are resident at once: 3.86 us (E = 8192: 6.3 -> 5.4 us, E = 16 384: 9.3 -> 8.7 us).  One block
    // per SM is faster still in a long chain (3.75 us: up to seven launches in flight) but a launch then takes 14 us from its first
    // warp to its last, which a chain of 10-20 steps pays for (20 steps: 4.2-4.4 us per step on three blocks, 4.4 on one, 5.3 on the
    // full grid; 10 steps: 4.7 / 5.3 / 5.5).  Large batches need every warp slot for their own latency hiding (E = 32 768: 17.1 us on
    // the full grid, 17.8 on three blocks per SM).  The latency shape (2-warp blocks): two blocks per SM - E = 1024 1.87 -> 1.76 us,
    // E = 2048 3.38 -> 2.32 us.  Sweeps: profiles/ab_r02_40.log .. ab_r02_46.log
    if (h->use_warp && h->warp->wpb == 2) h->grid_late = 2 * h->num_sms;
    if (h->use_warp && h->warp->wpb == 4) h->grid_late = cfg->num_envs <= 166 * (int64_t)h->num_sms ? 3 * h->num_sms : 0;
    // (default-ordering steps keep the full grid: half of it speeds up chains of them but costs an isolated step behind a policy
    // kernel up to 1 us, profiles/README.md)
    if (const char *gl = std::getenv("D2D_B200_LATE_GRID")) h->grid_late = std::max(0, std::atoi(gl));      // A/B
    if (const char *gs = std::getenv("D2D_B200_GRID"))      // tests: few blocks, so every block steps many envs
        if (std::atoi(gs) > 0) { h->grid = std::min(h->grid, std::atoi(gs)); h->many.grid = std::min(h->many.grid, std::atoi(gs)); }
    if (h->use_warp) {      // one ticket word per warp slot of the step geometry
        const size_t words = (size_t)h->grid * h->warp->wpb;
        cudaError_t et = cudaMalloc(&h->dTickets, words * sizeof(uint64_t));
        if (et == cudaSuccess) et = cudaMemset(h->dTickets, 0, words * sizeof(uint64_t));
        if (et != cudaSuccess) return bail(fail(D2D_ERR_CUDA, std::string("ticket buffer: ") + cudaGetErrorString(et)));
    }
    *out = h;
    return D2D_OK;
}

namespace {
void free_slot(d2d_host_slot &s) {
    cudaFree(s.dev);
    cudaFree(s.stage16);
    s.stage16 = nullptr;
    if (s.host) cudaFreeHost(s.host);
    s.dev = s.host = nullptr;
    s.bytes = s.out_offset = s.out_bytes = 0;
    s.mask = 0;
}
}  // namespace

D2D_API int d2d_destroy(d2d_handle_t *h) {
    if (!h) return D2D_OK;
    D2DDeviceGuard guard(h->cfg.cuda_device);
    cudaFree(h->dA); cudaFree(h->dB); cudaFree(h->dD); cudaFree(h->dMeta); cudaFree(h->dPwr); cudaFree(h->dPwrD); cudaFree(h->stage_pos);
    cudaFree(h->dRngStep); cudaFree(h->act_scratch); cudaFree(h->dTickets); cudaFree(h->dDenseOvf);
    for (auto &s : h->slot) {
        if (s.used && s.ev_out) cudaEventSynchronize(s.ev_out);
        free_slot(s);
        for (void *p : s.stage) cudaFree(p);
        if (h->pipe_ready) { cudaEventDestroy(s.ev_in); cudaEventDestroy(s.ev_kernel); cudaEventDestroy(s.ev_out); }
    }
    if (h->pipe_ready) { cudaStreamDestroy(h->s_in); cudaStreamDestroy(h->s_out); }
    delete h;
    return D2D_OK;
}

D2D_API int d2d_state_bytes(const d2d_handle_t *h, size_t *pos_bytes, size_t *step_bytes, size_t *stats_bytes) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_state_bytes: null handle");
    if (pos_bytes) *pos_bytes = (size_t)h->cfg.num_envs * h->V * 2 * sizeof(float);
    if (step_bytes) *step_bytes = (size_t)h->cfg.num_envs;
    if (stats_bytes) *stats_bytes = (size_t)D2D_STATS_REPLICAS * 8 * sizeof(double);
    return D2D_OK;
}

D2D_API int d2d_bind_state(d2d_handle_t *h, float *positions, uint8_t *step_count, double *stats) {
    if (!h || !positions) return fail(D2D_ERR_INVALID_ARG, "d2d_bind_state: positions buffer is required");
    if ((uintptr_t)positions % 16) return fail(D2D_ERR_INVALID_ARG, "d2d_bind_state: positions must be 16-byte aligned");
    if (positions != h->pos) h->last_kind = D2D_LAST_OTHER;      // new positions: nothing is known about who wrote them
    h->pos = positions;
    h->step_count = step_count;
    h->stats = stats;
    return D2D_OK;
}

D2D_API int d2d_bind_positions_f64(d2d_handle_t *h, double *positions_f64) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_bind_positions_f64: null handle");
    if (positions_f64 && ((uintptr_t)positions_f64 % 16))
        return fail(D2D_ERR_INVALID_ARG, "d2d_bind_positions_f64: buffer must be 16-byte aligned");
    h->pos64 = positions_f64;
    h->last_kind = D2D_LAST_OTHER;
    return D2D_OK;
}

D2D_API int d2d_bind_autoreset(d2d_handle_t *h, uint32_t *episode_index, uint64_t base_key) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_bind_autoreset: null handle");
    if (episode_index && !h->use_warp)
        return fail(D2D_ERR_UNSUPPORTED, "d2d_bind_autoreset: auto-reset runs on the warp kernel only (<= 32 CUEs, <= 32 DUE pairs, <= 64 RBs, "
                                         "no downlinks, no ShadowingPathLoss)");
    h->episode_index = episode_index;
    h->ar_base = base_key;
    return D2D_OK;
}

D2D_API int d2d_set_positions(d2d_handle_t *h, const double *src, int src_on_device, int64_t first_env, int64_t count,
                              void *stream) {
    if (!h || !src) return fail(D2D_ERR_INVALID_ARG, "d2d_set_positions: null argument");
    if (!h->pos) return fail(D2D_ERR_STATE, "d2d_set_positions: call d2d_bind_state first");
    if (first_env < 0 || count < 0 || first_env + count > h->cfg.num_envs)
        return fail(D2D_ERR_INVALID_ARG, "d2d_set_positions: env range out of bounds");
    if (count == 0) return D2D_OK;
    D2D_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const double *dsrc = src;
    if (!src_on_device) {
        if (h->stage_pos_envs < count) {
            cudaFree(h->stage_pos);
            h->stage_pos = nullptr; h->stage_pos_envs = 0;
            D2D_CUDA(cudaMalloc(&h->stage_pos, sizeof(double) * 2 * h->V * count));
            h->stage_pos_envs = count;
        }
        D2D_CUDA(cudaMemcpyAsync(h->stage_pos, src, sizeof(double) * 2 * h->V * count, cudaMemcpyHostToDevice, st));
        dsrc = h->stage_pos;
    }
    const int64_t total = count * h->V;
    const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)h->num_sms * 8);
    d2d_set_positions_kernel<<<grid, 256, 0, st>>>(dsrc, h->pos + first_env * h->V * 2,
                                                    h->pos64 ? h->pos64 + first_env * h->V * 2 : nullptr, count, h->V);
    D2D_CUDA(cudaGetLastError());
    ++h->launches;
    h->last_kind = D2D_LAST_OTHER; h->last_stream = stream;
    if (!src_on_device) D2D_CUDA(cudaStreamSynchronize(st));
    return D2D_OK;
}

D2D_API int d2d_get_positions(d2d_handle_t *h, float *dst, int dst_on_device, int64_t first_env, int64_t count, void *stream) {
    if (!h || !dst) return fail(D2D_ERR_INVALID_ARG, "d2d_get_positions: null argument");
    if (!h->pos) return fail(D2D_ERR_STATE, "d2d_get_positions: call d2d_bind_state first");
    if (first_env < 0 || count < 0 || first_env + count > h->cfg.num_envs)
        return fail(D2D_ERR_INVALID_ARG, "d2d_get_positions: env range out of bounds");
    if (count == 0) return D2D_OK;
    D2D_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t row = sizeof(float) * 2 * h->V;
    D2D_CUDA(cudaMemcpyAsync(dst, h->pos + first_env * h->V * 2, row * count, dst_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    if (!dst_on_device) D2D_CUDA(cudaStreamSynchronize(st));
    return D2D_OK;
}

namespace {

// Simulator.reset for every env in the mask; `total` units per launch stay below 2^32
int reset_launch(d2d_handle *h, uint64_t seed, uint64_t first_global_env, const uint8_t *env_mask, cudaStream_t st) {
    const int C = h->cfg.num_cues, D = h->cfg.num_due_pairs;
    const int64_t units = (C + 1) / 2 + D;
    const int64_t chunk = std::max<int64_t>(1, (int64_t)0x7fffffff / std::max<int64_t>(units, 2 * h->V));
    for (int64_t e0 = 0; e0 < h->cfg.num_envs; e0 += chunk) {
        const int64_t n = std::min<int64_t>(chunk, h->cfg.num_envs - e0);
        const int64_t total = n * units;
        const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)h->num_sms * 16);
        d2d_reset_kernel<<<grid, 256, 0, st>>>(h->pos + e0 * h->V * 2, h->pos64 ? h->pos64 + e0 * h->V * 2 : nullptr,
                                               h->step_count ? h->step_count + e0 : nullptr, env_mask ? env_mask + e0 : nullptr,
                                               (uint32_t)total, (uint32_t)C, (uint32_t)D, (float)h->cfg.cell_radius_m,
                                               (float)h->cfg.d2d_radius_m, seed, first_global_env + (uint64_t)e0,
                                               (uint32_t)((0x100000000ull + (uint64_t)units - 1) / (uint64_t)units));
        D2D_CUDA(cudaGetLastError());
        ++h->launches;
    }
    return D2D_OK;
}

int sample_launch(d2d_handle *h, int32_t *actions, uint64_t seed, uint32_t t, cudaStream_t st) {
    const int C = h->cfg.num_cues, D = h->cfg.num_due_pairs;
    const int64_t L = std::max(C, D);
    const int64_t chunk = std::max<int64_t>(1, (int64_t)0x7fffffff / std::max<int64_t>(L, h->N));
    for (int64_t e0 = 0; e0 < h->cfg.num_envs; e0 += chunk) {
        const int64_t n = std::min<int64_t>(chunk, h->cfg.num_envs - e0);
        const int64_t total = n * L;
        const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)h->num_sms * 16);
        d2d_sample_actions_kernel<<<grid, 256, 0, st>>>(actions + e0 * h->N, (uint32_t)total, (uint32_t)C, (uint32_t)D, (uint32_t)h->N,
                                                        (uint32_t)(h->cfg.num_rbs * h->cfg.n_pwr_cue), (uint32_t)(h->cfg.num_rbs * h->cfg.n_pwr_due),
                                                        seed, h->cfg.first_global_env + (uint64_t)e0, t);
        D2D_CUDA(cudaGetLastError());
        ++h->launches;
    }
    return D2D_OK;
}

}  // namespace

D2D_API int d2d_reset(d2d_handle_t *h, uint64_t seed, uint64_t first_global_env, const uint8_t *env_mask, void *stream) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_reset: null handle");
    if (!h->pos) return fail(D2D_ERR_STATE, "d2d_reset: call d2d_bind_state first");
    D2D_GUARD(h);
    h->last_kind = D2D_LAST_OTHER; h->last_stream = stream;
    return reset_launch(h, seed, first_global_env, env_mask, (cudaStream_t)stream);
}

D2D_API int d2d_sample_actions(d2d_handle_t *h, int32_t *actions, uint64_t seed, uint32_t step_index, void *stream) {
    if (!h || !actions) return fail(D2D_ERR_INVALID_ARG, "d2d_sample_actions: null argument");
    D2D_GUARD(h);
    h->last_kind = D2D_LAST_OTHER; h->last_stream = stream;      // it writes actions: the next step orders itself the default way
    return sample_launch(h, actions, seed, step_index, (cudaStream_t)stream);
}

namespace {

// per-agent rewards (SHANNON / CUE_SINR_SHANNON always; SYSTEM_CAPACITY when the caller asked for the broadcast): one more
// small kernel over `total` env-steps of io; `with_stats`: the reward statistics of the per-agent functions; `autoreset`: rows
// whose step counter is 0 after the step were reset by it (D2D_STEP_AUTORESET) and score nothing
int agent_reward_launch(d2d_handle *h, const d2d_step_io_t *io, int64_t total, bool with_stats, cudaStream_t st, bool autoreset = false) {
    if (!io->obs || !io->reward || !io->actions) return fail(D2D_ERR_INVALID_ARG, "per-agent rewards need the actions, obs and reward buffers");
    const bool warp_team = h->N <= 64;
    const int teams = warp_team ? 8 : 1;
    const int grid = (int)std::min<int64_t>((total + teams - 1) / teams, (int64_t)h->num_sms * 8);
    // only CueSinrShannon keeps per-RB counters in shared memory (opt-in done by d2d_create)
    const size_t smem = h->cfg.reward_fn == D2D_REWARD_CUE_SINR_SHANNON ? (size_t)teams * h->cfg.num_rbs * sizeof(uint32_t) : 0;
    double *stats = with_stats && h->cfg.reward_fn != D2D_REWARD_SYSTEM_CAPACITY ? h->stats : nullptr;
    const uint8_t *counters = autoreset ? h->step_count : nullptr;
    if (warp_team)
        d2d_agent_reward_kernel<32><<<grid, 256, smem, st>>>(io->actions, io->obs, io->agent_reward, io->reward, stats, total, h->N,
                                                            h->dMeta, h->cfg.num_rbs, h->cfg.reward_fn, (float)h->cfg.reward_param, counters);
    else
        d2d_agent_reward_kernel<256><<<grid, 256, smem, st>>>(io->actions, io->obs, io->agent_reward, io->reward, stats, total, h->N,
                                                             h->dMeta, h->cfg.num_rbs, h->cfg.reward_fn, (float)h->cfg.reward_param, counters);
    D2D_CUDA(cudaGetLastError());
    ++h->launches;
    return D2D_OK;
}

int step_launch(d2d_handle *h, const d2d_step_io_t *io, int T, int mode, void *stream, const EpisodeArgs &ea = EpisodeArgs()) {
    const D2DStepPlan pl = d2d_plan_step(h, io, mode, stream, ea);
    D2DParams P = make_params(h, io);
    P.T = T;
    P.t_stride = h->cfg.num_envs;
    P.ep_seed = ea.ep_seed; P.act_seed = ea.act_seed; P.act_t0 = ea.act_t0;
    P.flags = pl.flags | (ea.draw_actions ? D2D_PF_DRAW_ACTIONS : 0u) | (ea.no_reset ? D2D_PF_NO_RESET : 0u);
    if (pl.tok_sign) { P.tickets = h->dTickets; P.tok_wait = pl.tok_wait; P.tok_sign = pl.tok_sign; }
    cudaStream_t st = (cudaStream_t)stream;
    for (int64_t e0 = 0; e0 < h->cfg.num_envs; e0 += pl.chunk) {
        const int64_t n = std::min<int64_t>(pl.chunk, h->cfg.num_envs - e0);
        if (e0 > 0) {
            const int64_t dl = pl.chunk * h->N;
            P.first_global_env += (uint64_t)pl.chunk;
            if (P.actions) P.actions += dl;
            P.pos += pl.chunk * h->V * 2; P.pos_out += pl.chunk * h->V * 2;
            if (P.pos64) P.pos64 += pl.chunk * h->V * 2;
            if (P.step_count) P.step_count += pl.chunk;
            if (P.episode_index) P.episode_index += pl.chunk;
            if (P.obs) P.obs += dl * 6;
            if (P.obs_dyn) P.obs_dyn += dl;
            if (P.cap) P.cap += dl;
            if (P.reward) P.reward += pl.chunk;
            if (P.done) P.done += pl.chunk;
            if (P.rate) P.rate += dl;
            if (P.rb_out) P.rb_out += dl;
            if (P.pwr_out) P.pwr_out += dl;
            // a later chunk of the same step follows a kernel that passed its wait (or was itself entitled to skip it)
            if (h->pdl) P.flags &= ~D2D_PF_INPUTS_FRESH;
        }
        P.num_envs = n;
#ifdef D2D_TIMELINE
        P.tl_slot = (int32_t)(h->launches % D2D_TL_SLOTS);
#endif
        const bool alt = mode != MODE_STEP && h->many.warp;      // fused multi-step launches of large batches: their own shape
        const D2DWarpShape *warp = alt ? h->many.warp : h->warp;
        const int epb = alt ? h->many.envs_per_block : h->envs_per_block;
        const int grid = (int)std::min<int64_t>(alt ? h->many.grid : pl.grid, (n + epb - 1) / epb);
        if (h->use_warp) { const int64_t warps = (int64_t)grid * warp->wpb; P.envs_per_warp = (uint32_t)(n / warps); P.envs_extra = (uint32_t)(n % warps); }
        D2DLaunchSel sel;
        sel.many = mode == MODE_MANY; sel.episode = mode == MODE_EPISODE;
        sel.no_reset = ea.no_reset;
        sel.autoreset = pl.autoreset;
        sel.fast = mode == MODE_EPISODE && ea.draw_actions && !io->actions_out;
        sel.exact = h->pos64 != nullptr;
        // FULL: exactly the core outputs were passed, so the kernel tests no output pointer on its hot path
        sel.full = io->obs && io->capacity_mbps && io->reward && io->done && !io->rate_bps && !io->rb && !io->tx_pwr_dBm && !io->obs_dyn &&
                   h->step_count && h->cfg.reward_fn == D2D_REWARD_SYSTEM_CAPACITY;
        cudaError_t err;
        if (h->use_warp) err = warp->launch(h, P, grid, sel, st, h->pdl);
        else if (h->dense_bt) err = d2d_dense_launch(h, P, grid, sel, st, h->pdl);
        else err = d2d_block_launch(h, P, grid, st, h->pdl);
        if (err != cudaSuccess) return fail(D2D_ERR_CUDA, std::string("step kernel launch: ") + cudaGetErrorString(err));
        ++h->launches;
    }
    D2D_CUDA(cudaGetLastError());
    h->last_stream = stream;
    h->last_kind = pl.last_kind;
    if (h->dRngStep) {      // ShadowingPathLoss: the next call draws fresh values, also when this one is replayed from a CUDA graph
        d2d_advance_counter_kernel<<<1, 1, 0, st>>>(h->dRngStep, (uint64_t)T);
        D2D_CUDA(cudaGetLastError());
    }
    if (mode != MODE_EPISODE && (h->cfg.reward_fn != D2D_REWARD_SYSTEM_CAPACITY || io->agent_reward))
        return agent_reward_launch(h, io, (int64_t)T * h->cfg.num_envs, true, st, pl.autoreset);
    return D2D_OK;
}

int check_step_args(const d2d_handle_t *h, const d2d_step_io_t *io, const char *who, bool need_actions = true, bool autoreset_ok = false) {
    if (!h || !io || (need_actions && !io->actions)) return fail(D2D_ERR_INVALID_ARG, std::string(who) + ": handle, io and io->actions are required");
    if (io->flags & D2D_STEP_AUTORESET) {
        if (!autoreset_ok || !h->use_warp)
            return fail(D2D_ERR_UNSUPPORTED, std::string(who) + ": D2D_STEP_AUTORESET applies to d2d_step on warp-kernel configurations only");
        if (!h->episode_index || !h->step_count)
            return fail(D2D_ERR_STATE, std::string(who) + ": D2D_STEP_AUTORESET needs d2d_bind_autoreset and a bound step counter");
    }
    if (!h->pos) return fail(D2D_ERR_STATE, std::string(who) + ": call d2d_bind_state first");
    if (io->flags & D2D_STEP_ACTIONS_I16)      // (d2d_step_host_async clears the flag on the device-side io it passes down)
        return fail(D2D_ERR_INVALID_ARG, std::string(who) + ": D2D_STEP_ACTIONS_I16 applies to d2d_step_host / d2d_step_host_async only");
    if (io->obs && ((uintptr_t)io->obs % 8)) return fail(D2D_ERR_INVALID_ARG, std::string(who) + ": obs must be 8-byte aligned");
    if (io->obs_dyn && ((uintptr_t)io->obs_dyn % 8)) return fail(D2D_ERR_INVALID_ARG, std::string(who) + ": obs_dyn must be 8-byte aligned");
    return D2D_OK;
}

// d2d_episode / d2d_rollout: the per-agent reward pass and the composed path read drawn actions back; when the caller does not
// record them, they go to handle-owned scratch of `slices` x E x N actions
int reserve_act_scratch(d2d_handle *h, int64_t slices, cudaStream_t st) {
    const size_t need = (size_t)slices * h->cfg.num_envs * h->N;
    if (h->act_scratch_elems >= need) return D2D_OK;
    D2D_CUDA(cudaStreamSynchronize(st));
    cudaFree(h->act_scratch);
    h->act_scratch = nullptr; h->act_scratch_elems = 0;
    D2D_CUDA(cudaMalloc(&h->act_scratch, need * sizeof(int32_t)));
    h->act_scratch_elems = need;
    return D2D_OK;
}

// io advanced by `steps` slices of E envs
void advance_io(d2d_step_io_t &cur, int64_t steps, int64_t E, int N) {
    const int64_t dl = steps * E * N, de = steps * E;
    if (cur.actions) cur.actions += dl;
    if (cur.obs) cur.obs += dl * 6;
    if (cur.obs_dyn) cur.obs_dyn += dl * 2;
    if (cur.capacity_mbps) cur.capacity_mbps += dl;
    if (cur.reward) cur.reward += de;
    if (cur.done) cur.done += de;
    if (cur.rate_bps) cur.rate_bps += dl;
    if (cur.rb) cur.rb += dl;
    if (cur.tx_pwr_dBm) cur.tx_pwr_dBm += dl;
    if (cur.agent_reward) cur.agent_reward += dl;
    if (cur.actions_out) cur.actions_out += dl;
}

}  // namespace

D2D_API int d2d_step(d2d_handle_t *h, const d2d_step_io_t *io, void *stream) {
    int rc = check_step_args(h, io, "d2d_step", true, true);
    if (rc) return rc;
    D2D_GUARD(h);
    return step_launch(h, io, 1, MODE_STEP, stream);
}

D2D_API int d2d_step_many(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, void *stream) {
    int rc = check_step_args(h, io, "d2d_step_many");
    if (rc) return rc;
    if (num_steps < 1) return fail(D2D_ERR_INVALID_ARG, "d2d_step_many: num_steps must be >= 1");
    D2D_GUARD(h);
    const int64_t E = h->cfg.num_envs;
    // fused launches of as many steps as 32-bit indices allow (all of them unless T E N is astronomically large);
    // configurations served by the block kernel take one launch per step
    const int64_t fuse = h->use_warp ? std::clamp<int64_t>(d2d_max_launch_envs(h) / E, 1, num_steps) : 1;
    d2d_step_io_t cur = *io;
    for (int64_t t0 = 0; t0 < num_steps; t0 += fuse) {
        const int T = (int)std::min<int64_t>(fuse, num_steps - t0);
        rc = step_launch(h, &cur, T, T > 1 ? MODE_MANY : MODE_STEP, stream);
        if (rc) return rc;
        advance_io(cur, T, E, h->N);
    }
    return D2D_OK;
}

D2D_API int d2d_episode(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, uint64_t reset_seed, uint64_t action_seed,
                        uint32_t episode_flags, void *stream) {
    const bool draw = (episode_flags & D2D_EPISODE_DRAW_ACTIONS) != 0u;
    int rc = check_step_args(h, io, "d2d_episode", !draw);
    if (rc) return rc;
    if (num_steps < 0 || num_steps > 254) return fail(D2D_ERR_INVALID_ARG, "d2d_episode: num_steps must be in [0, 254]");
    if (!h->step_count) return fail(D2D_ERR_STATE, "d2d_episode: a step-counter buffer must be bound");
    D2D_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t E = h->cfg.num_envs;
    const int T1 = num_steps + 1;
    const bool agent_pass = h->cfg.reward_fn != D2D_REWARD_SYSTEM_CAPACITY || io->agent_reward;
    d2d_step_io_t cur = *io;
    const bool fused = h->use_warp && (int64_t)T1 * E <= d2d_max_launch_envs(h);
    if (draw && !cur.actions_out && (agent_pass || !fused)) {
        rc = reserve_act_scratch(h, fused ? T1 : 1, st);
        if (rc) return rc;
    }
    if (fused) {
        if (draw && !cur.actions_out && agent_pass) cur.actions_out = h->act_scratch;
        EpisodeArgs ea;
        ea.ep_seed = reset_seed; ea.act_seed = action_seed; ea.draw_actions = draw;
        rc = step_launch(h, &cur, T1, MODE_EPISODE, stream, ea);
        if (rc) return rc;
        if (agent_pass) {
            if (draw) cur.actions = cur.actions_out;
            rc = agent_reward_launch(h, &cur, E, false, st);                    // slice 0: the reset step enters no statistic
            if (rc || num_steps == 0) return rc;
            advance_io(cur, 1, E, h->N);
            return agent_reward_launch(h, &cur, (int64_t)num_steps * E, true, st);
        }
        return D2D_OK;
    }
    // composed: d2d_reset, then per slice d2d_sample_actions (when drawing) + d2d_step; the reset step is not counted
    h->last_kind = D2D_LAST_OTHER; h->last_stream = stream;
    rc = reset_launch(h, reset_seed, h->cfg.first_global_env, nullptr, st);
    if (rc) return rc;
    uint8_t *counters = h->step_count;
    double *stats = h->stats;
    for (int t = 0; t < T1; ++t) {
        d2d_step_io_t one = cur;
        one.actions_out = nullptr;
        if (draw) {
            int32_t *dst = cur.actions_out ? cur.actions_out : h->act_scratch;
            rc = sample_launch(h, dst, action_seed, (uint32_t)t, st);
            if (rc) return rc;
            one.actions = dst;
            h->last_kind = D2D_LAST_OTHER;
        }
        if (t == 0) { h->step_count = nullptr; h->stats = nullptr; }          // envs/d2d_env.py:50: simulator.step, no num_steps += 1
        rc = step_launch(h, &one, 1, MODE_STEP, stream);
        h->step_count = counters; h->stats = stats;
        if (rc) return rc;
        advance_io(cur, 1, E, h->N);
    }
    return D2D_OK;
}

D2D_API int d2d_rollout(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, uint64_t action_seed, uint32_t first_step_index,
                        void *stream) {
    int rc = check_step_args(h, io, "d2d_rollout", false);
    if (rc) return rc;
    if (num_steps < 1) return fail(D2D_ERR_INVALID_ARG, "d2d_rollout: num_steps must be >= 1");
    D2D_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t E = h->cfg.num_envs;
    const bool agent_pass = h->cfg.reward_fn != D2D_REWARD_SYSTEM_CAPACITY || io->agent_reward;
    d2d_step_io_t cur = *io;
    cur.actions = nullptr;
    // (with an fp64 position shadow bound the steps must run the shadow-aware instantiation: composed path)
    const bool fused = h->use_warp && !h->pos64 && (int64_t)num_steps * E <= d2d_max_launch_envs(h);
    if (!cur.actions_out && (agent_pass || !fused)) {
        rc = reserve_act_scratch(h, fused ? num_steps : 1, st);
        if (rc) return rc;
    }
    if (fused) {
        if (!cur.actions_out && agent_pass) cur.actions_out = h->act_scratch;
        EpisodeArgs ea;
        ea.act_seed = action_seed; ea.act_t0 = first_step_index; ea.draw_actions = true; ea.no_reset = true;
        rc = step_launch(h, &cur, num_steps, MODE_EPISODE, stream, ea);
        if (rc || !agent_pass) return rc;
        cur.actions = cur.actions_out;
        return agent_reward_launch(h, &cur, (int64_t)num_steps * E, true, st);
    }
    for (int t = 0; t < num_steps; ++t) {
        d2d_step_io_t one = cur;
        one.actions_out = nullptr;
        int32_t *dst = cur.actions_out ? cur.actions_out : h->act_scratch;
        rc = sample_launch(h, dst, action_seed, first_step_index + (uint32_t)t, st);
        if (rc) return rc;
        one.actions = dst;
        h->last_kind = D2D_LAST_OTHER;
        rc = step_launch(h, &one, 1, MODE_STEP, stream);
        if (rc) return rc;
        advance_io(cur, 1, E, h->N);
    }
    return D2D_OK;
}

// ---- host-buffer steps: a two-slot pipeline (copy-in stream -> caller's stream for the kernel -> copy-out stream) ----
namespace {

int host_pipeline_init(d2d_handle *h) {
    if (h->pipe_ready) return D2D_OK;
    D2D_CUDA(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
    D2D_CUDA(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
    for (auto &s : h->slot) {
        D2D_CUDA(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
        D2D_CUDA(cudaEventCreateWithFlags(&s.ev_kernel, cudaEventDisableTiming));
        D2D_CUDA(cudaEventCreateWithFlags(&s.ev_out, cudaEventDisableTiming));
    }
    h->pipe_ready = true;
    return D2D_OK;
}

// the buffers of a d2d_step_io_t in a fixed order: actions, then the outputs
void io_pointers(const d2d_step_io_t *io, void *out[D2D_NUM_IO_BUFFERS]) {
    out[0] = (void *)io->actions; out[1] = io->obs; out[2] = io->obs_dyn; out[3] = io->capacity_mbps; out[4] = io->reward;
    out[5] = io->done; out[6] = io->rate_bps; out[7] = io->rb; out[8] = io->tx_pwr_dBm; out[9] = io->agent_reward;
}
void io_from_pointers(void *const p[D2D_NUM_IO_BUFFERS], d2d_step_io_t *io) {
    io->actions = (const int32_t *)p[0]; io->obs = (float *)p[1]; io->obs_dyn = (float *)p[2]; io->capacity_mbps = (float *)p[3];
    io->reward = (float *)p[4]; io->done = (uint8_t *)p[5]; io->rate_bps = (float *)p[6]; io->rb = (int16_t *)p[7];
    io->tx_pwr_dBm = (int16_t *)p[8]; io->agent_reward = (float *)p[9];
}
void io_sizes(const d2d_handle *h, size_t bytes[D2D_NUM_IO_BUFFERS]) {
    const size_t E = (size_t)h->cfg.num_envs, EN = E * h->N;
    const size_t b[D2D_NUM_IO_BUFFERS] = {EN * 4, EN * 24, EN * 8, EN * 4, E * 4, E, EN * 4, EN * 2, EN * 2, EN * 4};
    std::memcpy(bytes, b, sizeof(b));
}
const uint32_t kIoMask[D2D_NUM_IO_BUFFERS] = {0u, D2D_OUT_OBS, D2D_OUT_OBS_DYN, D2D_OUT_CAPACITY, D2D_OUT_REWARD, D2D_OUT_DONE,
                                              D2D_OUT_RATE, D2D_OUT_RB, D2D_OUT_TX_PWR, D2D_OUT_AGENT_REWARD};

}  // namespace

D2D_API int d2d_host_slot_buffers(d2d_handle_t *h, int slot, uint32_t outputs, d2d_step_io_t *host_io) {
    if (!h || !host_io || slot < 0 || slot >= D2D_HOST_SLOTS) return fail(D2D_ERR_INVALID_ARG, "d2d_host_slot_buffers: bad handle, slot or io");
    if (!(outputs & (D2D_OUT_OBS | D2D_OUT_OBS_DYN | D2D_OUT_CAPACITY | D2D_OUT_REWARD | D2D_OUT_DONE | D2D_OUT_RATE | D2D_OUT_RB |
                     D2D_OUT_TX_PWR | D2D_OUT_AGENT_REWARD)))
        return fail(D2D_ERR_INVALID_ARG, "d2d_host_slot_buffers: empty output mask");
    D2D_GUARD(h);
    int rc = host_pipeline_init(h);
    if (rc) return rc;
    d2d_host_slot &s = h->slot[slot];
    if (s.host && s.mask == outputs) { *host_io = s.host_io; return D2D_OK; }
    if (s.used) D2D_CUDA(cudaEventSynchronize(s.ev_out));
    free_slot(s);
    size_t bytes[D2D_NUM_IO_BUFFERS], off[D2D_NUM_IO_BUFFERS] = {}, total = 0;
    io_sizes(h, bytes);
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    total = align(bytes[0]);
    s.out_offset = total;
    for (int i = 1; i < D2D_NUM_IO_BUFFERS; ++i)
        if (outputs & kIoMask[i]) { off[i] = total; total = align(total + bytes[i]); }
    s.out_bytes = total - s.out_offset;
    D2D_CUDA(cudaMalloc(&s.dev, total));
    D2D_CUDA(cudaHostAlloc(&s.host, total, cudaHostAllocDefault));
    std::memset(s.host, 0, total);
    s.bytes = total; s.mask = outputs;
    void *hp[D2D_NUM_IO_BUFFERS] = {}, *dp[D2D_NUM_IO_BUFFERS] = {};
    hp[0] = s.host; dp[0] = s.dev;
    for (int i = 1; i < D2D_NUM_IO_BUFFERS; ++i)
        if (outputs & kIoMask[i]) { hp[i] = (char *)s.host + off[i]; dp[i] = (char *)s.dev + off[i]; }
    s.host_io = d2d_step_io_t{}; s.dev_io = d2d_step_io_t{};
    io_from_pointers(hp, &s.host_io);
    io_from_pointers(dp, &s.dev_io);
    *host_io = s.host_io;
    return D2D_OK;
}

D2D_API int d2d_step_host_async(d2d_handle_t *h, const d2d_step_io_t *hio, int slot, void *stream) {
    if (!h || !hio || !hio->actions) return fail(D2D_ERR_INVALID_ARG, "d2d_step_host_async: handle, io and io->actions are required");
    if (slot < 0 || slot >= D2D_HOST_SLOTS) return fail(D2D_ERR_INVALID_ARG, "d2d_step_host_async: slot must be in [0, D2D_HOST_SLOTS)");
    if (hio->flags & D2D_STEP_AUTORESET) return fail(D2D_ERR_UNSUPPORTED, "d2d_step_host_async: D2D_STEP_AUTORESET applies to d2d_step only");
    if (!h->pos) return fail(D2D_ERR_STATE, "d2d_step_host_async: call d2d_bind_state first");
    D2D_GUARD(h);
    int rc = host_pipeline_init(h);
    if (rc) return rc;
    d2d_host_slot &s = h->slot[slot];
    cudaStream_t st = (cudaStream_t)stream;
    size_t bytes[D2D_NUM_IO_BUFFERS];
    io_sizes(h, bytes);
    void *host[D2D_NUM_IO_BUFFERS], *mine[D2D_NUM_IO_BUFFERS];
    io_pointers(hio, host);
    io_pointers(&s.host_io, mine);
    // the slot's own pinned output buffers (d2d_host_slot_buffers): ONE copy back for all of them; the actions may come from
    // the slot's pinned action buffer or from any other host buffer of the caller's (a ring of pre-filled ones, say)
    const bool packed = s.host && std::memcmp(host + 1, mine + 1, sizeof(host) - sizeof(host[0])) == 0;
    d2d_step_io_t dio{};
    if (packed) dio = s.dev_io;
    else {
        void *dp[D2D_NUM_IO_BUFFERS] = {};
        for (int i = 0; i < D2D_NUM_IO_BUFFERS; ++i) {
            if (host[i] && !s.stage[i]) D2D_CUDA(cudaMalloc(&s.stage[i], bytes[i]));
            dp[i] = host[i] ? s.stage[i] : nullptr;
        }
        io_from_pointers(dp, &dio);
    }
    // the actions arrive by a copy on another stream: never D2D_STEP_INPUTS_STABLE
    dio.flags = 0;
    // copy-in: this slot's action staging is free once the kernel that last read it has run
    if (s.used) D2D_CUDA(cudaStreamWaitEvent(h->s_in, s.ev_kernel, 0));
    if (hio->flags & D2D_STEP_ACTIONS_I16) {
        // half the upload: int16 actions, widened on the copy-in stream (so ev_in covers the widening too)
        if (!s.stage16) D2D_CUDA(cudaMalloc(&s.stage16, bytes[0] / 2));
        D2D_CUDA(cudaMemcpyAsync(s.stage16, host[0], bytes[0] / 2, cudaMemcpyHostToDevice, h->s_in));
        const int64_t count = (int64_t)(bytes[0] / 4);
        d2d_widen_actions_kernel<<<(unsigned)std::min<int64_t>(4 * h->num_sms, (count / 2 + 255) / 256 + 1), 256, 0, h->s_in>>>(
            (const int16_t *)s.stage16, (int32_t *)dio.actions, count);
        D2D_CUDA(cudaGetLastError());
    } else {
        D2D_CUDA(cudaMemcpyAsync((void *)dio.actions, host[0], bytes[0], cudaMemcpyHostToDevice, h->s_in));
    }
    D2D_CUDA(cudaEventRecord(s.ev_in, h->s_in));
    // kernel on the caller's stream (steps stay ordered there): needs the actions in, and this slot's previous
    // outputs copied out
    D2D_CUDA(cudaStreamWaitEvent(st, s.ev_in, 0));
    if (s.used) D2D_CUDA(cudaStreamWaitEvent(st, s.ev_out, 0));
    rc = check_step_args(h, &dio, "d2d_step_host_async");
    if (!rc) rc = step_launch(h, &dio, 1, MODE_STEP, stream);
    if (rc) return rc;
    D2D_CUDA(cudaEventRecord(s.ev_kernel, st));
    // copy-out
    D2D_CUDA(cudaStreamWaitEvent(h->s_out, s.ev_kernel, 0));
    if (packed) {
        D2D_CUDA(cudaMemcpyAsync((char *)s.host + s.out_offset, (char *)s.dev + s.out_offset, s.out_bytes, cudaMemcpyDeviceToHost, h->s_out));
    } else {
        void *dp[D2D_NUM_IO_BUFFERS];
        io_pointers(&dio, dp);
        for (int i = 1; i < D2D_NUM_IO_BUFFERS; ++i)
            if (host[i]) D2D_CUDA(cudaMemcpyAsync(host[i], dp[i], bytes[i], cudaMemcpyDeviceToHost, h->s_out));
    }
    D2D_CUDA(cudaEventRecord(s.ev_out, h->s_out));
    s.used = true;
    return D2D_OK;
}

D2D_API int d2d_step_host_wait(d2d_handle_t *h, int slot) {
    if (!h || slot < 0 || slot >= D2D_HOST_SLOTS) return fail(D2D_ERR_INVALID_ARG, "d2d_step_host_wait: bad handle or slot");
    if (!h->slot[slot].used) return D2D_OK;
    D2D_GUARD(h);
    D2D_CUDA(cudaEventSynchronize(h->slot[slot].ev_out));
    return D2D_OK;
}

D2D_API int d2d_step_host(d2d_handle_t *h, const d2d_step_io_t *hio, void *stream) {
    int rc = d2d_step_host_async(h, hio, 0, stream);
    if (rc) return rc;
    return d2d_step_host_wait(h, 0);
}

D2D_API int d2d_per_agent_obs(d2d_handle_t *h, const float *table, float *out, int64_t num_envs, void *stream) {
    if (!h || !table || !out) return fail(D2D_ERR_INVALID_ARG, "d2d_per_agent_obs: null argument");
    if (num_envs < 0 || num_envs > h->cfg.num_envs) return fail(D2D_ERR_INVALID_ARG, "d2d_per_agent_obs: bad num_envs");
    if (num_envs == 0) return D2D_OK;
    if (num_envs * h->N > 0x7fffffffLL) return fail(D2D_ERR_UNSUPPORTED, "d2d_per_agent_obs: num_envs * N exceeds the grid limit");
    D2D_GUARD(h);
    d2d_per_agent_obs_kernel<<<(unsigned)(num_envs * h->N), 128, 0, (cudaStream_t)stream>>>(table, out, h->N);
    D2D_CUDA(cudaGetLastError());
    ++h->launches;
    return D2D_OK;
}

D2D_API int d2d_stats_reset(d2d_handle_t *h, void *stream) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_stats_reset: null handle");
    if (!h->stats) return fail(D2D_ERR_STATE, "d2d_stats_reset: no stats buffer bound");
    D2D_GUARD(h);
    D2D_CUDA(cudaMemsetAsync(h->stats, 0, (size_t)D2D_STATS_REPLICAS * 8 * sizeof(double), (cudaStream_t)stream));
    return D2D_OK;
}

#ifdef D2D_TIMELINE
// instrumented build only (profiles/timeline.py): copies the stamp table to the host
D2D_API int d2d_debug_timeline(void *host_out, size_t bytes, int wpb) {
    D2D_CUDA(cudaDeviceSynchronize());
    D2D_CUDA(d2d_warp_shape(wpb)->timeline(host_out, bytes));
    return D2D_OK;
}
#endif
D2D_API int64_t d2d_launch_count(const d2d_handle_t *h) { return h ? h->launches : -1; }

D2D_API int d2d_step_geometry(const d2d_handle_t *h, int32_t *grid, int32_t *block, int32_t *smem_bytes, int32_t *envs_per_block) {
    if (!h) return fail(D2D_ERR_INVALID_ARG, "d2d_step_geometry: null handle");
    if (grid) *grid = h->grid;
    if (block) *block = h->block;
    if (smem_bytes) *smem_bytes = h->smem;
    if (envs_per_block) *envs_per_block = h->envs_per_block;
    return D2D_OK;
}
