// d2d_common.cuh - shared device types and math for the sm_100a step kernels.
//
// The arithmetic contract is SURVEY.md Appendix A (reference simulator.py:89-154).  The kernels work in
// the LINEAR power domain in fp32 and only go to dB for the two quantities the reference reports in dB:
//
//   w_k     = 10^(p_k/10) * 10^((eo_k - K)/10)          interferer EIRP minus the path-loss constant [mW]
//   g(d)    = d^-ple                                    (= 1/d^2 for ple = 2: no transcendental)
//   I_j     = sum_{k != j, rb_k = rb_j} w_k * g(|tx_k - rx_j|)            simulator.py:95-101
//   snr_lin = 10^(p_j/10) * a_j * g(d_j),  a_j = 10^((eo + ro - K - noise)/10)   simulator.py:93,115
//   r       = snr_lin / (1 + I_j / noise_lin)           = 10^(SINR_dB/10)        simulator.py:106-107
//   SINR_dB = 10 log10(r);  SNR_dB = p + snr0_dB - 5 ple log10(d^2)
//   rate    = log2(1 + r);  cap = bw_MHz * rate  (both gated by SINR_dB > sensitivity) simulator.py:118-154
//
// fp32 keeps ~1e-6 dB absolute error; links whose SINR falls within `rescue_band_dB` of 0 dB (where a
// pure relative tolerance on a dB value is ill-conditioned) are recomputed in fp64 from the same inputs
// (d2d_rescue_fp64 below).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define D2D_MAX_PWR_LEVELS 128     // entries of the integer-dBm -> mW table
#define D2D_WARP_MAX_LINKS 64      // warp-per-env kernel: 2 link slots per lane
#define D2D_INACTIVE_KEY 0x80000000u
#ifndef D2D_RESCUE_ENABLED
#define D2D_RESCUE_ENABLED 1
#endif

// fp32 per-link constants (SoA of two float4 so a lane fetches each with one conflict-free LDS.128)
struct __align__(16) D2DLinkA {
    float tx_lin0;    // 10^((eo_t - K)/10)
    float a_lin;      // 10^((eo_t + ro_v - K - noise_v)/10)
    float inv_noise;  // 10^(-noise_v/10)
    float snr0_dB;    // eo_t + ro_v - K - noise_v
};
struct __align__(16) D2DLinkB {
    float sens_dBm;   // receiver sensitivity (compared with SINR_dB as the reference does)
    float bw_MHz;     // 1e-6 * rb_bandwidth_kHz * 1000
    int32_t tx_dev;   // device index of the transmitter
    int32_t rx_dev;   // device index of the receiver
};
// fp64 per-link constants for the rescue path (same folding as D2DLinkA, kept in double)
struct D2DLinkD {
    double a_lin;     // 10^((eo_t + ro_v - K - noise_v)/10)
    double t_lin;     // 10^((eo_t - K)/10)
    double inv_noise; // 10^(-noise_v/10)
    double bw_MHz;
};

struct D2DParams {
    int64_t num_envs;
    int32_t N, V, C, R;
    int32_t n_pwr_cue, n_pwr_due;
    int32_t episode_length;
    int32_t nbins;               // block kernel: number of RB bins
    int32_t bin_cap;             // dense kernel: record slots per RB bin
    int32_t align4;              // warp kernel: every env's DUE (tx, rx) pair is a 16-byte aligned float4
    int32_t reward_fn;           // d2d_reward_fn: per-agent reward functions take their reward statistics from the post-pass kernel
    int32_t uniform;             // every CUE link shares one set of constants, and every DUE link (u_cue / u_due below)
    void *dense_ovf;             // dense kernel: [grid][N] float4 overflow records, then [grid][N] u16 RBs (handle-owned scratch)
    int32_t T;                   // d2d_step_many: steps per env in this launch (1 for d2d_step)
    uint32_t envs_per_warp;      // warp kernel: floor(num_envs / (grid * warps per block)), divided on the host (a 20-instruction
                                 // sequence ahead of every warp's first load otherwise) ...
    uint32_t envs_extra;         // ... and the remainder: warps [0, envs_extra) step one env more (contiguous ranges, balanced to +-1)
    int64_t t_stride;            // d2d_step_many: envs between consecutive step slices of the io buffers
    uint32_t magic_cue, magic_due;  // d2d_div_magic(n_pwr_cue / n_pwr_due): rb = umulhi(a, magic) + (a & npw1)
    uint32_t npw1_cue, npw1_due;    // 0xffffffff when n_pwr == 1 (then magic = 0 and rb = a), else 0
    float ple;                   // path-loss exponent
    float neg_half_ple;          // -ple/2           : g = exp2(neg_half_ple * log2(d^2))
    float snr_slope;             // 5*ple*log10(2)   : SNR_dB = p + snr0 - snr_slope*log2(d^2)
    float min_cap;               // SystemCapacityRewardFunction.min_capacity_mbps
    float rescue_band_dB;        // |SINR_dB| or |SNR_dB| below rescue_band_dB + rescue_c / d_min is recomputed in fp64
    float rescue_c;              // 0 unless an fp64 position shadow is bound (covers the fp32 rounding of positions)
    float rescue_dmin2;          // with a shadow: links with a distance^2 below this are always recomputed
    // per-agent reward functions (envs/reward_fn.py:47-78) compare a link's SINR_dB with a threshold: links within thr_band of it
    // take the fp64 pass, whose stored fp32 value falls on the float64 value's side of the threshold (d2d_sinr_store)
    float thr_dB, thr_band;      // thr_band = 0: no threshold (SystemCapacityRewardFunction)
    double thr_d;
    float4 u_cue, u_due;         // default-shape kernel: the one D2DLinkA of every CUE link / every DUE link (constant bank)
    float2 us_cue, us_due;       // ... and the (sens_dBm, bw_MHz) of D2DLinkB
    D2DLinkD ud_cue, ud_due;     // ... and their fp64 twins for the fp64 pass (valid when `uniform`)
    // ShadowingPathLoss (path_loss.py:69-81; general-topology kernel only): gauss(0, chi) added beyond d0 at EVERY path-loss
    // evaluation.  Counter-based draws: Philox4x32-10 keyed by rng_seed, counter (global env, victim | source << 16, kind, rng_step)
    float shadow_chi_dB;         // 0 = no shadowing
    float shadow_d0sq;           // d0^2
    uint64_t rng_seed, first_global_env, rng_step;
    const uint64_t *rng_step_dev; // ShadowingPathLoss: the step-call counter in device memory (added to rng_step), advanced on the stream
                                 // after every step so that a replayed CUDA graph draws fresh values each time
    uint32_t flags;              // D2D_PF_*
    // Per-warp tickets (warp kernel, single-launch d2d_step): see d2d_ticket_wait below
    uint64_t *tickets;           // [grid * warps per block] one word per warp slot of the launch geometry, or nullptr
    uint64_t tok_wait;           // != 0: wait for this token in the warp's ticket word instead of executing griddepcontrol.wait
    uint64_t tok_sign;           // != 0: the token this launch's warps publish when their stores are done
    // d2d_episode (warp kernel, EPISODE instantiation): Simulator.reset + the uncounted reset step + T counted steps in one launch
    uint64_t ep_seed;            // Philox key of this episode's position draws (d2d_reset's `seed`)
    uint64_t act_seed;           // Philox key of the on-device action draws
    uint32_t act_t0;             // step index of slice 0 in the action draws (d2d_rollout continues an episode's sequence)
    float cell_radius, d2d_radius;
    int32_t *actions_out;        // [T + 1][E][N] optional record of the drawn actions
    float *pos_out;              // = pos (the episode's positions become the bound state)
    double shadow_chi_d, shadow_d0sq_d;   // unrounded copies for the fp64 rescue path
    double ple_d;                // fp64 copy for the rescue path
    const D2DLinkA *linkA;       // [N]
    const D2DLinkB *linkB;       // [N]
    const D2DLinkD *linkD;       // [N]
    const int32_t *link_meta;    // [N] general-topology kernel: power levels of the link's action space | (1 << 16 if SIDELINK)
    const float *pwr_lin;        // [D2D_MAX_PWR_LEVELS] 10^(p/10), correctly rounded from fp64
    const double *pwr_lin_d;     // same table in fp64 (rescue path)
    // state
    const float *pos;            // [E][V][2]
    const double *pos64;         // [E][V][2] optional fp64 shadow of caller-supplied positions (rescue path only)
    uint8_t *step_count;         // [E]
    double *stats;               // [D2D_NUM_STATS] or nullptr
    // step io
    const int32_t *actions;      // [E][N]
    float *obs;                  // [E][N][6]
    float2 *obs_dyn;             // [E][N] (sinr_dB, snr_dB): the per-step part of the observation table alone
    float *cap;                  // [E][N]
    float *reward;               // [E]
    uint8_t *done;               // [E]
    float *rate;                 // [E][N]
    int16_t *rb_out;             // [E][N]
    int16_t *pwr_out;            // [E][N]
#ifdef D2D_TIMELINE
    int32_t tl_slot;             // instrumented build (profiles/timeline.py): which d2d_tl_buf slot this launch stamps
#endif
    // d2d_step with D2D_STEP_AUTORESET (warp kernel, MODE 5).  Last in the struct, so every other kernel's parameter offsets stay put.
    uint32_t *episode_index;     // [E] episodes each env has begun since the last full reset (caller-owned)
    uint64_t ar_base;            // base of the per-env reset keys: env e's n-th auto-reset draws under d2d_autoreset_key(ar_base, n)
};

#ifdef D2D_TIMELINE
// Instrumented build only: every warp of the warp kernel stamps (globaltimer at entry, clock64 at entry / before
// griddepcontrol.wait / after it / at its end, SM id) so that profiles/timeline.py can lay consecutive launches side by side,
// and counts what the warp did: envs stepped, flagged links recomputed in fp64 before / after its wait, envs that took the
// overflow pass (an RB above D2D_BIN_CAP links).
#define D2D_TL_SLOTS 64
#define D2D_TL_WARPS 4096
struct D2DTlRec { unsigned long long g0, c0, c1, c2, c3, smid, n_env, n_pre, n_post, n_ovf; };
__device__ D2DTlRec d2d_tl_buf[D2D_TL_SLOTS][D2D_TL_WARPS];
__device__ __forceinline__ unsigned long long d2d_tl_clock() { return (unsigned long long)clock64(); }
__device__ __forceinline__ unsigned long long d2d_tl_gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned d2d_tl_smid() { unsigned s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s; }
#endif

__device__ __forceinline__ float d2d_lg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float d2d_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float d2d_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Programmatic dependent launch (PDL; the ordering rule is spelled out in include/d2d_b200.h).  A step kernel is launched
// with programmatic stream serialisation, so it may start while the previous kernel in its stream is still running.
// What it may touch before griddepcontrol.wait depends on D2D_PF_INPUTS_FRESH:
//   set (the default):  something other than this handle's own step kernels may have written this step's actions or the
//       positions (a policy kernel, a copy, d2d_reset ...).  The kernel waits FIRST - every earlier kernel's memory is
//       then complete and visible - and only then releases its own dependents and loads anything.  PDL still hides the
//       launch latency and the block scheduling, nothing else.
//   clear (the caller's D2D_STEP_INPUTS_STABLE promise, honoured only when the previous kernel this handle enqueued on
//       the stream was one of its own step kernels):  a step kernel never writes actions or positions, so the inputs are
//       loaded and the whole env-step computed right away; the wait comes only before the first access to memory a
//       previous STEP wrote - the step counters and the output buffers.  By induction every such kernel starts after
//       the last "fresh" kernel passed its wait (that one releases its dependents only afterwards), so whatever wrote
//       the inputs before that point is complete and visible.
#define D2D_PF_INPUTS_FRESH 1u
#define D2D_PF_DRAW_ACTIONS 2u     // d2d_episode / d2d_rollout: actions drawn on the device instead of read from P.actions
#define D2D_PF_LATE_WAIT 8u        // d2d_step after a d2d_step whose output buffers this one does not touch: the per-link outputs are stored
                                   // AHEAD of griddepcontrol.wait; only the step counters and the per-env scalars come after it (d2d_abi.cu)
#define D2D_PF_NO_RESET 4u         // d2d_rollout: the EPISODE instantiation continues from the bound state (no position draw, every slice counted)
__device__ __forceinline__ void d2d_pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void d2d_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// kernel entry: see above
__device__ __forceinline__ void d2d_pdl_entry(uint32_t flags) {
    if (flags & D2D_PF_INPUTS_FRESH) d2d_pdl_wait();
    d2d_pdl_launch_dependents();
}
// Per-warp tickets.  griddepcontrol.wait orders a launch after ALL of its predecessor, although env e of step k + 1 depends only on
// env e of step k (its step counter, its output rows), which the SAME warp slot of the same launch geometry stepped.  When the
// host knows that the previous kernel in the stream was this handle's single-launch d2d_step with the same geometry (and the
// caller made the D2D_STEP_INPUTS_STABLE promise), launch k + 1 carries tok_wait = the token launch k's warps publish with a
// gpu-scope RELEASE store after their last store; warp w of launch k + 1 ACQUIRE-spins on its own ticket word in place of the
// grid-wide wait.  A token is (chain id, position in the chain) - unique per launch of a chain, baked into the launch parameters,
// so it survives CUDA-graph replays (the word holds the chain's LAST token between replays, never a waited-for one: a chain
// with a waiter has at least two launches).  Every warp of launch k is resident or finished before a block of launch k + 1 can
// start (a dependent launches only after every block of its predecessor has executed launch_dependents), so the spin cannot
// deadlock; and launch k + 1 cannot complete before every warp of launch k has published, so a later consumer ordered after
// launch k + 1 - by stream order or by its own griddepcontrol.wait - sees launch k's stores as well.
// The spin is bounded (~10 ms): should a token ever fail to arrive - a host-side bookkeeping bug, not a legal state - the warp falls
// back to griddepcontrol.wait, which is always sufficient, and counts the event in statistic D2D_STAT_TICKET_TIMEOUTS (tests assert 0).
__device__ __forceinline__ bool d2d_ticket_wait(const uint64_t *word, uint64_t token) {
    uint64_t v;
    for (uint32_t spin = 0; spin < 200000u; ++spin) {
        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(word) : "memory");
        if (v == token) return true;
        __nanosleep(40);
    }
    d2d_pdl_wait();
    return false;
}
__device__ __forceinline__ void d2d_ticket_sign(uint64_t *word, uint64_t token) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(word), "l"(token) : "memory");
}

// envs/d2d_env.py:95: rb = a // n_pwr for a >= 0.  n_pwr is a runtime value, so divide by multiplying
// with magic = ceil(2^32 / n) (exact for a < 2^32 / n; n = 1 has no 32-bit magic and is passed through).
__host__ __device__ __forceinline__ uint32_t d2d_div_magic(int n) {
    return n <= 1 ? 0u : (uint32_t)((0x100000000ull + (uint32_t)n - 1) / (uint32_t)n);
}
__device__ __forceinline__ int d2d_div(int a, uint32_t magic) {
    return magic ? (int)__umulhi((uint32_t)a, magic) : a;
}

// Philox4x32-R (Salmon et al. 2011); same constants as the oracle's restatement.  R = 10 is the standard strength (positions,
// shadowing); R = 7 is the smallest round count the paper reports as passing BigCrush and is used for the per-step action draws,
// which are made inside the step kernel's hot loop.
template <int ROUNDS>
__device__ __forceinline__ uint4 d2d_philox4x32(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
__device__ __forceinline__ uint4 d2d_philox4x32_10(uint4 c, uint2 k) { return d2d_philox4x32<10>(c, k); }

// ---- counter-based draws of the device-side reset and of the on-device action sampling -------------------------------------
// (restated value for value by oracle/d2d_oracle.c: d2d_oracle_reset_positions / d2d_oracle_sample_actions; the reference
// draws from Python's global Mersenne Twister - position.py:18-45, envs/d2d_env.py:54-60 - so only distributions can match.)
//
// Reset.  An env's devices are drawn in UNITS of one Philox block (four 32-bit words = two uniform-in-disc draws):
//   unit u < CU = ceil(C / 2):  CUE 2u from words (x, y), CUE 2u + 1 from words (z, w)
//   unit CU + d:                DUE pair d - attempt 0: transmitter from (x, y), first receiver offset from (z, w);
//                               attempt a >= 1: receiver offsets 2a - 1 from (x, y) and 2a from (z, w)
//   block(u, a) = Philox4x32-10(counter = (global env lo, hi, u, a), key = seed)
// position.py:24-28: theta = 2 pi u1, r = radius sqrt(u2); 24-bit uniforms centred in their cell, so u is never 0 (r = 0 would
// put a receiver on its transmitter).  The products are rounded separately (no FMA contraction) so that every kernel that
// inlines these helpers draws bit-identical positions.
#define D2D_RESET_MAX_OFFSETS 64u
__device__ __forceinline__ uint4 d2d_reset_block(uint64_t seed, uint64_t genv, uint32_t unit, uint32_t attempt) {
    return d2d_philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), unit, attempt),
                             make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
__device__ __forceinline__ float2 d2d_disc_from_words(uint32_t w0, uint32_t w1, float radius) {
    const float u1 = __fmul_rn((float)(w0 >> 8) + 0.5f, 1.0f / 16777216.0f), u2 = __fmul_rn((float)(w1 >> 8) + 0.5f, 1.0f / 16777216.0f);
    float s, c;
    __sincosf(__fmul_rn(6.283185307179586f, u1), &s, &c);
    const float r = __fmul_rn(radius, __fsqrt_rn(u2));
    return make_float2(__fmul_rn(r, c), __fmul_rn(r, s));
}
// CUE j of global env genv
__device__ __forceinline__ float2 d2d_draw_cue(uint64_t seed, uint64_t genv, uint32_t j, float cell_radius) {
    const uint4 b = d2d_reset_block(seed, genv, j >> 1, 0u);
    return (j & 1u) ? d2d_disc_from_words(b.z, b.w, cell_radius) : d2d_disc_from_words(b.x, b.y, cell_radius);
}
// DUE pair d: (tx_x, tx_y, rx_x, rx_y); the receiver is re-drawn around the transmitter until it falls inside the cell
// (position.py:38-44; bounded to D2D_RESET_MAX_OFFSETS candidates)
__device__ __forceinline__ float4 d2d_draw_due(uint64_t seed, uint64_t genv, uint32_t cu, uint32_t d, float cell_radius, float d2d_radius) {
    uint4 b = d2d_reset_block(seed, genv, cu + d, 0u);
    const float2 tx = d2d_disc_from_words(b.x, b.y, cell_radius);
    const float r2max = __fmul_rn(cell_radius, cell_radius);
    float2 rx = tx;
    for (uint32_t k = 0; k < D2D_RESET_MAX_OFFSETS; ++k) {
        if (k && (k & 1u)) b = d2d_reset_block(seed, genv, cu + d, (k + 1u) >> 1);
        const float2 o = (k & 1u) ? d2d_disc_from_words(b.x, b.y, d2d_radius) : d2d_disc_from_words(b.z, b.w, d2d_radius);
        rx = make_float2(__fadd_rn(tx.x, o.x), __fadd_rn(tx.y, o.y));
        if (__fadd_rn(__fmul_rn(rx.x, rx.x), __fmul_rn(rx.y, rx.y)) <= r2max) break;
    }
    return make_float4(tx.x, tx.y, rx.x, rx.y);
}
// Actions (envs/d2d_env.py:54-60: Discrete(n).sample(), uniform over 0 .. n - 1).  One Philox block serves the CUE and the DUE
// link of pair index l (CUE l / DUE pair l) for two consecutive steps:
//   block(l, t) = Philox4x32-7(counter = (global env lo, hi, l, t >> 1), key = action seed ^ D2D_ACTION_KEY)
//   word        = 2 (t & 1) + (1 if the link is a DUE pair);   a = floor(word * n / 2^32)
#define D2D_ACTION_KEY 0xA511E9B3u
__device__ __forceinline__ uint4 d2d_action_block(uint64_t act_seed, uint64_t genv, uint32_t l, uint32_t t) {
    return d2d_philox4x32<7>(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32), l, t >> 1),
                             make_uint2((uint32_t)act_seed ^ D2D_ACTION_KEY, (uint32_t)(act_seed >> 32)));
}
__device__ __forceinline__ uint32_t d2d_action_word(const uint4 &b, uint32_t t, bool due) {
    return (t & 1u) ? (due ? b.w : b.z) : (due ? b.y : b.x);
}

// Auto-reset (D2D_STEP_AUTORESET): the Philox key of an env's n-th episode since the last full reset, key(base, n) =
// splitmix64(base + n * 0x9E3779B97F4A7C15) with splitmix64 the output function of Steele et al.'s SplitMix64.  Philox's counter
// carries the global env, so the draws depend on (base, global env, n) only.  Mirrored by VecD2DEnv.autoreset_key.
__host__ __device__ __forceinline__ uint64_t d2d_autoreset_key(uint64_t base, uint64_t n) {
    uint64_t z = base + n * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// The N(0,1) draw of one ShadowingPathLoss evaluation (kind 0: the terms of the SINR, 1: the SNR's own-link evaluation): Box-Muller
// on two 24-bit uniforms of one Philox block.  Restated value for value by the oracle (d2d_oracle_shadow_normal).
__device__ __forceinline__ uint2 d2d_shadow_bits(const D2DParams &P, uint64_t genv, uint32_t victim, uint32_t source, uint32_t kind) {
    const uint64_t step = P.rng_step + (P.rng_step_dev ? *P.rng_step_dev : 0ull);
    const uint4 o = d2d_philox4x32_10(make_uint4((uint32_t)genv, (uint32_t)(genv >> 32) ^ (kind << 31) ^ ((uint32_t)(step >> 32) << 8),
                                                 victim | (source << 16), (uint32_t)step),
                                      make_uint2((uint32_t)P.rng_seed ^ 0x5bd1e995u, (uint32_t)(P.rng_seed >> 32)));
    return make_uint2(o.x >> 8, o.y >> 8);
}
__device__ __forceinline__ float d2d_shadow_normal(const D2DParams &P, uint64_t genv, uint32_t victim, uint32_t source, uint32_t kind) {
    const uint2 b = d2d_shadow_bits(P, genv, victim, source, kind);
    const float u1 = ((float)b.x + 0.5f) * (1.0f / 16777216.0f), u2 = ((float)b.y + 0.5f) * (1.0f / 16777216.0f);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}
__device__ __forceinline__ double d2d_shadow_normal_f64(const D2DParams &P, uint64_t genv, uint32_t victim, uint32_t source, uint32_t kind) {
    const uint2 b = d2d_shadow_bits(P, genv, victim, source, kind);
    const double u1 = ((double)b.x + 0.5) * (1.0 / 16777216.0), u2 = ((double)b.y + 0.5) * (1.0 / 16777216.0);
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}
// linear gain factor 10^(-chi z / 10) of one evaluation at squared distance d2 (1 within d0, path_loss.py:75-81)
__device__ __forceinline__ float d2d_shadow_factor(const D2DParams &P, float d2, uint64_t genv, uint32_t victim, uint32_t source, uint32_t kind) {
    if (!(P.shadow_chi_dB > 0.f) || !(d2 > P.shadow_d0sq)) return 1.0f;
    return exp2f(-0.33219280948873623f * P.shadow_chi_dB * d2d_shadow_normal(P, genv, victim, source, kind));
}
__device__ __forceinline__ double d2d_shadow_factor_f64(const D2DParams &P, double d2, uint64_t genv, uint32_t victim, uint32_t source, uint32_t kind) {
    if (!(P.shadow_chi_dB > 0.f) || !(d2 > P.shadow_d0sq_d)) return 1.0;
    return exp2(-0.33219280948873623 * P.shadow_chi_d * d2d_shadow_normal_f64(P, genv, victim, source, kind));
}

// Path gain g(d^2) = d^-ple.  PLE2: one MUFU.RCP; otherwise MUFU.LG2 + MUFU.EX2.
template <bool PLE2>
__device__ __forceinline__ float d2d_gain(float d2, float neg_half_ple) {
    if (PLE2) return d2d_rcp(d2);
    return d2d_ex2(neg_half_ple * d2d_lg2(d2));
}

// log2(1 + r) with full relative accuracy for small r (the reference's log2(1 + 10^(sinr/10)),
// simulator.py:124,151).  For r < 0.25 the MUFU path would lose the low bits of r in 1 + r, so use
// log1p(r) = 2 atanh(r / (2 + r)) with a 4-term odd series (|s| <= 1/9: truncation < 3e-9 relative).
__device__ __forceinline__ float d2d_log2_1p(float r) {
    if (r < 0.25f) {
        float s = r * d2d_rcp(2.0f + r);
        // one Newton step on the quotient keeps s at ~1 ulp (rcp.approx alone is 1-2 ulp: fine, but cheap)
        float s2 = s * s;
        float poly = fmaf(s2, fmaf(s2, fmaf(s2, (1.0f / 7.0f), 0.2f), (1.0f / 3.0f)), 1.0f);
        return 2.8853900817779268f * s * poly;   // 2 / ln 2
    }
    return d2d_lg2(1.0f + r);
}

struct D2DLinkOut {
    float sinr_dB, snr_dB, rate, cap;
};

// The fp32 image of a float64 SINR_dB.  ShannonRewardFunction / CueSinrShannonRewardFunction (envs/reward_fn.py:55,72) compare
// the float64 value with a threshold; the post-pass kernel compares the stored fp32 value with the fp32 threshold, so the
// stored value is moved by at most one ulp onto the float64 value's side of it when plain rounding would cross.
__device__ __forceinline__ float d2d_sinr_store(double sinr, const D2DParams &P) {
    float v = (float)sinr;
    if (P.thr_band > 0.f) {
        const bool ge = sinr >= P.thr_d;
        if ((v >= P.thr_dB) != ge) v = ge ? P.thr_dB : nextafterf(P.thr_dB, -3.0e38f);
    }
    return v;
}

// Per-link epilogue in fp32 (Appendix A).  p_lin = 10^(p/10); g = d^-ple of the own link as the SINR sees it, g_snr as the SNR
// sees it (the same value unless ShadowingPathLoss draws the two evaluations separately);
// I = interference [mW]; cA = (tx_lin0, a_lin, inv_noise, snr0_dB); sb = (sens_dBm, bw_MHz).
// SNR_dB is taken from the LINEAR ratio like SINR_dB: its absolute error is then ~1e-6 dB near 0 dB, where the pure relative
// 1e-4 bound bites.  (The dB-domain form p + snr0 - 5 ple log10 d^2 subtracts two ~60 dB numbers: 1e-5 dB of rounding,
// 1.5e-4 relative at 0.064 dB - found by tests/test_gpu_round2.py::test_band_edge_sweep_of_sinr_and_snr.)
template <bool PLE2>
__device__ __forceinline__ D2DLinkOut d2d_link_epilogue(int p, float p_lin, float g_snr, float g, float I, const float4 &cA,
                                                        const float2 &sb, const D2DParams &P) {
    D2DLinkOut o;
    const float snr_lin = p_lin * cA.y * g;
    const float r = snr_lin * d2d_rcp(fmaf(I, cA.z, 1.0f));
    o.snr_dB = 3.0102999566398120f * d2d_lg2(p_lin * cA.y * g_snr);
    o.sinr_dB = 3.0102999566398120f * d2d_lg2(r);
    const bool ok = o.sinr_dB > sb.x;
    const float rate = d2d_log2_1p(r);
    o.rate = ok ? rate : 0.0f;
    o.cap = ok ? sb.y * rate : 0.0f;
    return o;
}

// ---- fp64 rescue ------------------------------------------------------------------------------------
// A pure relative tolerance on a dB value is ill-conditioned where the value crosses 0: fp32 leaves
// ~1e-6 dB of absolute error, and - when the caller supplied float64 positions that had to be rounded to
// the fp32 device state - up to ~8.7 * ulp / d dB more for a link or interferer d metres away.  A link is
// therefore recomputed in fp64 when   |SINR_dB| or |SNR_dB| < rescue_band_dB + rescue_c / d_min
// (d_min = the smallest distance that entered its sums), or d_min^2 < rescue_dmin2.  rescue_c and
// rescue_dmin2 are 0 unless an fp64 shadow of the positions is bound (d2d_bind_positions_f64), in which
// case the recomputation also reads the unrounded positions.  The kernels run it AFTER the env's outputs
// are stored, when nothing else is live, and overwrite that link's four values.  It is written without
// libm calls on purpose: log10/pow would raise the whole kernel's register allocation for a rare path.

// ln(r) for r in [0.7, 1.55]: 2 atanh((r-1)/(r+1)), odd series to s^19 (truncation < 1e-16 relative)
__device__ __forceinline__ double d2d_ln_near1(double r) {
    const double s = (r - 1.0) / (r + 1.0), s2 = s * s;
    double q = 1.0 / 19.0;
    q = fma(q, s2, 1.0 / 17.0); q = fma(q, s2, 1.0 / 15.0); q = fma(q, s2, 1.0 / 13.0);
    q = fma(q, s2, 1.0 / 11.0); q = fma(q, s2, 1.0 / 9.0);  q = fma(q, s2, 1.0 / 7.0);
    q = fma(q, s2, 1.0 / 5.0);  q = fma(q, s2, 1.0 / 3.0);  q = fma(q, s2, 1.0);
    return 2.0 * s * q;
}
// ln(x), x > 0 normal: exponent split so the mantissa lies in [0.75, 1.5)
__device__ __forceinline__ double d2d_ln_f64(double x) {
    int hi = __double2hiint(x), lo = __double2loint(x);
    int ex = ((hi >> 20) & 0x7ff) - 1023;
    hi = (hi & 0x000fffff) | 0x3ff00000;
    double m = __hiloint2double(hi, lo);
    if (m >= 1.5) { m *= 0.5; ++ex; }
    return fma((double)ex, 0.6931471805599453094, d2d_ln_near1(m));
}
// exp(y) for |y| < 700: Cody-Waite reduction + degree-13 Taylor on |f| <= ln2/2
__device__ __forceinline__ double d2d_exp_f64(double y) {
    const double n = rint(y * 1.4426950408889634074);
    const double f = fma(-n, 1.9082149292705877e-10, fma(-n, 0.693147180369123816490, y));
    double q = 1.0 / 6227020800.0;
    q = fma(q, f, 1.0 / 479001600.0); q = fma(q, f, 1.0 / 39916800.0); q = fma(q, f, 1.0 / 3628800.0);
    q = fma(q, f, 1.0 / 362880.0);    q = fma(q, f, 1.0 / 40320.0);    q = fma(q, f, 1.0 / 5040.0);
    q = fma(q, f, 1.0 / 720.0);       q = fma(q, f, 1.0 / 120.0);      q = fma(q, f, 1.0 / 24.0);
    q = fma(q, f, 1.0 / 6.0);         q = fma(q, f, 0.5);              q = fma(q, f, 1.0);
    q = fma(q, f, 1.0);
    return q * __hiloint2double(((int)n + 1023) << 20, 0);
}
template <bool PLE2>
__device__ __forceinline__ double d2d_gain_f64(double d2, double ple) {
    if (PLE2) return 1.0 / d2;
    return d2d_exp_f64(-0.5 * ple * d2d_ln_f64(d2));
}
// integer Tx power of link k re-derived from the env's raw action row (envs/d2d_env.py:96)
__device__ __forceinline__ int d2d_pwr_of(const int32_t *act_env, int k, const D2DParams &P) {
    const int a = act_env[k];
    const int npw = P.link_meta[k] & 0xffff;
    return (a - (a / npw) * npw) & (D2D_MAX_PWR_LEVELS - 1);
}
__device__ __forceinline__ int d2d_tx_dev(int k, int C) { return k < C ? 1 + k : 1 + C + 2 * (k - C); }
__device__ __forceinline__ int d2d_rx_dev(int k, int C) { return k < C ? 0 : 2 + C + 2 * (k - C); }
// position of device v of this env: the fp64 shadow when bound, else the fp32 state (exact in that case)
__device__ __forceinline__ double2 d2d_pos_f64(const float2 *pe32, const double2 *pe64, int v) {
    if (pe64) return pe64[v];
    const float2 p = pe32[v];
    return make_double2((double)p.x, (double)p.y);
}
// interferer k's fp64 contribution at receiver rx: w_k * g(d)
template <bool PLE2>
__device__ __forceinline__ double d2d_ix_term_f64(int k, double2 rx, const float2 *pe32, const double2 *pe64,
                                                  const int32_t *act_env, const D2DParams &P, uint64_t genv = 0, int victim = 0) {
    const double2 tk = d2d_pos_f64(pe32, pe64, P.linkB[k].tx_dev);
    const double ex = tk.x - rx.x, ey = tk.y - rx.y, d2 = ex * ex + ey * ey;
    return P.pwr_lin_d[d2d_pwr_of(act_env, k, P)] * P.linkD[k].t_lin * d2d_gain_f64<PLE2>(d2, P.ple_d) *
           d2d_shadow_factor_f64(P, d2, genv, (uint32_t)victim, (uint32_t)k, 0);
}
// all four outputs of link j from its fp64 interference sum (simulator.py:93,106-107,115,118-154)
template <bool PLE2>
__device__ __forceinline__ D2DLinkOut d2d_link_f64(int j, double2 tx, double2 rx, double I, float sens_dBm,
                                                   const int32_t *act_env, const D2DParams &P, uint64_t genv = 0) {
    const D2DLinkD Lj = P.linkD[j];
    const double dx = tx.x - rx.x, dy = tx.y - rx.y, d2 = dx * dx + dy * dy;
    const double S0 = P.pwr_lin_d[d2d_pwr_of(act_env, j, P)] * Lj.a_lin * d2d_gain_f64<PLE2>(d2, P.ple_d);
    // under ShadowingPathLoss the SINR's and the SNR's own-link evaluations draw separately (simulator.py:93 and :113)
    const double S = S0 * d2d_shadow_factor_f64(P, d2, genv, (uint32_t)j, (uint32_t)j, 1);
    const double r = S0 * d2d_shadow_factor_f64(P, d2, genv, (uint32_t)j, (uint32_t)j, 0) / fma(I, Lj.inv_noise, 1.0);   // a_lin already carries 1/noise
    const double sinr = 4.3429448190325182765 * d2d_ln_f64(r); // 10 log10
    const double rate = 1.4426950408889634074 * d2d_ln_f64(1.0 + r);
    const bool ok = sinr > (double)sens_dBm;
    D2DLinkOut o;
    o.sinr_dB = d2d_sinr_store(sinr, P);
    o.snr_dB = (float)(4.3429448190325182765 * d2d_ln_f64(S));
    o.rate = ok ? (float)rate : 0.0f;
    o.cap = ok ? (float)(Lj.bw_MHz * rate) : 0.0f;
    return o;
}
// does this link need the fp64 pass?  dmin2 = smallest squared distance that entered its sums (EXACT only).  THR: the
// instantiation also serves per-agent reward functions, whose hard SINR threshold is a second ill-conditioned point.
template <bool EXACT, bool THR = true>
__device__ __forceinline__ bool d2d_needs_rescue(const D2DLinkOut &o, float dmin2, const D2DParams &P) {
    const float lo = fminf(fabsf(o.sinr_dB), fabsf(o.snr_dB));
    const bool thr = THR && fabsf(o.sinr_dB - P.thr_dB) < P.thr_band;
    if (!EXACT) return lo < P.rescue_band_dB || thr;
    return lo < fmaf(P.rescue_c, rsqrtf(dmin2), P.rescue_band_dB) || dmin2 < P.rescue_dmin2 || thr;
}
// ---- cheap fp64 building blocks of the rescue passes (no division or libm subroutines) ------------------------------------
// 1 / x in fp64 from the fp32 reciprocal and three Newton steps (x normal, > 0): no division subroutine
__device__ __forceinline__ double d2d_rcp_f64(double x) {
    double y = (double)d2d_rcp((float)x);
    y = fma(y, fma(-x, y, 1.0), y);
    y = fma(y, fma(-x, y, 1.0), y);
    y = fma(y, fma(-x, y, 1.0), y);
    return y;
}
template <bool PLE2>
__device__ __forceinline__ double d2d_gain_f64_fast(double d2, double ple) {
    if (PLE2) return d2d_rcp_f64(d2);
    return d2d_exp_f64(-0.5 * ple * d2d_ln_f64(d2));
}
// ln(x) in fp64.  |x - 1| < 1/16 - every value the fp32 trigger sends here unless an fp64 position shadow is bound -
// needs no exponent split and five series terms; everything else takes the general d2d_ln_f64.
// 10 log10(x) in fp64 for |x - 1| < 1/16: no exponent split, five series terms
__device__ __forceinline__ double d2d_db_near1(double x) {
    const double s = (x - 1.0) * d2d_rcp_f64(x + 1.0), s2 = s * s;      // |s| < 1/31: s^11 / 11 < 1e-17
    double q = 1.0 / 9.0;
    q = fma(q, s2, 1.0 / 7.0); q = fma(q, s2, 1.0 / 5.0); q = fma(q, s2, 1.0 / 3.0); q = fma(q, s2, 1.0);
    return 8.6858896380650365530 * s * q;                               // 2 * 10 / ln 10
}
