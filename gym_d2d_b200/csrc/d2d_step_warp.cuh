// d2d_step_warp.cuh - fused env.step, one warp per environment, for C <= 32 CUEs, D <= 32 DUE pairs and
// R <= 64 RBs (the reference's default 25/25/25 configuration and everything around it).
//
// Replaces, for E environments at once, the reference call chain
//   D2DEnv.step (envs/d2d_env.py:62-71) -> _decode_action (:93-101) -> Simulator.step (simulator.py:77-154)
//   -> LinearObsFunction (envs/obs_fn.py:43-61) -> SystemCapacityRewardFunction (envs/reward_fn.py:27-44).
//
// Mapping: lane l owns CUE link l (slot A) and DUE pair l (slot B).
//
// The kernel is bound by the SM's load/store data pipe (shared-memory + global wavefronts, profiles/README.md), so
// the design minimises wavefronts per env, not instructions: inputs go straight to registers (LDG, software-pipelined
// one env ahead; staging them through shared memory with cp.async was measured and costs 60 more wavefronts per env),
// peer-record loads are predicated on the record being a real co-channel peer, dead lanes count into private dummy
// words, and the default EnvConfig reads its link constants from the constant bank.
//
// GROUPING.  The masked per-RB interference sum (Actions.get_actions_by_rb, actions.py:27-31 + simulator.py:95-101)
// is a segmented reduction over links grouped by RB.  The grouping is a per-warp BINNED table in shared memory:
//   rank = atomicAdd(count[rb], 1)                 one shared atomic per link
//   bin[rb][rank] = (tx_x, tx_y, w, u)             the link's peer record, D2D_BIN_CAP record slots per RB
// after which a victim's co-channel peers are the first count[rb] records of ITS bin: no prefix scan, no offsets, no
// scatter pass.  The first D2D_WALK_INLINE records are handled branch-free (immediate-offset LDS, predicated terms, so
// the loads and gains of a lane's two victims overlap); fuller bins take a short serial loop.  An RB that holds more
// than D2D_BIN_CAP links (~0.4 % of envs at the default load, but a policy may put every agent on one RB) keeps its
// first D2D_BIN_CAP links in the bin; the links ranked beyond it add their terms in a shuffle pass over just those links.
//
// All CUE links share one receiver (the MBS at the origin), so there an interferer contributes a per-link scalar
// u_k = w_k g(|tx_k|) computed once, and a CUE victim's walk is a sum of u_k; a DUE victim evaluates
// w_k g(|tx_k - rx|).  The victim is excluded from its own bin by index - never subtracted from a per-RB total,
// which would cancel a weak interferer against a 70 dB stronger self term.
//
// SHAPE.  D2DShape<true> instantiates the kernel for the reference's default EnvConfig (25 RBs, 25 CUEs, 25 DUE
// pairs, 24 / 21 power levels: envs/env_config.py:12-27, envs/d2d_env.py:31-35) with every count, stride and division
// magic an immediate; D2DShape<false> reads them from the launch parameters.  Same code, same results.
//
// HBM traffic per env-step is the compulsory 32N + 8V + 5 bytes (DESIGN.md): one coalesced pass over the env's
// actions and positions, one over its outputs; nothing is re-read.
#pragma once

#include "d2d_common.cuh"

// Launch shapes, picked by the host from the batch size (measured on B200, profiles/README.md):
//   WPB = 2: latency shape - a batch of well under one wave (E <= D2D_LATENCY_ENVS); the rare fp64 pass runs BEFORE
//            griddepcontrol.wait (see d2d_rescue_warp), so nothing but stores follows the wait
//   WPB = 4: finest block granularity at full occupancy - best when the batch is about one wave (E = 4096)
//   WPB = 8: best sustained throughput for batches of many waves
#ifndef D2D_MINB8
#define D2D_MINB8 3
#endif
#ifndef D2D_MINB4
#define D2D_MINB4 7
#endif
#ifndef D2D_MINB2
#define D2D_MINB2 14
#endif
#ifndef D2D_LATENCY_ENVS
#define D2D_LATENCY_ENVS 2048
#endif
#ifndef D2D_WPB_MID
#define D2D_WPB_MID 4          // warps per block of the one-wave shape (build knob of the A/B harness)
#endif
#define D2D_WARP_MIN_BLOCKS(WPB) ((WPB) == 2 ? D2D_MINB2 : (WPB) == D2D_WPB_MID ? D2D_MINB4 : D2D_MINB8)
#ifndef D2D_STATS_REPLICAS
#define D2D_STATS_REPLICAS 1024
#endif
#ifndef D2D_BIN_CAP
#define D2D_BIN_CAP 8          // peer records per RB bin on the fast path
#endif
#ifndef D2D_WALK_INLINE
#define D2D_WALK_INLINE 5      // records handled branch-free before the serial loop
#endif

// ---- shared memory layout ---------------------------------------------------------------------------------------------
// block:    pwr_lin[128] f32 | linkA[64] float4 (slot A: lane, slot B: 32 + lane) | linkS[64] float2 (sens, bw)
// per warp: R bins of D2D_BIN_STRIDE bytes | 64 dummy counter pairs (8 B each: slot A lanes, then slot B lanes) | a zero record
// A bin = D2D_BIN_CAP records of 16 B + a 16 B tail: {link count, 1 if a SIDELINK is on this RB}; the odd stride also
// spreads consecutive bins over the banks.  Dead lanes (no link, or agent absent this step) run the same straight-line
// code: they count into their own dummy word (no same-address serialisation) and store / load no record.
#define D2D_BLK_PWR 0u
#define D2D_BLK_LINKA (D2D_MAX_PWR_LEVELS * 4u)
#define D2D_BLK_LINKS (D2D_BLK_LINKA + 64u * 16u)
#define D2D_BLK_BYTES (D2D_BLK_LINKS + 64u * 8u)
#define D2D_DUMMY_BYTES 528u
#define D2D_BIN_STRIDE (D2D_BIN_CAP * 16u + 16u)
#define D2D_BIN_CNT (D2D_BIN_CAP * 16u)
__host__ __device__ inline uint32_t d2d_warp_smem_per_warp(int R) { return (uint32_t)R * D2D_BIN_STRIDE + D2D_DUMMY_BYTES + (((uint32_t)R * 8u + 15u) & ~15u); }
__host__ __device__ inline uint32_t d2d_warp_smem_bytes(int R, int wpb) { return D2D_BLK_BYTES + (uint32_t)wpb * d2d_warp_smem_per_warp(R); }

// Link / device / RB counts of the batch: immediates for the default EnvConfig, launch parameters otherwise.
template <bool SPEC>
struct D2DShape {
    uint32_t c_, n_, v_, r_, npc_, npd_, mc_, md_, n1c_, n1d_;
    __device__ __forceinline__ explicit D2DShape(const D2DParams &P) {
        if (!SPEC) {
            c_ = (uint32_t)P.C; n_ = (uint32_t)P.N; v_ = (uint32_t)P.V; r_ = (uint32_t)P.R;
            npc_ = (uint32_t)P.n_pwr_cue; npd_ = (uint32_t)P.n_pwr_due;
            mc_ = P.magic_cue; md_ = P.magic_due; n1c_ = P.npw1_cue; n1d_ = P.npw1_due;
        }
    }
    __device__ __forceinline__ uint32_t C() const { return SPEC ? 25u : c_; }
    __device__ __forceinline__ uint32_t N() const { return SPEC ? 50u : n_; }
    __device__ __forceinline__ uint32_t D() const { return SPEC ? 25u : n_ - c_; }
    __device__ __forceinline__ uint32_t V() const { return SPEC ? 76u : v_; }
    __device__ __forceinline__ uint32_t R() const { return SPEC ? 25u : r_; }
    __device__ __forceinline__ uint32_t npc() const { return SPEC ? 24u : npc_; }
    __device__ __forceinline__ uint32_t npd() const { return SPEC ? 21u : npd_; }
    // envs/d2d_env.py:95: rb = a // n_pwr for 0 <= a <= R n_pwr, by the multiply-high magic of d2d_div_magic
    __device__ __forceinline__ uint32_t rb_cue(uint32_t a) const {
        return SPEC ? __umulhi(a, 178956971u) : __umulhi(a, mc_) + (a & n1c_);      // ceil(2^32 / 24)
    }
    __device__ __forceinline__ uint32_t rb_due(uint32_t a) const {
        return SPEC ? __umulhi(a, 204522253u) : __umulhi(a, md_) + (a & n1d_);      // ceil(2^32 / 21)
    }
};

// Explicit ld/st.shared on 32-bit shared-window addresses: the compiler never re-derives generic addresses.
__device__ __forceinline__ void d2d_sts128(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void d2d_sts128_if(bool p, uint32_t a, float x, float y, float z, float w) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.v4.f32 [%1], {%2, %3, %4, %5}; }"
                 ::"r"((uint32_t)p), "r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void d2d_sts32_if(bool p, uint32_t a, uint32_t x) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.u32 [%1], %2; }" ::"r"((uint32_t)p), "r"(a), "r"(x) : "memory");
}
__device__ __forceinline__ void d2d_sts64_if(bool p, uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.v2.u32 [%1], {%2, %3}; }" ::"r"((uint32_t)p), "r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void d2d_sts64f(uint32_t a, float x, float y) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory");
}
__device__ __forceinline__ float4 d2d_lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float2 d2d_lds64(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float d2d_lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}
// same, with a compile-time byte offset folded into the instruction (no address add per access)
template <int OFF>
__device__ __forceinline__ float4 d2d_lds128_at(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a), "n"(OFF) : "memory");
    return v;
}
template <int OFF>
__device__ __forceinline__ float d2d_lds32_at(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF) : "memory");
    return v;
}
template <int OFF>
__device__ __forceinline__ uint2 d2d_lds64u_at(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];" : "=r"(v.x), "=r"(v.y) : "r"(a), "n"(OFF) : "memory");
    return v;
}
template <int OFF>
__device__ __forceinline__ uint32_t d2d_lds32u_at(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF) : "memory");
    return v;
}
template <int OFF>
__device__ __forceinline__ uint32_t d2d_atoms_inc_at(uint32_t a) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1+%2], 1;" : "=r"(old) : "r"(a), "n"(OFF) : "memory");
    return old;
}
// cp.async (LDGSTS): predicated per-lane global -> shared copies of 4 / 8 / 16 bytes
__device__ __forceinline__ void d2d_cp4_if(bool p, uint32_t dst, const void *src) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q cp.async.ca.shared.global [%1], [%2], 4; }" ::"r"((uint32_t)p), "r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void d2d_cp8_if(bool p, uint32_t dst, const void *src) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q cp.async.ca.shared.global [%1], [%2], 8; }" ::"r"((uint32_t)p), "r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void d2d_cp16_if(bool p, uint32_t dst, const void *src) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q cp.async.cg.shared.global [%1], [%2], 16; }" ::"r"((uint32_t)p), "r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void d2d_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void d2d_cp_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// warp-wide integer sum in one instruction (REDUX)
__device__ __forceinline__ uint32_t d2d_redux_add(uint32_t x) {
    uint32_t r;
    asm volatile("redux.sync.add.u32 %0, %1, 0xffffffff;" : "=r"(r) : "r"(x));
    return r;
}
// index of the highest set bit (FLO) and removal of that bit - rescue path only
__device__ __forceinline__ uint32_t d2d_pop_bit(uint32_t &mask) {
    uint32_t k;
    asm("bfind.u32 %0, %1;" : "=r"(k) : "r"(mask));
    mask ^= 1u << k;
    return k;
}

// One interferer's term at a general receiver: w_k g(|tx_k - rx|)
template <bool PLE2, bool EXACT>
__device__ __forceinline__ float d2d_term_rx(const float4 r, bool valid, float rxx, float rxy, float nhp, float &dmin2) {
    const float dx = r.x - rxx, dy = r.y - rxy;
    const float d2 = fmaf(dx, dx, dy * dy);
    if (EXACT) dmin2 = valid ? fminf(dmin2, d2) : dmin2;
    return valid ? r.z * d2d_gain<PLE2>(d2, nhp) : 0.0f;
}
// A victim's co-channel records are the first records of its bin; `valid` has bit t set when record t exists and is
// not the victim itself (at most D2D_BIN_CAP bits on the fast path).  A lane whose record t is not a peer reads the
// warp's all-zero record instead (`zrec`: one address for every such lane, so a broadcast, not a bank conflict): the
// load / store data pipe, not instruction issue, bounds this kernel, and 60 % of the (lane, t) pairs are not peers.
template <bool PLE2, bool EXACT, int T>
__device__ __forceinline__ void d2d_inline_rx(float &I, uint32_t bin, uint32_t zrec, uint32_t valid, float rxx, float rxy, float nhp,
                                              float &dmin2) {
    if constexpr (T < D2D_WALK_INLINE) {
        const bool v = valid & (1u << T);
        I += d2d_term_rx<PLE2, EXACT>(d2d_lds128(v ? bin + 16u * T : zrec), v, rxx, rxy, nhp, dmin2);
        d2d_inline_rx<PLE2, EXACT, T + 1>(I, bin, zrec, valid, rxx, rxy, nhp, dmin2);
    }
}
template <bool PLE2, bool EXACT>
__device__ __forceinline__ float d2d_walk_rx(uint32_t bin, uint32_t zrec, uint32_t valid, float rxx, float rxy, float nhp, float &dmin2) {
    float I = 0.0f;
    d2d_inline_rx<PLE2, EXACT, 0>(I, bin, zrec, valid, rxx, rxy, nhp, dmin2);
    valid >>= D2D_WALK_INLINE;
    for (uint32_t a = bin + 16u * D2D_WALK_INLINE; valid; valid >>= 1, a += 16u)   // > D2D_WALK_INLINE links on one RB
        if (valid & 1u) I += d2d_term_rx<PLE2, EXACT>(d2d_lds128(a), true, rxx, rxy, nhp, dmin2);
    return I;
}
// Interference at the MBS: the records carry u_k = w_k g(|tx_k|) in .w (the zero record adds nothing)
template <int T>
__device__ __forceinline__ void d2d_inline_mbs(float &I, uint32_t bin, uint32_t zrec, uint32_t valid) {
    if constexpr (T < D2D_WALK_INLINE) {
        I += d2d_lds32((valid & (1u << T)) ? bin + (16u * T + 12u) : zrec);
        d2d_inline_mbs<T + 1>(I, bin, zrec, valid);
    }
}
__device__ __forceinline__ float d2d_walk_mbs(uint32_t bin, uint32_t zrec, uint32_t valid) {
    float I = 0.0f;
    d2d_inline_mbs<0>(I, bin, zrec, valid);
    valid >>= D2D_WALK_INLINE;
    for (uint32_t a = bin + 16u * D2D_WALK_INLINE + 12u; valid; valid >>= 1, a += 16u)
        if (valid & 1u) I += d2d_lds32(a);
    return I;
}

// Predicated global stores (no branch, no reconvergence bookkeeping around a two-line body)
__device__ __forceinline__ void d2d_stg64_if(bool p, void *ptr, float x, float y) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.global.v2.f32 [%1], {%2, %3}; }" ::"r"((uint32_t)p), "l"(ptr), "f"(x), "f"(y) : "memory");
}
__device__ __forceinline__ void d2d_stg32_if(bool p, void *ptr, float x) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.global.f32 [%1], %2; }" ::"r"((uint32_t)p), "l"(ptr), "f"(x) : "memory");
}
__device__ __forceinline__ void d2d_stg16_if(bool p, void *ptr, int x) {
    asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.global.u16 [%1], %2; }" ::"r"((uint32_t)p), "l"(ptr), "h"((short)x) : "memory");
}

// One env's inputs as a lane sees them: its CUE action + transmitter (device 1 + l), its DUE action + (tx, rx) pair
// (devices 1 + C + 2l, + 1).  Lanes without a link keep benign values (action -1 = absent, unit distances).
struct D2DLaneIn {
    uint32_t aA, aB;
    float2 tA;        // CUE transmitter (its receiver is the MBS at the origin)
    float4 pB;        // DUE (tx_x, tx_y, rx_x, rx_y)
};
// iA = e N + lane, qA = e V + 1 + lane
template <bool SPEC>
__device__ __forceinline__ D2DLaneIn d2d_load_inputs(const D2DParams &P, const D2DShape<SPEC> &S, uint32_t iA, uint32_t qA, uint32_t lane,
                                                      bool hasA, bool hasB) {
    D2DLaneIn in;
    in.aA = 0xffffffffu; in.aB = 0xffffffffu;
    in.tA = make_float2(1.f, 0.f);
    in.pB = make_float4(1.f, 0.f, 0.f, 0.f);
    const float2 *pos = reinterpret_cast<const float2 *>(P.pos);
    if (hasA) { in.aA = (uint32_t)__ldg(P.actions + iA); in.tA = __ldg(pos + qA); }
    if (hasB) {
        in.aB = (uint32_t)__ldg(P.actions + (iA + S.C()));
        const float2 *pq = pos + (qA + S.C() + lane);
        if (SPEC || P.align4) {
            in.pB = __ldg(reinterpret_cast<const float4 *>(pq));
        } else {
            const float2 t = __ldg(pq), r = __ldg(pq + 1);
            in.pB = make_float4(t.x, t.y, r.x, r.y);
        }
    }
    return in;
}

// d2d_step_many: the next step's two actions of the same env (positions stay in registers)
template <bool SPEC>
__device__ __forceinline__ void d2d_load_actions(const D2DParams &P, const D2DShape<SPEC> &S, uint32_t iA, bool hasA, bool hasB,
                                                 D2DLaneIn &in) {
    in.aA = 0xffffffffu; in.aB = 0xffffffffu;
    if (hasA) in.aA = (uint32_t)__ldg(P.actions + iA);
    if (hasB) in.aB = (uint32_t)__ldg(P.actions + (iA + S.C()));
}

// log2(1 + r), branch-free form of d2d_log2_1p (both sides are a handful of instructions; a divergent branch costs more)
__device__ __forceinline__ float d2d_log2_1p_sel(float r) {
    const float s = r * d2d_rcp(2.0f + r);
    const float s2 = s * s;
    const float poly = fmaf(s2, fmaf(s2, fmaf(s2, (1.0f / 7.0f), 0.2f), (1.0f / 3.0f)), 1.0f);
    const float small = (2.8853900817779268f * s) * poly;
    const float big = d2d_lg2(1.0f + r);
    return r < 0.25f ? small : big;
}
// Per-link epilogue in fp32 (Appendix A), dead lanes zeroed.  Same arithmetic as d2d_link_epilogue (d2d_common.cuh).
// SNR_dB comes from the linear ratio, like SINR_dB (see d2d_link_epilogue).
__device__ __forceinline__ D2DLinkOut d2d_link_epilogue_warp(bool live, float p_lin, float g, float I, const float4 &cA, const float2 &sb) {
    D2DLinkOut o;
    const float snr_lin = p_lin * cA.y * g;
    const float r = snr_lin * d2d_rcp(fmaf(I, cA.z, 1.0f));
    const float snr = 3.0102999566398120f * d2d_lg2(snr_lin);
    const float sinr = 3.0102999566398120f * d2d_lg2(r);
    const bool ok = live && sinr > sb.x;
    const float rate = d2d_log2_1p_sel(r);
    o.snr_dB = live ? snr : 0.0f;
    o.sinr_dB = live ? sinr : 0.0f;
    o.rate = ok ? rate : 0.0f;
    o.cap = ok ? sb.y * rate : 0.0f;
    return o;
}

// ---- rare paths -----------------------------------------------------------------------------------------------------------

// Some RB holds more links than a bin has record slots: the links ranked D2D_BIN_CAP and above have no record, and this pass
// adds their terms by shuffle (the bin walk has already added those of the records).  Source keys: the RB of a live slot of
// rank >= D2D_BIN_CAP, the slot's unique inactive key otherwise; victim keys: the RB of every live slot.  A term counts when
// the keys match and it is not the victim itself.  The terms go on top of the bin walk's sums IA / IB (and, with EXACT, its
// distances dmin2A / dmin2B), in lane order.
// Only lanes that hold such a source are visited, in lane order: at the default load one lane, rarely two (an RB of 9 or 10
// links); with every link on one RB at most 25.  Any other lane matches no victim but itself, so skipping it changes no bit.
#ifndef D2D_RARE_ATTR
#define D2D_RARE_ATTR __forceinline__     // A/B knob: __noinline__ moves the rare paths out of the hot loop's code
#endif
template <bool PLE2, bool EXACT>
__device__ D2D_RARE_ATTR void d2d_overflow_warp(uint32_t lane, uint32_t keyA, uint32_t keyB, uint32_t srcA, uint32_t srcB, float4 recA,
                                                   float4 pB, float wB, float uB, float nhp, float &IA, float &IB, float &dminA, float &dminB) {
#pragma unroll 1
    for (uint32_t src = __ballot_sync(0xffffffffu, (srcA & srcB & D2D_INACTIVE_KEY) == 0u); src; src &= src - 1u) {
        const uint32_t k = (uint32_t)__ffs((int)src) - 1u;
        const uint32_t kA = __shfl_sync(0xffffffffu, srcA, k), kB = __shfl_sync(0xffffffffu, srcB, k);
        const float4 ra = make_float4(__shfl_sync(0xffffffffu, recA.x, k), __shfl_sync(0xffffffffu, recA.y, k),
                                      __shfl_sync(0xffffffffu, recA.z, k), __shfl_sync(0xffffffffu, recA.w, k));
        const float4 rb = make_float4(__shfl_sync(0xffffffffu, pB.x, k), __shfl_sync(0xffffffffu, pB.y, k),
                                      __shfl_sync(0xffffffffu, wB, k), __shfl_sync(0xffffffffu, uB, k));
        if (EXACT) {
            IA += d2d_term_rx<PLE2, true>(ra, kA == keyA && k != lane, 0.f, 0.f, nhp, dminA);
            IA += d2d_term_rx<PLE2, true>(rb, kB == keyA, 0.f, 0.f, nhp, dminA);
        } else {
            IA += (kA == keyA && k != lane) ? ra.w : 0.f;
            IA += (kB == keyA) ? rb.w : 0.f;
        }
        IB += d2d_term_rx<PLE2, EXACT>(ra, kA == keyB, pB.z, pB.w, nhp, dminB);
        IB += d2d_term_rx<PLE2, EXACT>(rb, kB == keyB && k != lane, pB.z, pB.w, nhp, dminB);
    }
}

__device__ __forceinline__ double d2d_shfl_f64(double v, int src) {
    return __hiloint2double(__shfl_sync(0xffffffffu, __double2hiint(v), src), __shfl_sync(0xffffffffu, __double2loint(v), src));
}
__device__ __forceinline__ double d2d_shfl_xor_f64(double v, int m) {
    return __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(v), m), __shfl_xor_sync(0xffffffffu, __double2loint(v), m));
}

// fp64 recomputation of the links flagged by needA / needB (see d2d_common.cuh for why and when).  Per flagged link the
// whole warp cooperates: every lane evaluates its own two links' interference terms at the victim's receiver in fp64
// (positions are exact in fp64: they ARE the fp32 state, or the bound fp64 shadow), a butterfly sums them, and the
// victim's own lane recomputes that link's outputs.  Two placements (d2d_step_warp_kernel picks by launch shape):
//   STORE = false: the new values replace the lane's registers (oA / oB) BEFORE the env's outputs are stored.  The pass touches
//                  only inputs (positions, actions, constant tables), so it runs ahead of griddepcontrol.wait like the rest of the
//                  env's arithmetic - after the wait it sat on the critical path of every back-to-back launch of a one-wave batch
//                  (profiles/timeline.py: the ~7 % of warps with a flagged link ended 2 us after the others and held the block
//                  slots of the next launch).  Costs the hot loop a few spilled registers.
//   STORE = true:  the pass runs after the env's stores and overwrites the link's outputs in global memory - no live output
//                  registers across it; the throughput shape (many envs per warp, one wait per warp).
// Nothing of the hot loop's shared-memory state is used: only the lane's own inputs.
// Without a position shadow a dB value is rewritten only when its linear ratio is within 1/16 of one - the only place the
// fp32 value is ill-conditioned; rate and capacity are well conditioned there and are rewritten only if the sensitivity
// gate (simulator.py:123,149) could sit inside that band.  With a shadow every output of the link is rewritten.
// AR (d2d_step with auto-reset): `drawn` marks an env whose positions this launch drew; the shadow rows still hold the finished
// episode's, so the pass takes the lane's fp32 registers - the values the launch stores to the shadow.
// Returns the number of links recomputed.
// 10^(p/10) in fp64 for the warp kernel's fp64 pass: the constant bank instead of a global table (filled by d2d_create)
static __constant__ double d2d_pwr_lin_c[D2D_MAX_PWR_LEVELS];    // one copy per translation unit (d2d_tu_warp.cu)

template <bool PLE2, bool EXACT, bool SPEC, bool STORE, bool THR, bool AR = false>
__device__ __forceinline__ int d2d_rescue_warp(const D2DParams &P, const D2DShape<SPEC> &S, uint32_t e, uint32_t lane, uint32_t jA,
                                               uint32_t keyA, uint32_t keyB, bool needA, bool needB, uint32_t pA, uint32_t pB_,
                                               const float2 &tA, const float4 &pB, D2DLinkOut &oA, D2DLinkOut &oB, bool drawn = false) {
    const uint32_t C = S.C(), V = S.V();
    // Without an fp64 shadow the positions ARE the fp32 state the lane already holds; with uniform link constants (one set per
    // link type: every default-shape batch) those come from the constant bank, like the power table: then the pass reads
    // no global memory at all - its dependent round trips were most of its ~2 us per link (profiles/timeline.py).
    const bool uni = SPEC || P.uniform != 0;
    // this lane's two transmitters and the DUE receiver, in fp64
    double2 txA = make_double2((double)tA.x, (double)tA.y), txB = make_double2((double)pB.x, (double)pB.y);
    double2 rxB = make_double2((double)pB.z, (double)pB.w);
    if (EXACT && !(AR && drawn)) {
        const double2 *pe64 = reinterpret_cast<const double2 *>(P.pos64) + (int64_t)e * V;
        if (lane < C) txA = pe64[1u + lane];
        if (lane < S.D()) { txB = pe64[1u + C + 2u * lane]; rxB = pe64[2u + C + 2u * lane]; }
    }
    // radiated weights w = 10^(p/10) 10^((eo - K)/10) in fp64
    const double wA = d2d_pwr_lin_c[pA & (D2D_MAX_PWR_LEVELS - 1)] * (uni ? P.ud_cue.t_lin : lane < C ? P.linkD[lane].t_lin : 0.0);
    const double wB = d2d_pwr_lin_c[pB_ & (D2D_MAX_PWR_LEVELS - 1)] * (uni ? P.ud_due.t_lin : lane < S.D() ? P.linkD[C + lane].t_lin : 0.0);
    int done = 0;
#pragma unroll 1
    for (int s = 0; s < 2; ++s) {
        uint32_t todo = __ballot_sync(0xffffffffu, s ? needB : needA);
        while (todo) {
            const int L = (int)d2d_pop_bit(todo);
            const uint32_t key = __shfl_sync(0xffffffffu, s ? keyB : keyA, L);
            const double rxx = s ? d2d_shfl_f64(rxB.x, L) : 0.0, rxy = s ? d2d_shfl_f64(rxB.y, L) : 0.0;   // MBS at the origin
            double I = 0.0;
            if (keyA == key && !(s == 0 && (int)lane == L)) {
                const double ex = txA.x - rxx, ey = txA.y - rxy;
                I += wA * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
            }
            if (keyB == key && !(s == 1 && (int)lane == L)) {
                const double ex = txB.x - rxx, ey = txB.y - rxy;
                I += wB * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
            }
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) I += d2d_shfl_xor_f64(I, sh);
            if ((int)lane == L) {
                const uint32_t j = s ? C + lane : lane;
                D2DLinkD Lj = s ? P.ud_due : P.ud_cue;
                float sens = s ? P.us_due.x : P.us_cue.x;
                if (!uni) { Lj = P.linkD[j]; sens = P.linkB[j].sens_dBm; }
                const double2 tx = s ? txB : txA;
                const double dx = tx.x - rxx, dy = tx.y - rxy;
                const double Sg = d2d_pwr_lin_c[(s ? pB_ : pA) & (D2D_MAX_PWR_LEVELS - 1)] * Lj.a_lin * d2d_gain_f64_fast<PLE2>(dx * dx + dy * dy, P.ple_d);
                const double r = Sg * d2d_rcp_f64(fma(I, Lj.inv_noise, 1.0));          // a_lin already carries 1 / noise
                const bool r1 = fabs(r - 1.0) < 0.0625, s1 = fabs(Sg - 1.0) < 0.0625;
                const uint32_t row = s ? jA + C : jA;
                D2DLinkOut o;
                if (!STORE) o = s ? oB : oA;
                double sinr = 0.0;
                if (EXACT || r1 || (THR && P.thr_band > 0.f)) {
                    sinr = r1 ? d2d_db_near1(r) : 4.3429448190325182765 * d2d_ln_f64(r);
                    o.sinr_dB = THR ? d2d_sinr_store(sinr, P) : (float)sinr;
                    if (STORE && P.obs) P.obs[(uint64_t)row * 6u + 4u] = o.sinr_dB;
                    if (STORE && P.obs_dyn) P.obs_dyn[row].x = o.sinr_dB;
                }
                if (EXACT || s1) {
                    o.snr_dB = (float)(s1 ? d2d_db_near1(Sg) : 4.3429448190325182765 * d2d_ln_f64(Sg));
                    if (STORE && P.obs) P.obs[(uint64_t)row * 6u + 5u] = o.snr_dB;
                    if (STORE && P.obs_dyn) P.obs_dyn[row].y = o.snr_dB;
                }
                if (EXACT || (r1 && fabsf(sens) < 0.5f)) {
                    const double rate = sinr > (double)sens ? 1.4426950408889634074 * d2d_ln_f64(1.0 + r) : 0.0;
                    o.cap = (float)(Lj.bw_MHz * rate);
                    o.rate = (float)rate;
                    if (STORE && P.cap) P.cap[row] = o.cap;
                    if (STORE && P.rate) P.rate[row] = o.rate;
                }
                if (!STORE) { if (s) oB = o; else oA = o; }
                ++done;
            }
        }
    }
    return (int)__reduce_add_sync(0xffffffffu, (unsigned)done);
}

// the throughput shapes' call of the pass (after the stores): one place to take it out of line
template <bool PLE2, bool EXACT, bool SPEC, bool THR, bool AR = false>
__device__ D2D_RARE_ATTR int d2d_rescue_warp_late(const D2DParams &P, const D2DShape<SPEC> &S, uint32_t e, uint32_t lane, uint32_t jA,
                                                  uint32_t keyA, uint32_t keyB, bool needA, bool needB, uint32_t pA, uint32_t pB_,
                                                  float2 tA, float4 pB, bool drawn = false) {
    D2DLinkOut oA, oB;       // unused by the storing variant
    return d2d_rescue_warp<PLE2, EXACT, SPEC, true, THR, AR>(P, S, e, lane, jA, keyA, keyB, needA, needB, pA, pB_, tA, pB, oA, oB, drawn);
}

// FULL: the caller passed exactly the core outputs (obs, capacity, reward, done) and a step counter is bound - the
// VecD2DEnv default - so no pointer is tested on the hot path; otherwise every output is optional and checked.
// MANY: d2d_step_many - P.T consecutive steps per env in ONE launch (the agent loop of examples/simple_env.py:20-33
// with the actions of all T steps given up front).  An env's positions are read once and stay in registers for its T
// steps; step t reads actions[t][e] and writes the [t][e] slice of every output (slices P.t_stride envs apart).
// MODE 0: d2d_step.  MODE 1 (MANY): d2d_step_many.  MODE 2 (EPISODE): d2d_episode - D2DEnv.reset (envs/d2d_env.py:45-52) and the
// agent loop after it in ONE launch: slice 0 of every output is the uncounted reset step on freshly drawn positions
// (Simulator.reset, simulator.py:61-75; the draws of d2d_reset, d2d_common.cuh), slices 1 .. P.T - 1 are the counted steps.  The
// positions are drawn in registers and written to the bound state once; the actions of every step are either read from
// actions [P.T][E][N] or (D2D_PF_DRAW_ACTIONS) drawn on the device like envs/d2d_env.py:54-60 - the kernel then reads nothing
// but its constant tables.  MODE 2 reads its variant from P.flags (given or drawn actions, d2d_episode or d2d_rollout, any
// set of outputs); MODE 3 (episode) and MODE 4 (rollout) are the instantiations of the common case - drawn actions, exactly
// the core outputs (FULL) - with those choices compiled in: 490 instead of 590 warp-instructions per env-step.
// MODE 5 (AR): d2d_step with D2D_STEP_AUTORESET.  An env whose step counter is below episode_length at entry steps exactly as in
// MODE 0; one at or past it (its previous step returned done) is reset instead, as D2DEnv.reset does it (envs/d2d_env.py:45-52):
// positions drawn like d2d_reset and actions like d2d_sample_actions(step 0), both under d2d_autoreset_key(ar_base, n) with n its
// incremented episode index, then one uncounted step on them.  Its outputs are that step's with reward = done = 0; its counter
// becomes 0, the drawn positions the bound state.  The launch always waits at entry (the host never flags it INPUTS_STABLE or
// LATE_WAIT), so each group's counters and episode indices are read into lanes before the group's first env is computed.
template <bool PLE2, bool EXACT, int WPB, bool FULL, bool SPEC, int MODE>
__global__ void __launch_bounds__(WPB * 32, D2D_WARP_MIN_BLOCKS(WPB))
d2d_step_warp_kernel(const __grid_constant__ D2DParams P) {
    extern __shared__ __align__(16) unsigned char d2d_warp_smem[];
    constexpr bool AR = MODE == 5;
    constexpr bool MANY = MODE != 0 && !AR, EPI = MODE >= 2 && !AR, EPI_FAST = MODE == 3 || MODE == 4;
    static_assert(!EPI_FAST || FULL, "the fast episode / rollout instantiations write exactly the core outputs");
    const D2DShape<SPEC> S(P);
    // latency shape: the fp64 pass runs before griddepcontrol.wait
    constexpr bool RESCUE_EARLY = WPB == 2;
    // statistics flushed with the warp's last env, ahead of the wait - the shapes where a warp steps one or a few envs; the
    // throughput shape flushes after its loop (the per-env test costs its 37-env warps more than the late atomics)
    constexpr bool FLUSH_EARLY = WPB != 8;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t C = S.C(), N = S.N(), V = S.V(), R = S.R();
#ifdef D2D_TIMELINE
    const unsigned long long tl_g0 = d2d_tl_gtime(), tl_c0 = d2d_tl_clock();
    unsigned long long tl_c1 = 0, tl_c2 = 0;
    uint32_t tl_env = 0, tl_pre = 0, tl_post = 0, tl_ovf = 0;      // envs, fp64 links before / after the wait, overflow envs
    bool tl_waited = false;
#endif
    d2d_pdl_entry(P.flags);
    uint32_t blk = (uint32_t)__cvta_generic_to_shared(d2d_warp_smem);
    asm volatile("mov.u32 %0, %0;" : "+r"(blk));      // opaque: keep the base in a register instead of re-deriving it
    const uint32_t bins = blk + D2D_BLK_BYTES + warp * d2d_warp_smem_per_warp((int)R);
    const uint32_t dumA = bins + R * D2D_BIN_STRIDE + (lane << 3);        // this lane's dummy (count, flag) pairs: A, B at + 256
    const uint32_t zrec = bins + R * D2D_BIN_STRIDE + 512u;               // the warp's all-zero peer record
    const bool hasA = lane < C, hasB = lane < S.D();

    const uint32_t num_envs = (uint32_t)P.num_envs;
    const uint32_t gw = blockIdx.x * WPB + warp;
    const uint32_t e0 = min(gw * P.envs_per_warp + min(gw, P.envs_extra), num_envs),
                   e_end = min(e0 + P.envs_per_warp + (gw < P.envs_extra ? 1u : 0u), num_envs);
    uint32_t e = e0;
    uint32_t iA = e * N + lane;                                    // slot-A link index of the env being computed
    uint32_t qN = e * V + 1u + lane;                               // slot-A device index of the env being prefetched
    // the first env's inputs go out before anything else: their latency overlaps the table loads of the prologue instead of
    // following them (a warp of a one-wave batch steps a single env: two serial memory round trips were a tenth of its life)
    D2DLaneIn nxt;
    const bool draw_actions = EPI_FAST || (EPI && (P.flags & D2D_PF_DRAW_ACTIONS) != 0u);
    const bool ep_reset = MODE == 3 || (MODE == 2 && (P.flags & D2D_PF_NO_RESET) == 0u);     // d2d_episode (true) or d2d_rollout (false)
    if (EPI) {
        nxt.aA = nxt.aB = 0xffffffffu; nxt.tA = make_float2(1.f, 0.f); nxt.pB = make_float4(1.f, 0.f, 0.f, 0.f);
        if (e < e_end && !draw_actions) d2d_load_actions<SPEC>(P, S, iA, hasA, hasB, nxt);
    } else if (e < e_end) nxt = d2d_load_inputs<SPEC>(P, S, iA, qN, lane, hasA, hasB);

    // ---- prologue (constant tables only: nothing a previous kernel in the stream may have written) ------------------
    // block tables: 10^(p/10) for integer dBm, and the per-link constants by lane slot (zeros where there is no link)
    for (uint32_t i = threadIdx.x; i < D2D_MAX_PWR_LEVELS / 4u; i += WPB * 32u) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(P.pwr_lin) + i);
        d2d_sts128(blk + D2D_BLK_PWR + (i << 4), v.x, v.y, v.z, v.w);
    }
    for (uint32_t i = threadIdx.x; !SPEC && i < 64u; i += WPB * 32u) {
        const uint32_t l = i & 31u, j = i < 32u ? l : C + l;
        const bool has = i < 32u ? l < C : l < S.D();
        const float4 a = has ? __ldg(reinterpret_cast<const float4 *>(P.linkA) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float2 b = has ? __ldg(reinterpret_cast<const float2 *>(P.linkB + j)) : make_float2(0.f, 0.f);
        d2d_sts128(blk + D2D_BLK_LINKA + (i << 4), a.x, a.y, a.z, a.w);
        d2d_sts64f(blk + D2D_BLK_LINKS + (i << 3), b.x, b.y);
    }
    // this warp's bins: every counter starts at zero; each env re-zeroes them after use (the dummy words just run on)
    // the RBs' (link count, SIDELINK flag) pairs: a compact array behind the bins, 8 bytes per RB, so that the 25 counters of the
    // default shape spread over 16 bank pairs (in the bins' tails - 144-byte stride - they fell onto 8 banks: ATOMS took 6.5
    // wavefronts instead of ~3)
    const uint32_t cb = bins + R * D2D_BIN_STRIDE + D2D_DUMMY_BYTES;
    for (uint32_t r = lane; r < R; r += 32u) d2d_sts64_if(true, cb + (r << 3), 0u, 0u);
    d2d_sts64_if(true, dumA, 0u, 0u);
    d2d_sts64_if(true, dumA + 256u, 0u, 0u);
    if (lane < 4u) d2d_sts32_if(true, zrec + (lane << 2), 0u);
    __syncthreads();

    const uint32_t lkA = blk + D2D_BLK_LINKA + (lane << 4), lkS = blk + D2D_BLK_LINKS + (lane << 3);
    const uint32_t zero0 = cb + (lane << 3);                                  // this lane's share of the counter re-zeroing
    // a valid action is 0 <= a < R n_pwr (envs/d2d_env.py:36-40); anything else marks the agent absent this step.
    // The sentinel action R n_pwr decodes to (rb = R, p = 0): a valid table index and an address inside the warp's slice.
    const uint32_t limA = R * S.npc(), limB = R * S.npd();

    // per-warp partial statistics (fp32 over the few envs one warp visits; flushed once as fp64 atomics)
    float st_reward = 0.f, st_cap = 0.f, st_reward2 = 0.f;
    uint32_t st_pen = 0, st_resc = 0;

    // 32-bit indexing: the host launches at most 2^31 / max(6N, 2V) envs per call (d2d_step chunks larger batches).
    // Each warp steps a CONTIGUOUS range of envs, so the per-env scalars (step counter, reward, done) are kept in
    // registers - env i of a group of 32 lives in lane i - and read / written once per group as full sectors.  (One byte
    // per env read and written by 32 different warps per sector cost a quarter of the kernel's time in L2 read-modify-
    // write stalls: profiles/README.md.)
    uint32_t g = 0;                                                // position of env e in its group of 32
    int ns_keep = 0;                                               // lane i: step counter of the group's env i
    float rew_keep = 0.f;                                          // lane i: reward of the group's env i
    uint32_t ep_keep = 0;                                          // AR, lane i: episode index of the group's env i ...
    bool rs_keep = false;                                          // ... and whether this launch resets it
    uint32_t st_steps = 0;                                         // AR: counted env-steps of this warp
    // d2d_step_many state: step index inside the env, the link / env offsets of output slice t, the env's positions
    uint32_t t = 0, tN = 0, tE = 0;
    const uint32_t T = MANY ? (uint32_t)P.T : 1u, strideE = MANY ? (uint32_t)P.t_stride : 0u, strideN = strideE * N;
    float2 tA_keep = make_float2(1.f, 0.f);
    float4 pB_keep = make_float4(1.f, 0.f, 0.f, 0.f);
    uint4 ablk = make_uint4(0u, 0u, 0u, 0u);                       // EPISODE: the lane's action block of steps t & ~1, t | 1
    // Programmatic dependent launch: the kernel BEFORE this one in the stream may still be running.  If it is one of this
    // library's step kernels it never writes actions or positions (and anything else - a policy kernel, a reset, a copy -
    // does not release its dependents early), so this env-step's inputs are read and its whole chain computed right away;
    // griddepcontrol.wait comes only before the first access to memory a previous step wrote: the step counters and the
    // output buffers.  Back-to-back steps thus overlap one step's tail with the next step's loads and arithmetic.
    while (e < e_end) {
        // ---- one coalesced pass over the env's inputs, software-pipelined: the NEXT env's (or step's) loads are in
        // flight while this one computes, so a warp hides its own HBM latency -------------------------------------------
        uint32_t aA = nxt.aA, aB = nxt.aB;
        if (EPI) {
            const uint64_t genv = P.first_global_env + (uint64_t)e;
            if (t == 0u) {
                tA_keep = make_float2(1.f, 0.f); pB_keep = make_float4(1.f, 0.f, 0.f, 0.f);
                if (ep_reset) {                                     // Simulator.reset (simulator.py:61-75): this env's new positions
                    if (hasA) tA_keep = d2d_draw_cue(P.ep_seed, genv, lane, P.cell_radius);
                    if (hasB) pB_keep = d2d_draw_due(P.ep_seed, genv, (C + 1u) >> 1, lane, P.cell_radius, P.d2d_radius);
                } else {                                            // d2d_rollout: the bound positions, read once for the T steps
                    const float2 *pe = reinterpret_cast<const float2 *>(P.pos) + (uint64_t)e * V;
                    if (hasA) tA_keep = __ldg(pe + 1u + lane);
                    if (hasB) {
                        const float2 tx = __ldg(pe + 1u + C + 2u * lane), rx = __ldg(pe + 2u + C + 2u * lane);
                        pB_keep = make_float4(tx.x, tx.y, rx.x, rx.y);
                    }
                }
            }
            if (draw_actions) {                                     // envs/d2d_env.py:54-60: Discrete(R n_pwr).sample() per agent
                const uint32_t ts = t + P.act_t0;
                if ((ts & 1u) == 0u || t == 0u) ablk = d2d_action_block(P.act_seed, genv, lane, ts);
                aA = hasA ? __umulhi(d2d_action_word(ablk, ts, false), limA) : 0xffffffffu;
                aB = hasB ? __umulhi(d2d_action_word(ablk, ts, true), limB) : 0xffffffffu;
            }
        } else if (!MANY || t == 0u) { tA_keep = nxt.tA; pB_keep = nxt.pB; }
        // AR: this env is reset instead of stepped.  Every use below reads (AR && ar_rst): a bare runtime flag, although constant
        // false in the other modes, changed their instruction schedule
        bool ar_rst = false;
        if constexpr (AR) {
            if (g == 0u) {
                ns_keep = e + lane < e_end ? (int)P.step_count[e + lane] : 0;
                ep_keep = e + lane < e_end ? P.episode_index[e + lane] : 0u;
            }
            ar_rst = __shfl_sync(0xffffffffu, ns_keep, (int)g) >= P.episode_length;
            if (ar_rst) {                                           // (the prefetched positions and actions of this env go unused)
                const uint64_t genv = P.first_global_env + (uint64_t)e;
                const uint64_t key = d2d_autoreset_key(P.ar_base, (uint64_t)(__shfl_sync(0xffffffffu, ep_keep, (int)g) + 1u));
                tA_keep = hasA ? d2d_draw_cue(key, genv, lane, P.cell_radius) : make_float2(1.f, 0.f);
                pB_keep = hasB ? d2d_draw_due(key, genv, (C + 1u) >> 1, lane, P.cell_radius, P.d2d_radius) : make_float4(1.f, 0.f, 0.f, 0.f);
                const uint4 ab = d2d_action_block(key, genv, lane, 0u);
                aA = hasA ? __umulhi(d2d_action_word(ab, 0u, false), limA) : 0xffffffffu;
                aB = hasB ? __umulhi(d2d_action_word(ab, 0u, true), limB) : 0xffffffffu;
            }
        }
        const float2 tA = tA_keep;
        const float4 pB = pB_keep;
        const uint32_t jA = iA + tN, jB = jA + C;                   // this env-step's link indices (outputs)
        const bool last_t = !MANY || t + 1u == T;
        if (EPI) {
            if (!draw_actions) {
                if (!last_t) d2d_load_actions<SPEC>(P, S, jA + strideN, hasA, hasB, nxt);
                else if (e + 1u < e_end) d2d_load_actions<SPEC>(P, S, iA + N, hasA, hasB, nxt);
            }
        } else if (last_t) {
            qN += V;
            if (e + 1u < e_end) nxt = d2d_load_inputs<SPEC>(P, S, iA + N, qN, lane, hasA, hasB);
        } else {
            d2d_load_actions<SPEC>(P, S, jA + strideN, hasA, hasB, nxt);
        }
        const bool liveA = hasA && aA < limA, liveB = hasB && aB < limB;   // has a link AND the agent acts this step

        // ---- envs/d2d_env.py:93-101: rb = a // n_pwr, p = a % n_pwr; rank inside the RB (actions.py:27-31) -------------
        const uint32_t asA = liveA ? aA : limA, asB = liveB ? aB : limB;      // dead lanes -> (rb = R, p = 0)
        const uint32_t rbA = S.rb_cue(asA), rbB = S.rb_due(asB);
        const uint32_t pA = asA - rbA * S.npc(), pB_ = asB - rbB * S.npd();
        const uint32_t binA = bins + rbA * D2D_BIN_STRIDE, binB = bins + rbB * D2D_BIN_STRIDE;
        const uint32_t cntA = liveA ? cb + (rbA << 3) : dumA, cntB = liveB ? cb + (rbB << 3) : dumA + 256u;
        const uint32_t rankA = d2d_atoms_inc_at<0>(cntA);
        const uint32_t rankB = d2d_atoms_inc_at<0>(cntB);
        d2d_sts32_if(liveB, cntB + 4u, 1u);                                     // a SIDELINK is on this RB (reward_fn.py:31-37)
        const float plA = d2d_lds32(blk + D2D_BLK_PWR + (pA << 2));            // 10^(p/10)
        const float plB = d2d_lds32(blk + D2D_BLK_PWR + (pB_ << 2));
        // (tx_lin0, a_lin, inv_noise, snr0_dB): the default EnvConfig has one set per link type, held in the constant bank
        const float4 cA = SPEC ? P.u_cue : d2d_lds128_at<0>(lkA), cB = SPEC ? P.u_due : d2d_lds128_at<512>(lkA);

        // ---- peer records: position, radiated weight w, and its value u at the MBS -------------------------------
        const float d2A = fmaf(tA.x, tA.x, tA.y * tA.y);                       // CUE -> MBS distance^2 (own link)
        const float gA = d2d_gain<PLE2>(d2A, P.neg_half_ple);
        const float wA = plA * cA.x;
        const float d2Bm = fmaf(pB.x, pB.x, pB.y * pB.y);                      // DUE tx -> MBS distance^2 (as interferer)
        const float wB = plB * cB.x;
        const float uA = wA * gA, uB = wB * d2d_gain<PLE2>(d2Bm, P.neg_half_ple);
        const float dxB = pB.x - pB.z, dyB = pB.y - pB.w;                      // DUE own link
        const float d2B = fmaf(dxB, dxB, dyB * dyB);
        const float gB = d2d_gain<PLE2>(d2B, P.neg_half_ple);
        d2d_sts128_if(liveA && rankA < D2D_BIN_CAP, binA + (rankA << 4), tA.x, tA.y, wA, uA);
        d2d_sts128_if(liveB && rankB < D2D_BIN_CAP, binB + (rankB << 4), pB.x, pB.y, wB, uB);
        __syncwarp();

        // ---- simulator.py:95-101: interference at each victim's receiver (a dead lane has an empty range) ----------
        const uint2 ctA = d2d_lds64u_at<0>(cntA);                              // (links on the victim's RB, SIDELINK flag)
        const uint32_t nA = ctA.x, nB = d2d_lds32u_at<0>(cntB);
        float dminA = 3.0e38f, dminB = 3.0e38f;
        // bit t of valid <=> record t of the victim's bin exists and is not the victim (dead lane: 0).  An RB of more than
        // D2D_BIN_CAP links has D2D_BIN_CAP records; a victim ranked beyond them has none to exclude.
        const uint32_t validA = liveA ? (((1u << min(nA, (uint32_t)D2D_BIN_CAP)) - 1u) & ~(rankA < D2D_BIN_CAP ? 1u << rankA : 0u)) : 0u;
        const uint32_t validB = liveB ? (((1u << min(nB, (uint32_t)D2D_BIN_CAP)) - 1u) & ~(rankB < D2D_BIN_CAP ? 1u << rankB : 0u)) : 0u;
        float IA = EXACT ? d2d_walk_rx<PLE2, true>(binA, zrec, validA, 0.f, 0.f, P.neg_half_ple, dminA) : d2d_walk_mbs(binA, zrec, validA);
        float IB = d2d_walk_rx<PLE2, EXACT>(binB, zrec, validB, pB.z, pB.w, P.neg_half_ple, dminB);
        const bool ovfA = liveA && rankA >= D2D_BIN_CAP, ovfB = liveB && rankB >= D2D_BIN_CAP;
        if (__any_sync(0xffffffffu, ovfA || ovfB)) {
            // rare: some RB holds more links than a bin has record slots - add the links without a record
            const uint32_t keyA = liveA ? rbA : (D2D_INACTIVE_KEY | lane), keyB = liveB ? rbB : (D2D_INACTIVE_KEY | 32u | lane);
            const uint32_t srcA = ovfA ? rbA : (D2D_INACTIVE_KEY | lane), srcB = ovfB ? rbB : (D2D_INACTIVE_KEY | 32u | lane);
            d2d_overflow_warp<PLE2, EXACT>(lane, keyA, keyB, srcA, srcB, make_float4(tA.x, tA.y, wA, uA), pB, wB, uB, P.neg_half_ple,
                                           IA, IB, dminA, dminB);
#ifdef D2D_TIMELINE
            ++tl_ovf;
#endif
        }

        // ---- per-link epilogue (simulator.py:93,106-107,110-127,144-154); dead lanes are zeroed ------------------------
        const float2 sA = SPEC ? P.us_cue : d2d_lds64(lkS), sB = SPEC ? P.us_due : d2d_lds64(lkS + 256u);   // (sensitivity, RB bandwidth in MHz)
        const D2DLinkOut oA32 = d2d_link_epilogue_warp(liveA, plA, gA, IA, cA, sA);
        const D2DLinkOut oB32 = d2d_link_epilogue_warp(liveB, plB, gB, IB, cB, sB);
        const bool needA = liveA && d2d_needs_rescue<EXACT, !FULL>(oA32, fminf(dminA, d2A), P);
        const bool needB = liveB && d2d_needs_rescue<EXACT, !FULL>(oB32, fminf(dminB, d2B), P);

        // ---- envs/reward_fn.py:27-44 -----------------------------------------------------------------------------------
        const bool bad = __any_sync(0xffffffffu, liveA && ctA.y != 0u && oA32.cap <= P.min_cap);
        const uint32_t n_act = d2d_redux_add((liveA ? 1u : 0u) + (liveB ? 1u : 0u));
        float cap_sum = oA32.cap + oB32.cap;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) cap_sum += __shfl_xor_sync(0xffffffffu, cap_sum, s);
        const float reward = bad ? -1.0f : cap_sum * d2d_rcp((float)n_act);
        // every lane has read its counters (its capacity fed the reduction above): clear them for the next env
        __syncwarp();
        d2d_sts64_if(lane < R, zero0, 0u, 0u);
        if (!SPEC && R > 32u) d2d_sts64_if(lane + 32u < R, zero0 + 256u, 0u, 0u);

        // ---- rare: fp64 recomputation of flagged links (latency shape: here, replacing the link's values in oA / oB; the
        // reward and the statistics keep the fp32 capacities either way) -------------------------------------------------
        D2DLinkOut oA = oA32, oB = oB32;
        if (D2D_RESCUE_ENABLED && RESCUE_EARLY && __any_sync(0xffffffffu, needA || needB)) {
            const uint32_t keyA = liveA ? rbA : (D2D_INACTIVE_KEY | lane), keyB = liveB ? rbB : (D2D_INACTIVE_KEY | 32u | lane);
            const uint32_t nr = (uint32_t)d2d_rescue_warp<PLE2, EXACT, SPEC, false, !FULL, AR>(P, S, e, lane, jA, keyA, keyB, needA, needB, pA, pB_, tA, pB,
                                                                                                oA, oB, (AR && ar_rst));
            st_resc += ((ep_reset && t == 0u) || (AR && ar_rst)) ? 0u : nr;   // the reset step enters no statistic
#ifdef D2D_TIMELINE
            (tl_waited ? tl_post : tl_pre) += nr;
#endif
        }

        // ---- per-warp statistics; flushed with the warp's LAST env, ahead of the wait and of that env's stores: the reductions
        // commute with every other launch's, and a warp (hence its block's slot) is not retired before its outstanding atomics
        // are acknowledged - issued at the very end they cost 0.3 us per launch of a one-wave batch (profiles/README.md) --------
        if ((!ep_reset || t != 0u) && !(AR && ar_rst)) {                    // the reset step (envs/d2d_env.py:50) earns no reward
            if (P.reward_fn == 0) { st_reward += reward; st_reward2 = fmaf(reward, reward, st_reward2); }
            st_cap += cap_sum;
            st_pen += bad ? 1u : 0u;
            if (AR) ++st_steps;
        }
        if (FLUSH_EARLY && P.stats && last_t && e + 1u == e_end && lane < (RESCUE_EARLY ? 6u : 5u)) {
            // one fire-and-forget fp64 reduction per statistic and warp, spread over the replicas
            const float vf = lane == 0 ? st_reward : lane == 1 ? st_cap : st_reward2;
            const uint32_t vi = lane == 3 ? (AR ? st_steps : (e_end - e0) * (ep_reset ? T - 1u : T))  // env-steps this warp made
                              : lane == 4 ? st_pen : st_resc;
            const double v = lane < 3u ? (double)vf : (double)vi;              // (two conversions instead of six)
            if (v != 0.0) atomicAdd(P.stats + ((blockIdx.x * WPB + warp) % D2D_STATS_REPLICAS) * 8 + lane, v);
        }

        // griddepcontrol.wait: everything above read only inputs (no step kernel writes actions or positions); from here on every
        // earlier kernel's memory is complete.  What is left after it is the step-counter load, the stores and the exit - the part
        // of a launch that cannot overlap its predecessor (profiles/timeline.py).
        // (single-launch d2d_step after a d2d_step of the same geometry: this warp waits for ITS predecessor only - d2d_ticket_wait)
#ifdef D2D_TIMELINE
        if (e == e0 && t == 0u) tl_c1 = d2d_tl_clock();
#endif
        // LATE: the host found that this launch's per-link outputs (observation table, capacities, info) alias nothing its predecessor
        // - another d2d_step of this handle - writes: they go out right away, and the wait moves in front of the only accesses that
        // do depend on the predecessor, the step counters and the per-env scalars of the warp's first group (see below).  At one wave
        // of envs every warp's stores used to queue up behind the grid-wide release.
        const bool LATE = !MANY && !AR && (P.flags & D2D_PF_LATE_WAIT) != 0u;
        if (e == e0 && t == 0u && !LATE) {
            if (!MANY && P.tok_wait != 0ull) {
                if (lane == 0u && !d2d_ticket_wait(P.tickets + (blockIdx.x * WPB + warp), P.tok_wait) && P.stats)
                    atomicAdd(P.stats + 6, 1.0);                           // D2D_STAT_TICKET_TIMEOUTS
                __syncwarp();
            } else {
                d2d_pdl_wait();
            }
        }
#ifdef D2D_TIMELINE
        if (e == e0 && t == 0u) tl_c2 = d2d_tl_clock();
        if (e == e0 && t == 0u && !LATE) tl_waited = true;
#endif
        if (!AR && !LATE && !ep_reset && g == 0u && t == 0u && (FULL || P.step_count)) ns_keep = e + lane < e_end ? (int)P.step_count[e + lane] : 0;   // consumed at the group's end
        // ---- outputs: compact observation table (envs/obs_fn.py:55-61), capacity, optional info.  Rows of absent
        // agents carry their positions and zeros (the reference has no row for them). ---------------------------------
        // (one divergent branch per slot: cheaper than predicating every store, and the two merge when C == D)
        if ((ep_reset && t == 0u) || (AR && ar_rst)) {
            // the drawn positions become the bound state (after the wait: an earlier step kernel may still be reading it)
            float2 *pe = reinterpret_cast<float2 *>(P.pos_out) + (uint64_t)e * V;
            double2 *pe64 = P.pos64 ? reinterpret_cast<double2 *>(const_cast<double *>(P.pos64)) + (uint64_t)e * V : nullptr;
            if (lane == 0u) { pe[0] = make_float2(0.f, 0.f); if (pe64) pe64[0] = make_double2(0.0, 0.0); }     // simulator.py:63-64
            if (hasA) { pe[1u + lane] = tA; if (pe64) pe64[1u + lane] = make_double2((double)tA.x, (double)tA.y); }
            if (hasB) {
                const uint32_t q = 1u + C + 2u * lane;
                pe[q] = make_float2(pB.x, pB.y); pe[q + 1u] = make_float2(pB.z, pB.w);
                if (pe64) { pe64[q] = make_double2((double)pB.x, (double)pB.y); pe64[q + 1u] = make_double2((double)pB.z, (double)pB.w); }
            }
        }
        if (EPI && !EPI_FAST && P.actions_out) {
            if (hasA) P.actions_out[jA] = (int32_t)aA;
            if (hasB) P.actions_out[jB] = (int32_t)aB;
        }
        if (hasA) {
            if (FULL || P.obs) {
                float2 *oa = reinterpret_cast<float2 *>(reinterpret_cast<char *>(P.obs) + (uint64_t)jA * 24u);
                oa[0] = make_float2(tA.x, tA.y); oa[1] = make_float2(0.f, 0.f); oa[2] = make_float2(oA.sinr_dB, oA.snr_dB);
            }
            if (FULL || P.cap) P.cap[jA] = oA.cap;
            if (!FULL) {
                if (P.obs_dyn) P.obs_dyn[jA] = make_float2(oA.sinr_dB, oA.snr_dB);
                if (P.rate) P.rate[jA] = oA.rate;
                if (P.rb_out) P.rb_out[jA] = (int16_t)(liveA ? rbA : 0u);
                if (P.pwr_out) P.pwr_out[jA] = (int16_t)(liveA ? pA : 0u);
            }
        }
        if (hasB) {
            if (FULL || P.obs) {
                float2 *ob = reinterpret_cast<float2 *>(reinterpret_cast<char *>(P.obs) + (uint64_t)jB * 24u);
                ob[0] = make_float2(pB.x, pB.y); ob[1] = make_float2(pB.z, pB.w); ob[2] = make_float2(oB.sinr_dB, oB.snr_dB);
            }
            if (FULL || P.cap) P.cap[jB] = oB.cap;
            if (!FULL) {
                if (P.obs_dyn) P.obs_dyn[jB] = make_float2(oB.sinr_dB, oB.snr_dB);
                if (P.rate) P.rate[jB] = oB.rate;
                if (P.rb_out) P.rb_out[jB] = (int16_t)(liveB ? rbB : 0u);
                if (P.pwr_out) P.pwr_out[jB] = (int16_t)(liveB ? pB_ : 0u);
            }
        }

        // ---- the other shapes: the rare fp64 pass after the env's per-link stores (it overwrites them) ---------------------------
        const auto rescue_late = [&]() {
            if (D2D_RESCUE_ENABLED && !RESCUE_EARLY && __any_sync(0xffffffffu, needA || needB)) {
                const uint32_t keyA = liveA ? rbA : (D2D_INACTIVE_KEY | lane), keyB = liveB ? rbB : (D2D_INACTIVE_KEY | 32u | lane);
                const uint32_t nr = (uint32_t)d2d_rescue_warp_late<PLE2, EXACT, SPEC, !FULL, AR>(P, S, e, lane, jA, keyA, keyB, needA, needB, pA, pB_,
                                                                                                  tA, pB, (AR && ar_rst));
                st_resc += ((ep_reset && t == 0u) || (AR && ar_rst)) ? 0u : nr;
#ifdef D2D_TIMELINE
                (tl_waited ? tl_post : tl_pre) += nr;
#endif
            }
        };
        // d2d_step: right here, before the group end.  A late launch stored the per-link outputs ahead of the wait, so the pass of
        // the env that closes the warp's first group runs ahead of it too: after the wait it was on the critical path of every
        // back-to-back launch of a one-wave batch (profiles/timeline.py).  Its count goes out with the warp's last env, not at the
        // exit, where an outstanding atomic holds the warp's block slot.  (The multi-step modes keep the pass after the group's
        // scalars and the count at the exit: measured faster for d2d_rollout, which has no wait in its loop.)
        if (!MANY) rescue_late();
        if (!MANY && FLUSH_EARLY && !RESCUE_EARLY && P.stats && e + 1u == e_end && lane == 5u && st_resc != 0u)
            atomicAdd(P.stats + ((blockIdx.x * WPB + warp) % D2D_STATS_REPLICAS) * 8 + 5u, (double)st_resc);
        if (MANY && T <= 32u) {
            // per-step scalars: lane t keeps slice t's reward until the env's last step, then T lanes store their slices at once
            // (two strided stores per env instead of two single-lane stores per step)
            rew_keep = lane == t ? reward : rew_keep;
            if (last_t) {
                // num_steps before this launch: lane g of the group holds it (episode: num_steps = 0 at reset, slice 0 uncounted)
                const int ns0 = ep_reset ? -1 : __shfl_sync(0xffffffffu, ns_keep, (int)g);
                if (lane < T) {
                    if (FULL || P.reward) P.reward[lane * strideE + e] = rew_keep;
                    if (FULL || P.done) P.done[lane * strideE + e] = min(ns0 + (int)lane + 1, 255) >= P.episode_length ? 1 : 0;
                }
                if (lane == g) ns_keep = min(ns0 + (int)T, 255);
            }
        } else if (MANY) {
            // (more than 32 steps per launch) per-step scalars straight to slice t (write-only, so partial sectors merge in L2);
            // the step counter stays in the group's registers until the env's last step
            if (lane == g) {
                // EPISODE: num_steps = 0 at reset (envs/d2d_env.py:46) and slice 0 is the uncounted reset step
                const int ns = ep_reset ? (int)min(t, 255u) : min(ns_keep + (int)t + 1, 255);
                if (FULL || P.reward) P.reward[tE + e] = reward;
                if (FULL || P.done) P.done[tE + e] = ns >= P.episode_length ? 1 : 0;
                if (last_t) ns_keep = ns;
            }
        } else {
            rew_keep = lane == g ? ((AR && ar_rst) ? 0.f : reward) : rew_keep;
            if (AR) rs_keep = lane == g ? (AR && ar_rst) : rs_keep;
        }
        if (last_t && (g == 31u || e + 1u == e_end)) {
            if (LATE) {
#ifdef D2D_TIMELINE
                if (e - g == e0) tl_c1 = d2d_tl_clock();
#endif
                if (e - g == e0) d2d_pdl_wait();                       // (the warp's first group: once per warp)
#ifdef D2D_TIMELINE
                if (e - g == e0) { tl_c2 = d2d_tl_clock(); tl_waited = true; }
#endif
                ns_keep = ((FULL || P.step_count) && lane <= g) ? (int)P.step_count[e - g + lane] : 0;
            }
            // envs/d2d_env.py:65,68 for the whole group: num_steps += 1; done = num_steps >= EPISODE_LENGTH
            if (lane <= g) {
                const uint32_t eg = e - g + lane;
                const int ns = MANY ? ns_keep : (AR && rs_keep) ? 0 : min(ns_keep + 1, 255);
                if (FULL || P.step_count) P.step_count[eg] = (uint8_t)ns;
                if (AR && rs_keep) P.episode_index[eg] = ep_keep + 1u;
                if (!MANY && (FULL || P.reward)) P.reward[eg] = rew_keep;
                if (!MANY && (FULL || P.done)) P.done[eg] = ns >= P.episode_length ? 1 : 0;
            }
        }

        if (MANY) rescue_late();
#ifdef D2D_TIMELINE
        tl_env += last_t ? 1u : 0u;
#endif
        if (last_t) {
            g = (g + 1u) & 31u;
            if (e + 1u == e_end) g = 0u;
            t = 0u; tN = 0u; tE = 0u;
            ++e; iA += N;
        } else {
            ++t; tN += strideN; tE += strideE;
        }
        __syncwarp();     // every lane is done with this env's records and counters before the next env's are written
    }

    // this warp's stores are done: publish the launch's token for the same warp slot of the next launch (d2d_ticket_wait).  A warp
    // without envs still has to wait for its predecessor first, or its token could overtake an unfinished one's.
    if (!MANY && P.tok_sign != 0ull) {
        __syncwarp();
        if (lane == 0u) {
            uint64_t *word = P.tickets + (blockIdx.x * WPB + warp);
            if (e0 >= e_end && P.tok_wait != 0ull && !d2d_ticket_wait(word, P.tok_wait) && P.stats) atomicAdd(P.stats + 6, 1.0);
            d2d_ticket_sign(word, P.tok_sign);
        }
    }
#ifdef D2D_TIMELINE
    if (lane == 0u && blockIdx.x * WPB + warp < D2D_TL_WARPS) {
        D2DTlRec r; r.g0 = tl_g0; r.c0 = tl_c0; r.c1 = tl_c1; r.c2 = tl_c2; r.c3 = d2d_tl_clock(); r.smid = d2d_tl_smid();
        r.n_env = tl_env; r.n_pre = tl_pre; r.n_post = tl_post; r.n_ovf = tl_ovf;
        d2d_tl_buf[P.tl_slot & (D2D_TL_SLOTS - 1)][blockIdx.x * WPB + warp] = r;
    }
#endif
    if (!FLUSH_EARLY) {
        if (P.stats && lane < 6u) {
            const float vf = lane == 0 ? st_reward : lane == 1 ? st_cap : st_reward2;
            const uint32_t vi = lane == 3 ? (AR ? st_steps : (e_end - e0) * (ep_reset ? T - 1u : T)) : lane == 4 ? st_pen : st_resc;
            const double v = lane < 3u ? (double)vf : (double)vi;
            if (v != 0.0) atomicAdd(P.stats + ((blockIdx.x * WPB + warp) % D2D_STATS_REPLICAS) * 8 + lane, v);
        }
    } else if (MANY && !RESCUE_EARLY && P.stats && lane == 5u && st_resc != 0u) {
        atomicAdd(P.stats + ((blockIdx.x * WPB + warp) % D2D_STATS_REPLICAS) * 8 + 5u, (double)st_resc);
    }
}
