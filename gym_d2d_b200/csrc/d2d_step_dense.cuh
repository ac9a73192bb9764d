// d2d_step_dense.cuh - fused env.step for 65 <= N <= 1024 links, one thread block per environment, ONE block barrier per env
// (BASELINE config #3: 100 RBs / 100 CUEs / 500 DUE pairs -> N = 600, V = 1101).
//
// Same arithmetic contract as d2d_step_warp.cuh (SURVEY Appendix A; simulator.py:89-154).  What differs from the sorting block
// kernel (d2d_step_block.cuh: count -> scan -> scatter -> walk, four barriers per env) is the same-RB grouping of
// Actions.get_actions_by_rb (actions.py:27-31): like the warp kernel it is a BINNED table - rank = atomicAdd(count[rb]) and the
// link's 16-byte peer record goes straight to bin[rb][rank] - so there is no scan and no scatter pass, and the tables are
// multi-buffered so that consecutive envs overlap inside a block:
//
//   per env e (bins buffer e & 1, counter buffer e % 3):
//     phase 1  take the env's inputs (prefetched into registers one env ahead), decode (envs/d2d_env.py:93-101), rank, record
//     barrier  (the only one)
//     deferred the reward / done / statistics of env e - 1 (its warps' partial sums are complete now), zero env e - 1's counters
//     phase 2  every victim walks its RB's bin (simulator.py:95-101), epilogue, rare warp-cooperative fp64 pass, stores,
//              per-warp partial sums of the reward reduction (envs/reward_fn.py:27-44)
//
// A warp that is still in phase 2 of env e never collides with one that already fills the tables of env e + 1 (other
// buffers); the counters of env e - 1 are cleared after the barrier of env e and reused by env e + 2, after the barrier of
// env e + 1.  A bin holds `bin_cap` records (mean + 4 sigma of the per-RB load, odd so that consecutive bins start on different
// banks); links beyond that (a crowded RB: 0.7 % of the dense envs, or a policy that puts everyone on one RB) go to a
// per-env overflow list that only the victims of an overflowing RB scan; an env that used it ends with a second barrier,
// so the list needs one buffer only.
//
// A record is (tx_x, tx_y, w, who): w = 10^(p/10) 10^((eo-K)/10) is the radiated weight, who = link | Tx power << 16 (read by
// the fp64 pass only).  CUE victims - whose receiver is the MBS - take the same walk as DUE victims with rx = (0, 0).
#pragma once

#include "d2d_common.cuh"

#define D2D_DENSE_MAX_LPT 5
#define D2D_DENSE_MAX_WARPS 16
#define D2D_DENSE_WALK_BAND_DB 0.0075f      // rescue band per sqrt(peer) of a long walk: 2 sqrt(n) ulp of SINR, 1.45x margin to 1e-4
// blocks per SM the register allocation has to allow (80 registers at 256 threads)
#define D2D_DENSE_MINB(BT) ((BT) <= 128 ? 6 : (BT) <= 160 ? 5 : (BT) <= 192 ? 4 : 3)

// What the out-of-line fp64 pass needs of the launch parameters, copied to shared memory once per block: read through the
// reference to the __grid_constant__ parameter struct every field was a generic-address global load - a quarter of the pass's
// cycles were long-scoreboard stalls on them (profiles/README.md), and the block's other warps wait for the pass at the barrier.
struct D2DDenseRC {
    D2DLinkD ud_cue, ud_due;     // the two link types' fp64 constants (uniform)
    double ple_d, thr_d;
    const double *pos64;         // fp64 position shadow or nullptr
    const D2DLinkD *linkD;       // per-link tables (per-device overrides)
    const D2DLinkB *linkB;
    float sens_cue, sens_due, thr_dB, thr_band;
    uint32_t C, V, CAP, uniform;
};

struct D2DDenseLayout {
    uint32_t bins, pwr, pwr_d, cnt, red, sst, rc, mbar, sact, spos, grp, total, cnt_words;
};

__host__ __device__ inline D2DDenseLayout d2d_dense_layout(int N, int R, int cap, int bt, int V) {
    D2DDenseLayout L;
    uint32_t b = 0;
    L.pwr_d = b; b += D2D_MAX_PWR_LEVELS * 8u;                            // 10^(p/10) in fp64 (the fp64 pass)  (fixed offsets first)
    L.pwr = b;   b += D2D_MAX_PWR_LEVELS * 4u;                            // 10^(p/10)
    L.red = b;   b += 2u * 4u * D2D_DENSE_MAX_WARPS * 4u;                 // [2][4][warps]: capacity, acting agents, rescues, penalty
    L.sst = b;   b += 8u * 8u;                                            // the block's statistics (one thread adds to them per env)
    L.rc = b;    b += (uint32_t)((sizeof(D2DDenseRC) + 15u) & ~15u);      // the fp64 pass's constants
    L.mbar = b;  b += 16u;                                                // the staging buffer's mbarrier
    L.sact = b;  b += (((uint32_t)N * 4u + 15u) & ~15u) + 16u;            // the next env's actions: its 16-byte aligned window of the global array
    L.spos = b;  b += (((uint32_t)V * 8u + 15u) & ~15u) + 16u;            // and its V positions
    L.grp = b;   b += 2u * (uint32_t)bt * 4u;                        // [2][BT]: reward and step counter of the envs of the current group of BT
    L.cnt_words = ((uint32_t)R + 2u + 3u) & ~3u;                          // per buffer: R counters (links | SIDELINKs << 16), overflow count
    L.cnt = b;   b += 3u * L.cnt_words * 4u;
    b = (b + 127u) & ~127u;
    L.bins = b;  b += 2u * (uint32_t)R * (uint32_t)cap * 16u;            // [2][R][cap] float4 peer records; 128-byte aligned, cap % 8 == 0
    L.total = b + 112u;                                                   // the kernel rounds the dynamic window's base up to 128 bytes
    return L;
}

// bin capacity for an expected per-RB load of N / R links: mean + 3.5 sigma rounded up to a multiple of 8 (the walk's conflict-free
// rotation works on 128-byte groups of 8 records)
__host__ inline int d2d_dense_bin_cap(int N, int R) {
    const double m = (double)N / (double)(R > 0 ? R : 1);
    int cap = (int)(m + 3.5 * sqrt(m) + 1.0);
    if (cap > N) cap = N;
    if (cap < 8) cap = 8;
    return (cap + 7) & ~7;
}

// interferer record rk's fp64 term at receiver rxd (the cooperative fp64 pass); pwd = the fp64 power table in shared memory
template <bool PLE2>
__device__ __forceinline__ double d2d_dense_term_f64(const float4 rk, const double2 rxd, const double2 *pe64, const double *pwd, const D2DDenseRC &rc) {
    const uint32_t wk = __float_as_uint(rk.w), kk = wk & 0xffffu;
    const double2 tk = pe64 ? pe64[d2d_tx_dev((int)kk, (int)rc.C)] : make_double2((double)rk.x, (double)rk.y);
    const double ex = tk.x - rxd.x, ey = tk.y - rxd.y;
    const double t_lin = rc.uniform ? (kk < rc.C ? rc.ud_cue.t_lin : rc.ud_due.t_lin) : rc.linkD[kk].t_lin;
    return pwd[wk >> 16] * t_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, rc.ple_d);
}

// What the fp64 pass changes of a link's outputs: flag 1 = sinr_dB, 2 = snr_dB, 4 = rate and capacity
struct D2DDenseFix {
    float sinr_dB, snr_dB, rate, cap;
    uint32_t flags;
};

// Warp-cooperative fp64 recomputation of link vj of env e (rb, slot in its bin and Tx power given): the lanes split the RB's
// peer records, a butterfly sums their terms, every lane returns the same result.  Kept out of line: rare, and its fp64
// registers must not count against the hot loop's allocation.
template <bool PLE2, bool THR>
__device__ __noinline__ D2DDenseFix d2d_dense_rescue(const D2DDenseRC &rc, uint32_t e, uint32_t vj, uint32_t vrb, uint32_t vself, uint32_t vpw,
                                                     const float4 *bp, const uint32_t *cn, const float4 *ovrec,
                                                     const uint16_t *ovrb, const double *pwd, uint32_t ovn, uint32_t lane, float vrx_x, float vrx_y) {
    // (without an fp64 shadow of the positions and with uniform link constants the pass reads no global memory: the victim's
    // receiver comes from its lane's registers, the transmitters from the peer records, the tables and constants from shared
    // memory - the pass sits between two block barriers, so its latency is what the other warps wait for)
    const uint32_t C = rc.C, V = rc.V, CAP = rc.CAP;
    const bool exact = rc.pos64 != nullptr;
    const double2 *pe64 = exact ? reinterpret_cast<const double2 *>(rc.pos64) + (int64_t)e * V : nullptr;
    const float4 own = vself < CAP ? bp[vrb * CAP + vself] : ovrec[vself - CAP];                 // the victim's own record: (tx_x, tx_y, ..)
    const double2 txd = exact ? pe64[d2d_tx_dev((int)vj, (int)C)] : make_double2((double)own.x, (double)own.y);
    double2 rxd = make_double2(0.0, 0.0);                                                          // a CUE's receiver: the MBS at the origin
    if (vj >= C) rxd = exact ? pe64[d2d_rx_dev((int)vj, (int)C)] : make_double2((double)vrx_x, (double)vrx_y);
    const uint32_t vn = cn[vrb] & 0xffffu, vnb = min(vn, CAP);
    const float4 *vbase = bp + vrb * CAP;
    double I64 = 0.0;
    for (uint32_t q = lane; q < vnb; q += 32u)
        if (q != vself) I64 += d2d_dense_term_f64<PLE2>(vbase[q], rxd, pe64, pwd, rc);
    if (vn > CAP)
#pragma unroll 1
        for (uint32_t q = lane; q < ovn; q += 32u)
            if (ovrb[q] == (uint16_t)vrb && CAP + q != vself) I64 += d2d_dense_term_f64<PLE2>(ovrec[q], rxd, pe64, pwd, rc);
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1)
        I64 += __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(I64), sh), __shfl_xor_sync(0xffffffffu, __double2loint(I64), sh));
    const D2DLinkD Lj = rc.uniform ? (vj < C ? rc.ud_cue : rc.ud_due) : rc.linkD[vj];
    const float sens = rc.uniform ? (vj < C ? rc.sens_cue : rc.sens_due) : rc.linkB[vj].sens_dBm;
    const double ex = txd.x - rxd.x, ey = txd.y - rxd.y;
    const double Sg = pwd[vpw] * Lj.a_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, rc.ple_d);
    const double r = Sg * d2d_rcp_f64(fma(I64, Lj.inv_noise, 1.0));
    const bool r1 = fabs(r - 1.0) < 0.0625, s1 = fabs(Sg - 1.0) < 0.0625;
    D2DDenseFix f = {0.f, 0.f, 0.f, 0.f, 0u};
    double sinr = 0.0;
    if (exact || r1 || (THR && rc.thr_band > 0.f)) {
        sinr = r1 ? d2d_db_near1(r) : 4.3429448190325182765 * d2d_ln_f64(r);
        float sv = (float)sinr;
        if (THR && rc.thr_band > 0.f) {             // d2d_sinr_store: the fp32 image stays on the float64 value's side of the reward threshold
            const bool ge = sinr >= rc.thr_d;
            if ((sv >= rc.thr_dB) != ge) sv = ge ? rc.thr_dB : nextafterf(rc.thr_dB, -3.0e38f);
        }
        f.sinr_dB = sv; f.flags |= 1u;
    }
    if (exact || s1) { f.snr_dB = (float)(s1 ? d2d_db_near1(Sg) : 4.3429448190325182765 * d2d_ln_f64(Sg)); f.flags |= 2u; }
    if (exact || (r1 && fabsf(sens) < 0.5f)) {
        const double rate = sinr > (double)sens ? 1.4426950408889634074 * d2d_ln_f64(1.0 + r) : 0.0;
        f.rate = (float)rate; f.cap = (float)(Lj.bw_MHz * rate); f.flags |= 4u;
    }
    return f;
}

// FULL: exactly the core outputs (obs, capacity, reward, done) and the step counters are bound and every link of a type shares
// one set of constants (no per-device overrides) - the VecD2DEnv default - so the hot path tests no pointer and selects its
// constants from the constant bank.  EXACT: an fp64 shadow of the positions is bound (the fp64 pass then needs d_min).
#define D2D_DENSE_SPEC_N 600u
#define D2D_DENSE_SPEC_C 100u
#define D2D_DENSE_SPEC_R 100u
#define D2D_DENSE_SPEC_CAP 16u
template <bool PLE2, int LPT, int BT, bool FULL, bool EXACT, bool SPEC = false>
__global__ void __launch_bounds__(BT, D2D_DENSE_MINB(BT)) d2d_step_dense_kernel(const __grid_constant__ D2DParams P) {
    extern __shared__ __align__(16) unsigned char d2d_dense_smem[];
    constexpr uint32_t NW = BT / 32;
    // SPEC: BASELINE config #3 itself (100 RBs / 100 CUEs / 500 DUE pairs, the reference's default power levels: envs/env_config.py:12-27,
    // envs/d2d_env.py:31-35) with every count, stride, shared-memory offset and division magic an immediate - and, because no link of
    // a thread's second slot can be a CUE, that slot's code without the link-type selects: 738 -> 666 us
    const uint32_t N = SPEC ? D2D_DENSE_SPEC_N : (uint32_t)P.N, C = SPEC ? D2D_DENSE_SPEC_C : (uint32_t)P.C,
                   V = SPEC ? 1u + D2D_DENSE_SPEC_C + 2u * (D2D_DENSE_SPEC_N - D2D_DENSE_SPEC_C) : (uint32_t)P.V,
                   R = SPEC ? D2D_DENSE_SPEC_R : (uint32_t)P.R, CAP = SPEC ? D2D_DENSE_SPEC_CAP : (uint32_t)P.bin_cap;
    const uint32_t npc = SPEC ? 24u : (uint32_t)P.n_pwr_cue, npd = SPEC ? 21u : (uint32_t)P.n_pwr_due;
    const uint32_t mgc = SPEC ? 178956971u : P.magic_cue, mgd = SPEC ? 204522253u : P.magic_due;      // ceil(2^32 / 24), ceil(2^32 / 21)
    const uint32_t n1c = SPEC ? 0u : P.npw1_cue, n1d = SPEC ? 0u : P.npw1_due;
    const D2DDenseLayout L = d2d_dense_layout((int)N, (int)R, (int)CAP, BT, (int)V);
    // the bins sit on 128-byte boundaries of the shared window (see the walk): round the dynamic region's base up
    unsigned char *const sm = d2d_dense_smem + ((0u - (uint32_t)__cvta_generic_to_shared(d2d_dense_smem)) & 127u);
    float4 *bins = reinterpret_cast<float4 *>(sm + L.bins);
    // the overflow list of a crowded RB's links lives in a handle-owned global scratch (N records per block; L2-resident and
    // touched by 2-3 % of the envs): in shared memory it cost 11 KB
    float4 *ovrec = reinterpret_cast<float4 *>(P.dense_ovf) + (uint64_t)blockIdx.x * N;
    uint16_t *ovrb = reinterpret_cast<uint16_t *>(reinterpret_cast<float4 *>(P.dense_ovf) + (uint64_t)gridDim.x * N) + (uint64_t)blockIdx.x * N;
    float *pwr = reinterpret_cast<float *>(sm + L.pwr);
    double *pwd = reinterpret_cast<double *>(sm + L.pwr_d);
    uint32_t *cnt = reinterpret_cast<uint32_t *>(sm + L.cnt);
    float *red = reinterpret_cast<float *>(sm + L.red);
    // block-level scalars in shared memory rather than in registers that would live across the whole env loop (and spill):
    // the statistics of the envs this block stepped, and the reward / step counter of every env of the current group
    double *sst = reinterpret_cast<double *>(sm + L.sst);
    float *grew = reinterpret_cast<float *>(sm + L.grp);
    int32_t *gns = reinterpret_cast<int32_t *>(sm + L.grp) + BT;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint32_t sact_sa = (uint32_t)__cvta_generic_to_shared(sm + L.sact), spos_sa = (uint32_t)__cvta_generic_to_shared(sm + L.spos);
    const uint32_t mbar_sa = (uint32_t)__cvta_generic_to_shared(sm + L.mbar);
    d2d_pdl_entry(P.flags);

    for (uint32_t i = tid; i < D2D_MAX_PWR_LEVELS; i += BT) { pwr[i] = P.pwr_lin[i]; pwd[i] = P.pwr_lin_d[i]; }
    for (uint32_t i = tid; i < 3u * L.cnt_words; i += BT) cnt[i] = 0u;
    if (tid < 8u) sst[tid] = 0.0;
    D2DDenseRC *rcs = reinterpret_cast<D2DDenseRC *>(sm + L.rc);
    if (tid == 32u) {
        rcs->ud_cue = P.ud_cue; rcs->ud_due = P.ud_due; rcs->ple_d = P.ple_d; rcs->thr_d = P.thr_d; rcs->pos64 = P.pos64;
        rcs->linkD = P.linkD; rcs->linkB = P.linkB; rcs->sens_cue = P.us_cue.x; rcs->sens_due = P.us_due.x; rcs->thr_dB = P.thr_dB;
        rcs->thr_band = P.thr_band; rcs->C = C; rcs->V = V; rcs->CAP = CAP; rcs->uniform = (uint32_t)P.uniform;
    }
    bool has[LPT], cue[LPT];
#pragma unroll
    for (int k = 0; k < LPT; ++k) {
        const uint32_t j = tid + k * BT;
        has[k] = j < N; cue[k] = j < C && !(SPEC && k * BT >= (int)D2D_DENSE_SPEC_C);
    }
    // link constants (tx_lin0, a_lin, inv_noise, snr0_dB) and (sens, bw): one set per link type from the constant bank unless
    // a device-config file overrode single devices (then the per-link tables, through L1)
    auto link_cA = [&](uint32_t j, bool is_cue) -> float4 {
        return (FULL || P.uniform) ? (is_cue ? P.u_cue : P.u_due) : __ldg(reinterpret_cast<const float4 *>(P.linkA) + j);
    };
    auto link_sB = [&](uint32_t j, bool is_cue) -> float2 {
        return (FULL || P.uniform) ? (is_cue ? P.us_cue : P.us_due) : __ldg(reinterpret_cast<const float2 *>(P.linkB + j));
    };
    // The next env's inputs - N actions, V positions: two contiguous rows of the global arrays - are STAGED in shared memory one
    // env ahead by the bulk-copy engine: thread 0 issues one cp.async.bulk per row for the row's 16-byte aligned interior and
    // 4-byte cp.asyncs for the (at most three) words on either side of it, and every thread waits for both on an mbarrier at the
    // top of phase 1.  Nothing is prefetched into registers: held there across the walk the values were what the compiler spilled at
    // the kernel's 64-register cap - with the spill store waiting for the load right behind its issue (20 % of all stall
    // samples) - and 60 LDG with their 64-bit address arithmetic per env are gone.  A row keeps its alignment modulo 16 in the
    // staging buffer (element i of the row at buffer + (row address & 15) + i * size).
    auto stage_row = [&](const char *row, uint32_t bytes, uint32_t dst_sa) -> uint32_t {      // thread 0; returns the bulk copy's bytes
        const uint64_t a0 = (uint64_t)row, a1 = a0 + bytes;
        const uint64_t w0 = (a0 + 15ull) & ~15ull, w1 = a1 & ~15ull;
        const uint32_t d0 = dst_sa + ((uint32_t)a0 & 15u);
        for (uint64_t x = a0; x < (w0 < a1 ? w0 : a1); x += 4ull)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + (uint32_t)(x - a0)), "l"(x) : "memory");
        for (uint64_t x = (w1 > w0 ? w1 : w0); x < a1; x += 4ull)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + (uint32_t)(x - a0)), "l"(x) : "memory");
        return w1 > w0 ? (uint32_t)(w1 - w0) : 0u;
    };
    auto stage_inputs = [&](uint32_t e) {
        if (tid == 0u) {
            const char *arow = reinterpret_cast<const char *>(P.actions + (uint64_t)e * N), *prow = reinterpret_cast<const char *>(P.pos) + (uint64_t)e * V * 8ull;
            const uint32_t ba = stage_row(arow, N * 4u, sact_sa), bpz = stage_row(prow, V * 8u, spos_sa);
            // two arrivals complete a phase: this thread's word copies (cp.async; fires at once when there were none) and the
            // expect_tx one, which the bulk copies' bytes then complete
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(mbar_sa) : "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar_sa), "r"(ba + bpz) : "memory");
            if (ba) {
                const uint64_t w0 = ((uint64_t)arow + 15ull) & ~15ull;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(sact_sa + ((uint32_t)(uint64_t)arow & 15u) + (uint32_t)(w0 - (uint64_t)arow)), "l"(w0), "r"(ba), "r"(mbar_sa) : "memory");
            }
            if (bpz) {
                const uint64_t w0 = ((uint64_t)prow + 15ull) & ~15ull;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(spos_sa + ((uint32_t)(uint64_t)prow & 15u) + (uint32_t)(w0 - (uint64_t)prow)), "l"(w0), "r"(bpz), "r"(mbar_sa) : "memory");
            }
        }
    };
    auto staged_wait = [&](uint32_t parity) {
        uint32_t done = 0u;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(mbar_sa), "r"(parity) : "memory");
    };
    const uint32_t num_envs = (uint32_t)P.num_envs;
    const uint32_t per_block = (num_envs + gridDim.x - 1u) / gridDim.x;
    const uint32_t e0 = min(blockIdx.x * per_block, num_envs), e_end = min(e0 + per_block, num_envs);
    uint32_t g = 0;                  // position of the env in its group of BT

    // reward / statistics of env `ep` (buffer pb of red), by the thread that owns it; the group's scalars when it is complete
    auto finalise = [&](uint32_t ep, uint32_t gp, bool flush) {
        if (tid == gp) {
            const float *rd = red + (ep & 1u) * 4u * D2D_DENSE_MAX_WARPS;
            float cs = 0.f, na = 0.f, rs = 0.f, bd = 0.f;
#pragma unroll
            for (uint32_t w2 = 0; w2 < NW; ++w2) {
                cs += rd[w2]; na += rd[D2D_DENSE_MAX_WARPS + w2]; rs += rd[2 * D2D_DENSE_MAX_WARPS + w2]; bd += rd[3 * D2D_DENSE_MAX_WARPS + w2];
            }
            const bool any_bad = bd != 0.f;
            const float reward = any_bad ? -1.0f : cs / na;
            grew[gp] = reward;
            // (one thread per env, and consecutive envs' threads are a barrier apart: plain read-modify-writes)
            if (P.reward_fn == 0) { sst[0] += (double)reward; sst[2] += (double)reward * (double)reward; }
            sst[1] += (double)cs;
            sst[3] += 1.0; sst[4] += any_bad ? 1.0 : 0.0; sst[5] += (double)rs;
        }
        if (flush) {
            __syncthreads();                                     // (block-uniform) the last env's reward is in grew
            if (tid <= gp) {
                // envs/d2d_env.py:65,68 for the whole group: num_steps += 1; done = num_steps >= EPISODE_LENGTH
                const uint32_t eg = ep - gp + tid;
                const int ns = min(gns[tid] + 1, 255);
                if (FULL || P.step_count) P.step_count[eg] = (uint8_t)ns;
                if (FULL || P.reward) P.reward[eg] = grew[tid];
                if (FULL || P.done) P.done[eg] = ns >= P.episode_length ? 1 : 0;
            }
        }
    };

    if (tid == 0u) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 2;" ::"r"(mbar_sa) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (e0 < e_end) stage_inputs(e0);
    __syncthreads();
    // (griddepcontrol.wait comes before the first access to memory an earlier step wrote - see d2d_step_warp.cuh)

    uint32_t c3 = 0;                 // e % 3 without the division
    for (uint32_t e = e0; e < e_end; ++e) {
        uint32_t *cn = cnt + c3 * L.cnt_words;
        float4 *bp = bins + (e & 1u) * R * CAP;

        // ---- phase 1: inputs (the next env's loads go out first), decode, rank inside the RB, peer record --------------------
        uint32_t a[LPT];
        float2 tx[LPT], rx[LPT];
        staged_wait((e - e0) & 1u);
        {
            const uint32_t sa = sact_sa + ((uint32_t)(uint64_t)(P.actions + (uint64_t)e * N) & 15u);
            const uint32_t sp = spos_sa + ((uint32_t)((uint64_t)P.pos + (uint64_t)e * V * 8ull) & 15u);
#pragma unroll
            for (int k = 0; k < LPT; ++k) {
                const uint32_t j = min(tid + k * BT, N - 1u);         // (a thread without a link in slot k re-reads the last link and never uses it)
                const uint32_t txd = cue[k] ? 1u + j : 1u + C + 2u * (j - C);
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(a[k]) : "r"(sa + j * 4u) : "memory");
                asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(tx[k].x), "=f"(tx[k].y) : "r"(sp + txd * 8u) : "memory");
                asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(rx[k].x), "=f"(rx[k].y) : "r"(sp + (cue[k] ? 0u : txd + 1u) * 8u) : "memory");      // a CUE's receiver: the MBS (device 0)
            }
        }
        // what phase 2 needs of a link besides its positions, in ONE register (the kernel runs at its 64-register cap):
        // rb | Tx power << 9 | slot in the bin (or bin_cap + place in the overflow list) << 16 | valid action << 31
        float d2own[LPT];
        uint32_t st[LPT];
        // (griddepcontrol.wait comes before the first access to memory an earlier step wrote or read: this phase already stores
        // the position columns of the env's observation rows, which do not depend on the step)
        if (e == e0) d2d_pdl_wait();
#pragma unroll
        for (int k = 0; k < LPT; ++k) {
            const uint32_t j = tid + k * BT;
            const uint32_t npw = cue[k] ? npc : npd;
            {
                const float dxo = tx[k].x - rx[k].x, dyo = tx[k].y - rx[k].y;       // own link (a CUE's receiver is the MBS at the origin)
                d2own[k] = fmaf(dxo, dxo, dyo * dyo);
            }
            if (has[k] && (FULL || P.obs)) {
                float2 *ob = reinterpret_cast<float2 *>(reinterpret_cast<char *>(P.obs) + (uint64_t)(e * N + j) * 24u);
                ob[0] = tx[k];                                       // an absent agent's row keeps its positions (sinr = snr = 0)
                ob[1] = rx[k];
            }
            const bool lv = has[k] && a[k] < R * npw;             // valid actions: 0 <= a < R n_pwr (envs/d2d_env.py:36-40)
            const uint32_t as = lv ? a[k] : 0u;
            const uint32_t rbk = __umulhi(as, cue[k] ? mgc : mgd) + (as & (cue[k] ? n1c : n1d));
            const uint32_t pwk = as - rbk * npw;
            const float plk = lv ? pwr[pwk] : 0.0f;
            uint32_t sq = 0u;
            if (lv) {
                const uint32_t rank = atomicAdd(&cn[rbk], cue[k] ? 1u : 0x10001u) & 0xffffu;      // high half counts the SIDELINKs
                const float4 rec = make_float4(tx[k].x, tx[k].y, plk * link_cA(j, cue[k]).x, __uint_as_float(j | (pwk << 16)));
                if (rank < CAP) {
                    sq = rank;
                    bp[rbk * CAP + rank] = rec;
                } else {                                                                         // crowded RB: the env's overflow list
                    const uint32_t s = atomicAdd(&cn[R], 1u);
                    sq = CAP + s;
                    ovrec[s] = rec;
                    ovrb[s] = (uint16_t)rbk;
                }
            }
            st[k] = rbk | (pwk << 9) | (sq << 16) | (lv ? 0x80000000u : 0u);
        }
        __syncthreads();

        // ---- deferred: env e - 1 is complete (every warp's partial sums are in), its counters can go ------------------------
        if (e > e0) finalise(e - 1u, g == 0u ? BT - 1u : g - 1u, g == 0u);
        if (g == 0u) gns[tid] = ((FULL || P.step_count) && e + tid < e_end) ? (int)P.step_count[e + tid] : 0;   // consumed at the group's flush
        {
            uint32_t *cprev = cnt + (c3 == 0u ? 2u : c3 - 1u) * L.cnt_words;
            for (uint32_t i = tid; i <= R; i += BT) cprev[i] = 0u;
        }
        const uint32_t ovn = cn[R];                               // block-uniform: the env spilled into the overflow list
        // the next env's inputs: in flight during this env's walk (issued here rather than before phase 1: the previous env's
        // stores, which read the registers these loads reuse, have drained by now)
        if (e + 1u < e_end) stage_inputs(e + 1u);

        // ---- phase 2: interference walk (simulator.py:95-101), epilogue, outputs --------------------------------------------------
        float cap_part = 0.0f;
        float capk[LPT];
        uint32_t n_act = 0, resc = 0, badbits = 0, needbits = 0;     // needbits: bit k = slot k needs the fp64 pass, bit 8 + k = it is a CUE sharing its RB with a SIDELINK
#pragma unroll
        for (int k = 0; k < LPT; ++k) {
            const uint32_t j = tid + k * BT;
            const bool lv = (int32_t)st[k] < 0;
            const uint32_t rbk = st[k] & 0x1ffu, pwk = (st[k] >> 9) & 0x7fu, sq = (st[k] >> 16) & 0x7fffu;
            D2DLinkOut o = {0.f, 0.f, 0.f, 0.f};
            bool need = false, side = false;
            float2 sBk = make_float2(0.f, 0.f);
            // The walk (simulator.py:95-101).  A record's 16-byte bank group is its slot modulo 8 (bins start on 128-byte boundaries),
            // whatever the RB.  Lane l therefore visits the 8 slots of a group in the order (l & 7) ^ i: in every iteration the
            // eight lanes of a quarter-warp - the unit LDS.128 is served in - read eight different bank groups, so the random
            // RBs of a warp's 32 victims cost no bank conflicts (in slot order they cost 6.2 wavefronts per load where 2.6
            // would do).  Slots 8.. are taken four at a time, and only while some lane of the warp still has records there.
            uint32_t pb = 0u, pend = 0u, pself = 0u, n = 0u;
            if (lv) {
                const uint32_t cw = cn[rbk];
                n = cw & 0xffffu;
                side = (cw >> 16) != 0u;
                pb = (uint32_t)__cvta_generic_to_shared(bp + rbk * CAP);
                pend = pb + min(n, CAP) * 16u; pself = pb + sq * 16u;
            }
            float I = 0.0f, dmin2 = 3.0e38f;
            {
                uint64_t nrx;                                                   // (-rx.x, -rx.y) for the packed subtract
                asm("mov.b64 %0, {%1, %2};" : "=l"(nrx) : "f"(-rx[k].x), "f"(-rx[k].y));
                auto term = [&](uint32_t pa) {
                    if (pa < pend) {
                        float4 rk;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(rk.x), "=f"(rk.y), "=f"(rk.z), "=f"(rk.w) : "r"(pa));
                        uint64_t t, dd;
                        float qx, qy;
                        asm("mov.b64 %0, {%1, %2};" : "=l"(t) : "f"(rk.x), "f"(rk.y));
                        asm("add.rn.f32x2 %0, %1, %2;" : "=l"(dd) : "l"(t), "l"(nrx));
                        asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(dd) : "l"(dd));
                        asm("mov.b64 {%0, %1}, %2;" : "=f"(qx), "=f"(qy) : "l"(dd));
                        const float d2 = qx + qy;
                        const float gq = d2d_gain<PLE2>(d2, P.neg_half_ple);
                        I = fmaf(rk.z, pa == pself ? 0.0f : gq, I);
                        if (EXACT) dmin2 = fminf(dmin2, d2);
                    }
                };
                const uint32_t rot8 = (lane & 7u) << 4, rot4 = (lane & 3u) << 4;
#pragma unroll
                for (uint32_t i = 0; i < 8u; ++i) term(pb | (rot8 ^ (i << 4)));
                for (uint32_t base = 128u; base < CAP * 16u; base += 64u) {
                    if (!__any_sync(0xffffffffu, pb + base < pend)) break;
#pragma unroll
                    for (uint32_t i = 0; i < 4u; ++i) term((pb + base) | (rot4 ^ (i << 4)));
                }
            }
            if (lv) {
                if (n > CAP) {
#pragma unroll 1
                    for (uint32_t q = 0; q < ovn; ++q) {
                        if (ovrb[q] != (uint16_t)rbk || CAP + q == sq) continue;
                        const float4 rk = ovrec[q];
                        const float dx = rk.x - rx[k].x, dy = rk.y - rx[k].y;
                        const float d2 = fmaf(dx, dx, dy * dy);
                        I = fmaf(rk.z, d2d_gain<PLE2>(d2, P.neg_half_ple), I);
                        dmin2 = fminf(dmin2, d2);
                    }
                }
                const float gown = d2d_gain<PLE2>(d2own[k], P.neg_half_ple);
                sBk = link_sB(j, cue[k]);
                o = d2d_link_epilogue<PLE2>((int)pwk, pwr[pwk] /* 10^(p/10) again: a table read costs less than a register held across the barrier */, gown, gown, I, link_cA(j, cue[k]), sBk, P);
                need = D2D_RESCUE_ENABLED && d2d_needs_rescue<EXACT, !FULL>(o, fminf(dmin2, d2own[k]), P);
                // the fp32 running sum over n peers drifts by ~sqrt(n) ulp: on crowded RBs the band widens with the walk
                // (n = 1024: 0.24 dB, where the pass still rewrites the SINR; DESIGN.md 4.4)
                if (D2D_RESCUE_ENABLED && n > 64u && fabsf(o.sinr_dB) < D2D_DENSE_WALK_BAND_DB * sqrtf((float)n)) need = true;
            }
            if (lv) {
                cap_part += o.cap;
                ++n_act;
                if (cue[k] && side && o.cap <= P.min_cap) badbits |= 1u << k;      // envs/reward_fn.py:30-39
                if (need) needbits |= 1u << k;
                if (cue[k] && side) needbits |= 0x100u << k;
            }
            capk[k] = o.cap;
            if (has[k]) {
                const uint32_t gi = e * N + j;
                if (FULL || P.obs) {
                    float2 *ob = reinterpret_cast<float2 *>(reinterpret_cast<char *>(P.obs) + (uint64_t)gi * 24u);
                    ob[2] = make_float2(o.sinr_dB, o.snr_dB);
                }
                if (FULL || P.cap) P.cap[gi] = o.cap;
                if (!FULL) {
                    if (P.obs_dyn) P.obs_dyn[gi] = make_float2(o.sinr_dB, o.snr_dB);
                    if (P.rate) P.rate[gi] = o.rate;
                    if (P.rb_out) P.rb_out[gi] = lv ? (int16_t)rbk : (int16_t)0;
                    if (P.pwr_out) P.pwr_out[gi] = lv ? (int16_t)pwk : (int16_t)0;
                }
            }
        }

        // ---- rare fp64 pass (d2d_common.cuh; same policy as d2d_rescue_warp): ~0.2 % of the links, about one per dense env.
        // The victim's warp takes it together - its lanes split the RB's peer records, a butterfly sums their terms - so the
        // block's other warps are not held up at the next barrier by one thread's serial fp64 loop.  The victim's lane then
        // rewrites (after its own stores above) what fp32 could not deliver.
        if (D2D_RESCUE_ENABLED && __any_sync(0xffffffffu, (needbits & 0xffu) != 0u)) {
#pragma unroll
            for (int k = 0; k < LPT; ++k) {
                uint32_t mask = __ballot_sync(0xffffffffu, (needbits >> k) & 1u);
                while (mask) {
                    const int src = __ffs((int)mask) - 1;
                    mask &= mask - 1u;
                    ++resc;
                    const uint32_t vj = (tid - lane) + (uint32_t)src + k * BT;
                    const uint32_t vst = __shfl_sync(0xffffffffu, st[k], src);
                    const D2DDenseFix f = d2d_dense_rescue<PLE2, !FULL>(*rcs, e, vj, vst & 0x1ffu, (vst >> 16) & 0x7fffu, (vst >> 9) & 0x7fu, bp, cn, ovrec, ovrb, pwd, ovn, lane,
                                                                 __shfl_sync(0xffffffffu, rx[k].x, src), __shfl_sync(0xffffffffu, rx[k].y, src));
                    if ((int)lane == src) {
                        const uint64_t gi = (uint64_t)e * N + vj;
                        if ((f.flags & 1u) && (FULL || P.obs)) P.obs[gi * 6u + 4u] = f.sinr_dB;
                        if ((f.flags & 2u) && (FULL || P.obs)) P.obs[gi * 6u + 5u] = f.snr_dB;
                        if (!FULL && P.obs_dyn) {
                            if (f.flags & 1u) P.obs_dyn[gi].x = f.sinr_dB;
                            if (f.flags & 2u) P.obs_dyn[gi].y = f.snr_dB;
                        }
                        if (f.flags & 4u) {
                            if (FULL || P.cap) P.cap[gi] = f.cap;
                            if (!FULL && P.rate) P.rate[gi] = f.rate;
                            cap_part += f.cap - capk[k];
                            badbits &= ~(1u << k);
                            if (((needbits >> (8 + k)) & 1u) && f.cap <= P.min_cap) badbits |= 1u << k;
                        }
                    }
                }
            }
        }

        // ---- per-warp partial sums of the reward reduction (envs/reward_fn.py:27-44); the env's owner adds them up after the
        // next barrier (finalise) ----------------------------------------------------------------------------------------------------
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) cap_part += __shfl_xor_sync(0xffffffffu, cap_part, s);
        const uint32_t n_act_w = __reduce_add_sync(0xffffffffu, n_act);
        const bool bad_w = __any_sync(0xffffffffu, badbits != 0u);
        if (lane == 0) {
            float *rd = red + (e & 1u) * 4u * D2D_DENSE_MAX_WARPS;
            rd[warp] = cap_part; rd[D2D_DENSE_MAX_WARPS + warp] = (float)n_act_w;
            rd[2 * D2D_DENSE_MAX_WARPS + warp] = (float)resc; rd[3 * D2D_DENSE_MAX_WARPS + warp] = bad_w ? 1.f : 0.f;     // resc is warp-uniform
        }
        if (ovn != 0u) __syncthreads();      // the overflow list has one buffer: everybody is done with it before the next env fills it
        g = g + 1u == BT ? 0u : g + 1u;
        c3 = c3 == 2u ? 0u : c3 + 1u;
    }
    __syncthreads();
    if (e_end > e0) finalise(e_end - 1u, g == 0u ? BT - 1u : g - 1u, true);

    if (P.stats) {
        // block totals of the six statistics -> one fp64 atomic each
        __syncthreads();
        if (tid < 6 && sst[tid] != 0.0) atomicAdd(P.stats + (blockIdx.x % D2D_STATS_REPLICAS) * 8 + tid, sst[tid]);
    }
}
