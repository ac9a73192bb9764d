// d2d_step_block.cuh - fused env.step, one thread block per environment, for N > 64 links
// (BASELINE config #3: 100 RBs / 100 CUEs / 500 DUE pairs -> N = 600, V = 1101).
//
// Same arithmetic contract as d2d_step_warp.cuh.  The same-RB grouping of Actions.get_actions_by_rb
// (actions.py:27-31) is a shared-memory counting sort by RB: count -> exclusive scan -> scatter; each
// victim link then walks its own bin (expected N/R peers) instead of all N links, so the work per
// env-step is O(N + N^2/R) pair evaluations, like the reference, not the dense N*Q product.
//
// Two kernels: d2d_step_block_kernel<PLE2, LPT> keeps a thread's <= LPT links in registers between the phases and
// scatters full peer records (N <= 256 LPT, LPT <= 4: every configuration up to 1024 links, incl. config #3);
// d2d_step_block_generic_kernel stages everything in shared memory, takes any N <= 65535 and any link topology (each
// link's transmitter / receiver device and action space come from tables): it also serves envs with DOWNLINK actions.
#pragma once

#include "d2d_common.cuh"

#define D2D_BLOCK_THREADS 256

// dynamic shared memory layout (sizes depend on N and nbins), see d2d_block_smem_bytes()
struct D2DBlockSmemView {
    float4 *rec;       // [N] (tx_x, tx_y, w, key)
    float4 *aux;       // [N] (rx_x, rx_y, p_lin, p as int bits)
    float4 *linkA;     // [N]
    float4 *linkB;     // [N]
    float *pwr_lin;    // [D2D_MAX_PWR_LEVELS]
    int32_t *bin_cnt;  // [nbins]
    int32_t *bin_off;  // [nbins]
    int32_t *slot;     // [N] position of the link inside its bin
    uint16_t *sorted;  // [N] link indices grouped by bin
    float *red;        // [32] reduction scratch
};

__host__ __device__ inline size_t d2d_block_smem_bytes(int N, int nbins) {
    size_t b = 0;
    b += (size_t)4 * N * sizeof(float4);
    b += D2D_MAX_PWR_LEVELS * sizeof(float);
    b += (size_t)2 * nbins * sizeof(int32_t);
    b += (size_t)N * sizeof(int32_t);
    b += 32 * sizeof(float);
    b += ((size_t)N * sizeof(uint16_t) + 15) & ~(size_t)15;
    return b;
}

__device__ __forceinline__ D2DBlockSmemView d2d_block_carve(unsigned char *raw, int N, int nbins) {
    D2DBlockSmemView v;
    v.rec = reinterpret_cast<float4 *>(raw);
    v.aux = v.rec + N;
    v.linkA = v.aux + N;
    v.linkB = v.linkA + N;
    v.pwr_lin = reinterpret_cast<float *>(v.linkB + N);
    v.bin_cnt = reinterpret_cast<int32_t *>(v.pwr_lin + D2D_MAX_PWR_LEVELS);
    v.bin_off = v.bin_cnt + nbins;
    v.slot = v.bin_off + nbins;
    v.red = reinterpret_cast<float *>(v.slot + N);
    v.sorted = reinterpret_cast<uint16_t *>(v.red + 32);
    return v;
}

template <bool PLE2>
__global__ void __launch_bounds__(D2D_BLOCK_THREADS) d2d_step_block_generic_kernel(const D2DParams P) {
    extern __shared__ __align__(16) unsigned char d2d_smem_raw[];
    const int N = P.N, V = P.V, nbins = P.nbins;
    D2DBlockSmemView S = d2d_block_carve(d2d_smem_raw, N, nbins);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    d2d_pdl_entry(P.flags);

    for (int i = tid; i < N; i += D2D_BLOCK_THREADS) {
        S.linkA[i] = reinterpret_cast<const float4 *>(P.linkA)[i];
        S.linkB[i] = reinterpret_cast<const float4 *>(P.linkB)[i];
    }
    for (int i = tid; i < D2D_MAX_PWR_LEVELS; i += D2D_BLOCK_THREADS) S.pwr_lin[i] = P.pwr_lin[i];

    double st_reward = 0.0, st_cap = 0.0, st_reward2 = 0.0, st_pen = 0.0, st_resc = 0.0, st_n = 0.0;
    d2d_pdl_wait();

    for (int64_t e = blockIdx.x; e < P.num_envs; e += gridDim.x) {
        const int32_t *act = P.actions + e * N;
        const float2 *pe = reinterpret_cast<const float2 *>(P.pos) + e * V;
        const uint64_t genv = P.first_global_env + (uint64_t)e;         // ShadowingPathLoss draws are keyed by the global env
        for (int i = tid; i < nbins; i += D2D_BLOCK_THREADS) S.bin_cnt[i] = 0;
        __syncthreads();

        // phase 1: decode (envs/d2d_env.py:93-101), stage link records, count links per RB bin.  Transmitter / receiver
        // devices and the action space's power levels come from the link tables (envs/d2d_env.py:80-91: by tx membership)
        for (int j = tid; j < N; j += D2D_BLOCK_THREADS) {
            const int meta = P.link_meta[j], npw = meta & 0xffff;
            const int txd = __float_as_int(S.linkB[j].z), rxd = __float_as_int(S.linkB[j].w);
            const int a = __ldg(act + j);
            const float2 t = __ldg(pe + txd), r = __ldg(pe + rxd);
            const bool active = a >= 0 && a < P.R * npw;         // valid actions: 0 <= a < R n_pwr (envs/d2d_env.py:36-40)
            const int rb = active ? a / npw : 0, p = active ? a - rb * npw : 0;
            // key: the RB, bit 29 marks a SIDELINK (reward_fn.py:31-37); absent agents get a key nobody shares
            const uint32_t key = active ? (uint32_t)rb | ((uint32_t)(meta >> 16) << 29) : (D2D_INACTIVE_KEY | (uint32_t)j);
            const float pl = active ? S.pwr_lin[p & (D2D_MAX_PWR_LEVELS - 1)] : 0.0f;
            S.rec[j] = make_float4(t.x, t.y, pl * S.linkA[j].x, __uint_as_float(key));
            S.aux[j] = make_float4(r.x, r.y, pl, __int_as_float(active ? p : -1));
            if (active) S.slot[j] = atomicAdd(&S.bin_cnt[rb % nbins], 1);
        }
        __syncthreads();

        // exclusive scan of the bin counts (first warp; nbins is small)
        if (warp == 0) {
            const int chunk = (nbins + 31) >> 5, lo = lane * chunk, hi = min(lo + chunk, nbins);
            int sum = 0;
            for (int i = lo; i < hi; ++i) sum += S.bin_cnt[i];
            int incl = sum;
#pragma unroll
            for (int s = 1; s < 32; s <<= 1) {
                const int n = __shfl_up_sync(0xffffffffu, incl, s);
                if (lane >= s) incl += n;
            }
            int run = incl - sum;
            for (int i = lo; i < hi; ++i) { S.bin_off[i] = run; run += S.bin_cnt[i]; }
        }
        __syncthreads();
        for (int j = tid; j < N; j += D2D_BLOCK_THREADS) {
            const uint32_t key = __float_as_uint(S.rec[j].w);
            if (!(key & D2D_INACTIVE_KEY)) S.sorted[S.bin_off[(key & 0x1fffffffu) % (uint32_t)nbins] + S.slot[j]] = (uint16_t)j;
        }
        __syncthreads();

        // phase 2: per-victim interference walk + epilogue + outputs
        float cap_part = 0.0f;
        int n_act = 0, bad = 0, resc = 0;
        for (int j = tid; j < N; j += D2D_BLOCK_THREADS) {
            const float4 rj = S.rec[j], xj = S.aux[j];
            const uint32_t key = __float_as_uint(rj.w);
            const int p = __float_as_int(xj.w);
            const bool active = p >= 0;
            D2DLinkOut o = {0.f, 0.f, 0.f, 0.f};
            if (active) {
                const uint32_t rbkey = key & 0x1fffffffu;
                const int b = rbkey % (uint32_t)nbins, beg = S.bin_off[b], end = beg + S.bin_cnt[b];
                // the sum is accumulated in fp64: an RB may hold over a thousand links, and an fp32 running sum of n terms drifts by
                // ~sqrt(n) ulp - at n = 1 100, 1e-4 relative of a SINR just outside the 0.0625 dB band of the fp64 pass (DESIGN.md 4.4)
                double Id = 0.0;
                float dmin2 = 3.0e38f;
                bool side = false;
                for (int q = beg; q < end; ++q) {
                    const int k = S.sorted[q];
                    const float4 rk = S.rec[k];
                    if (k != j && (__float_as_uint(rk.w) & 0x9fffffffu) == rbkey) {
                        const float dx = rk.x - xj.x, dy = rk.y - xj.y;
                        const float d2 = fmaf(dx, dx, dy * dy);
                        Id += (double)(rk.z * (d2d_gain<PLE2>(d2, P.neg_half_ple) * d2d_shadow_factor(P, d2, genv, (uint32_t)j, (uint32_t)k, 0)));
                        dmin2 = fminf(dmin2, d2);
                        side |= (__float_as_uint(rk.w) >> 29) & 1u;
                    }
                }
                const float4 Av = S.linkA[j], Bv = S.linkB[j];
                const float2 sb = make_float2(Bv.x, Bv.y);
                const float dx = rj.x - xj.x, dy = rj.y - xj.y;
                const float d2own = fmaf(dx, dx, dy * dy);
                const float gown = d2d_gain<PLE2>(d2own, P.neg_half_ple);
                o = d2d_link_epilogue<PLE2>(p, xj.z, gown, gown * d2d_shadow_factor(P, d2own, genv, (uint32_t)j, (uint32_t)j, 0), (float)Id, Av, sb, P);
                if (P.shadow_chi_dB > 0.f && d2own > P.shadow_d0sq)      // the SNR's own evaluation of the path loss (simulator.py:113)
                    o.snr_dB -= P.shadow_chi_dB * d2d_shadow_normal(P, genv, (uint32_t)j, (uint32_t)j, 1);
                if (D2D_RESCUE_ENABLED && d2d_needs_rescue<true>(o, fminf(dmin2, d2own), P)) {   // rare: fp64 pass (d2d_common.cuh)
                    const double2 *pe64 = P.pos64 ? reinterpret_cast<const double2 *>(P.pos64) + e * V : nullptr;
                    const double2 rx = d2d_pos_f64(pe, pe64, __float_as_int(Bv.w));
                    double I64 = 0.0;
                    for (int q = beg; q < end; ++q) {
                        const int k = S.sorted[q];
                        if (k != j && (__float_as_uint(S.rec[k].w) & 0x9fffffffu) == rbkey) I64 += d2d_ix_term_f64<PLE2>(k, rx, pe, pe64, act, P, genv, j);
                    }
                    o = d2d_link_f64<PLE2>(j, d2d_pos_f64(pe, pe64, __float_as_int(Bv.z)), rx, I64, sb.x, act, P, genv);
                    ++resc;
                }
                cap_part += o.cap;
                ++n_act;
                bad |= (!((key >> 29) & 1u) && side && o.cap <= P.min_cap);   // envs/reward_fn.py:30-39: a non-SIDELINK link
            }
            const int64_t g = e * N + j;
            if (P.obs) {
                float2 *ob = reinterpret_cast<float2 *>(P.obs + g * 6);
                ob[0] = make_float2(rj.x, rj.y);      // an absent agent's row keeps its positions (sinr = snr = 0)
                ob[1] = make_float2(xj.x, xj.y);
                ob[2] = make_float2(o.sinr_dB, o.snr_dB);
            }
            if (P.obs_dyn) P.obs_dyn[g] = make_float2(o.sinr_dB, o.snr_dB);
            if (P.cap) P.cap[g] = o.cap;
            if (P.rate) P.rate[g] = o.rate;
            if (P.rb_out) P.rb_out[g] = active ? (int16_t)(key & 0x1fffffffu) : (int16_t)0;
            if (P.pwr_out) P.pwr_out[g] = active ? (int16_t)p : (int16_t)0;
        }

        // block reduction for the reward (envs/reward_fn.py:27-44)
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) cap_part += __shfl_xor_sync(0xffffffffu, cap_part, s);
        const int n_act_w = __reduce_add_sync(0xffffffffu, n_act);
        const int resc_w = __reduce_add_sync(0xffffffffu, resc);
        if (lane == 0) { S.red[warp] = cap_part; S.red[8 + warp] = (float)n_act_w; S.red[16 + warp] = (float)resc_w; }
        const int any_bad = __syncthreads_or(bad);   // barrier: S.red is visible to thread 0 below
        if (tid == 0) {
            float cs = 0.f, na = 0.f, rs = 0.f;
            for (int w2 = 0; w2 < D2D_BLOCK_THREADS / 32; ++w2) { cs += S.red[w2]; na += S.red[8 + w2]; rs += S.red[16 + w2]; }
            const float reward = any_bad ? -1.0f : cs / na;
            int ns = P.step_count ? (int)P.step_count[e] + 1 : 1;
            if (ns > 255) ns = 255;
            if (P.step_count) P.step_count[e] = (uint8_t)ns;
            if (P.reward) P.reward[e] = reward;
            if (P.done) P.done[e] = ns >= P.episode_length ? 1 : 0;
            if (P.reward_fn == 0) { st_reward += reward; st_reward2 += (double)reward * reward; }
            st_cap += cs;
            st_pen += any_bad ? 1.0 : 0.0; st_resc += rs; st_n += 1.0;
        }
        __syncthreads();
    }

    if (P.stats && tid == 0) {
        double *dst = P.stats + (blockIdx.x % 32) * 8;
        atomicAdd(dst + 0, st_reward); atomicAdd(dst + 1, st_cap); atomicAdd(dst + 2, st_reward2);
        atomicAdd(dst + 3, st_n); atomicAdd(dst + 4, st_pen); atomicAdd(dst + 5, st_resc);
    }
}


// ---- register-resident block kernel ------------------------------------------------------------------------------------------
// Per env (4 block barriers):
//   1. every thread loads its <= LPT links' inputs (coalesced), decodes them and takes a rank in its RB's counter
//   2. warp 0 turns the counts into offsets (exclusive scan) and re-zeroes the counters for the next env
//   3. every link writes its 16-byte peer record (tx_x, tx_y, w, u) at offset[rb] + rank: an RB's records are contiguous
//   4. every victim walks its RB's range - a CUE victim sums the u scalars (all CUE links share the MBS receiver), a DUE
//      victim evaluates w g(|tx - rx|) - then the epilogue, the stores and the block reduction for the reward.
// A block steps a CONTIGUOUS range of envs; the per-env scalars (step counter, reward, done) of a group of 256 envs live
// in the registers of thread (env - group start) and are read / written as full sectors, like the warp kernel does.
#define D2D_BLOCK_MAX_LPT 4
#define D2D_BLOCK_RESQ 32          // links per env the cooperative fp64 pass takes (more are recomputed inline by their thread)

__host__ __device__ inline size_t d2d_block2_smem_bytes(int N, int nbins) {
    size_t b = (size_t)N * sizeof(float4);                        // rec
    b += D2D_MAX_PWR_LEVELS * sizeof(float);                      // pwr_lin
    b += ((size_t)(nbins + 1) * 2 * sizeof(uint32_t) + 15) & ~(size_t)15;   // cnt (count | SIDELINK count << 16), off
    b += ((size_t)N * sizeof(uint32_t) + 15) & ~(size_t)15;       // who: (link index | Tx power << 16) of each sorted record (fp64 pass only)
    b += 2 * (D2D_BLOCK_RESQ * 8 + 4) * sizeof(uint32_t);         // resq[2]: links queued for the cooperative fp64 pass
    b += 2 * 32 * sizeof(float);                                  // red[2][32]
    return b;
}

template <bool PLE2, int LPT>
__global__ void __launch_bounds__(D2D_BLOCK_THREADS, LPT <= 2 ? 4 : 3) d2d_step_block_kernel(const __grid_constant__ D2DParams P) {
    extern __shared__ __align__(16) unsigned char d2d_smem_raw[];
    const uint32_t N = (uint32_t)P.N, C = (uint32_t)P.C, V = (uint32_t)P.V, nbins = (uint32_t)P.nbins;
    float4 *rec = reinterpret_cast<float4 *>(d2d_smem_raw);
    float *pwr = reinterpret_cast<float *>(rec + N);
    uint32_t *cnt = reinterpret_cast<uint32_t *>(pwr + D2D_MAX_PWR_LEVELS);
    uint32_t *off = cnt + (nbins + 1);
    float *red = reinterpret_cast<float *>(d2d_smem_raw + d2d_block2_smem_bytes((int)N, (int)nbins) - 2 * 32 * sizeof(float));
    uint32_t *resq = reinterpret_cast<uint32_t *>(red) - 2 * (D2D_BLOCK_RESQ * 8 + 4);      // [2][4 + 32 * 8]: word 0 = count
    uint32_t *who = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(resq) - (((size_t)N * sizeof(uint32_t) + 15) & ~(size_t)15));
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    d2d_pdl_entry(P.flags);

    for (uint32_t i = tid; i < D2D_MAX_PWR_LEVELS; i += D2D_BLOCK_THREADS) pwr[i] = P.pwr_lin[i];
    for (uint32_t i = tid; i <= nbins; i += D2D_BLOCK_THREADS) cnt[i] = 0u;
    if (tid < 2u) resq[tid * (D2D_BLOCK_RESQ * 8 + 4)] = 0u;
    // this thread's links and their constants (fixed for the whole launch)
    bool has[LPT], cue[LPT];
#pragma unroll
    for (int k = 0; k < LPT; ++k) {
        const uint32_t j = tid + k * D2D_BLOCK_THREADS;
        has[k] = j < N; cue[k] = j < C;
    }
    // link constants (tx_lin0, a_lin, inv_noise, snr0_dB) and (sens, bw): one set per link type from the constant bank unless
    // a device-config file overrode single devices (then the per-link tables, through L1)
    auto link_cA = [&](uint32_t j, bool is_cue) -> float4 {
        return P.uniform ? (is_cue ? P.u_cue : P.u_due) : __ldg(reinterpret_cast<const float4 *>(P.linkA) + j);
    };
    auto link_sB = [&](uint32_t j, bool is_cue) -> float2 {
        return P.uniform ? (is_cue ? P.us_cue : P.us_due) : __ldg(reinterpret_cast<const float2 *>(P.linkB + j));
    };
    float st_reward = 0.f, st_cap = 0.f, st_reward2 = 0.f, st_pen = 0.f, st_resc = 0.f, st_n = 0.f;   // of the envs this thread owns

    const uint32_t num_envs = (uint32_t)P.num_envs;
    const uint32_t per_block = (num_envs + gridDim.x - 1u) / gridDim.x;
    const uint32_t e0 = min(blockIdx.x * per_block, num_envs), e_end = min(e0 + per_block, num_envs);
    uint32_t g = 0;                  // position of the env in its group of 256
    int ns_keep = 0;                 // thread i: step counter of the group's env i
    float rew_keep = 0.f;            // thread i: reward of the group's env i
    __syncthreads();
    // (griddepcontrol.wait comes before the first access to memory an earlier step wrote - see d2d_step_warp.cuh)

    for (uint32_t e = e0; e < e_end; ++e) {
        const int32_t *act = P.actions + e * N;
        const float2 *pe = reinterpret_cast<const float2 *>(P.pos) + e * V;

        // ---- phase 1: inputs, decode (envs/d2d_env.py:93-101), rank inside the RB (actions.py:27-31) ---------------
        float2 tx[LPT], rx[LPT];
        float pl[LPT];
        uint32_t rb[LPT], pw[LPT], rank[LPT];
        bool live[LPT];
#pragma unroll
        for (int k = 0; k < LPT; ++k) {
            const uint32_t j = tid + k * D2D_BLOCK_THREADS;
            uint32_t a = 0xffffffffu;
            tx[k] = make_float2(1.f, 0.f); rx[k] = make_float2(0.f, 0.f);
            if (has[k]) {
                a = (uint32_t)__ldg(act + j);
                const uint32_t txd = cue[k] ? 1u + j : 1u + C + 2u * (j - C);
                tx[k] = __ldg(pe + txd);
                if (!cue[k]) rx[k] = __ldg(pe + txd + 1u);
            }
            const uint32_t npw = (uint32_t)(cue[k] ? P.n_pwr_cue : P.n_pwr_due);
            live[k] = has[k] && a < (uint32_t)P.R * npw;            // valid actions: 0 <= a < R n_pwr (envs/d2d_env.py:36-40)
            const uint32_t as = live[k] ? a : 0u;
            rb[k] = __umulhi(as, cue[k] ? P.magic_cue : P.magic_due) + (as & (cue[k] ? P.npw1_cue : P.npw1_due));
            pw[k] = as - rb[k] * npw;
            pl[k] = live[k] ? pwr[pw[k]] : 0.0f;
            rank[k] = 0u;
            if (live[k]) rank[k] = atomicAdd(&cnt[rb[k]], cue[k] ? 1u : 0x10001u) & 0xffffu;        // high half counts the SIDELINKs
        }
        __syncthreads();

        // ---- phase 2: counts -> offsets (warp 0), counters cleared for the next env ------------------------------------
        if (warp == 0) {
            const uint32_t chunk = (nbins + 31u) >> 5, lo = lane * chunk, hi = min(lo + chunk, nbins);
            uint32_t sum = 0;
            for (uint32_t i = lo; i < hi; ++i) sum += cnt[i] & 0xffffu;
            uint32_t incl = sum;
#pragma unroll
            for (int s = 1; s < 32; s <<= 1) {
                const uint32_t n = __shfl_up_sync(0xffffffffu, incl, s);
                if (lane >= (uint32_t)s) incl += n;
            }
            uint32_t run = incl - sum;
            for (uint32_t i = lo; i < hi; ++i) {
                const uint32_t c = cnt[i];
                off[i] = run | (c & 0xffff0000u);        // offset in the low half, the RB's SIDELINK count above it
                run += c & 0xffffu;
                cnt[i] = 0u;
            }
            if (lane == 31u) off[nbins] = run;
        }
        __syncthreads();

        // ---- phase 3: peer records, grouped by RB -------------------------------------------------------------------------
        uint32_t beg[LPT], end[LPT], self[LPT];
        bool side[LPT];
        float gown[LPT];
#pragma unroll
        for (int k = 0; k < LPT; ++k) {
            beg[k] = 0u; end[k] = 0u; self[k] = 0u; side[k] = false;
            const float dxo = tx[k].x - rx[k].x, dyo = tx[k].y - rx[k].y;       // own link (a CUE's receiver is the MBS at the origin)
            const float d2own = fmaf(dxo, dxo, dyo * dyo);
            gown[k] = d2d_gain<PLE2>(d2own, P.neg_half_ple);
            if (live[k]) {
                const uint32_t o = off[rb[k]];
                beg[k] = o & 0xffffu; end[k] = off[rb[k] + 1u] & 0xffffu; side[k] = (o >> 16) != 0u;
                self[k] = beg[k] + rank[k];
                const float w = pl[k] * link_cA(tid + k * D2D_BLOCK_THREADS, cue[k]).x;
                const float u = w * (cue[k] ? gown[k] : d2d_gain<PLE2>(fmaf(tx[k].x, tx[k].x, tx[k].y * tx[k].y), P.neg_half_ple));
                rec[self[k]] = make_float4(tx[k].x, tx[k].y, w, u);             // u = this link's interference at the MBS
                who[self[k]] = (tid + k * D2D_BLOCK_THREADS) | (pw[k] << 16);
            }
        }
        __syncthreads();

        // ---- phase 4: interference walk (simulator.py:95-101), epilogue, outputs ----------------------------------------------
        if (e == e0) d2d_pdl_wait();
        if (g == 0u && P.step_count) ns_keep = e + tid < e_end ? (int)P.step_count[e + tid] : 0;      // consumed at the group's end
        uint32_t *rq = resq + (e & 1u) * (D2D_BLOCK_RESQ * 8 + 4);      // this env's queue; the other one is cleared below
        float cap_part = 0.0f;
        uint32_t n_act = 0, resc = 0;
        bool bad = false;
#pragma unroll
        for (int k = 0; k < LPT; ++k) {
            const uint32_t j = tid + k * D2D_BLOCK_THREADS;
            D2DLinkOut o = {0.f, 0.f, 0.f, 0.f};
            if (live[k]) {
                // fp64 accumulation, as in the general kernel: an RB may hold all 1024 links of an env
                double Id = 0.0;
                float dmin2 = 3.0e38f;
                if (cue[k] && !P.pos64) {
                    for (uint32_t q = beg[k]; q < end[k]; ++q)
                        if (q != self[k]) Id += (double)rec[q].w;
                } else {
                    for (uint32_t q = beg[k]; q < end[k]; ++q) {
                        if (q == self[k]) continue;
                        const float4 rk = rec[q];
                        const float dx = rk.x - rx[k].x, dy = rk.y - rx[k].y;
                        const float d2 = fmaf(dx, dx, dy * dy);
                        Id += (double)(rk.z * d2d_gain<PLE2>(d2, P.neg_half_ple));
                        dmin2 = fminf(dmin2, d2);
                    }
                }
                const float dxo = tx[k].x - rx[k].x, dyo = tx[k].y - rx[k].y;
                const float2 sBk = link_sB(j, cue[k]);
                o = d2d_link_epilogue<PLE2>((int)pw[k], pl[k], gown[k], gown[k], (float)Id, link_cA(j, cue[k]), sBk, P);
                uint32_t qslot = D2D_BLOCK_RESQ;
                const bool need = D2D_RESCUE_ENABLED && d2d_needs_rescue<true>(o, fminf(dmin2, fmaf(dxo, dxo, dyo * dyo)), P);
                if (need) {
                    // fp64 pass (d2d_common.cuh; same policy as d2d_rescue_warp): ~0.2 % of the links, i.e. about one per dense
                    // env.  A thread recomputing its link alone would stall the other 255 at the next barrier, so the link is
                    // queued and a whole warp takes it after the barrier (below); only a full queue is served inline.
                    qslot = atomicAdd(rq, 1u);
                    ++resc;
                    if (qslot < D2D_BLOCK_RESQ) {
                        uint32_t *q8 = rq + 4 + qslot * 8;
                        q8[0] = j | (pw[k] << 16); q8[1] = beg[k] | (end[k] << 16); q8[2] = self[k];
                        q8[3] = __float_as_uint(tx[k].x); q8[4] = __float_as_uint(tx[k].y);
                        q8[5] = __float_as_uint(rx[k].x); q8[6] = __float_as_uint(rx[k].y);
                    }
                }
                if (need && qslot >= D2D_BLOCK_RESQ) {
                    const double2 *pe64 = P.pos64 ? reinterpret_cast<const double2 *>(P.pos64) + (int64_t)e * V : nullptr;
                    const bool exact = pe64 != nullptr;
                    const double2 rxd = exact ? pe64[d2d_rx_dev((int)j, (int)C)] : make_double2((double)rx[k].x, (double)rx[k].y);
                    const double2 txd = exact ? pe64[d2d_tx_dev((int)j, (int)C)] : make_double2((double)tx[k].x, (double)tx[k].y);
                    double I64 = 0.0;
                    for (uint32_t q = beg[k]; q < end[k]; ++q) {
                        if (q == self[k]) continue;
                        const uint32_t wk = who[q], kk = wk & 0xffffu;
                        const float4 rk = rec[q];
                        const double2 tk = exact ? pe64[d2d_tx_dev((int)kk, (int)C)] : make_double2((double)rk.x, (double)rk.y);
                        const double ex = tk.x - rxd.x, ey = tk.y - rxd.y;
                        I64 += P.pwr_lin_d[wk >> 16] * P.linkD[kk].t_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
                    }
                    const D2DLinkD Lj = P.linkD[j];
                    const double ex = txd.x - rxd.x, ey = txd.y - rxd.y;
                    const double Sg = P.pwr_lin_d[pw[k]] * Lj.a_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
                    const double r = Sg * d2d_rcp_f64(fma(I64, Lj.inv_noise, 1.0));
                    const bool r1 = fabs(r - 1.0) < 0.0625, s1 = fabs(Sg - 1.0) < 0.0625;
                    double sinr = (double)o.sinr_dB;
                    if (exact || r1 || P.thr_band > 0.f) { sinr = r1 ? d2d_db_near1(r) : 4.3429448190325182765 * d2d_ln_f64(r); o.sinr_dB = d2d_sinr_store(sinr, P); }
                    if (exact || s1) o.snr_dB = (float)(s1 ? d2d_db_near1(Sg) : 4.3429448190325182765 * d2d_ln_f64(Sg));
                    if (exact || (r1 && fabsf(sBk.x) < 0.5f)) {
                        const double rate = sinr > (double)sBk.x ? 1.4426950408889634074 * d2d_ln_f64(1.0 + r) : 0.0;
                        o.rate = (float)rate; o.cap = (float)(Lj.bw_MHz * rate);
                    }
                }
                cap_part += o.cap;
                ++n_act;
                bad |= cue[k] && side[k] && o.cap <= P.min_cap;      // envs/reward_fn.py:30-39
            }
            if (has[k]) {
                const uint32_t gi = e * N + j;
                if (P.obs) {
                    float2 *ob = reinterpret_cast<float2 *>(reinterpret_cast<char *>(P.obs) + (uint64_t)gi * 24u);
                    ob[0] = tx[k];                                   // an absent agent's row keeps its positions (sinr = snr = 0)
                    ob[1] = rx[k];
                    ob[2] = make_float2(o.sinr_dB, o.snr_dB);
                }
                if (P.obs_dyn) P.obs_dyn[gi] = make_float2(o.sinr_dB, o.snr_dB);
                if (P.cap) P.cap[gi] = o.cap;
                if (P.rate) P.rate[gi] = o.rate;
                if (P.rb_out) P.rb_out[gi] = live[k] ? (int16_t)rb[k] : (int16_t)0;
                if (P.pwr_out) P.pwr_out[gi] = live[k] ? (int16_t)pw[k] : (int16_t)0;
            }
        }

        // ---- block reduction for the reward (envs/reward_fn.py:27-44); the env's owner thread keeps the scalars ------------
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) cap_part += __shfl_xor_sync(0xffffffffu, cap_part, s);
        const uint32_t n_act_w = __reduce_add_sync(0xffffffffu, n_act), resc_w = __reduce_add_sync(0xffffffffu, resc);
        float *rd = red + (e & 1u) * 32u;                                // double-buffered: no barrier after the owner's read
        if (lane == 0) { rd[warp] = cap_part; rd[8 + warp] = (float)n_act_w; rd[16 + warp] = (float)resc_w; }
        const int any_bad = __syncthreads_or(bad ? 1 : 0);
        // ---- cooperative fp64 pass: warp w takes queued links w, w + 8, ...; its lanes split the RB's peer records, a
        // butterfly sums their terms, lane 0 rewrites what fp32 could not deliver (after the owner's stores above) --------
        {
            const uint32_t nq = min(rq[0], (uint32_t)D2D_BLOCK_RESQ);
            if (tid == 0) resq[((e & 1u) ^ 1u) * (D2D_BLOCK_RESQ * 8 + 4)] = 0u;      // the next env's queue
            const double2 *pe64 = P.pos64 ? reinterpret_cast<const double2 *>(P.pos64) + (int64_t)e * V : nullptr;
            const bool exact = pe64 != nullptr;
            for (uint32_t i = warp; i < nq; i += D2D_BLOCK_THREADS / 32) {
                const uint32_t *q8 = rq + 4 + i * 8;
                const uint32_t j = q8[0] & 0xffffu, pwj = q8[0] >> 16, qb = q8[1] & 0xffffu, qe = q8[1] >> 16, qs = q8[2];
                const double2 txd = exact ? pe64[d2d_tx_dev((int)j, (int)C)]
                                          : make_double2((double)__uint_as_float(q8[3]), (double)__uint_as_float(q8[4]));
                const double2 rxd = exact ? pe64[d2d_rx_dev((int)j, (int)C)]
                                          : make_double2((double)__uint_as_float(q8[5]), (double)__uint_as_float(q8[6]));
                double I64 = 0.0;
                for (uint32_t q = qb + lane; q < qe; q += 32u) {
                    if (q == qs) continue;
                    const uint32_t wk = who[q], kk = wk & 0xffffu;
                    const float4 rk = rec[q];
                    const double2 tk = exact ? pe64[d2d_tx_dev((int)kk, (int)C)] : make_double2((double)rk.x, (double)rk.y);
                    const double ex = tk.x - rxd.x, ey = tk.y - rxd.y;
                    I64 += P.pwr_lin_d[wk >> 16] * P.linkD[kk].t_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
                }
#pragma unroll
                for (int sh = 16; sh > 0; sh >>= 1)
                    I64 += __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(I64), sh), __shfl_xor_sync(0xffffffffu, __double2loint(I64), sh));
                if (lane == 0) {
                    const D2DLinkD Lj = P.linkD[j];
                    const float sens = link_sB(j, j < C).x;
                    const double ex = txd.x - rxd.x, ey = txd.y - rxd.y;
                    const double Sg = P.pwr_lin_d[pwj] * Lj.a_lin * d2d_gain_f64_fast<PLE2>(ex * ex + ey * ey, P.ple_d);
                    const double r = Sg * d2d_rcp_f64(fma(I64, Lj.inv_noise, 1.0));
                    const bool r1 = fabs(r - 1.0) < 0.0625, s1 = fabs(Sg - 1.0) < 0.0625;
                    const uint64_t gi = (uint64_t)e * N + j;
                    double sinr = 0.0;
                    if (exact || r1 || P.thr_band > 0.f) {
                        sinr = r1 ? d2d_db_near1(r) : 4.3429448190325182765 * d2d_ln_f64(r);
                        const float sv = d2d_sinr_store(sinr, P);
                        if (P.obs) P.obs[gi * 6u + 4u] = sv;
                        if (P.obs_dyn) P.obs_dyn[gi].x = sv;
                    }
                    if (exact || s1) {
                        const float snr = (float)(s1 ? d2d_db_near1(Sg) : 4.3429448190325182765 * d2d_ln_f64(Sg));
                        if (P.obs) P.obs[gi * 6u + 5u] = snr;
                        if (P.obs_dyn) P.obs_dyn[gi].y = snr;
                    }
                    if (exact || (r1 && fabsf(sens) < 0.5f)) {
                        const double rate = sinr > (double)sens ? 1.4426950408889634074 * d2d_ln_f64(1.0 + r) : 0.0;
                        if (P.cap) P.cap[gi] = (float)(Lj.bw_MHz * rate);
                        if (P.rate) P.rate[gi] = (float)rate;
                    }
                }
            }
        }
        if (tid == g) {
            float cs = 0.f, na = 0.f, rs = 0.f;
#pragma unroll
            for (int w2 = 0; w2 < D2D_BLOCK_THREADS / 32; ++w2) { cs += rd[w2]; na += rd[8 + w2]; rs += rd[16 + w2]; }
            const float reward = any_bad ? -1.0f : cs / na;
            rew_keep = reward;
            if (P.reward_fn == 0) { st_reward += reward; st_reward2 = fmaf(reward, reward, st_reward2); }
            st_cap += cs;
            st_pen += any_bad ? 1.f : 0.f; st_resc += rs; st_n += 1.f;
        }
        if (g == D2D_BLOCK_THREADS - 1u || e + 1u == e_end) {
            // envs/d2d_env.py:65,68 for the whole group: num_steps += 1; done = num_steps >= EPISODE_LENGTH
            if (tid <= g) {
                const uint32_t eg = e - g + tid;
                const int ns = min(ns_keep + 1, 255);
                if (P.step_count) P.step_count[eg] = (uint8_t)ns;
                if (P.reward) P.reward[eg] = rew_keep;
                if (P.done) P.done[eg] = ns >= P.episode_length ? 1 : 0;
            }
            g = 0u;
        } else {
            ++g;
        }
    }

    if (P.stats) {
        // block totals of the six statistics -> one fp64 atomic each
        float v[6] = {st_reward, st_cap, st_reward2, st_n, st_pen, st_resc};
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 6; ++i) {
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], s);
            if (lane == 0) red[i * 8 + warp] = v[i];
        }
        __syncthreads();
        if (tid < 6) {
            double t = 0.0;
            for (int w2 = 0; w2 < D2D_BLOCK_THREADS / 32; ++w2) t += (double)red[tid * 8 + w2];
            if (t != 0.0) atomicAdd(P.stats + (blockIdx.x % D2D_STATS_REPLICAS) * 8 + tid, t);
        }
    }
}
