// d2d_aux.cuh - the kernels either side of the step: position upload, device-side reset, and the
// optional per-agent observation materialisation.
#pragma once

#include "d2d_common.cuh"

// Device.set_position over a batch (device.py:82-83): float64 [count][V][2] -> float32 state.
// Device 0 (the MBS) is pinned to the origin like simulator.py:63-64.
__global__ void d2d_set_positions_kernel(const double *__restrict__ src, float *__restrict__ dst,
                                         double *__restrict__ dst64, int64_t count, int V) {
    const int64_t total = count * V;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int v = (int)(i % V);
        double2 s = reinterpret_cast<const double2 *>(src)[i];
        if (v == 0) s = make_double2(0.0, 0.0);
        reinterpret_cast<float2 *>(dst)[i] = make_float2((float)s.x, (float)s.y);
        if (dst64) reinterpret_cast<double2 *>(dst64)[i] = s;      // unrounded shadow for the fp64 rescue path
    }
}

// Simulator.reset (simulator.py:61-75): one thread per (env, draw unit) - a pair of CUEs or one DUE pair, one Philox block each
// (d2d_common.cuh) - writing 16 bytes.  Both kinds of unit run the SAME instruction stream - two uniform-in-disc draws from the
// block's four words, the second one with the cell radius (a CUE) or as an offset of d2d radius from the first (a DUE receiver) -
// so a warp that holds both kinds does not execute two divergent halves; only the in-cell re-draw of a receiver
// (position.py:31-45, a few per cent of the pairs) diverges.  units = ceil(C / 2) + D per env; `total` = num_envs * units
// < 2^32 per launch (the host chunks); `magic` = ceil(2^32 / units) turns the env index into one multiply.
__global__ void d2d_reset_kernel(float *__restrict__ pos, double *__restrict__ pos64, uint8_t *__restrict__ step_count,
                                 const uint8_t *__restrict__ env_mask, uint32_t total, uint32_t C, uint32_t D, float cell_radius,
                                 float d2d_radius, uint64_t seed, uint64_t first_global_env, uint32_t magic) {
    const uint32_t CU = (C + 1u) >> 1, U = CU + D, V = 1u + C + 2u * D;
    const float r2max = __fmul_rn(cell_radius, cell_radius);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        uint32_t e = __umulhi(i, magic);
        e -= (e * U > i) ? 1u : 0u;                              // (the magic may overshoot by one for large i)
        const uint32_t u = i - e * U;
        if (env_mask && !env_mask[e]) continue;
        float2 *pe = reinterpret_cast<float2 *>(pos) + (uint64_t)e * V;
        double2 *pe64 = pos64 ? reinterpret_cast<double2 *>(pos64) + (uint64_t)e * V : nullptr;
        const uint64_t g = first_global_env + (uint64_t)e;
        if (u == 0u) {
            pe[0] = make_float2(0.f, 0.f);                       // simulator.py:63-64
            if (pe64) pe64[0] = make_double2(0.0, 0.0);
            if (step_count) step_count[e] = 0;                   // envs/d2d_env.py:46
        }
        const bool due = u >= CU;
        uint4 b = d2d_reset_block(seed, g, u, 0u);
        const float2 p0 = d2d_disc_from_words(b.x, b.y, cell_radius);
        float2 p1 = d2d_disc_from_words(b.z, b.w, due ? d2d_radius : cell_radius);
        if (due) {
            p1 = make_float2(__fadd_rn(p0.x, p1.x), __fadd_rn(p0.y, p1.y));
            // position.py:38-44: re-draw the receiver until it falls inside the cell (the same candidates as d2d_draw_due)
            for (uint32_t k = 1; k < D2D_RESET_MAX_OFFSETS && __fadd_rn(__fmul_rn(p1.x, p1.x), __fmul_rn(p1.y, p1.y)) > r2max; ++k) {
                if (k & 1u) b = d2d_reset_block(seed, g, u, (k + 1u) >> 1);
                const float2 o = (k & 1u) ? d2d_disc_from_words(b.x, b.y, d2d_radius) : d2d_disc_from_words(b.z, b.w, d2d_radius);
                p1 = make_float2(__fadd_rn(p0.x, o.x), __fadd_rn(p0.y, o.y));
            }
        }
        // devices 1 + 2u, 2 + 2u (CUEs; the second one may not exist) or 1 + C + 2d, 2 + C + 2d (a DUE pair)
        const uint32_t t = due ? 1u + C + 2u * (u - CU) : 1u + 2u * u;
        const bool two = due || 2u * u + 1u < C;
        if (two && (((uintptr_t)(pe + t)) & 15u) == 0u) *reinterpret_cast<float4 *>(pe + t) = make_float4(p0.x, p0.y, p1.x, p1.y);
        else { pe[t] = p0; if (two) pe[t + 1u] = p1; }
        if (pe64) { pe64[t] = make_double2((double)p0.x, (double)p0.y); if (two) pe64[t + 1u] = make_double2((double)p1.x, (double)p1.y); }
    }
}

// Discrete(n).sample() for every agent of every env (envs/d2d_env.py:54-60), step index t of the episode (0 = the reset step):
// the same draws the EPISODE instantiation of the warp kernel makes in registers (d2d_common.cuh).  One thread per (env, pair
// index l): CUE l and DUE pair l share a Philox block.  Links beyond the uplinks and sidelinks (DOWNLINK 'mbs:cueXX', never
// sampled by the reference's reset) are marked absent (-1).
__global__ void d2d_sample_actions_kernel(int32_t *__restrict__ actions, uint32_t total, uint32_t C, uint32_t D, uint32_t N,
                                          uint32_t n_cue, uint32_t n_due, uint64_t act_seed, uint64_t first_global_env, uint32_t t) {
    const uint32_t L = max(C, D), X = N - C - D;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint32_t e = i / L, l = i - e * L;
        const uint4 b = d2d_action_block(act_seed, first_global_env + (uint64_t)e, l, t);
        int32_t *a = actions + (uint64_t)e * N;
        if (l < C) a[l] = (int32_t)__umulhi(d2d_action_word(b, t, false), n_cue);
        if (l < D) a[C + l] = (int32_t)__umulhi(d2d_action_word(b, t, true), n_due);
        if (l < X) a[C + D + l] = -1;
    }
}

// D2D_STEP_ACTIONS_I16: the host uploaded int16 actions; the step kernels read int32 (sign-extended: < 0 stays "absent")
__global__ void d2d_widen_actions_kernel(const int16_t *__restrict__ src, int32_t *__restrict__ dst, int64_t count) {
    const int64_t pairs = count >> 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += (int64_t)gridDim.x * blockDim.x) {
        const short2 v = reinterpret_cast<const short2 *>(src)[i];
        reinterpret_cast<int2 *>(dst)[i] = make_int2((int)v.x, (int)v.y);
    }
    if ((count & 1) && blockIdx.x == 0 && threadIdx.x == 0) dst[count - 1] = (int32_t)src[count - 1];
}

// ShadowingPathLoss: the step-call counter lives in device memory and advances on the stream (so does a replayed CUDA graph's)
__global__ void d2d_advance_counter_kernel(uint64_t *counter, uint64_t by) { *counter += by; }

// LinearObsFunction.get_state (envs/obs_fn.py:43-53): agent i's vector = its own row, then every other
// row in link order.  One block per (env, agent); float2 granularity (3 per row).
__global__ void d2d_per_agent_obs_kernel(const float *__restrict__ table, float *__restrict__ out, int N) {
    const int64_t e = blockIdx.x / N;
    const int i = (int)(blockIdx.x - e * N);
    const float2 *src = reinterpret_cast<const float2 *>(table) + e * N * 3;
    float2 *dst = reinterpret_cast<float2 *>(out) + (e * N + i) * (int64_t)N * 3;
    for (int m = threadIdx.x; m < 3 * N; m += blockDim.x) {
        const int row = m / 3, part = m - row * 3;
        const int link = row == 0 ? i : (row - 1 < i ? row - 1 : row);
        dst[m] = src[link * 3 + part];
    }
}


// Per-agent rewards from a step's results (SURVEY 8f-3), one TEAM of threads per env (a warp for N <= 64, a block beyond):
//   mode 0  SystemCapacityRewardFunction's scalar broadcast to the acting agents (envs/reward_fn.py:44)
//   mode 1  ShannonRewardFunction (envs/reward_fn.py:47-57): log2(1 + 10^(sinr/10)) if sinr >= param else -1
//   mode 2  CueSinrShannonRewardFunction (envs/reward_fn.py:60-78): -1 if some OTHER action on the agent's RB is a
//           non-SIDELINK link with sinr < param, else log2(1 + 10^(sinr/10))
// Reads the decoded step results (sinr_dB from the observation table - after the fp64 pass, so threshold decisions see the
// rescued values) and re-derives the RB from the raw action (envs/d2d_env.py:93-101).  For modes 1 / 2 reward[e] becomes
// the mean agent reward and the reward statistics are accumulated here (the step kernel skips them).
// reset_rows (D2D_STEP_AUTORESET, else NULL): the step counters after the step.  A row at 0 was reset by the step, whose actions are
// not the caller's: it has no acting agent - agent_reward 0, reward 0, nothing added to the statistics.
template <int TEAM>
__global__ void d2d_agent_reward_kernel(const int32_t *__restrict__ actions, const float *__restrict__ obs,
                                        float *__restrict__ agent_reward, float *__restrict__ reward, double *__restrict__ stats,
                                        int64_t num_envs, int N, const int32_t *__restrict__ link_meta, int R, int mode, float param,
                                        const uint8_t *__restrict__ reset_rows) {
    extern __shared__ uint32_t d2d_weak_smem[];
    const int teams = blockDim.x / TEAM, team = threadIdx.x / TEAM, tl = threadIdx.x % TEAM;
    uint32_t *weak = d2d_weak_smem + (size_t)team * R;         // mode 2 only (the launch requests no shared memory otherwise)
    auto team_sync = [&]() { if (TEAM == 32) __syncwarp(); else __syncthreads(); };
    float st_r = 0.f, st_r2 = 0.f;
    const int64_t rounds = (num_envs + (int64_t)gridDim.x * teams - 1) / ((int64_t)gridDim.x * teams);
    for (int64_t it = 0; it < rounds; ++it) {
        const int64_t e = (it * gridDim.x + blockIdx.x) * teams + team;
        const bool in = e < num_envs;                 // whole teams drop out together; barriers stay uniform per block
        const bool acts = in && !(reset_rows && reset_rows[e] == 0);
        const int32_t *act = actions + (in ? e : 0) * N;
        const float *ob = obs + (in ? e : 0) * N * 6;
        if (mode == 2) {
            for (int r = tl; r < R; r += TEAM) weak[r] = 0u;
            team_sync();
            for (int j = tl; acts && j < N; j += TEAM) {
                const int meta = link_meta[j], npw = meta & 0xffff;          // power levels | SIDELINK << 16
                const uint32_t a = (uint32_t)act[j];
                if (!(meta >> 16) && a < (uint32_t)(R * npw) && ob[j * 6 + 4] < param) atomicAdd(&weak[a / (uint32_t)npw], 1u);
            }
            team_sync();
        }
        float sum = 0.f;
        int n_act = 0;
        for (int j = tl; in && j < N; j += TEAM) {
            const int meta = link_meta[j], npw = meta & 0xffff;
            const uint32_t a = (uint32_t)act[j];
            const bool live = acts && a < (uint32_t)(R * npw);
            float rw = 0.f;
            if (live) {
                const float sinr = ob[j * 6 + 4];
                const float shannon = d2d_log2_1p(d2d_ex2(sinr * 0.33219280948873623f));     // log2(1 + 10^(sinr/10))
                if (mode == 0) rw = reward[e];
                else if (mode == 1) rw = sinr >= param ? shannon : -1.0f;
                else rw = weak[a / (uint32_t)npw] - ((!(meta >> 16) && sinr < param) ? 1u : 0u) > 0u ? -1.0f : shannon;
                sum += rw;
                ++n_act;
            }
            if (agent_reward) agent_reward[e * N + j] = rw;
        }
        if (mode != 0) {
            // mean over the acting agents -> reward[e]; team reduction through the warp, then shared memory for blocks
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, s); n_act += __shfl_xor_sync(0xffffffffu, n_act, s); }
            if (TEAM > 32) {
                __shared__ float red_s[8];
                __shared__ int red_n[8];
                team_sync();
                if ((tl & 31) == 0) { red_s[tl >> 5] = sum; red_n[tl >> 5] = n_act; }
                team_sync();
                sum = 0.f; n_act = 0;
                for (int w = 0; w < TEAM / 32; ++w) { sum += red_s[w]; n_act += red_n[w]; }
            }
            if (in && tl == 0) {
                const float r = n_act ? sum / (float)n_act : 0.f;
                reward[e] = r;
                st_r += r; st_r2 = fmaf(r, r, st_r2);
            }
        }
        team_sync();
    }
    if (mode != 0 && stats && tl == 0 && (st_r != 0.f || st_r2 != 0.f)) {
        double *dst = stats + ((blockIdx.x * teams + team) % 32) * 8;
        atomicAdd(dst + 0, (double)st_r);
        atomicAdd(dst + 2, (double)st_r2);
    }
}
