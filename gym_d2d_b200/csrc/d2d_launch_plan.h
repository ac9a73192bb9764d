// d2d_launch_plan.h - how a step launch is ordered behind the kernels before it (include/d2d_b200.h, "Ordering rule"; DESIGN.md
// 4.7).  Host-only and free of CUDA calls, so that a test can compile it without a GPU (tests/test_launch_plan.py).
#pragma once

#include "d2d_internal.h"

enum { MODE_STEP = 0, MODE_MANY = 1, MODE_EPISODE = 2 };

// One launch (per chunk of envs) makes T consecutive steps: MODE_STEP (T = 1) is d2d_step; MODE_MANY / MODE_EPISODE need
// the warp kernel (T slices per env; the episode's slice 0 is the uncounted reset step).
struct EpisodeArgs {
    uint64_t ep_seed = 0, act_seed = 0;
    uint32_t act_t0 = 0;         // step index of slice 0 in the action draws
    bool draw_actions = false;
    bool no_reset = false;       // d2d_rollout: continue from the bound state, every slice counted
};

// The step kernels index with 32 bits: at most this many env-slices per launch (> 7 million default envs)
inline int64_t d2d_max_launch_envs(const d2d_handle *h) {
    return std::max<int64_t>(1, (int64_t)0x7fffffff / std::max(6 * h->N, 2 * h->V));
}

// Per-warp tickets from 5 QUARTER envs per warp (1.25 envs).  Measured (profiles/README.md): the hand-off wins as soon as warps
// step more than one env per launch (E = 6 144, 1.5 envs per warp: 7.6 -> 5.3 us; E = 16 384: 12.4 -> 9.4 us; E = 131 072:
// 69.5 -> 65.9 us) and loses at exactly one (E = 4 096: 5.4 -> 6.8 us; E = 1 024: 2.7 -> 9.5 us), where the hardware's grid-wide
// wait is cheaper than the release / acquire hand-off (two L2 round trips) - and where the launches do not publish tokens
// either (the release store holds a warp's block slot for an L2 round trip: 5.4 -> 10 us at E = 4 096)
constexpr int64_t kTicketMinQuarterEnvs = 5;

struct D2DStepPlan {
    bool autoreset = false;      // d2d_step with D2D_STEP_AUTORESET
    uint32_t flags = 0;          // D2D_PF_INPUTS_FRESH | D2D_PF_LATE_WAIT
    int grid = 0;                // block cap of the step geometry's launches: the full grid, or h->grid_late under the late wait
    uint64_t tok_wait = 0, tok_sign = 0;   // per-warp tickets (D2DParams); tok_sign = 0: this launch takes no part in a chain
    int64_t chunk = 0;           // envs per launch
    int last_kind = 0;           // D2D_LAST_* of the handle once the launch is enqueued
};

inline D2DStepPlan d2d_plan_step(d2d_handle *h, const d2d_step_io_t *io, int mode, void *stream, const EpisodeArgs &ea) {
    D2DStepPlan pl;
    const int64_t E = h->cfg.num_envs;
    // D2D_STEP_AUTORESET (d2d_step only): always the default ordering - wait at entry, no late wait, no tickets, the full grid
    pl.autoreset = mode == MODE_STEP && (io->flags & D2D_STEP_AUTORESET) != 0u;
    // batches beyond the 32-bit bound go in chunks; the fused launches' callers checked that their T slices fit
    pl.chunk = mode != MODE_STEP ? E : h->chunk_override > 0 ? std::min(d2d_max_launch_envs(h), h->chunk_override) : d2d_max_launch_envs(h);
    // a single-kernel plain step: a d2d_step of the warp kernel in one launch, with no post-pass kernel after it (per-agent
    // rewards, the ShadowingPathLoss counter) - the next step's predecessor in the stream is then this step's kernel itself
    const bool single = h->use_warp && mode == MODE_STEP && !pl.autoreset && h->cfg.reward_fn == D2D_REWARD_SYSTEM_CAPACITY &&
                        !io->agent_reward && !h->dRngStep && pl.chunk >= E;
    // Inputs may be read ahead of griddepcontrol.wait only on the caller's promise AND when the kernel before this one (for this
    // handle, in this stream) was a step kernel, which writes neither actions nor positions.  An episode that draws its own
    // actions reads no input at all; a rollout reads the positions like a step does.
    bool stable = h->pdl && h->last_stream == stream;
    const bool reads_positions = mode != MODE_EPISODE || ea.no_reset;
    if (!reads_positions && ea.draw_actions) stable = h->pdl;
    else if (!reads_positions) stable = stable && (io->flags & D2D_STEP_INPUTS_STABLE) && h->last_kind != D2D_LAST_OTHER;
    else stable = stable && (io->flags & D2D_STEP_INPUTS_STABLE) && h->last_kind == D2D_LAST_STEP && !pl.autoreset;
    // Late wait (d2d_step_warp.cuh): a flagged single-kernel step right behind another one of this handle, whose per-link output
    // buffers alias none of the previous step's, stores them ahead of griddepcontrol.wait - nothing the predecessor does can
    // collide with them, and whatever was enqueued before the predecessor is complete (a kernel that is not a step kernel never
    // lets its successor start early).  The step counters and per-env scalars stay behind the wait.
    // (measured, profiles/ab_r02_25 .. 28.log: a win at every batch size - E = 1 024: 2.55 -> 1.94 us, 4 096: 5.42 -> 4.94 us,
    // 4 608: 7.76 -> 4.75 us, and level with or ahead of the per-warp tickets beyond one wave (E = 32 768: 17.8 -> 17.3 us) - except
    // where two launches of 2-warp blocks fill the SM's warp slots exactly: E = 2 048 3.46 -> 4.22 us)
    const size_t EN = (size_t)E * h->N;
    const uintptr_t cur[6][2] = {{(uintptr_t)io->obs, EN * 24}, {(uintptr_t)io->obs_dyn, EN * 8}, {(uintptr_t)io->capacity_mbps, EN * 4},
                                 {(uintptr_t)io->rate_bps, EN * 4}, {(uintptr_t)io->rb, EN * 2}, {(uintptr_t)io->tx_pwr_dBm, EN * 2}};
    bool late = single && stable && h->late_wait_on && h->prev_out_valid && h->last_kind == D2D_LAST_STEP &&
                !(h->warp->wpb == 2 && E > 1792 && h->grid_late == 0);
    for (int a = 0; late && a < 6; ++a)
        for (int b = 0; b < 6; ++b)
            if (cur[a][0] && h->prev_out[b][0] && cur[a][0] < h->prev_out[b][1] && h->prev_out[b][0] < cur[a][0] + cur[a][1]) late = false;
    h->prev_out_valid = single;
    for (int a = 0; a < 6; ++a) { h->prev_out[a][0] = cur[a][0]; h->prev_out[a][1] = cur[a][0] ? cur[a][0] + cur[a][1] : 0; }
    pl.flags = (stable ? 0u : D2D_PF_INPUTS_FRESH) | (late ? D2D_PF_LATE_WAIT : 0u);
    pl.grid = late && h->grid_late > 0 ? std::min(h->grid, h->grid_late) : h->grid;
    // Per-warp tickets (d2d_common.cuh): a single-kernel step publishes a token per warp; the next one - same stream, same
    // geometry, inputs declared stable - waits per warp for that token instead of for the whole grid.  Only for steps that write
    // buffers their predecessor wrote: the late wait serves the others.
    const int grid1 = (int)std::min<int64_t>(pl.grid, (E + h->envs_per_block - 1) / h->envs_per_block);
    if (single && !late && h->dTickets && h->pdl && h->tickets_on && 4 * E >= kTicketMinQuarterEnvs * grid1 * h->warp->wpb) {
        const bool follow = stable && h->chain_seq > 0 && h->chain_seq < 0xffffu && h->chain_grid == grid1 && h->last_stream == stream;
        if (!follow) { ++h->chain_id; h->chain_seq = 0; h->chain_grid = grid1; }
        pl.tok_wait = follow ? ((h->chain_id << 16) | h->chain_seq) : 0ull;
        pl.tok_sign = (h->chain_id << 16) | (h->chain_seq + 1u);
        ++h->chain_seq;
    } else {
        h->chain_seq = 0;
    }
    // (an auto-reset step writes positions: the next step reads them after its wait, as after an episode)
    pl.last_kind = (mode == MODE_EPISODE && !ea.no_reset) || pl.autoreset ? D2D_LAST_EPISODE : D2D_LAST_STEP;
    return pl;
}
