"""The ordering policy of step launches (gym_d2d_b200/csrc/d2d_launch_plan.h: d2d_plan_step), checked on the CPU.

The GPU ordering tests compare outputs with D2D_B200_PDL=0, and those outputs are the same whether a launch read its inputs
early, took the late wait or handed over per warp; only the step time shows it.  Here the real d2d_plan_step is compiled
with nvcc into a host-only program that builds a handle, runs a sequence of calls on it and prints each plan.  The handles
carry the geometry d2d_create plans on a B200 (148 SMs): E = 4096 on 4-warp blocks, 1024 blocks of 7 x 148 resident,
late-wait steps on 3 x 148.
"""
from __future__ import annotations

import shutil
import subprocess
from pathlib import Path
from typing import List, NamedTuple

import pytest

ROOT = Path(__file__).resolve().parent.parent

FRESH, LATE = 1, 8                 # D2D_PF_INPUTS_FRESH, D2D_PF_LATE_WAIT
LAST_STEP, LAST_EPISODE = 1, 2     # D2D_LAST_*
STEP, MANY, EPISODE = 0, 1, 2      # MODE_*
CHUNK = 0x7fffffff // (6 * 50)     # the 32-bit bound of the default EnvConfig (N = 50 links, V = 76 devices)

_PROBE = r'''
#include "d2d_launch_plan.h"
#include <cstdio>
#include <cstring>
// handle E wpb grid envs_per_block grid_late pdl late_wait_on tickets_on chunk_override reward_fn
// step mode stream outputs stable autoreset agent_reward draw_actions no_reset
int main() {
    static const D2DWarpShape shapes[3] = {{2}, {4}, {8}};
    d2d_handle *h = nullptr;
    char cmd[16];
    while (std::scanf("%15s", cmd) == 1) {
        if (!std::strcmp(cmd, "handle")) {
            delete h;
            h = new d2d_handle();
            long long E, chunk;
            int wpb, pdl, late, tickets, reward;
            if (std::scanf("%lld %d %d %d %d %d %d %d %lld %d", &E, &wpb, &h->grid, &h->envs_per_block, &h->grid_late, &pdl, &late,
                           &tickets, &chunk, &reward) != 10) return 1;
            h->cfg.num_envs = E; h->cfg.reward_fn = reward;
            h->N = 50; h->V = 76;
            h->use_warp = true; h->warp = &shapes[wpb == 2 ? 0 : wpb == 4 ? 1 : 2];
            h->pdl = pdl; h->late_wait_on = late; h->tickets_on = tickets; h->chunk_override = chunk;
            h->dTickets = reinterpret_cast<uint64_t *>(uintptr_t{1} << 44);
        } else {
            int mode, outputs, stable, autoreset, agent, draw, no_reset;
            unsigned long long stream;
            if (std::scanf("%d %llu %d %d %d %d %d %d", &mode, &stream, &outputs, &stable, &autoreset, &agent, &draw, &no_reset) != 8) return 1;
            d2d_step_io_t io{};
            const uintptr_t base = (uintptr_t)outputs << 40;      // output set k: core outputs at their own addresses
            io.obs = reinterpret_cast<float *>(base);
            io.capacity_mbps = reinterpret_cast<float *>(base + (uintptr_t{1} << 36));
            io.reward = reinterpret_cast<float *>(base + (uintptr_t{2} << 36));
            io.done = reinterpret_cast<uint8_t *>(base + (uintptr_t{3} << 36));
            io.agent_reward = agent ? reinterpret_cast<float *>(base + (uintptr_t{4} << 36)) : nullptr;
            io.flags = (stable ? D2D_STEP_INPUTS_STABLE : 0u) | (autoreset ? D2D_STEP_AUTORESET : 0u);
            EpisodeArgs ea;
            ea.draw_actions = draw; ea.no_reset = no_reset;
            const D2DStepPlan pl = d2d_plan_step(h, &io, mode, reinterpret_cast<void *>(stream), ea);
            h->last_stream = reinterpret_cast<void *>(stream); h->last_kind = pl.last_kind;      // as step_launch does once enqueued
            std::printf("%u %d %llu %llu %lld %d\n", pl.flags, pl.grid, (unsigned long long)pl.tok_wait, (unsigned long long)pl.tok_sign,
                        (long long)pl.chunk, pl.last_kind);
        }
    }
    delete h;
    return 0;
}
'''


class Plan(NamedTuple):
    flags: int
    grid: int
    tok_wait: int = 0
    tok_sign: int = 0
    chunk: int = CHUNK
    last_kind: int = LAST_STEP


def tok(chain: int, seq: int) -> int:
    return (chain << 16) | seq


@pytest.fixture(scope='module')
def probe(tmp_path_factory):
    nvcc = shutil.which('nvcc') or ('/usr/local/cuda/bin/nvcc' if Path('/usr/local/cuda/bin/nvcc').exists() else None)
    if nvcc is None:
        pytest.skip('nvcc not found')
    d = tmp_path_factory.mktemp('plan')
    (d / 'plan_probe.cu').write_text(_PROBE)
    subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-std=c++17', '-diag-suppress', '159',
                    '-I', str(ROOT / 'gym_d2d_b200' / 'csrc'), '-o', str(d / 'plan_probe'), str(d / 'plan_probe.cu')],
                   check=True, capture_output=True)
    return d / 'plan_probe'


def handle(E=4096, wpb=4, grid=1024, epb=4, grid_late=444, pdl=1, late_wait=1, tickets=1, chunk=0, reward=0) -> str:
    return f'handle {E} {wpb} {grid} {epb} {grid_late} {pdl} {late_wait} {tickets} {chunk} {reward}'


def step(outputs=1, stream=1, stable=1, mode=STEP, autoreset=0, agent_reward=0, draw=0, no_reset=0) -> str:
    return f'step {mode} {stream} {outputs} {stable} {autoreset} {agent_reward} {draw} {no_reset}'


def plans(probe, *lines: str) -> List[Plan]:
    res = subprocess.run([str(probe)], input='\n'.join(lines) + '\n', check=True, capture_output=True, text=True)
    return [Plan(*map(int, ln.split())) for ln in res.stdout.split('\n') if ln]


def test_first_step_on_a_stream_waits_at_entry(probe):
    assert plans(probe, handle(), step()) == [Plan(FRESH, 1024)]


def test_late_wait_behind_a_step_with_disjoint_outputs(probe):
    """Ping-pong output sets at one env per warp: every step after the first stores ahead of the wait, on 3 x 148 blocks."""
    assert plans(probe, handle(), step(1), step(2), step(1)) == [Plan(FRESH, 1024), Plan(LATE, 444), Plan(LATE, 444)]


def test_aliased_outputs_hand_over_per_warp_beyond_one_env_per_warp(probe):
    """E = 6144 (1.5 envs per warp on the full 1036-block grid): the first step opens chain 1, the late-wait step breaks it,
    the next step that writes its predecessor's buffers opens chain 2 and the one after it follows."""
    assert plans(probe, handle(E=6144, grid=1036), step(1), step(2), step(2), step(2), step(2, stable=0)) == [
        Plan(FRESH, 1036, 0, tok(1, 1)), Plan(LATE, 444), Plan(0, 1036, 0, tok(2, 1)), Plan(0, 1036, tok(2, 1), tok(2, 2)),
        Plan(FRESH, 1036, 0, tok(3, 1))]


def test_aliased_outputs_at_one_env_per_warp_take_no_tokens(probe):
    assert plans(probe, handle(), step(1), step(1), step(1)) == [Plan(FRESH, 1024), Plan(0, 1024), Plan(0, 1024)]


def test_autoreset_step_waits_at_entry_and_so_does_the_step_after_it(probe):
    assert plans(probe, handle(), step(1), step(2, autoreset=1), step(1), step(2)) == [
        Plan(FRESH, 1024), Plan(FRESH, 1024, last_kind=LAST_EPISODE), Plan(FRESH, 1024), Plan(LATE, 444)]


def test_per_agent_reward_post_pass_keeps_the_late_wait_off(probe):
    """The post-pass kernel is the next step's predecessor in the stream: neither step may store ahead of the wait."""
    assert plans(probe, handle(), step(1), step(2, agent_reward=1), step(1)) == [Plan(FRESH, 1024), Plan(0, 1024), Plan(0, 1024)]
    assert plans(probe, handle(reward=1), step(1), step(2), step(1)) == [Plan(FRESH, 1024), Plan(0, 1024), Plan(0, 1024)]


def test_stream_change_waits_at_entry(probe):
    assert plans(probe, handle(), step(1, stream=1), step(2, stream=2), step(1, stream=2)) == [
        Plan(FRESH, 1024), Plan(FRESH, 1024), Plan(LATE, 444)]
    assert plans(probe, handle(E=6144, grid=1036), step(1, stream=1), step(1, stream=1), step(1, stream=2)) == [
        Plan(FRESH, 1036, 0, tok(1, 1)), Plan(0, 1036, tok(1, 1), tok(1, 2)), Plan(FRESH, 1036, 0, tok(2, 1))]


def test_late_wait_off(probe):
    assert plans(probe, handle(late_wait=0), step(1), step(2)) == [Plan(FRESH, 1024), Plan(0, 1024)]
    assert plans(probe, handle(E=6144, grid=1036, late_wait=0), step(1), step(2)) == [
        Plan(FRESH, 1036, 0, tok(1, 1)), Plan(0, 1036, tok(1, 1), tok(1, 2))]


def test_two_warp_blocks_past_1792_envs_on_the_full_grid_keep_the_grid_wide_wait(probe):
    assert plans(probe, handle(E=2048, wpb=2, grid=1024, epb=2, grid_late=0), step(1), step(2)) == [Plan(FRESH, 1024), Plan(0, 1024)]
    assert plans(probe, handle(E=1792, wpb=2, grid=896, epb=2, grid_late=0), step(1), step(2)) == [Plan(FRESH, 896), Plan(LATE, 896)]
    assert plans(probe, handle(E=2048, wpb=2, grid=1024, epb=2, grid_late=296), step(1), step(2)) == [Plan(FRESH, 1024), Plan(LATE, 296)]


def test_chunked_batch_neither_waits_late_nor_takes_tokens(probe):
    assert plans(probe, handle(E=6144, grid=1036, chunk=1000), step(1), step(2)) == [Plan(FRESH, 1036, chunk=1000), Plan(0, 1036, chunk=1000)]


def test_episode_with_drawn_actions_on_another_stream(probe):
    """It reads no input, so it never waits at entry for one; it writes positions, so the next step does."""
    assert plans(probe, handle(), step(1, stream=1), step(2, stream=2, mode=EPISODE, draw=1, stable=0), step(1, stream=2), step(2, stream=2)) == [
        Plan(FRESH, 1024), Plan(0, 1024, chunk=4096, last_kind=LAST_EPISODE), Plan(FRESH, 1024), Plan(LATE, 444)]
    # a rollout and a fused d2d_step_many read the positions like a step: behind a step, ahead of the wait
    assert plans(probe, handle(), step(1), step(1, mode=EPISODE, draw=1, no_reset=1), step(1, mode=MANY)) == [
        Plan(FRESH, 1024), Plan(0, 1024, chunk=4096), Plan(0, 1024, chunk=4096)]


def test_without_pdl_every_step_waits_at_entry(probe):
    assert plans(probe, handle(E=6144, grid=1036, pdl=0), step(1), step(2), step(2)) == [Plan(FRESH, 1036)] * 3
