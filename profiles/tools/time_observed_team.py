"""Observation rows for one team (observed_team / NULL row pointers): what the single-team step saves, measured.

1. Step-kernel time per launch for observed_team 'both' / 'camera' / 'target', float32 and float16, on MATE-4v8-9 x 65 536,
   MATE-8v8-9 x 32 768 and MATE-4v2-9 x 65 536: bench.py's steady state (staggered episode clocks, settle and warm-up
   steps), CUDA events around `--steps` step launches, the six variants of a workload alternated over `--rounds` rounds in
   one process.  Each variant's share of the HBM peak uses its own algorithmic bytes (bench.algorithmic_bytes with the
   unobserved team's rows left out and the rows at 2 bytes for float16).
2. The README's MultiCamera stack (greedy targets, MoreTrainingInformation, RepeatedRewardIndividualDone,
   AuxiliaryCameraRewards) end to end on MATE-4v8-9 x 65 536, observed_team 'both' against 'camera', alternated.
3. mate_b200_step_host env-steps/s on the dense and the compacted leg, 'both' against 'camera'.

The card's name, power limit and maximum SM clock are printed beside the numbers.

    python profiles/tools/time_observed_team.py [--steps 200] [--rounds 3] [--e2e-steps 100] [--host-steps 10]
"""

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from mate_b200 import _abi  # noqa: E402
from mate_b200.config import flatten_config, read_config  # noqa: E402
from mate_b200.sim import BatchedSim  # noqa: E402
from time_obs_format import card  # noqa: E402

WORKLOADS = (('MATE-4v8-9.yaml', 65536), ('MATE-8v8-9.yaml', 32768), ('MATE-4v2-9.yaml', 65536))
TEAMS = ('both', 'camera', 'target')
FORMATS = {'float32': torch.float32, 'float16': torch.float16}


def team_row_bytes(cfg, team, dtype):
    nc, nt, no = cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']
    dc, dt = 22 + 5 * nt + 4 * no + 7 * nc, 27 + 7 * nc + 4 * no + 5 * nt
    size = 2 if dtype == torch.float16 else 4
    return {'camera': nc * dc * size, 'target': nt * dt * size}[team]


def algorithmic_bytes(cfg, team, dtype):
    """bench.algorithmic_bytes (float32 rows of both teams) with the rows this variant writes."""
    full = bench.algorithmic_bytes(cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles'])
    rows32 = team_row_bytes(cfg, 'camera', torch.float32) + team_row_bytes(cfg, 'target', torch.float32)
    written = sum(team_row_bytes(cfg, t, dtype) for t in ('camera', 'target') if team in ('both', t))
    return full - rows32 + written


def steady_sim(cfg, B, dtype, team, cams, tgts, settle):
    sim = BatchedSim(cfg, B, device=0, observation_dtype=dtype, observed_team=team)
    sim.reset(seed=0)
    steps0 = np.random.RandomState(1234).randint(0, cfg['max_episode_steps'] + 1, size=B).astype(np.int32)
    sim.set_state({'episode_step': steps0})
    sim.alloc_aux()
    for name, ctype, _, _ in _abi.AUX_FIELDS:   # the aux outputs bench.py's timed step keeps
        if name not in ('coverage', 'num_delivered'):
            setattr(sim._aux_struct, name, ctype())   # pylint: disable=protected-access
    for k in range(settle):
        sim.step(cams[k % len(cams)], tgts[k % len(tgts)], auto_reset=True, aux=True)
    return sim


def time_device(sim, cams, tgts, steps, warmup):
    ring = len(cams)
    for k in range(warmup):
        sim.step(cams[k % ring], tgts[k % ring], auto_reset=True, aux=True)
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(2_000_000)   # pylint: disable=protected-access  # the host runs ahead: no launch gap is timed
    start.record()
    for k in range(steps):
        sim.step(cams[k % ring], tgts[k % ring], auto_reset=True, aux=True)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / steps


def device_part(args, peak):
    out = {}
    for config, B in WORKLOADS:
        cfg = flatten_config(read_config(config))
        cams, tgts = bench.make_actions(cfg, B, torch.device('cuda', 0), 8, seed=0)
        variants = [(team, fmt) for fmt in FORMATS for team in TEAMS]
        times = {v: [] for v in variants}
        for r in range(args.rounds):
            for team, fmt in (variants if r % 2 == 0 else variants[::-1]):
                sim = steady_sim(cfg, B, FORMATS[fmt], team, cams, tgts, args.settle)
                ms = time_device(sim, cams, tgts, args.steps, args.warmup)
                sim.close()
                del sim
                times[(team, fmt)].append(ms)
                print(f'{config} x {B} round {r} {team} {fmt}: {ms * 1e3:.1f} us/step', flush=True)
        res = {}
        for (team, fmt), runs in times.items():
            ms = float(np.median(runs))
            A = algorithmic_bytes(cfg, team, FORMATS[fmt])
            achieved = A * B / (ms * 1e-3) / 1e9
            res[f'{team} {fmt}'] = {'us_per_step_median': 1e3 * ms, 'us_per_step_runs': [1e3 * t for t in runs],
                                    'spread_us': 1e3 * (max(runs) - min(runs)), 'algorithmic_bytes_per_env_step': A,
                                    'achieved_gbs': achieved, 'frac_of_hbm_peak': achieved / peak}
        out[f'{config.replace(".yaml", "")} x {B}'] = res
    return out


def camera_stack(team, B):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    return mate.make('MATE-4v8-9-v0', num_envs=B, observed_team=team, wrappers=[
        mate.MoreTrainingInformation, mate.RepeatedRewardIndividualDone,
        lambda e: mate.AuxiliaryCameraRewards(e, coefficients={'raw_reward': 1.0, 'coverage_rate': 1.0}, reduction='mean'),
        lambda e: mate.MultiCamera(e, target_agent=mate.GreedyTargetAgent(seed=0))])


def e2e_part(args):
    B = 65536
    gen = torch.Generator(device='cuda')
    gen.manual_seed(0)
    acts = [((torch.rand((B, 4, 2), device='cuda', generator=gen) * 2 - 1) * torch.tensor([5.0, 2.5], device='cuda')) for _ in range(8)]
    envs = {team: camera_stack(team, B) for team in ('both', 'camera')}
    for env in envs.values():
        env.reset(seed=0)
        for k in range(args.warmup):
            env.step(acts[k % 8])
    times = {team: [] for team in envs}
    for r in range(args.rounds):
        for team in (('both', 'camera') if r % 2 == 0 else ('camera', 'both')):
            env = envs[team]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(args.e2e_steps):
                env.step(acts[k % 8])
            torch.cuda.synchronize()
            times[team].append((time.perf_counter() - t0) / args.e2e_steps)
            print(f'MultiCamera stack round {r} {team}: {1e3 * times[team][-1]:.3f} ms/step', flush=True)
    for env in envs.values():
        env.unwrapped.close()
    return {team: {'ms_per_step_median': 1e3 * float(np.median(t)), 'ms_per_step_runs': [1e3 * x for x in t],
                   'env_steps_per_s': B / float(np.median(t))} for team, t in times.items()}


def host_part(args):
    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))
    B = 65536
    cams, tgts = bench.make_actions(cfg, B, torch.device('cuda', 0), 8, seed=0)
    host_cam = [c.cpu().pin_memory() for c in cams[:2]]
    host_tgt = [t.cpu().pin_memory() for t in tgts[:2]]
    out = {}
    for leg, compact in (('dense copy', '0'), ('compacted', '1')):
        for team in ('both', 'camera'):
            os.environ['MATE_B200_HOST_COMPACT'] = compact   # read once per simulator, by its first step_host call
            sim = steady_sim(cfg, B, torch.float32, team, cams, tgts, args.settle)
            rows = (torch.zeros((B, 4, sim.dc)).pin_memory(), torch.zeros((B, 8, sim.dt)).pin_memory() if team == 'both' else None,
                    torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
            for k in range(3):
                sim.step_host(host_cam[k % 2], host_tgt[k % 2], rows)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(args.host_steps):
                sim.step_host(host_cam[k % 2], host_tgt[k % 2], rows)
            seconds = time.perf_counter() - t0
            leg_used, link = sim.host_leg_info()
            sim.close()
            out.setdefault(leg, {})[team] = {'env_steps_per_s': B * args.host_steps / seconds, 'ms_per_step': 1e3 * seconds / args.host_steps,
                                             'leg': leg_used, 'row_bytes_on_link_last_step': link}
            print(f'step_host {leg} {team}: {json.dumps(out[leg][team])}', flush=True)
    return out


def main():
    parser = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    parser.add_argument('--steps', type=int, default=200, help='timed device steps per variant and round')
    parser.add_argument('--warmup', type=int, default=20)
    parser.add_argument('--settle', type=int, default=64)
    parser.add_argument('--rounds', type=int, default=3)
    parser.add_argument('--e2e-steps', type=int, default=100, help='timed steps of the MultiCamera stack per round (0 = skip)')
    parser.add_argument('--host-steps', type=int, default=10, help='timed step_host calls per leg and team (0 = skip)')
    parser.add_argument('--out', help='write the JSON result here too')
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_observed_team.py measures on a GPU; none is visible')
    peak, peak_source = bench.measured_peak_gbs()
    info = card()
    print('card:', json.dumps(info), flush=True)
    result = {'card': info, 'hbm_peak_gbs': peak, 'hbm_peak_source': peak_source,
              'method': f'staggered episode clocks, {args.settle} settle + {args.warmup} warm-up steps, CUDA events around '
                        f'{args.steps} step launches, variants alternated over {args.rounds} rounds',
              'device': device_part(args, peak)}
    if args.e2e_steps > 0:
        result['multicamera_stack'] = e2e_part(args)
    if args.host_steps > 0:
        result['step_host'] = host_part(args)
    result['card_after'] = card()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, 'w', encoding='UTF-8') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
