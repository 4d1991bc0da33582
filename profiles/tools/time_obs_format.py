"""float32 against float16 observation rows (mate_b200_set_observation_format), alternated in one process.

The device-resident step is timed with bench.py's method: 65 536 environments, episode clocks staggered uniformly over one
episode, `--settle` untimed steps, `--warmup` untimed steps, CUDA events around K step launches.  The two formats take
turns for `--rounds` rounds (the first format of a round alternates), so drift of the shared host or of the clocks falls
on both.  Each format's share of the HBM peak uses its own algorithmic bytes (bench.algorithmic_bytes with the rows at 2
bytes for float16).  Then mate_b200_step_host is timed for both formats on each device -> host leg.  The card's name, power
limit and maximum SM clock are printed beside the numbers.

    python profiles/tools/time_obs_format.py [--config MATE-4v8-9.yaml] [--envs 65536] [--steps 500] [--rounds 3]
"""

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from mate_b200.config import flatten_config, read_config  # noqa: E402
from mate_b200.sim import BatchedSim  # noqa: E402

FORMATS = {'float32': torch.float32, 'float16': torch.float16}
LEGS = {   # name -> (MATE_B200_HOST_COMPACT, rows_kept)
    'dense copy': ('0', False),
    'non-zero 16-byte chunks, rebuilt by host threads': ('1', False),
    'changed 64-byte groups patched into kept rows': ('1', True),
}


def card():
    query = 'name,power.limit,clocks.max.sm,driver_version'
    out = subprocess.run(['nvidia-smi', '--id=0', f'--query-gpu={query}', '--format=csv,noheader'],
                         capture_output=True, text=True, check=False).stdout.strip()
    return dict(zip(query.split(','), (x.strip() for x in out.split(',')))) if out else {'name': torch.cuda.get_device_name(0)}


def row_bytes(cfg, dtype):
    nc, nt, no = cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']
    dc, dt = 22 + 5 * nt + 4 * no + 7 * nc, 27 + 7 * nc + 4 * no + 5 * nt
    return (nc * dc + nt * dt) * (2 if dtype == torch.float16 else 4)


def algorithmic_bytes(cfg, dtype):
    nc, nt, no = cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']
    return bench.algorithmic_bytes(nc, nt, no) - row_bytes(cfg, torch.float32) + row_bytes(cfg, dtype)


def steady_sim(cfg, B, dtype, cams, tgts, settle):
    """A simulator in bench.py's steady state: staggered episode clocks, `settle` steps from the reset."""
    sim = BatchedSim(cfg, B, device=0, observation_dtype=dtype)
    sim.reset(seed=0)
    steps0 = np.random.RandomState(1234).randint(0, cfg['max_episode_steps'] + 1, size=B).astype(np.int32)
    sim.set_state({'episode_step': steps0})
    sim.alloc_aux()
    from mate_b200 import _abi  # pylint: disable=import-outside-toplevel

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


def time_host(cfg, B, dtype, cams, tgts, settle, compact, kept, steps):
    os.environ['MATE_B200_HOST_COMPACT'] = compact   # read once per simulator, by its first step_host call
    sim = steady_sim(cfg, B, dtype, cams, tgts, settle)
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    host_cam = [c.cpu().pin_memory() for c in cams[:2]]
    host_tgt = [t.cpu().pin_memory() for t in tgts[:2]]
    out = (torch.zeros((B, max(nc, 1), sim.dc), dtype=dtype).pin_memory(), torch.zeros((B, nt, sim.dt), dtype=dtype).pin_memory(),
           torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
    for k in range(3):
        sim.step_host(host_cam[k % 2], host_tgt[k % 2], out, auto_reset=True, rows_kept=kept)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        sim.step_host(host_cam[k % 2], host_tgt[k % 2], out, auto_reset=True, rows_kept=kept)
    seconds = time.perf_counter() - t0
    leg, link = sim.host_leg_info()
    sim.close()
    return {'env_steps_per_s': B * steps / seconds, 'ms_per_step': 1e3 * seconds / steps, 'leg': leg, 'row_bytes_on_link_last_step': link}


def main():
    parser = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    parser.add_argument('--config', default='MATE-4v8-9.yaml')
    parser.add_argument('--envs', type=int, default=65536)
    parser.add_argument('--steps', type=int, default=500, help='timed device steps per format and round')
    parser.add_argument('--warmup', type=int, default=20)
    parser.add_argument('--settle', type=int, default=64)
    parser.add_argument('--rounds', type=int, default=3)
    parser.add_argument('--host-steps', type=int, default=10, help='timed step_host calls per format and leg (0 = skip)')
    args = parser.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_obs_format.py measures on a GPU; none is visible')

    cfg = flatten_config(read_config(args.config))
    B = args.envs
    cams, tgts = bench.make_actions(cfg, B, torch.device('cuda', 0), 8, seed=0)
    peak, peak_source = bench.measured_peak_gbs()
    info = card()
    print('card:', json.dumps(info), flush=True)

    sims = {name: steady_sim(cfg, B, dtype, cams, tgts, args.settle) for name, dtype in FORMATS.items()}
    times = {name: [] for name in FORMATS}
    order = list(FORMATS)
    for r in range(args.rounds):
        for name in (order if r % 2 == 0 else order[::-1]):
            ms = time_device(sims[name], cams, tgts, args.steps, args.warmup)
            times[name].append(ms)
            print(f'round {r} {name}: {ms:.4f} ms/step', flush=True)
    for sim in sims.values():
        sim.close()

    device = {}
    for name, dtype in FORMATS.items():
        ms = float(np.median(times[name]))
        A = algorithmic_bytes(cfg, dtype)
        achieved = A * B / (ms * 1e-3) / 1e9
        device[name] = {'ms_per_step_median': ms, 'ms_per_step_runs': times[name], 'spread_ms': max(times[name]) - min(times[name]),
                        'env_steps_per_s': B / (ms * 1e-3), 'algorithmic_bytes_per_env_step': A, 'achieved_gbs': achieved,
                        'frac_of_hbm_peak': achieved / peak}
    host = {}
    if args.host_steps > 0:
        for leg, (compact, kept) in LEGS.items():
            for name, dtype in FORMATS.items():
                host.setdefault(leg, {})[name] = time_host(cfg, B, dtype, cams, tgts, args.settle, compact, kept, args.host_steps)
                print(f'step_host {leg} {name}: {json.dumps(host[leg][name])}', flush=True)
    f32, f16 = device['float32'], device['float16']
    print(json.dumps({
        'workload': f'{args.config.replace(".yaml", "")} x {B} envs', 'card': info, 'hbm_peak_gbs': peak, 'hbm_peak_source': peak_source,
        'method': f'staggered episode clocks, {args.settle} settle + {args.warmup} warm-up steps, CUDA events around {args.steps} '
                  f'step launches, formats alternated over {args.rounds} rounds',
        'device': device, 'step_host': host,
        'float16_faster_by_ms': f32['ms_per_step_median'] - f16['ms_per_step_median'],
        'larger_spread_ms': max(f32['spread_ms'], f16['spread_ms']),
    }))


if __name__ == '__main__':
    main()
