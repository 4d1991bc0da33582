"""Rendering time of `BatchedSim.render` / `MultiAgentTracking.render` (mate_b200_render, DESIGN.md section 7k).

Per preset (MATE-4v8-9, MATE-8v8-9, MATE-Navigation), a batch of 4096 environments after 50 live steps; K frames of
environments spread over the batch, K in {1, 16, 64}, at S in {256, 800, 1024}.  Device time of one call from CUDA
events around `reps` calls (fresh output tensors, as users get them) after a warm-up, best of `rounds`.  The written
bytes are K S^2 3; the card's name and power limit are read in the same call.  MATE-Navigation has no cameras, so its
frames have no field of view: its times are the cost of everything else in the picture.

    python profiles/tools/time_render.py [--reps 20] [--rounds 3] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PRESETS = ('MATE-4v8-9.yaml', 'MATE-8v8-9.yaml', 'MATE-Navigation.yaml')


def card():
    query = 'name,power.limit,clocks.max.sm,driver_version'
    out = subprocess.run(['nvidia-smi', '--id=0', f'--query-gpu={query}', '--format=csv,noheader'],
                         capture_output=True, text=True, check=False).stdout.strip()
    return dict(zip(query.split(','), (x.strip() for x in out.split(',')))) if out else {}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--envs', type=int, default=4096)
    parser.add_argument('--reps', type=int, default=20)
    parser.add_argument('--rounds', type=int, default=3)
    parser.add_argument('--out', default=None)
    args = parser.parse_args()
    sys.path.insert(0, ROOT)
    import torch  # pylint: disable=import-outside-toplevel

    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    assert torch.cuda.is_available(), 'time_render.py measures on a GPU'
    B = args.envs
    rows = []
    for preset in PRESETS:
        cfg = flatten_config(read_config(preset))
        sim = BatchedSim(cfg, B, device=0)
        sim.reset(seed=1)
        gen = torch.Generator(device='cuda')
        gen.manual_seed(0)
        nc, nt = int(cfg['num_cameras']), int(cfg['num_targets'])
        scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
        for _ in range(50):
            cam = (torch.rand((B, max(nc, 1), 2), generator=gen, device='cuda') * 2 - 1) * scale
            tgt = (torch.rand((B, nt, 2), generator=gen, device='cuda') * 2 - 1) * cfg['target_step_size']
            sim.step(cam[:, :nc].contiguous(), tgt, auto_reset=True)
        for K in (1, 16, 64):
            envs = torch.linspace(0, B - 1, K, device='cuda').to(torch.int32)
            for S in (256, 800, 1024):
                for _ in range(3):
                    sim.render(envs, size=S)
                torch.cuda.synchronize()
                best = float('inf')
                for _ in range(args.rounds):
                    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    start.record()
                    for _ in range(args.reps):
                        sim.render(envs, size=S)
                    stop.record()
                    stop.synchronize()
                    best = min(best, start.elapsed_time(stop) / args.reps)
                mb = K * S * S * 3 / 1e6
                rows.append({'preset': preset, 'K': K, 'S': S, 'ms': round(best, 4), 'MB': round(mb, 2),
                             'GB/s': round(mb / best, 1)})
                print(json.dumps(rows[-1]), flush=True)
        sim.close()
    result = {'card': card(), 'envs': B, 'reps': args.reps, 'rounds': args.rounds, 'rows': rows}
    print(json.dumps({'card': result['card']}))
    if args.out:
        with open(args.out, 'w', encoding='utf-8') as f:
            json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
