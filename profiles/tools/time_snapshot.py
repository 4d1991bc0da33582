"""Device-side state snapshots (mate_b200_save_state / mate_b200_load_state) against their yardsticks, in one process.

MATE-4v8-9 x 65 536 by default.  Cases:
  * full-batch save; full-batch load (scatter only: a handle without prepared resets, MATE_B200_REFILL=off);
  * full-batch load on a handle with prepared resets (the default): the load waits for the previous load's re-prepare
    of every environment, so back-to-back loads measure load + prepare;
  * a 64-entry snapshot loaded into every environment through a device map (the branching pattern);
  * a device-to-device cudaMemcpyAsync (tensor.copy_) of the full-batch payload bytes;
  * get_state / set_state of the full batch (host clock, they synchronise).
The device calls are timed with CUDA events: a sleep kernel first lets the host queue every call, so the events see
device time, not the enqueue.  "warm": `--reps` calls back to back (the 47 MB state and payload partly stay in the
126 MB L2); "cold": each call timed on its own after a 256 MB write that evicts the L2.  The card's name and power limit
are read in the same call and printed beside the numbers.

    python profiles/tools/time_snapshot.py [--config MATE-4v8-9.yaml] [--envs 65536] [--reps 200] [--out FILE]
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mate_b200 import _abi  # noqa: E402
from mate_b200.config import flatten_config, read_config  # noqa: E402
from mate_b200.sim import BatchedSim, _check, _dptr  # noqa: E402


def card():
    query = 'name,power.limit,clocks.max.sm,driver_version'
    out = subprocess.run(['nvidia-smi', '--id=0', f'--query-gpu={query}', '--format=csv,noheader'],
                         capture_output=True, text=True, check=False).stdout.strip()
    return dict(zip(query.split(','), (x.strip() for x in out.split(',')))) if out else {'name': torch.cuda.get_device_name(0)}


def timed(call, reps, flush=None):
    """Mean device time of `call` in microseconds: back to back (flush None) or each after `flush`."""
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps if flush else 1)]
    torch.cuda._sleep(200_000_000)   # ~0.1 s: the host queues everything below before the device reaches it
    if flush is None:
        events[0][0].record()
        for _ in range(reps):
            call()
        events[0][1].record()
        torch.cuda.synchronize()
        return events[0][0].elapsed_time(events[0][1]) * 1e3 / reps
    for start, end in events:
        flush()
        start.record()
        call()
        end.record()
    torch.cuda.synchronize()
    return float(np.mean([s.elapsed_time(e) for s, e in events])) * 1e3


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--config', default='MATE-4v8-9.yaml')
    parser.add_argument('--envs', type=int, default=65536)
    parser.add_argument('--reps', type=int, default=200)
    parser.add_argument('--out', default=None)
    args = parser.parse_args()
    info_card = card()
    cfg = flatten_config(read_config(args.config))
    B = args.envs
    sims = {}
    for refill in ('off', 'default'):
        if refill == 'off':
            os.environ['MATE_B200_REFILL'] = 'off'
        else:
            os.environ.pop('MATE_B200_REFILL', None)
        sim = BatchedSim(cfg, B, device=0)
        sim.reset(seed=0)
        gen = torch.Generator(device='cuda')
        gen.manual_seed(0)
        for _ in range(16):
            cam = (torch.rand((B, sim.nc, 2), generator=gen, device='cuda') * 2 - 1) * torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
            tgt = (torch.rand((B, sim.nt, 2), generator=gen, device='cuda') * 2 - 1) * cfg['target_step_size']
            sim.step(cam, tgt, auto_reset=True)
        sims[refill] = sim
    torch.cuda.synchronize()

    sim = sims['off']
    lib, stream = sim.lib, sim._stream()   # pylint: disable=protected-access
    full = sim.save_state()
    branch = sim.save_state(list(range(0, B, B // 64))[:64])
    src = torch.from_numpy(np.random.default_rng(0).integers(0, 64, B).astype(np.int32)).cuda()
    info_full, info_branch = full.info(), branch.info()
    copy_dst = torch.empty_like(full.payload)
    scrub = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def save(s):
        info = _abi.MateSnapshotInfo()
        return lambda: _check(lib, lib.mate_b200_save_state(s.handle, None, B, _dptr(full.payload), ctypes.byref(info), stream))

    def load(s, payload, info, index):
        return lambda: _check(lib, lib.mate_b200_load_state(s.handle, _dptr(payload), ctypes.byref(info), _dptr(index), 0, stream))

    cases = {
        'save, full batch': save(sim),
        'load, full batch (scatter only, refill off)': load(sim, full.payload, info_full, None),
        'load, full batch, with re-prepare (default refill)': load(sims['default'], full.payload, info_full, None),
        'load, 64-entry snapshot through src into every env': load(sim, branch.payload, info_branch, src),
        'device-to-device cudaMemcpyAsync of the payload bytes': lambda: copy_dst.copy_(full.payload),
    }
    results = {'card': info_card, 'config': args.config, 'envs': B, 'payload_bytes_full': full.payload_bytes,
               'payload_bytes_64': branch.payload_bytes, 'reps': args.reps, 'us': {}}
    for name, call in cases.items():
        reps = args.reps if 'prepare' not in name else max(10, args.reps // 10)
        warm = timed(call, reps)
        cold = timed(call, max(10, reps // 4), flush=lambda: scrub.zero_())
        results['us'][name] = {'warm': round(warm, 2), 'cold': round(cold, 2)}
        print(f'{name:60s} warm {warm:9.2f} us   cold {cold:9.2f} us', flush=True)
    for name in ('get_state', 'set_state'):
        state = sim.get_state()
        times = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if name == 'get_state':
                sim.get_state()
            else:
                sim.set_state(state)
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t0) * 1e6)
        results['us'][f'{name}, full batch (host clock)'] = {'min': round(min(times), 1), 'max': round(max(times), 1)}
        print(f'{name + ", full batch (host clock)":60s} {min(times):12.1f} - {max(times):.1f} us', flush=True)
    copy = results['us']['device-to-device cudaMemcpyAsync of the payload bytes']
    for name in ('save, full batch', 'load, full batch (scatter only, refill off)'):
        for kind in ('warm', 'cold'):
            print(f'{name} / memcpy ({kind}): {results["us"][name][kind] / copy[kind]:.2f}')
    print(json.dumps(results))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w', encoding='UTF-8') as f:
            json.dump(results, f, indent=1)
    for s in sims.values():
        s.close()


if __name__ == '__main__':
    main()
