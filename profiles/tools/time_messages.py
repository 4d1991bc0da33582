"""The tensor message channel (`MultiAgentTracking.exchange_messages`, DESIGN.md section 7i) against a torch composition
of the same work.

MATE-4v8-9 x 65 536 after 20 live steps, both teams, D in {8, 32, 128}, reduction none / sum / mean, a random recipients
mask (60 % of the pairs), with no filter and with range 1500 + dropout 0.25.  Per case, in one process and alternated
`--rounds` times:
  * kernel: `reps` calls of `env.exchange_messages` (fresh outputs each call, as users get them);
  * torch:  the same work composed of torch operations: the fp64 range mask, one `torch.rand` draw per pair, the inbox
    through `expand` / `where` (a batched product for sum / mean) and the edge adds.
Device time from CUDA events around `reps` calls queued behind a sleep kernel.  The inbox of every case but the smallest
is larger than the L2, so the writes reach HBM.  Algorithmic bytes: content read + mask read + output write + delivered
write; the fraction is of 6553 GB/s.  The card's name and power limit are read in the same call.

    python profiles/tools/time_messages.py [--reps 200] [--rounds 3] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PEAK_GBS = 6553.0


def card():
    query = 'name,power.limit,clocks.max.sm,driver_version'
    out = subprocess.run(['nvidia-smi', '--id=0', f'--query-gpu={query}', '--format=csv,noheader'],
                         capture_output=True, text=True, check=False).stdout.strip()
    return dict(zip(query.split(','), (x.strip() for x in out.split(',')))) if out else {}


def algorithmic_bytes(B, n, dim, reduction):
    out = n * n * dim if reduction == 'none' else n * dim
    return B * (n * dim * 4 + n * n + out * 4 + n * n)


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--envs', type=int, default=65536)
    parser.add_argument('--reps', type=int, default=200)
    parser.add_argument('--rounds', type=int, default=3)
    parser.add_argument('--out', default=None)
    args = parser.parse_args()
    sys.path.insert(0, ROOT)
    import numpy as np  # pylint: disable=import-outside-toplevel
    import torch  # pylint: disable=import-outside-toplevel

    import mate_b200  # pylint: disable=import-outside-toplevel

    assert torch.cuda.is_available(), 'time_messages.py measures on a GPU'
    B = args.envs
    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=B)
    env.reset(seed=1)
    gen = torch.Generator(device='cuda')
    gen.manual_seed(0)
    for _ in range(20):
        env.step((torch.rand((B, 4, 2), generator=gen, device='cuda') * 2 - 1, (torch.rand((B, 8, 2), generator=gen, device='cuda') * 2 - 1) * 20))

    def set_filter(restricted):
        env.message_rules = {'range_limit': [1500.0 if restricted else np.inf] * 2, 'keep_probability': [0.75 if restricted else 1.0] * 2}
        env.register_message_filter()

    def torch_exchange(team, content, mask, reduction, restricted, totals):
        xy = positions[team]
        deliver = mask
        if restricted:
            d = xy[:, :, None, :] - xy[:, None, :, :]
            deliver = deliver & (torch.sqrt((d * d).sum(-1)) <= 1500.0) & (torch.rand(mask.shape, device='cuda') < 0.75)
        by_recipient = deliver.transpose(1, 2)
        if reduction == 'none':
            inbox = torch.where(by_recipient[..., None], content[:, None].expand(-1, content.shape[1], -1, -1), 0.0)
        else:
            inbox = torch.bmm(by_recipient.float(), content)
            if reduction == 'mean':
                inbox = inbox / by_recipient.sum(-1, keepdim=True).clamp(min=1)
        totals += deliver
        return inbox, by_recipient

    def timed(call):
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(200_000_000)   # pylint: disable=protected-access  # the host queues every call before the device reaches them
        start.record()
        for _ in range(args.reps):
            call()
        end.record()
        torch.cuda.synchronize()
        return start.elapsed_time(end) * 1e3 / args.reps   # microseconds

    state = env.get_state()
    positions = [torch.from_numpy(state[name]).cuda() for name in ('cam_xy', 'tgt_xy')]
    cases = [(team, dim, reduction, restricted) for restricted in (False, True) for team in (0, 1) for dim in (8, 32, 128)
             for reduction in ('none', 'sum', 'mean')]
    rounds = {case: {'kernel_us': [], 'torch_us': []} for case in cases}
    for _ in range(args.rounds):
        for case in cases:
            team, dim, reduction, restricted = case
            n = (4, 8)[team]
            content = torch.randn((B, n, dim), generator=gen, device='cuda')
            mask = torch.rand((B, n, n), generator=gen, device='cuda') < 0.6
            totals = torch.zeros((B, n, n), dtype=torch.int32, device='cuda')
            set_filter(restricted)
            rounds[case]['kernel_us'].append(timed(lambda: env.exchange_messages(team, content, mask, reduction)))   # noqa: B023
            rounds[case]['torch_us'].append(timed(lambda: torch_exchange(team, content, mask, reduction, restricted, totals)))   # noqa: B023
            del content, mask, totals
            torch.cuda.empty_cache()
    results = []
    for case in cases:
        team, dim, reduction, restricted = case
        n = (4, 8)[team]
        kernel, baseline = float(np.median(rounds[case]['kernel_us'])), float(np.median(rounds[case]['torch_us']))
        nbytes = algorithmic_bytes(B, n, dim, reduction)
        results.append({'team': ('cameras', 'targets')[team], 'dim': dim, 'reduction': reduction,
                        'filter': 'range+dropout' if restricted else 'none', 'kernel_us': kernel, 'torch_us': baseline,
                        'kernel_rounds_us': rounds[case]['kernel_us'], 'torch_rounds_us': rounds[case]['torch_us'],
                        'bytes': nbytes, 'fraction_of_6553': nbytes / (kernel * 1e-6) / 1e9 / PEAK_GBS})
    report = {'card': card(), 'envs': B, 'reps': args.reps, 'rounds': args.rounds, 'results': results}
    text = json.dumps(report, indent=1)
    print(f"{report['card']}")
    print(f"{'team':8s} {'D':>4s} {'reduction':9s} {'filter':14s} {'kernel us':>10s} {'torch us':>10s} {'MB':>8s} {'of 6553':>8s}")
    for r in results:
        print(f"{r['team']:8s} {r['dim']:4d} {r['reduction']:9s} {r['filter']:14s} {r['kernel_us']:10.1f} {r['torch_us']:10.1f} "
              f"{r['bytes'] / 1e6:8.1f} {r['fraction_of_6553']:8.3f}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w', encoding='utf-8') as f:
            f.write(text)
    env.close()


if __name__ == '__main__':
    main()
