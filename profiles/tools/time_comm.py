"""The batched greedy teams with and without communication wrappers (DESIGN.md section 7h), against another tree.

Per configuration (MATE-4v8-9 x 65 536, MATE-8v8-9 x 32 768), after 50 live steps so that the agents' memories hold
real traffic:
  * each greedy kernel (mate_b200_greedy_target_actions / _camera_actions) on a fixed state, with
      none          no filter registered (the library's default),
      edges         an unrestricted filter with the edge tensors (what a batched environment registers by itself),
      range         range_limit 1500 + edges,
      range+drop    range_limit 1500, keep probability 0.75 + edges;
  * MultiCamera.step / MultiTarget.step with zero actions for the learning team, without a communication wrapper and
    with RestrictedCommunicationRange(RandomMessageDropout(env, 0.25), 1500).
Device time from CUDA events around `--reps` calls queued behind a sleep kernel.  A tree without
`BatchedSim.set_message_filter` (the parent) runs the cases that need no filter.  With `--parent DIR` the script runs
itself on this tree and on DIR in alternation (`--rounds`), each in a fresh process, and reports every round.  The card's
name and power limit are read in the same call.

    python profiles/tools/time_comm.py --parent /path/to/parent/tree [--rounds 3] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CONFIGS = (('MATE-4v8-9.yaml', 65536), ('MATE-8v8-9.yaml', 32768))


def card():
    query = 'name,power.limit,clocks.max.sm,driver_version'
    out = subprocess.run(['nvidia-smi', '--id=0', f'--query-gpu={query}', '--format=csv,noheader'],
                         capture_output=True, text=True, check=False).stdout.strip()
    return dict(zip(query.split(','), (x.strip() for x in out.split(',')))) if out else {}


def measure(tree, reps):
    sys.path.insert(0, tree)
    import torch  # pylint: disable=import-outside-toplevel

    import mate_b200  # pylint: disable=import-outside-toplevel
    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    def timed(call):
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(200_000_000)   # the host queues every call below before the device reaches them
        start.record()
        for _ in range(reps):
            call()
        end.record()
        torch.cuda.synchronize()
        return start.elapsed_time(end) * 1e3 / reps   # microseconds

    filtering = hasattr(BatchedSim, 'set_message_filter')
    results = {}
    for config, B in CONFIGS:
        sim = BatchedSim(flatten_config(read_config(config)), B, device=0)
        sim.reset(seed=1)
        sim.observe(aux=True)
        targets, cameras = mate_b200.GreedyTargetAgent(seed=2), mate_b200.GreedyCameraAgent(seed=3)
        targets.bind(sim)
        cameras.bind(sim)
        nt = sim.nt

        def tracked():
            return (sim.cam_obs[..., 26:22 + 5 * nt:5] > 0.5).to(torch.uint8)

        reset = True
        for _ in range(50):
            t_act = targets.act(reset_mask=reset).clone()
            c_act = cameras.act(tracked(), reset_mask=reset).clone()
            reset = None
            sim.step(c_act, t_act, auto_reset=True, aux=True)
        flags = tracked()
        delivered = tuple(torch.zeros(B, dtype=torch.int64, device=sim.device) for _ in range(2))
        totals = tuple(torch.zeros((B, n, n), dtype=torch.int32, device=sim.device) for n in (sim.nc, sim.nt))
        variants = {'none': {}}
        if filtering:
            edges = {'delivered': delivered, 'total_edges': totals}
            variants.update({'edges': edges, 'range': dict(edges, range_limit=(1500.0, 1500.0)),
                             'range+drop': dict(edges, range_limit=(1500.0, 1500.0), keep_probability=(0.75, 0.75))})
        for name, kwargs in variants.items():
            if filtering:
                sim.set_message_filter(**kwargs)
            results[f'{config} greedy_target_kernel {name}'] = timed(lambda: targets.act())
            results[f'{config} greedy_camera_kernel {name}'] = timed(lambda: cameras.act(flags))
        sim.close()
        for wrapped in ((False, True) if filtering else (False,)):
            for team in ('MultiCamera', 'MultiTarget'):
                def single_team(e, team=team, wrapped=wrapped):
                    if wrapped:
                        e = mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.25), range_limit=1500)
                    if team == 'MultiCamera':
                        return mate_b200.MultiCamera(e, target_agent=mate_b200.GreedyTargetAgent(seed=2))
                    return mate_b200.MultiTarget(e, camera_agent=mate_b200.GreedyCameraAgent(seed=3))

                env = mate_b200.make('MultiAgentTracking-v0', config=config, num_envs=B, wrappers=[single_team])
                env.reset(seed=1)
                base = env.unwrapped
                zeros = torch.zeros((B, base.num_cameras if team == 'MultiCamera' else base.num_targets, 2), device='cuda')
                for _ in range(50):
                    env.step(zeros)
                results[f'{config} {team}.step {"range+drop wrappers" if wrapped else "no wrapper"}'] = timed(lambda: env.step(zeros))
                env.close()
    return results


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument('--tree', default=None, help='measure the package of this tree in this process')
    parser.add_argument('--parent', default=None, help='alternate this tree and the parent tree, each in a fresh process')
    parser.add_argument('--rounds', type=int, default=3)
    parser.add_argument('--reps', type=int, default=200)
    parser.add_argument('--out', default=None)
    args = parser.parse_args()
    if args.tree is not None:
        print(json.dumps(measure(args.tree, args.reps)))
        return
    trees = {'this': ROOT}
    if args.parent:
        trees['parent'] = os.path.abspath(args.parent)
    rounds = []
    for r in range(args.rounds):
        for label, tree in trees.items():
            out = subprocess.run([sys.executable, os.path.abspath(__file__), '--tree', tree, '--reps', str(args.reps)],
                                 capture_output=True, text=True, check=True, cwd=tree).stdout
            rounds.append({'round': r, 'tree': label, 'us': json.loads(out.strip().splitlines()[-1])})
            print(json.dumps(rounds[-1]), flush=True)
    report = {'card': card(), 'reps': args.reps, 'rounds': rounds}
    if args.out:
        with open(args.out, 'w', encoding='UTF-8') as file:
            json.dump(report, file, indent=1)
    print(json.dumps(report['card']))


if __name__ == '__main__':
    main()
