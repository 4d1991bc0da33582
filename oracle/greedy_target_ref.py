"""NumPy restatement of ``GreedyTargetAgent`` (mate/agents/greedy.py:235-365) for a whole team, driven like
``group_step`` (mate/wrappers/single_team.py:79-92: observe -> communicate -> act) -- TEST INFRASTRUCTURE: the
checker of the CUDA kernel, itself pinned against recorded reference agents in ``tests/golden/agents_*.npz``."""

import numpy as np

WAREHOUSES = np.array([[925.0, 925.0], [-925.0, 925.0], [-925.0, -925.0], [925.0, -925.0]])   # constants.py:70-72


def communicated_non_empty(empty_bits, non_empty):
    """The remembered non-empty warehouse sets [Nt] after observe -> process_messages -> communicate, from the sets
    before the step; the goal choice of the act phase draws from these."""
    nt = len(empty_bits)
    non_empty = non_empty.copy()
    # observe -> process_messages (greedy.py:330-336)
    sends = np.zeros(nt, dtype=bool)
    for t in range(nt):
        seen = sum(1 << w for w in range(4) if empty_bits[t, w])
        if seen & non_empty[t]:
            non_empty[t] &= ~seen
            sends[t] = True
    # communicate: broadcasts reach every teammate (environment.py:1249-1269); greedy.py:338-365
    sent = [non_empty[t] for t in range(nt) if sends[t]]
    for t in range(nt):
        for s in sent:
            non_empty[t] &= s
    return non_empty


def team_step(xy, step_size, goal_bits, empty_bits, memory, draws, noise_scale):
    """One group_step of the Nt target agents of one environment.

    xy [Nt, 2], step_size [Nt], goal_bits [Nt, 4] (weights), empty_bits [Nt, 4] bool: the agents' private states;
    memory = dict(goal [Nt], non_empty [Nt] bit sets, prev_xy [Nt, 2], prev_noise [Nt, 2]) BEFORE the step;
    draws = dict(binomial [Nt], sample [Nt, 2], choice [Nt]) recorded outcomes.  Returns (actions [Nt, 2], memory after)."""
    nt = len(xy)
    goal = memory['goal'].copy()
    non_empty = communicated_non_empty(empty_bits, memory['non_empty'])
    # act (greedy.py:289-328)
    actions = np.zeros((nt, 2))
    noise_out = np.zeros((nt, 2))
    for t in range(nt):
        if goal_bits[t].any():
            goal[t] = int(np.flatnonzero(goal_bits[t])[0])
        if goal[t] < 0 or (not goal_bits[t].any() and not (non_empty[t] >> goal[t]) & 1):
            goal[t] = -1
            if non_empty[t] != 0:
                goal[t] = draws['choice'][t]
                assert goal[t] >= 0 and (non_empty[t] >> goal[t]) & 1
        prev_actual = xy[t] - memory['prev_xy'][t]
        action = WAREHOUSES[goal[t]] - xy[t] if goal[t] >= 0 else np.zeros(2)
        norm = np.linalg.norm(action)
        if norm > step_size[t]:
            action = action * (step_size[t] / norm)
        prob_high = not np.linalg.norm(prev_actual) > 0.2 * step_size[t]
        del prob_high   # the probability only matters for the live draw; the recorded outcome is replayed
        noise = noise_scale * draws['sample'][t] if draws['binomial'][t] else memory['prev_noise'][t]
        actions[t] = np.clip(action + noise, -step_size[t], step_size[t])   # the agent's own action space (base.py:176)
        noise_out[t] = noise
    return actions, {'goal': goal, 'non_empty': non_empty, 'prev_xy': xy.copy(), 'prev_noise': noise_out}
