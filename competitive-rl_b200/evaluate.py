"""evaluate_two_policies_in_batch on the device (competitive_rl/pong/evaluate.py:53-88; SURVEY section 8 row f3), and
evaluate_pool_in_batch, which plays every pairing of an opponent pool in one batch.

Same contract as the reference: two action functions play each other on a cPongDouble vec-env until `num_episodes`
episodes have finished; returns ([win, draw, lose, cumulative reward] of agent 0, the same for agent 1).  The per-env
bookkeeping (episode returns, win / draw / lose classification on done, zeroing finished envs) is tensor arithmetic on
the device instead of a Python loop over envs; the only host traffic per step is the finished-episode count that the
stopping rule needs."""
import numpy as np
import torch


def evaluate_two_policies_in_batch(compute_action0, compute_action1, envs, num_episodes):
    dev = envs.device
    n = envs.num_envs
    episode_rewards = torch.zeros((n, 2), dtype=torch.float64, device=dev)
    tally = torch.zeros(5, dtype=torch.float64, device=dev)     # wins0, draws, losses0, sum reward0, sum reward1
    total_episodes = 0
    obs = envs.reset()
    while True:
        a0 = torch.as_tensor(compute_action0(obs[0])).to(dev, dtype=torch.int32).reshape(-1)
        a1 = torch.as_tensor(compute_action1(obs[1])).to(dev, dtype=torch.int32).reshape(-1)
        obs, reward, done, info = envs.step(torch.stack([a0, a1], dim=1))
        done = done.bool()
        if done.ndim == 2:
            done = done.all(dim=1)
        episode_rewards += reward.to(torch.float64).reshape(n, 2)
        r0 = episode_rewards[:, 0]
        tally += torch.stack([(done & (r0 > 0)).sum(), (done & (r0 == 0)).sum(), (done & (r0 < 0)).sum(),
                              (r0 * done).sum(), (episode_rewards[:, 1] * done).sum()]).to(torch.float64)
        episode_rewards *= (~done).to(torch.float64).reshape(-1, 1)
        total_episodes += int(done.sum())                       # the one host sync of the step
        if total_episodes >= num_episodes:
            break
    w, d, l, s0, s1 = [float(x) for x in tally.tolist()]
    return [int(w), int(d), int(l), s0], [int(l), int(d), int(w), s1]


def evaluate_pool_in_batch(pool, envs, episodes_per_pair, pairs=None, networks=None, seed=0, resource_dir=None,
                           check_every=64, max_steps=None):
    """Win / draw / loss table of pool entries playing each other, every pairing in one batch.

    Both agents of every env are played by the league mode of the per-env opponent kernel (csrc/pong_opponent.cu,
    include/crl_b200.h crl_pong_opp_set_pairs): one launch per step evaluates both seats of every env, and env g plays
    pairing g mod P for the whole run.

    pool: up to 16 distinct names, resolved as TournamentEnvWrapper.set_opponents resolves them: "RULE_BASED", "RANDOM"
        and up to 8 LightActorCritic networks (WEAK / MEDIUM from their checkpoints, or names given in `networks`).
    envs: a 42x42 cPongDouble vec-env with frame_stack None and uint8 observations, at least one env per pairing.
        It is reset first.
    episodes_per_pair: the run stops once every pairing has at least this many finished episodes (checked every
        `check_every` steps, one host synchronisation each) or after `max_steps` steps.
    pairs: (seat 0, seat 1) pool indices or names; None = all M^2 ordered pairings, self-play included.  At most 256.
    networks: {name: state dict | module | checkpoint dict | path} of extra LightActorCritic networks.
    seed: keys RANDOM's actions.

    Returns {"pool", "pairs", "episodes", "wins", "draws", "losses", "steps"}: the tallies are int64 (M, M) arrays,
    row = seat 0's entry, column = seat 1's, counted from seat 0's side (> 0, == 0, < 0 summed clipped reward, as in
    evaluate_two_policies_in_batch); repeated pairings add up, pairings not played are 0."""
    from . import _native
    from .builtin_policies import pack_light_actor_critic, resolve_pairs, resolve_pool
    if envs.dim != 42 or envs.c != 1 or envs.f32 or envs.ring or getattr(envs, "n_agents", 2) != 2:
        raise ValueError("league evaluation needs a cPongDouble env with resized_dim=42, frame_stack=None and uint8 "
                         "observations")
    ext = _native.ext()
    added = {}
    for name, state in (networks or {}).items():
        if name in ("RULE_BASED", "RANDOM"):
            raise ValueError("%s is not a network" % name)
        if isinstance(state, str):
            state = torch.load(state, map_location="cpu", weights_only=True)
        added[name] = pack_light_actor_critic(state)
    pool, kinds, images = resolve_pool(pool, added, resource_dir)
    m = len(pool)
    if pairs is None:
        pairs = [(a, b) for a in range(m) for b in range(m)]
    idx = resolve_pairs(pairs, pool)
    p = len(idx)
    n = envs.num_envs
    if n < p:
        raise ValueError("%d pairings need at least as many envs (got %d)" % (p, n))
    if episodes_per_pair < 1 or check_every < 1 or (max_steps is not None and max_steps < 1):
        raise ValueError("episodes_per_pair, check_every and max_steps must be positive")

    dev = envs.device
    opp = ext.PongOpponents(n, int(dev.index), int(seed) & (2 ** 64 - 1), int(envs.first_env))
    try:
        for slot, image in enumerate(images):
            opp.load_net(slot, image)
        opp.set_pool(torch.tensor(kinds, dtype=torch.int32), None)
        opp.set_pairs(torch.tensor(idx, dtype=torch.int32))
        both = torch.zeros((n, 2), dtype=torch.int32, device=dev)
        envs.reset()
        rew = done = None
        steps = 0
        while True:
            # credits the episodes that the previous step ended, then acts for both seats
            opp.act_pairs(envs._obs[0], envs._obs[1], rew, done, both, None)
            if steps > 0 and (steps % check_every == 0 or steps == max_steps):
                st = np.array(opp.pair_stats(p), dtype=np.int64).reshape(p, 4)
                if st[:, 0].min() >= episodes_per_pair or steps == max_steps:
                    break
            envs.step(both)
            rew, done = envs._rew, envs._done
            steps += 1
    finally:
        torch.cuda.synchronize(dev)
        opp.close()
    out = {"pool": pool, "pairs": [tuple(k) for k in idx], "steps": steps}
    ab = np.array(idx, dtype=np.int64)
    for col, key in enumerate(("episodes", "wins", "draws", "losses")):
        t = np.zeros((m, m), np.int64)
        np.add.at(t, (ab[:, 0], ab[:, 1]), st[:, col])
        out[key] = t
    return out
