"""Randomised differential testing: random (valid) game configs, random placements and action streams, played on two
engine libraries through the same host code and compared step by step (tests/parity_common.compare_traces).

The generator only emits configurations the reference accepts (it aborts the process on invalid ones): modest
densities, ranges that exist, rules of the shapes both engines lower.  Everything derives from one integer seed.
"""
import numpy as np

import parity_common as pc

MANY_GROUPS_SEED = 70000     # seeds in [70000, 100000) draw 5-8 groups (up to 25 observation channels)
LARGE_MAP_SEED = 100000      # seeds from here on draw maps in large_map_mode (8 bands)
HUGE_MAP_SEED = 200000       # ... and from here on strips of more than 1000 x 1000 cells (16 bands)


def random_config(seed):
    import magent_b200 as magent
    gw = magent.gridworld
    rs = np.random.RandomState(seed)
    size_w, size_h = int(rs.randint(14, 40)), int(rs.randint(14, 40))
    if seed >= LARGE_MAP_SEED:
        # more than 99 x 99 cells: the reference's large_map_mode (GridWorld.cc:74-85, 403-438) -- movers and
        # turners are queued per vertical band (8 bands; 16 above 1000 x 1000 cells), band edges go to the
        # boundary buffer that runs last.  Strips keep the agent count (and the test time) small.
        if seed >= HUGE_MAP_SEED:
            size_w = int(rs.randint(4004, 5200))
            size_h = 1000 * 1000 // size_w + int(rs.randint(2, 12))
        else:
            size_w = int(rs.randint(100, 330))
            size_h = max(int(rs.randint(30, 100)), 99 * 99 // size_w + 1)
    turn = bool(rs.rand() < 0.3)
    food = bool(rs.rand() < 0.3)
    minimap = bool(rs.rand() < 0.6)
    cfg = gw.Config()
    cfg.set({"map_width": size_w, "map_height": size_h, "minimap_mode": minimap, "turn_mode": turn, "food_mode": food,
             "embedding_size": int(rs.randint(0, 12)), "goal_mode": bool(rs.rand() < 0.15)})
    n_groups = int(rs.randint(2, 5)) if seed < MANY_GROUPS_SEED or seed >= LARGE_MAP_SEED else int(rs.randint(5, 9))
    groups, bodies = [], []
    for g in range(n_groups):
        width, length = [(1, 1), (1, 1), (2, 2), (1, 2), (2, 1), (1, 3)][int(rs.randint(0, 6))]
        if not turn and rs.rand() < 0.5:
            width = length = max(1, min(width, length))
        def rng_range(lo, hi, body):
            r = float(rs.choice(np.arange(lo, hi, 0.5)))
            if rs.rand() < 0.35:
                return gw.SectorRange(max(r, 2.0), float(rs.choice([60, 90, 120, 150])))
            return gw.CircleRange(r)
        absorber = (seed % 3 == 2) and g == 0 and not food                       # train_arrange-style goals (Map.cc:341-349)
        if absorber:
            width = length = 1
        attrs = dict(
            width=width, length=length, hp=float(rs.choice([1.5, 3, 6, 10])), speed=float(rs.choice([0, 1, 1.5, 2, 3])),
            damage=float(rs.choice([0.5, 1, 2, 3.5])), step_recover=float(rs.choice([-0.3, -0.05, 0, 0.1, 0.5])),
            kill_supply=float(rs.choice([0, 0.5, 2])), eat_ability=float(rs.choice([0, 0.3, 1.2])),
            food_supply=float(rs.choice([0.05, 0.5, 2.5])), attack_in_group=int(rs.rand() < 0.3),
            view_range=rng_range(1.0, 6.5, width), attack_range=rng_range(0.5, 3.0, width),
            step_reward=float(rs.choice([-0.01, 0, 0.02])), kill_reward=float(rs.choice([0, 1, 5])),
            dead_penalty=float(rs.choice([-1, -0.1, 0])), attack_penalty=float(rs.choice([-0.1, -0.01, 0])))
        if absorber:
            attrs.update(can_absorb=1, damage=0.0, step_recover=0.0, attack_range=gw.CircleRange(0))
        t = cfg.register_agent_type("t%d" % g, attrs)
        groups.append(cfg.add_group(t))
        bodies.append((width, length))
    syms = [gw.AgentSymbol(g, index='any') for g in groups]
    for _ in range(int(rs.randint(0, 5))):
        i, j = rs.choice(n_groups, 2, replace=False)
        a, b = syms[i], syms[j]
        kind = int(rs.randint(0, 7 if seed % 3 == 1 and seed < LARGE_MAP_SEED else 6))   # pair rules are O(n^2): small maps only
        if kind == 0:
            cfg.add_reward_rule(gw.Event(a, 'attack', b), receiver=a, value=float(rs.choice([0.1, 0.2, 1])))
        elif kind == 1:
            cfg.add_reward_rule(gw.Event(a, 'kill', b), receiver=[a, b], value=[float(rs.choice([1, 2])), -0.5])
        elif kind == 2:
            cfg.add_reward_rule(gw.Event(a, 'collide', b), receiver=a, value=-0.05)
        elif kind == 3:
            cfg.add_reward_rule(gw.Event(a, 'attack', b) | gw.Event(a, 'kill', b), receiver=[a, gw.AgentSymbol(groups[i], 'all')],
                                value=[0.3, 0.01])
        elif kind == 4:
            x0, y0 = int(rs.randint(1, size_w // 2)), int(rs.randint(1, size_h // 2))
            cfg.add_reward_rule(gw.Event(a, 'in', ((x0, y0), (x0 + size_w // 3, y0 + size_h // 3))) & ~gw.Event(a, 'die'),
                                receiver=a, value=0.03)
        elif kind == 6:                                                           # two free subjects, one shared object (double_attack)
            k = int(rs.choice([x for x in range(n_groups) if x != i]))
            c = syms[k]
            a2 = gw.AgentSymbol(groups[i], index='any') if rs.rand() < 0.5 else b
            if a2 is b and k == j:
                a2 = gw.AgentSymbol(groups[i], index='any')
            cfg.add_reward_rule(gw.Event(a, 'attack', c) & gw.Event(a2, 'attack', c), receiver=[a, a2], value=[0.5, 0.5])
        else:
            cfg.add_reward_rule(gw.Event(a, 'die'), receiver=gw.AgentSymbol(groups[j], 'all'), value=0.25, terminal=bool(rs.rand() < 0.1))
    if 1000 <= seed < LARGE_MAP_SEED:
        general_rules(gw, cfg, rs, groups, syms, size_w, size_h)
    return cfg, dict(w=size_w, h=size_h, n_groups=n_groups, bodies=bodies, turn=turn)


def general_rules(gw, cfg, rs, groups, syms, size_w, size_h):
    """seeds >= 1000 add rules of the general shapes of the reference's binder (RewardEngine.cc:373-443): 'all' and
    fixed-index subjects, three free symbols, chains that re-bind a subject, group-quantified events"""
    n_groups = len(groups)

    def rect():
        if rs.rand() < 0.5:
            return ((0, 0), (size_w, size_h))                                     # everyone is inside
        x0, y0 = int(rs.randint(0, size_w // 2)), int(rs.randint(0, size_h // 2))
        return ((x0, y0), (x0 + int(rs.randint(3, size_w)), y0 + int(rs.randint(3, size_h))))

    for _ in range(int(rs.randint(1, 4))):
        i, j = (int(v) for v in rs.choice(n_groups, 2, replace=False))
        a, b = syms[i], syms[j]
        all_i, all_j = gw.AgentSymbol(groups[i], 'all'), gw.AgentSymbol(groups[j], 'all')
        fix_i = gw.AgentSymbol(groups[i], int(rs.randint(0, 6)))
        kind = int(rs.randint(0, 11))
        if kind == 0:
            cfg.add_reward_rule(gw.Event(all_i, 'in', rect()), receiver=all_i, value=0.07)
        elif kind == 1:
            cfg.add_reward_rule(gw.Event(all_i, 'die'), receiver=all_j, value=1.5, terminal=bool(rs.rand() < 0.5))
        elif kind == 2:
            cfg.add_reward_rule(gw.Event(fix_i, 'attack', b), receiver=[fix_i, b], value=[0.4, -0.2])
        elif kind == 3:                                                           # fixed subject, nothing inferred: never fires
            cfg.add_reward_rule(gw.Event(fix_i, 'in', rect()), receiver=fix_i, value=9.0)
        elif kind == 4:
            cfg.add_reward_rule(gw.Event(all_i, 'attack', b) | gw.Event(all_i, 'kill', b), receiver=[b, all_i], value=[-0.6, 0.2])
        elif kind == 5:                                                           # three free symbols
            k = int(rs.choice([x for x in range(n_groups) if x != i]))
            a2 = gw.AgentSymbol(groups[i], 'any')
            a3 = gw.AgentSymbol(groups[int(rs.randint(0, n_groups))], 'any')
            cfg.add_reward_rule(gw.Event(a, 'attack', syms[k]) & gw.Event(a2, 'attack', syms[k]) & gw.Event(a3, 'in', rect()),
                                receiver=[a, a2, a3], value=[0.5, 0.25, 0.125])
        elif kind == 6:
            cfg.add_reward_rule(gw.Event(all_i, 'in_a_line'), receiver=all_i, value=0.3)
        elif kind == 7:                                                           # chain: the later level re-binds an earlier subject
            if rs.rand() < 0.5:
                cfg.add_reward_rule(gw.Event(a, 'attack', b) & gw.Event(b, 'attack', a), receiver=[a, b], value=[0.2, 0.1])
            else:
                c = gw.AgentSymbol(groups[j], 'any')
                ev = gw.Event(c, 'attack', a) & gw.Event(a, 'attack', b) if rs.rand() < 0.5 else gw.Event(a, 'attack', b) & gw.Event(c, 'attack', a)
                cfg.add_reward_rule(ev, receiver=[a, b, c], value=[0.2, 0.1, 0.05])
        elif kind == 8:
            cfg.add_reward_rule(gw.Event(a, 'attack', gw.AgentSymbol(groups[j], int(rs.randint(0, 4)))), receiver=a, value=0.35)
        elif kind == 9:
            cfg.add_reward_rule(gw.Event(a, 'attack', b) & ~gw.Event(all_j, 'in', rect()), receiver=[a, all_j], value=[0.15, -0.01])
        else:                                                                     # 'all' level and fixed level next to a free one
            cfg.add_reward_rule((gw.Event(all_i, 'collide', b) | gw.Event(fix_i, 'attack', b)) & ~gw.Event(a, 'die'),
                                receiver=[a, b], value=[0.02, 0.04])


def make_env(lib, seed, **kw):
    import magent_b200 as magent
    cfg, info = random_config(seed)
    env = magent.GridWorld(cfg, _lib=lib, **kw)
    rs = np.random.RandomState(seed + 7919)
    env.set_seed(int(rs.randint(0, 10000)))
    env.reset()
    free = (info["w"] - 2) * (info["h"] - 2)
    env.add_walls(method="random", n=int(rs.randint(0, max(1, free // 25))))
    handles = env.get_handles()
    never = int(rs.randint(0, len(handles))) if seed % 7 == 6 else -1     # a group that stays empty for the whole episode
    for g, h in enumerate(handles):
        bw, bl = info["bodies"][g]
        if g == never:
            continue
        share = free * float(rs.choice([0.02, 0.06, 0.12] if seed % 3 != 1 else [0.1, 0.2, 0.3])) / (bw * bl) / info["n_groups"] * 2
        if seed >= LARGE_MAP_SEED:
            share *= 0.03 if seed >= HUGE_MAP_SEED else 0.4
        n = max(1, int(share))
        env.add_agents(h, method="random", n=n)
        if rs.rand() < 0.3:                                   # explicit placements, some of them blocked or off the map
            pos = [[int(rs.randint(1, info["w"] - 1)), int(rs.randint(1, info["h"] - 1)), int(rs.randint(0, 4))] for _ in range(6)]
            env.add_agents(h, method="custom", pos=pos)
    if seed % 5 == 4:                                         # rectangle fills (GridWorld.cc:180-290 "fill"): walls and agents,
        rf = np.random.RandomState(seed + 104729)             # partly on occupied cells and across the border
        for _ in range(int(rf.randint(1, 3))):
            x, y = int(rf.randint(0, info["w"] - 2)), int(rf.randint(0, info["h"] - 2))
            env.add_walls(method="fill", pos=(x, y), size=(int(rf.randint(1, 5)), int(rf.randint(1, 4))))
        for _ in range(int(rf.randint(1, 4))):
            h = handles[int(rf.randint(0, len(handles)))]
            x, y = int(rf.randint(1, info["w"] - 3)), int(rf.randint(1, info["h"] - 3))
            env.add_agents(h, method="fill", pos=(x, y), size=(int(rf.randint(1, 7)), int(rf.randint(1, 6))),
                           dir=int(rf.randint(0, 4)))
    return env


def trace(seed, lib, steps=25, **kw):
    """the random game of `seed` played on one engine library (pc.run_trace record list)"""
    rs = np.random.RandomState(seed)
    n_groups = len(make_env(lib, seed).get_handles())
    order = [int(g) for g in rs.permutation(n_groups)]
    acting = sorted(int(g) for g in rs.choice(n_groups, size=int(rs.randint(1, n_groups + 1)), replace=False))
    order = [g for g in order if g in acting]
    return pc.run_trace(make_env(lib, seed, **kw), steps, seed, keep_obs=True, act_groups=acting, order=order, stop_on_done=False)


def play(seed, lib_a, lib_b, steps=25, **kw):
    a = trace(seed, lib_a, steps)
    b = trace(seed, lib_b, steps, **kw)
    pc.compare_traces(a, b, what="fuzz seed %d" % seed)
    return a


def trace_irregular(env, steps, seed, acting, order):
    """like parity_common.run_trace, but the caller misbehaves the way real scripts do: clear_dead is skipped on some
    steps (dead agents keep their slots and still receive actions), agents are added in the middle of the episode,
    observations are not fetched every step"""
    handles = env.get_handles()
    rs = np.random.RandomState(seed ^ 0x5bd1)
    trace = []
    for t in range(steps):
        rec = {"num": [env.get_num(h) for h in handles]}
        obs = {}
        if rs.rand() < 0.7:
            for gi in acting:
                if rec["num"][gi] == 0:
                    continue
                v, f = env.get_observation(handles[gi])
                obs[gi] = (v.copy(), f.copy())
        rec["obs"] = obs
        rec["id"] = [env.get_agent_id(h).copy() for h in handles]
        rec["pos"] = [env.get_pos(h).copy() for h in handles]
        acts = {gi: rs.randint(0, env.get_action_space(handles[gi])[0], size=rec["num"][gi]).astype(np.int32) for gi in acting}
        for gi in order:
            env.set_action(handles[gi], acts[gi])
        rec["done"] = bool(env.step())
        rec["reward"] = [env.get_reward(h).copy() for h in handles]
        rec["alive"] = [env.get_alive(h).copy() for h in handles]
        rec["pos_after"] = [env.get_pos(h).copy() for h in handles]
        if rs.rand() < 0.65:
            env.clear_dead()
        if rs.rand() < 0.15:
            env.add_agents(handles[int(rs.randint(0, len(handles)))], method="random", n=int(rs.randint(1, 4)))
        if env.config.config_dict.get("goal_mode") and rs.rand() < 0.3:      # deprecated API: two RNG draws per agent
            env.set_goal(handles[int(rs.randint(0, len(handles)))], "random")
        trace.append(rec)
    return trace


def play_irregular(seed, lib_a, lib_b, steps=25, **kw):
    rs = np.random.RandomState(seed)
    n_groups = len(make_env(lib_a, seed).get_handles())
    order = [int(g) for g in rs.permutation(n_groups)]
    acting = sorted(int(g) for g in rs.choice(n_groups, size=int(rs.randint(1, n_groups + 1)), replace=False))
    order = [g for g in order if g in acting]
    a = trace_irregular(make_env(lib_a, seed), steps, seed, acting, order)
    b = trace_irregular(make_env(lib_b, seed, **kw), steps, seed, acting, order)
    pc.compare_traces(a, b, what="irregular fuzz seed %d" % seed)
    return a


def play_batch(seed, checker_lib, engine_lib, n_arenas=3, steps=15):
    """`_num_arenas` batch of the engine vs n_arenas independent checker environments (arena a is seeded seed0 + a;
    every setup call goes to all arenas).  Groups are presented as the concatenation over arenas."""
    import magent_b200 as magent
    cfg, info = random_config(seed)
    rs = np.random.RandomState(seed + 7919)
    seed0 = int(rs.randint(0, 10000))
    batch = magent.GridWorld(cfg, _lib=engine_lib, _num_arenas=n_arenas)
    singles = [magent.GridWorld(random_config(seed)[0], _lib=checker_lib) for _ in range(n_arenas)]
    batch.set_seed(seed0)
    batch.reset()
    for a, env in enumerate(singles):
        env.set_seed(seed0 + a)
        env.reset()
    free = (info["w"] - 2) * (info["h"] - 2)
    n_walls = int(rs.randint(0, max(1, free // 25)))
    for env in [batch] + singles:
        env.add_walls(method="random", n=n_walls)
    handles = batch.get_handles()
    for g, h in enumerate(handles):
        bw, bl = info["bodies"][g]
        n = max(1, int(free * float(rs.choice([0.02, 0.06, 0.12])) / (bw * bl) / info["n_groups"] * 2))
        for env in [batch] + singles:
            env.add_agents(env.get_handles()[g], method="random", n=n)
    G = len(handles)
    for t in range(steps):
        nums = [[env.get_num(env.get_handles()[g]) for g in range(G)] for env in singles]
        for g in range(G):
            tot = sum(n[g] for n in nums)
            assert batch.get_num(handles[g]) == tot, "step %d group %d num" % (t, g)
            if tot == 0:
                continue
            v, f = batch.get_observation(handles[g])
            parts = [env.get_observation(env.get_handles()[g]) for env in singles if env.get_num(env.get_handles()[g])]
            np.testing.assert_array_equal(v.view(np.uint32), np.concatenate([p[0] for p in parts]).view(np.uint32), err_msg="batch seed %d step %d view g%d" % (seed, t, g))
            np.testing.assert_array_equal(f.view(np.uint32), np.concatenate([p[1] for p in parts]).view(np.uint32), err_msg="batch seed %d step %d feat g%d" % (seed, t, g))
        for g in range(G):
            n_act = batch.get_action_space(handles[g])[0]
            acts = [rs.randint(0, n_act, size=n[g]).astype(np.int32) for n in nums]
            batch.set_action(handles[g], np.concatenate(acts) if acts else np.zeros((0,), np.int32))
            for env, a in zip(singles, acts):
                env.set_action(env.get_handles()[g], a)
        batch.step()
        for env in singles:
            env.step()
        for g in range(G):
            want_r = np.concatenate([env.get_reward(env.get_handles()[g]) for env in singles])
            want_p = np.concatenate([env.get_pos(env.get_handles()[g]).reshape(-1, 2) for env in singles])
            want_a = np.concatenate([env.get_alive(env.get_handles()[g]) for env in singles])
            np.testing.assert_allclose(batch.get_reward(handles[g]), want_r, atol=pc.REWARD_TOL, rtol=0, err_msg="batch seed %d step %d reward g%d" % (seed, t, g))
            np.testing.assert_array_equal(batch.get_pos(handles[g]).reshape(-1, 2), want_p, err_msg="batch seed %d step %d pos g%d" % (seed, t, g))
            np.testing.assert_array_equal(batch.get_alive(handles[g]), want_a, err_msg="batch seed %d step %d alive g%d" % (seed, t, g))
        batch.clear_dead()
        for env in singles:
            env.clear_dead()


def trace_chaotic_gen(env, steps, seed, acting, order, render_dir=None):
    """A caller that reads at every point of the loop: observations and rewards are fetched (from random groups, also
    non-acting ones) before set_action, between set_action calls, after step, after clear_dead and twice in a row;
    the acting subset changes from step to step; the episode is reset and repopulated once in the middle.  Every
    value read is recorded in call order, so two engines must agree on all of them (state-version caches of the
    observation pre-passes and host-side count caches are what this is after)."""
    handles = env.get_handles()
    rs = np.random.RandomState(seed ^ 0x2c1b3)
    log = []
    free = (env.config.config_dict["map_width"] - 2) * (env.config.config_dict["map_height"] - 2)
    attack_bias = float(rs.choice([0.0, 0.5, 0.85]))
    attack_base = []                                         # (not get_view2attack: it writes the attack cells into a
    for h in handles:                                        #  view-sized buffer, out of bounds when the attack range is
        import ctypes                                        #  the wider one -- in the reference as well)
        base = ctypes.c_int(0)
        env._lib.env_get_info(env.game, env._hv(h), b"attack_base", ctypes.cast(ctypes.byref(base), ctypes.c_void_p))
        attack_base.append(base.value)

    if render_dir is not None:
        env.set_render_dir(render_dir)
    W, H = env.config.config_dict["map_width"], env.config.config_dict["map_height"]

    def peek(tag):
        r = rs.rand()
        if render_dir is not None and r > 0.8:               # the cold path: replay frames, window queries, density maps
            q = rs.rand()
            if q < 0.4:
                if all(env.get_num(h) > 0 for h in handles):   # RenderGenerator.cc:151 reads agents[0] of every group
                    env.render()
            elif q < 0.7:
                x0, y0 = int(rs.randint(0, W - 3)), int(rs.randint(0, H - 3))
                info, events = env._get_render_info((x0, x0 + int(rs.randint(2, W))), (y0, y0 + int(rs.randint(2, H))))
                rows = np.array(sorted([k] + list(v) for k, v in info.items()), dtype=np.int64).reshape(-1, 4)
                log.append((tag + " window", rows, np.asarray(events, dtype=np.int64).reshape(-1, 3)))
            else:
                log.append((tag + " global_minimap", env.get_global_minimap(int(rs.randint(2, 9)), int(rs.randint(2, 9))).copy()))
            return
        if r < 0.45:
            gi = int(rs.randint(0, len(handles)))
            if env.get_num(handles[gi]) > 0:
                v, f = env.get_observation(handles[gi])
                log.append((tag + " obs g%d" % gi, v.copy(), f.copy()))
                if rs.rand() < 0.2:
                    v, f = env.get_observation(handles[gi])
                    log.append((tag + " obs again g%d" % gi, v.copy(), f.copy()))
                if rs.rand() < 0.25:                         # the compact hand-off on the same state: the engine's f16 call
                    if getattr(env._lib, "is_b200", False):  # against the checker's float32 observation rounded to f16
                        v, f = env.get_observation_f16(handles[gi])
                        log.append((tag + " obs f16 g%d" % gi, v.copy(), f.copy()))
                    else:
                        log.append((tag + " obs f16 g%d" % gi, v.astype(np.float16), f.astype(np.float16)))
        elif r < 0.65:
            gi = int(rs.randint(0, len(handles)))
            log.append((tag + " reward g%d" % gi, env.get_reward(handles[gi]).copy()))
        elif r < 0.8:
            gi = int(rs.randint(0, len(handles)))
            log.append((tag + " state g%d" % gi, env.get_pos(handles[gi]).copy(), env.get_agent_id(handles[gi]).copy(),
                        env.get_alive(handles[gi]).copy().astype(np.uint8)))

    for t in range(steps):
        if t == steps // 2:                                  # a new episode in the same process: the RNG stream goes on
            env.reset()
            for gi, h in enumerate(handles):
                env.add_agents(h, method="random", n=int(rs.randint(1, 2 + free // (40 * len(handles)))))
            log.append(("reset", np.array([env.get_num(h) for h in handles])))
        peek("t%d top" % t)
        yield
        now = [g for g in order if rs.rand() < 0.8]
        for gi in now:
            n = env.get_num(handles[gi])
            n_act = env.get_action_space(handles[gi])[0]
            act = rs.randint(0, n_act, size=n).astype(np.int32)
            if attack_bias > 0 and attack_base[gi] < n_act:   # bloodier episodes: kill chains, mutual and self kills
                hit = rs.rand(n) < attack_bias
                act[hit] = rs.randint(attack_base[gi], n_act, size=int(hit.sum()))
            env.set_action(handles[gi], act)
            peek("t%d after set_action g%d" % (t, gi))
            yield
            if rs.rand() < 0.06:                             # setup calls between set_action and step: the newcomers have
                gj = int(rs.randint(0, len(handles)))        # no action this step, walls may block queued moves
                env.add_agents(handles[gj], method="random", n=int(rs.randint(1, 3)))
                log.append(("t%d late add g%d" % (t, gj), np.array([env.get_num(h) for h in handles])))
                peek("t%d after late add" % t)
            if env.config.config_dict.get("goal_mode") and rs.rand() < 0.2:    # deprecated API: two RNG draws per agent
                env.set_goal(handles[int(rs.randint(0, len(handles)))], "random")
            if rs.rand() < 0.04:
                env.add_walls(method="random", n=int(rs.randint(1, 4)))
            if rs.rand() < 0.03:
                env.set_seed(int(rs.randint(0, 1000)))
        done = env.step()
        log.append(("t%d done" % t, np.array([int(done)] + [env.get_num(h) for h in handles])))
        peek("t%d after step" % t)
        peek("t%d after step (2)" % t)
        yield
        if rs.rand() < 0.8:
            env.clear_dead()
            peek("t%d after clear_dead" % t)
        for gi, h in enumerate(handles):
            log.append(("t%d end g%d" % (t, gi), env.get_pos(h).copy(), env.get_agent_id(h).copy()))
    if render_dir is not None:
        import os
        for name in sorted(os.listdir(render_dir)):
            log.append(("file " + name, np.frombuffer(open(os.path.join(render_dir, name), "rb").read(), dtype=np.uint8)))
    return log


def trace_chaotic(env, steps, seed, acting, order, render_dir=None):
    """trace_chaotic_gen run to its end (the generator yields between API calls so that two engines can be interleaved)"""
    g = trace_chaotic_gen(env, steps, seed, acting, order, render_dir=render_dir)
    try:
        while True:
            next(g)
    except StopIteration as e:
        return e.value


def chaotic_log(seed, lib, steps=24, **kw):
    """the chaotic caller of `seed` on one engine library (trace_chaotic record list)"""
    rs = np.random.RandomState(seed)
    n_groups = len(make_env(lib, seed).get_handles())
    order = [int(g) for g in rs.permutation(n_groups)]
    import shutil
    import tempfile
    # with more than 4 groups the reference indexes its 4-row colour table out of bounds (RenderGenerator.cc gen_config:
    # uninitialised stack in config.json)
    d = tempfile.mkdtemp() if n_groups <= 4 else None
    try:
        return trace_chaotic(make_env(lib, seed, **kw), steps, seed, None, order, render_dir=d)
    finally:
        if d is not None:
            shutil.rmtree(d, ignore_errors=True)


def play_chaotic(seed, lib_a, lib_b, steps=24, **kw):
    a = chaotic_log(seed, lib_a, steps)
    b = chaotic_log(seed, lib_b, steps, **kw)
    assert len(a) == len(b), "chaotic fuzz seed %d: %d vs %d records" % (seed, len(a), len(b))
    for ra, rb in zip(a, b):
        assert ra[0] == rb[0], "chaotic fuzz seed %d: %s vs %s" % (seed, ra[0], rb[0])
        for xa, xb in zip(ra[1:], rb[1:]):
            what = "chaotic fuzz seed %d: %s" % (seed, ra[0])
            assert xa.shape == xb.shape, what + " shape %s vs %s" % (xa.shape, xb.shape)
            if xa.dtype == np.float32 and " reward" in ra[0]:
                np.testing.assert_allclose(xa, xb, rtol=0, atol=pc.REWARD_TOL, err_msg=what)
            elif xa.dtype == np.float32:
                np.testing.assert_array_equal(xa.view(np.uint32), xb.view(np.uint32), err_msg=what)
            elif xa.dtype == np.float16:
                np.testing.assert_array_equal(xa.view(np.uint16), xb.view(np.uint16), err_msg=what)
            else:
                np.testing.assert_array_equal(xa, xb, err_msg=what)
    return a


def play_batch_chaotic(seed, checker_lib, engine_lib, n_arenas=3, steps=16):
    """The chaotic caller on an arena batch: `_num_arenas` arenas behind one engine handle against n_arenas independent
    checker environments (arena a seeded seed0 + a).  Reads happen at every point of the loop and are compared on the
    spot; the acting subset changes every step; clear_dead is skipped now and then; agents are added late to ALL arenas
    (random placement, each arena from its own RNG stream) or, through magent_b200_select_arena, to ONE arena at explicit
    positions; one reset in mid-run."""
    import magent_b200 as magent
    cfg, info = random_config(seed)
    rs = np.random.RandomState(seed + 15485863)
    seed0 = int(rs.randint(0, 10000))
    batch = magent.GridWorld(cfg, _lib=engine_lib, _num_arenas=n_arenas)
    singles = [magent.GridWorld(random_config(seed)[0], _lib=checker_lib) for _ in range(n_arenas)]
    both = [batch] + singles
    G = len(batch.get_handles())
    free = (info["w"] - 2) * (info["h"] - 2)
    what = "batch-chaotic seed %d" % seed

    def H(env, g):
        return env.get_handles()[g]

    def populate(scale):
        for g in range(G):
            bw, bl = info["bodies"][g]
            n = max(1, int(free * scale * float(rs.choice([0.03, 0.08])) / (bw * bl) / G * 2))
            for env in both:
                env.add_agents(H(env, g), method="random", n=n)

    batch.set_seed(seed0)
    batch.reset()
    for a, env in enumerate(singles):
        env.set_seed(seed0 + a)
        env.reset()
    n_walls = int(rs.randint(0, max(1, free // 30)))
    for env in both:
        env.add_walls(method="random", n=n_walls)
    populate(1.0)

    def cat(parts, shape_tail=None):
        parts = [p for p in parts if p.shape[0]]
        return np.concatenate(parts) if parts else None

    def peek(tag):
        r, g = rs.rand(), int(rs.randint(0, G))
        nums = [env.get_num(H(env, g)) for env in singles]
        assert batch.get_num(H(batch, g)) == sum(nums), "%s %s num g%d" % (what, tag, g)
        np.testing.assert_array_equal(batch.get_arena_nums(H(batch, g)), nums, err_msg="%s %s arena_num" % (what, tag))
        if sum(nums) == 0:
            return
        if r < 0.45:
            v, f = batch.get_observation(H(batch, g))
            parts = [env.get_observation(H(env, g)) for env, n in zip(singles, nums) if n]
            np.testing.assert_array_equal(v.view(np.uint32), np.concatenate([p[0] for p in parts]).view(np.uint32), err_msg="%s %s view g%d" % (what, tag, g))
            np.testing.assert_array_equal(f.view(np.uint32), np.concatenate([p[1] for p in parts]).view(np.uint32), err_msg="%s %s feature g%d" % (what, tag, g))
        elif r < 0.7:
            np.testing.assert_allclose(batch.get_reward(H(batch, g)), np.concatenate([env.get_reward(H(env, g)) for env in singles]),
                                       rtol=0, atol=pc.REWARD_TOL, err_msg="%s %s reward g%d" % (what, tag, g))
        else:
            np.testing.assert_array_equal(batch.get_pos(H(batch, g)).reshape(-1, 2), np.concatenate([env.get_pos(H(env, g)).reshape(-1, 2) for env in singles]), err_msg="%s %s pos g%d" % (what, tag, g))
            np.testing.assert_array_equal(batch.get_agent_id(H(batch, g)), np.concatenate([env.get_agent_id(H(env, g)) for env in singles]), err_msg="%s %s id g%d" % (what, tag, g))
            np.testing.assert_array_equal(batch.get_alive(H(batch, g)), np.concatenate([env.get_alive(H(env, g)) for env in singles]), err_msg="%s %s alive g%d" % (what, tag, g))

    for t in range(steps):
        if t == steps // 2:
            for env in both:
                env.reset()
            populate(0.5)
        peek("t%d top" % t)
        for g in [int(x) for x in rs.permutation(G) if rs.rand() < 0.8]:
            n_act = batch.get_action_space(H(batch, g))[0]
            acts = [rs.randint(0, n_act, size=env.get_num(H(env, g))).astype(np.int32) for env in singles]
            batch.set_action(H(batch, g), np.concatenate(acts))
            for env, a in zip(singles, acts):
                env.set_action(H(env, g), a)
            peek("t%d after set_action g%d" % (t, g))
            if rs.rand() < 0.08:
                gj, k = int(rs.randint(0, G)), int(rs.randint(1, 3))
                for env in both:
                    env.add_agents(H(env, gj), method="random", n=k)
            if rs.rand() < 0.08:                              # one arena only, explicit positions (some of them taken)
                a, gj = int(rs.randint(0, n_arenas)), int(rs.randint(0, G))
                pos = [[int(rs.randint(1, info["w"] - 1)), int(rs.randint(1, info["h"] - 1)), int(rs.randint(0, 4))] for _ in range(3)]
                batch.select_arena(a)
                batch.add_agents(H(batch, gj), method="custom", pos=pos)
                batch.select_arena(-1)
                singles[a].add_agents(H(singles[a], gj), method="custom", pos=pos)
        batch.step()
        dones = [env.step() for env in singles]
        np.testing.assert_array_equal(batch.get_arena_done() != 0, np.array(dones), err_msg="%s t%d done" % (what, t))
        peek("t%d after step" % t)
        peek("t%d after step (2)" % t)
        if rs.rand() < 0.8:
            for env in both:
                env.clear_dead()
            peek("t%d after clear_dead" % t)


def compare_chaotic_logs(a, b, what):
    assert len(a) == len(b), "%s: %d vs %d records" % (what, len(a), len(b))
    for ra, rb in zip(a, b):
        assert ra[0] == rb[0], "%s: %s vs %s" % (what, ra[0], rb[0])
        for xa, xb in zip(ra[1:], rb[1:]):
            w = "%s: %s" % (what, ra[0])
            assert xa.shape == xb.shape, w + " shape %s vs %s" % (xa.shape, xb.shape)
            if xa.dtype == np.float32 and " reward" in ra[0]:
                np.testing.assert_allclose(xa, xb, rtol=0, atol=pc.REWARD_TOL, err_msg=w)
            elif xa.dtype == np.float32:
                np.testing.assert_array_equal(xa.view(np.uint32), xb.view(np.uint32), err_msg=w)
            elif xa.dtype == np.float16:
                np.testing.assert_array_equal(xa.view(np.uint16), xb.view(np.uint16), err_msg=w)
            else:
                np.testing.assert_array_equal(xa, xb, err_msg=w)


def play_interleaved_engines(seed, checker_lib, engine_lib, n_engines=3, steps=16):
    """n_engines DIFFERENT random games alive in one process on the engine library, their chaotic callers advanced in
    random interleaving (a switch between any two API calls), each compared with the same game played alone on the
    checker: anything process-global in the backend (scratch buffers, cached launch configurations, the observation
    pre-pass products) must not leak between engines."""
    rs = np.random.RandomState(seed + 32452843)
    seeds = [seed * 10 + k for k in range(n_engines)]
    orders = []
    for sd in seeds:
        r = np.random.RandomState(sd)
        n_groups = len(make_env(checker_lib, sd).get_handles())
        orders.append([int(g) for g in r.permutation(n_groups)])
    want = [trace_chaotic(make_env(checker_lib, sd), steps, sd, None, o) for sd, o in zip(seeds, orders)]
    gens = [trace_chaotic_gen(make_env(engine_lib, sd), steps, sd, None, o) for sd, o in zip(seeds, orders)]
    got = [None] * n_engines
    live = list(range(n_engines))
    while live:
        k = live[int(rs.randint(0, len(live)))]
        try:
            next(gens[k])
        except StopIteration as e:
            got[k] = e.value
            live.remove(k)
    for k in range(n_engines):
        compare_chaotic_logs(want[k], got[k], "interleaved engines seed %d game %d" % (seed, k))
