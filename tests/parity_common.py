"""Shared helpers for the differential (parity) tests.

A *scenario* builds an environment on a given engine library, places walls/agents and returns the
env; `run_trace` then plays a pre-generated random action stream and records everything observable
through the ABI at every step.  Two traces (reference vs CUDA engine, or golden vs live) are compared
with `compare_traces`: integer state bit-exact, observations bit-exact (float32 byte equality),
rewards within 1e-6 (BASELINE.json north_star).
"""
import hashlib
import os

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LIB = os.path.join(REPO, "oracle", "_ref", "libmagent.so")
PORT_LIB = os.path.join(REPO, "oracle", "_build", "libmagent_oracle.so")
EMU_LIB = os.path.join(REPO, "tests", "_emu", "libmagent_emu.so")
CUDA_LIB = os.path.join(REPO, "magent_b200", "lib", "libmagent.so")
REWARD_TOL = 1e-6


def sha(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


def run_trace(env, steps, seed, act_groups=None, keep_obs=False, order=None, stop_on_done=True):
    """Play `steps` steps of uniform random actions; return a list of per-step dict records."""
    import magent_b200  # noqa: F401  (package must be importable)
    handles = env.get_handles()
    act_groups = list(range(len(handles))) if act_groups is None else act_groups
    order = act_groups if order is None else order
    rs = np.random.RandomState(seed)
    trace = []
    for _ in range(steps):
        rec = {"num": [env.get_num(h) for h in handles]}
        obs = {}
        for gi in act_groups:
            if rec["num"][gi] == 0:
                obs[gi] = (np.zeros((0,), np.float32), np.zeros((0,), np.float32))
                continue
            v, f = env.get_observation(handles[gi])
            obs[gi] = (v.copy(), f.copy()) if keep_obs else (sha(v), sha(f))
            if not keep_obs:
                rec.setdefault("hp_chan_sum", {})[gi] = float(np.asarray(v, dtype=np.float64).sum())
        rec["obs"] = obs
        rec["id"] = [env.get_agent_id(h).copy() for h in handles]
        rec["pos"] = [env.get_pos(h).copy() for h in handles]
        acts = {}
        for gi in act_groups:
            n_act = env.get_action_space(handles[gi])[0]
            acts[gi] = rs.randint(0, n_act, size=rec["num"][gi]).astype(np.int32)
        for gi in order:
            env.set_action(handles[gi], acts[gi])
        rec["done"] = bool(env.step())
        rec["reward"] = [env.get_reward(h).copy() for h in handles]
        rec["alive"] = [env.get_alive(h).copy() for h in handles]
        rec["pos_after"] = [env.get_pos(h).copy() for h in handles]
        env.clear_dead()
        trace.append(rec)
        if rec["done"] and stop_on_done:
            break
    return trace


def compare_traces(ta, tb, what="trace"):
    assert len(ta) == len(tb), "%s: length %d vs %d" % (what, len(ta), len(tb))
    for t, (a, b) in enumerate(zip(ta, tb)):
        tag = "%s step %d" % (what, t)
        assert a["num"] == b["num"], "%s num %s vs %s" % (tag, a["num"], b["num"])
        for g in range(len(a["num"])):
            np.testing.assert_array_equal(a["id"][g], b["id"][g], err_msg=tag + " id g%d" % g)
            np.testing.assert_array_equal(a["pos"][g], b["pos"][g], err_msg=tag + " pos g%d" % g)
            np.testing.assert_array_equal(a["alive"][g], b["alive"][g], err_msg=tag + " alive g%d" % g)
            np.testing.assert_array_equal(a["pos_after"][g], b["pos_after"][g], err_msg=tag + " pos_after g%d" % g)
            np.testing.assert_allclose(a["reward"][g], b["reward"][g], rtol=0, atol=REWARD_TOL,
                                       err_msg=tag + " reward g%d" % g)
        assert a["done"] == b["done"], tag + " done"
        for g in a["obs"]:
            va, fa = a["obs"][g]
            vb, fb = b["obs"][g]
            if isinstance(va, str):
                assert fa == fb, tag + " feature hash g%d" % g
                assert va == vb, tag + " view hash g%d" % g
            else:
                np.testing.assert_array_equal(fa.view(np.uint32), fb.view(np.uint32), err_msg=tag + " feature g%d" % g)
                np.testing.assert_array_equal(va.view(np.uint32), vb.view(np.uint32), err_msg=tag + " view g%d" % g)


# ------------------------------------------------------------------ scenarios (SURVEY.md §8d configs)
def make_battle(lib, map_size=40, n=60, seed=0, **kw):
    import magent_b200 as magent
    env = magent.GridWorld("battle", map_size=map_size, _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[0], method="random", n=n)
    env.add_agents(h[1], method="random", n=n)
    return env


def make_battle_blocks(lib, map_size=40, **kw):
    """the dense two-block layout of examples/train_battle.py:15-40"""
    import math
    import magent_b200 as magent
    env = magent.GridWorld("battle", map_size=map_size, _lib=lib, **kw)
    env.reset()
    h = env.get_handles()
    width = height = map_size
    init_num = map_size * map_size * 0.04
    gap = 3
    side = int(math.sqrt(init_num)) * 2
    pos = [[x, y, 0] for x in range(width // 2 - gap - side, width // 2 - gap, 2)
           for y in range((height - side) // 2, (height - side) // 2 + side, 2)]
    env.add_agents(h[0], method="custom", pos=pos)
    pos = [[x, y, 0] for x in range(width // 2 + gap, width // 2 + gap + side, 2)
           for y in range((height - side) // 2, (height - side) // 2 + side, 2)]
    env.add_agents(h[1], method="custom", pos=pos)
    return env


def make_pursuit(lib, map_size=40, seed=0, **kw):
    """config 1 of BASELINE.json: 40x40, 48 walls, 16 predators, 32 prey"""
    import magent_b200 as magent
    env = magent.GridWorld("pursuit", map_size=map_size, _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=map_size * map_size * 0.03)
    env.add_agents(h[0], method="random", n=map_size * map_size * 0.01)
    env.add_agents(h[1], method="random", n=map_size * map_size * 0.02)
    return env


def gather_config(size):
    """the config of examples/train_gather.py:14-43 (packaged as magent_b200.builtin.config.gather)"""
    from magent_b200.builtin.config import gather
    return gather.get_config(size)


def make_gather(lib, map_size=40, seed=0, n_agent=40, n_food=120, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(gather_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[1], method="random", n=n_agent)
    env.add_agents(h[0], method="random", n=n_food)
    return env


def make_builtin(lib, game, map_size=30, seed=3, n0=120, n1=60, **kw):
    """forest / double_attack: deer (group 0) and tigers (group 1), random placement"""
    import magent_b200 as magent
    env = magent.GridWorld(game, map_size=map_size, _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[0], method="random", n=n0)
    env.add_agents(h[1], method="random", n=n1)
    return env


def mixed_config(size):
    """synthetic config that stresses what the shipped games do not: three groups, a 2x2 body next to 1x1
    bodies, a 19x19 view (> 256 cells), starvation, kill_supply, attack_in_group, minimap + embedding, and a
    rule set using kill / collide / in / die / not / or / and with agent, object and whole-group receivers"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "embedding_size": 5})
    big = cfg.register_agent_type("big", dict(
        width=2, length=2, hp=8, speed=1, damage=3, step_recover=0.05, kill_supply=1,
        view_range=gw.CircleRange(9), attack_range=gw.CircleRange(2),
        step_reward=-0.01, kill_reward=3, dead_penalty=-2, attack_penalty=-0.05))
    small = cfg.register_agent_type("small", dict(
        width=1, length=1, hp=4, speed=2, damage=1, step_recover=-0.05, kill_supply=2,
        view_range=gw.CircleRange(4), attack_range=gw.CircleRange(1.5),
        step_reward=0.02, kill_reward=1, dead_penalty=-1, attack_penalty=-0.02))
    tank = cfg.register_agent_type("tank", dict(
        width=1, length=1, hp=12, speed=1, damage=5, step_recover=0.2, attack_in_group=1,
        view_range=gw.CircleRange(3), attack_range=gw.CircleRange(1),
        kill_reward=4, dead_penalty=-3, attack_penalty=-0.1))
    g0, g1, g2 = cfg.add_group(big), cfg.add_group(small), cfg.add_group(tank)
    a, b, c = (gw.AgentSymbol(g, index='any') for g in (g0, g1, g2))
    cfg.add_reward_rule(gw.Event(a, 'kill', b), receiver=[a, gw.AgentSymbol(g0, 'all')], value=[2, 0.25])
    cfg.add_reward_rule(gw.Event(b, 'attack', a) | gw.Event(b, 'kill', a), receiver=[b, a], value=[0.5, -0.5])
    cfg.add_reward_rule(gw.Event(c, 'collide', b), receiver=c, value=-0.125)
    cfg.add_reward_rule(gw.Event(b, 'in', ((3, 3), (size // 2, size // 2))) & ~gw.Event(b, 'die'), receiver=b, value=0.0625)
    cfg.add_reward_rule(gw.Event(c, 'attack', c2 := gw.AgentSymbol(g2, index='any')), receiver=[c, c2], value=[0.3, -0.3])
    return cfg


def make_mixed(lib, map_size=36, seed=6, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(mixed_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=30)
    env.add_agents(h[0], method="random", n=25)
    env.add_agents(h[1], method="random", n=160)
    env.add_agents(h[2], method="random", n=60)
    return env


def sector_config(size):
    """SectorRange views and attacks (angle < 180; reference Range.h:104-144, AgentType.cc:86-105): a 120-degree
    view cone + 90-degree attack cone on 1x1 bodies against 2x2 bodies with a 60-degree view / 150-degree attack"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "embedding_size": 6})
    scout = cfg.register_agent_type("scout", dict(
        width=1, length=1, hp=6, speed=2, damage=2, step_recover=0.1, kill_supply=1,
        view_range=gw.SectorRange(7, 120), attack_range=gw.SectorRange(2, 90),
        step_reward=-0.005, kill_reward=2, dead_penalty=-1, attack_penalty=-0.05))
    brute = cfg.register_agent_type("brute", dict(
        width=2, length=2, hp=9, speed=1, damage=3, step_recover=0.05,
        view_range=gw.SectorRange(5, 60), attack_range=gw.SectorRange(3, 150),
        step_reward=0.0, kill_reward=1, dead_penalty=-0.5, attack_penalty=-0.1))
    g0, g1 = cfg.add_group(scout), cfg.add_group(brute)
    a, b = gw.AgentSymbol(g0, index='any'), gw.AgentSymbol(g1, index='any')
    cfg.add_reward_rule(gw.Event(a, 'attack', b), receiver=a, value=0.2)
    cfg.add_reward_rule(gw.Event(b, 'attack', a), receiver=[b, a], value=[0.3, -0.1])
    return cfg


def make_sector(lib, map_size=34, seed=4, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(sector_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=20)
    env.add_agents(h[0], method="random", n=140)
    env.add_agents(h[1], method="random", n=40)
    return env


def turn_config(size):
    """turn_mode (deprecated in the reference, no shipped config): agents carry a direction, the action space is
    [moves][turn left, turn right][attacks], views / attacks / moves are relative to the heading, long bodies
    (2x1, 1x3, 2x2) pivot about their head and can be blocked (Map::do_turn, Map.cc:361-406)"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "turn_mode": True, "minimap_mode": True, "embedding_size": 8})
    lancer = cfg.register_agent_type("lancer", dict(
        width=1, length=3, hp=7, speed=2, damage=2, step_recover=0.1, kill_supply=1,
        view_range=gw.SectorRange(6, 100), attack_range=gw.SectorRange(3, 60),
        step_reward=-0.005, kill_reward=2, dead_penalty=-1, attack_penalty=-0.05))
    cart = cfg.register_agent_type("cart", dict(
        width=2, length=1, hp=9, speed=1, damage=3, step_recover=0.05,
        view_range=gw.CircleRange(4), attack_range=gw.CircleRange(1.5),
        step_reward=0.0, kill_reward=1, dead_penalty=-0.5, attack_penalty=-0.1))
    foot = cfg.register_agent_type("foot", dict(
        width=1, length=1, hp=5, speed=1, damage=1, step_recover=0.1,
        view_range=gw.CircleRange(5), attack_range=gw.SectorRange(2, 120),
        step_reward=0.01, kill_reward=0.5, dead_penalty=-0.2, attack_penalty=-0.02))
    g0, g1, g2 = cfg.add_group(lancer), cfg.add_group(cart), cfg.add_group(foot)
    a, b, c = (gw.AgentSymbol(g, index='any') for g in (g0, g1, g2))
    cfg.add_reward_rule(gw.Event(a, 'attack', b), receiver=a, value=0.2)
    cfg.add_reward_rule(gw.Event(b, 'attack', c), receiver=[b, c], value=[0.3, -0.1])
    cfg.add_reward_rule(gw.Event(c, 'collide', a), receiver=c, value=-0.05)
    return cfg


def make_turn(lib, map_size=36, seed=8, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(turn_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=25)
    env.add_agents(h[0], method="random", n=60)
    env.add_agents(h[1], method="random", n=60)
    env.add_agents(h[2], method="random", n=80)
    # explicit headings as well: custom takes (x, y, dir), fill takes dir
    env.add_agents(h[2], method="custom", pos=[[3, 3, 0], [5, 3, 1], [7, 3, 2], [9, 3, 3]])
    env.add_agents(h[1], method="fill", pos=(12, 2), size=(4, 4), dir=0)
    return env


def food_config(size):
    """food_mode (deprecated in the reference, no shipped config): a killed agent leaves food_supply units of food on
    the ATTACKED cell; food blocks movement and placement, shows up in its own channel, and is eaten by whoever
    attacks that cell (eat_ability per bite, any group, gone below 0.1) -- Map.cc:245,276-303"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "food_mode": True, "minimap_mode": True, "embedding_size": 6})
    wolf = cfg.register_agent_type("wolf", dict(
        width=2, length=2, hp=6, speed=1, damage=3, step_recover=-0.15, kill_supply=0.5, eat_ability=1.5, food_supply=2.0,
        view_range=gw.CircleRange(5), attack_range=gw.CircleRange(2),
        step_reward=-0.01, kill_reward=2, dead_penalty=-1, attack_penalty=-0.03))
    deer = cfg.register_agent_type("deer", dict(
        width=1, length=1, hp=2.5, speed=2, damage=1, step_recover=0.05, eat_ability=0.4, food_supply=3.3,
        view_range=gw.CircleRange(4), attack_range=gw.CircleRange(1.5),
        step_reward=0.01, kill_reward=1, dead_penalty=-0.5, attack_penalty=-0.01))
    crow = cfg.register_agent_type("crow", dict(
        width=1, length=1, hp=1.5, speed=3, damage=0.6, step_recover=-0.02, eat_ability=0.75, food_supply=0.25, attack_in_group=1,
        view_range=gw.CircleRange(3), attack_range=gw.CircleRange(1),
        kill_reward=0.5, dead_penalty=-0.1, attack_penalty=-0.02))
    g0, g1, g2 = cfg.add_group(wolf), cfg.add_group(deer), cfg.add_group(crow)
    a, b, c = (gw.AgentSymbol(g, index='any') for g in (g0, g1, g2))
    cfg.add_reward_rule(gw.Event(a, 'kill', b), receiver=a, value=1)
    cfg.add_reward_rule(gw.Event(b, 'attack', a), receiver=[b, a], value=[0.2, -0.2])
    cfg.add_reward_rule(gw.Event(c, 'attack', b), receiver=c, value=0.1)
    return cfg


def make_food(lib, map_size=30, seed=6, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(food_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=20)
    env.add_agents(h[0], method="random", n=30)
    env.add_agents(h[1], method="random", n=220)
    env.add_agents(h[2], method="random", n=120)
    return env


def make_battle_rect(lib, width=56, height=34, n=120, seed=2, **kw):
    """non-square map: map_width != map_height (minimap scales, feature x/W y/H, bounds all differ per axis)"""
    import magent_b200 as magent
    cfg = magent.builtin.config.battle.get_config(40)
    cfg.set({"map_width": width, "map_height": height})
    env = magent.GridWorld(cfg, _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    for h in env.get_handles():
        env.add_agents(h, method="random", n=n)
    return env


def multi4_config(size):
    """two armies of two unit types each: 4 groups, 13 channels, 16 rules (values of examples/train_multi.py:19-73)"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "embedding_size": 10})
    common = dict(width=1, length=1, damage=2, step_recover=0.1, attack_in_group=True,
                  step_reward=-0.01, kill_reward=0, dead_penalty=-0.1, attack_penalty=-1)
    melee = cfg.register_agent_type("melee", dict(common, hp=10, speed=1, view_range=gw.CircleRange(6),
                                                  attack_range=gw.CircleRange(1)))
    ranged = cfg.register_agent_type("ranged", dict(common, hp=3, speed=2, view_range=gw.CircleRange(6),
                                                    attack_range=gw.CircleRange(2)))
    groups = [cfg.add_group(t) for t in (melee, ranged, melee, ranged)]
    sym = [gw.AgentSymbol(g, index='any') for g in groups]
    for verb, value in (('attack', 2), ('kill', 100)):
        for mine, theirs in (((0, 1), (2, 3)), ((2, 3), (0, 1))):
            for m in mine:
                for t in theirs:
                    cfg.add_reward_rule(gw.Event(sym[m], verb, sym[t]), receiver=sym[m], value=value)
    return cfg


def make_multi4(lib, map_size=40, seed=8, n=70, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(multi4_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    for h in env.get_handles():
        env.add_agents(h, method="random", n=n)
    return env


def arrange_config(size):
    """absorbing goals (values of examples/train_arrange.py:180-212): a mover that bumps into a free goal dies
    into it (Map.cc:341-349), the goal doubles its hp and ignores later visitors"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "embedding_size": 12})
    goal = cfg.register_agent_type("goal", {'width': 1, 'length': 1, 'can_absorb': True})
    agent = cfg.register_agent_type("agent", {'width': 1, 'length': 1, 'hp': 10, 'speed': 2,
                                              'view_range': gw.CircleRange(6), 'step_recover': -10.0 / 400,
                                              'step_reward': 0})
    g_goal, g_agent = cfg.add_group(goal), cfg.add_group(agent)
    g, a = gw.AgentSymbol(g_goal, 'any'), gw.AgentSymbol(g_agent, 'any')
    cfg.add_reward_rule(gw.Event(a, 'collide', g), receiver=a, value=10)
    return cfg


def make_arrange(lib, map_size=30, seed=12, n_goal=70, n_agent=160, **kw):
    import magent_b200 as magent
    env = magent.GridWorld(arrange_config(map_size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    h = env.get_handles()
    env.add_walls(method="random", n=25)
    env.add_agents(h[0], method="random", n=n_goal)
    env.add_agents(h[1], method="random", n=n_agent)
    return env


def general_rules_config(size=16):
    """rule shapes beyond the shipped games (RewardEngine.cc:373-443): 'all' subjects of attack / in_a_line / die /
    at, a fixed-index subject, a fixed-index object (Agent::index is refreshed by clear_dead only), three free symbols"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "embedding_size": 6})
    statue = cfg.register_agent_type("statue", dict(width=1, length=1, hp=4, speed=0, damage=0.5, step_recover=0.0,
                                                    view_range=gw.CircleRange(3), attack_range=gw.CircleRange(1),
                                                    step_reward=0, kill_reward=0, dead_penalty=-1, attack_penalty=0))
    target = cfg.register_agent_type("target", dict(width=1, length=1, hp=1000, speed=0, damage=0, step_recover=0.0,
                                                    view_range=gw.CircleRange(2), attack_range=gw.CircleRange(0),
                                                    step_reward=0, kill_reward=0, dead_penalty=0, attack_penalty=0))
    queue = cfg.register_agent_type("queue", dict(width=1, length=1, hp=2, speed=0, damage=0, step_recover=0.0,
                                                  view_range=gw.CircleRange(2), attack_range=gw.CircleRange(0),
                                                  step_reward=0, kill_reward=0, dead_penalty=-2, attack_penalty=0))
    rover = cfg.register_agent_type("rover", dict(width=1, length=1, hp=6, speed=2, damage=1, step_recover=0.05,
                                                  view_range=gw.CircleRange(4), attack_range=gw.CircleRange(1.5),
                                                  step_reward=-0.005, kill_reward=1, dead_penalty=-0.5, attack_penalty=-0.01))
    S, T, Q, R = (cfg.add_group(t) for t in (statue, target, queue, rover))
    t_any, q_any, r_any = (gw.AgentSymbol(g, 'any') for g in (T, Q, R))
    r2, r3 = gw.AgentSymbol(R, 'any'), gw.AgentSymbol(R, 'any')
    all_s, all_t, all_q, all_r = (gw.AgentSymbol(g, 'all') for g in (S, T, Q, R))
    cfg.add_reward_rule(gw.Event(all_s, 'attack', t_any), receiver=[t_any, all_s], value=[-0.25, 0.5])
    cfg.add_reward_rule(gw.Event(all_q, 'in_a_line'), receiver=all_q, value=0.3)
    r_fix = gw.AgentSymbol(R, 2)
    cfg.add_reward_rule(gw.Event(r_fix, 'attack', q_any), receiver=[r_fix, q_any], value=[0.7, -0.1])
    cfg.add_reward_rule(gw.Event(r_any, 'kill', gw.AgentSymbol(Q, 1)), receiver=r_any, value=5.0)
    cfg.add_reward_rule(gw.Event(r_any, 'attack', gw.AgentSymbol(Q, 0)), receiver=r_any, value=0.11)
    cfg.add_reward_rule(gw.Event(all_t, 'at', (6, 5)), receiver=all_t, value=0.01)
    cfg.add_reward_rule(gw.Event(r_any, 'attack', q_any) & gw.Event(r2, 'attack', q_any) & gw.Event(r3, 'in', ((0, 0), (size, size // 2))),
                        receiver=[r_any, r2, r3], value=[0.2, 0.1, 0.05])
    cfg.add_reward_rule(gw.Event(gw.AgentSymbol(S, 0), 'in', ((0, 0), (size, size))), receiver=all_s, value=99.0)   # never fires
    cfg.add_reward_rule(gw.Event(all_q, 'die'), receiver=all_r, value=10.0, terminal=True)
    return cfg


def make_general_rules(lib, seed=21, size=16, n_rover=40, **kw):
    """two statues flank one immobile target (both must hit it in the same step for the 'all' attack rule), a vertical
    queue that rovers attack until the line breaks, rovers added before AND after the first clear_dead"""
    import magent_b200 as magent
    env = magent.GridWorld(general_rules_config(size), _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    S, T, Q, R = env.get_handles()
    env.add_agents(S, method="custom", pos=[[5, 5, 0], [7, 5, 0]])
    env.add_agents(T, method="custom", pos=[[6, 5, 0]])
    env.add_agents(Q, method="custom", pos=[[12, 8 + i, 0] for i in range(4)])
    env.add_agents(R, method="random", n=n_rover)
    return env


def make_many_rules(lib, size=30, n=120, seed=5, n_rules=40, **kw):
    """battle with 40 reward rules (the reference has no limit; the device keeps the rule table in HBM)"""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = magent.builtin.config.battle.get_config(size)
    a, b = gw.AgentSymbol(0, 'any'), gw.AgentSymbol(1, 'any')
    for k in range(n_rules):
        s, o = (a, b) if k % 2 == 0 else (b, a)
        ev = gw.Event(s, 'attack', o) if k % 3 else gw.Event(s, 'in', ((k % 7, k % 5), (size - k % 4, size - k % 6)))
        cfg.add_reward_rule(ev, receiver=s, value=0.001 * (k + 1))
    env = magent.GridWorld(cfg, _lib=lib, **kw)
    env.set_seed(seed)
    env.reset()
    for h in env.get_handles():
        env.add_agents(h, method="random", n=n)
    return env


# ------------------------------------------------------------------ the cold info getters (GridWorld.cc:717-894)
def info_snapshot(env, with_mean=True):
    """everything env_get_info serves besides num/id/pos/alive: spaces, view2attack + attack_base, groups_info,
    walls_info, global_minimap (two shapes, every group as the viewer's channel 0), mean_info"""
    import ctypes
    out = {}
    hs = env.get_handles()
    out["groups_info"] = env._get_groups_info().copy()
    out["walls_info"] = env._get_walls_info().copy()
    for h in hs:
        g = env._hv(h)
        out["spaces", g] = (env.get_view_space(h), env.get_feature_space(h), env.get_action_space(h))
        base, v2a = env.get_view2attack(h)
        out["view2attack", g] = (base, v2a.copy())
        for shape in ((5, 7), (10, 10)):
            buf = np.empty(shape + (len(hs),), dtype=np.float32)
            buf[0, 0, 0], buf[0, 0, 1] = shape
            env._lib.env_get_info(env.game, g, b"global_minimap", buf.ctypes.data)
            out["global_minimap", g, shape] = buf
        if with_mean and env.get_num(h) > 0:
            out["mean_info", g] = env.get_mean_info(h).copy()
    return out


def compare_info_snapshots(a, b, what=""):
    assert a.keys() == b.keys(), what
    for k in a:
        if k[0] == "spaces":
            assert a[k] == b[k], "%s %s" % (what, k)
        elif k[0] == "view2attack":
            assert a[k][0] == b[k][0], "%s attack_base %s" % (what, k)
            np.testing.assert_array_equal(a[k][1], b[k][1], err_msg="%s %s" % (what, k))
        elif k[0] in ("global_minimap", "mean_info"):
            np.testing.assert_array_equal(a[k].view(np.uint32), b[k].view(np.uint32), err_msg="%s %s" % (what, k))
        else:
            np.testing.assert_array_equal(a[k], b[k], err_msg="%s %s" % (what, k))


def info_log(make, lib, steps=6, seed=3):
    """[(what, info_snapshot)] before the first step and after every step and clear_dead of a random-action game"""
    env = make(lib)
    log = [("before the first step", info_snapshot(env, with_mean=False))]
    rs = np.random.RandomState(seed)
    for t in range(steps):
        for h in env.get_handles():
            env.set_action(h, rs.randint(0, env.get_action_space(h)[0], size=env.get_num(h)).astype(np.int32))
        env.step()
        log.append(("after step %d" % t, info_snapshot(env)))
        env.clear_dead()
        log.append(("after clear_dead %d" % t, info_snapshot(env)))
    return log


def play_and_compare_info(make, lib_a, lib_b, steps=6, seed=3):
    for (what, a), (_, b) in zip(info_log(make, lib_a, steps, seed), info_log(make, lib_b, steps, seed)):
        compare_info_snapshots(a, b, what)


# ------------------------------------------------------------------ extensions: select_arena, event counters
def play_selected_arenas(engine_lib, checker_lib, steps=40, n=160):
    """3 battle arenas behind one handle, set up DIFFERENTLY per arena through magent_b200_select_arena (own seed,
    own walls, own extra agents), against 3 independent checker environments set up the same way; also checks the
    per-arena cold getters and the device event counters (agent_steps, kills + starved = deaths, steps)."""
    import magent_b200 as magent
    A, size = 3, 28
    seeds = [5, 40, 7]
    extra = {0: [[3, 3, 0], [4, 3, 0], [5, 3, 0]], 2: [[20, 20, 0]]}
    walls = {1: [[10, y, 0] for y in range(5, 15)], 2: [[x, 9, 0] for x in range(12, 18)]}
    batch = magent.GridWorld("battle", map_size=size, _lib=engine_lib, _num_arenas=A)
    singles = [magent.GridWorld("battle", map_size=size, _lib=checker_lib) for _ in range(A)]
    batch.reset()
    for a, env in enumerate(singles):
        env.set_seed(seeds[a]); env.reset()
        batch.select_arena(a); batch.set_seed(seeds[a])
        if a in walls:
            env.add_walls(method="custom", pos=walls[a]); batch.add_walls(method="custom", pos=walls[a])
    batch.select_arena(-1)
    for g in range(2):
        for env in singles:
            env.add_agents(env.get_handles()[g], method="random", n=n)
        batch.add_agents(batch.get_handles()[g], method="random", n=n)
    for a, pos in extra.items():
        batch.select_arena(a)
        batch.add_agents(batch.get_handles()[1], method="custom", pos=pos)
        singles[a].add_agents(singles[a].get_handles()[1], method="custom", pos=pos)
        np.testing.assert_array_equal(batch._get_walls_info(), singles[a]._get_walls_info())
    batch.select_arena(-1)
    hs = batch.get_handles()
    c0 = batch.get_counters()
    rs = np.random.RandomState(2)
    agent_steps = deaths = 0
    for t in range(steps):
        nums = [batch.get_arena_nums(h) for h in hs]
        for g, h in enumerate(hs):
            assert list(nums[g]) == [s.get_num(s.get_handles()[g]) for s in singles]
            v, f = batch.get_observation(h)
            off = np.concatenate([[0], np.cumsum(nums[g])])
            for a, s in enumerate(singles):
                rv, rf = s.get_observation(s.get_handles()[g])
                np.testing.assert_array_equal(v[off[a]:off[a + 1]].view(np.uint32), rv.view(np.uint32))
                np.testing.assert_array_equal(f[off[a]:off[a + 1]].view(np.uint32), rf.view(np.uint32))
            act = rs.randint(0, 21, size=int(nums[g].sum())).astype(np.int32)
            batch.set_action(h, act)
            agent_steps += act.size
            for a, s in enumerate(singles):
                s.set_action(s.get_handles()[g], np.ascontiguousarray(act[off[a]:off[a + 1]]))
        batch.step()
        for s in singles:
            s.step()
        for g, h in enumerate(hs):
            alive = batch.get_alive(h)
            deaths += int((~alive.astype(bool)).sum())
            np.testing.assert_array_equal(alive, np.concatenate([s.get_alive(s.get_handles()[g]) for s in singles]))
            np.testing.assert_array_equal(batch.get_pos(h), np.concatenate([s.get_pos(s.get_handles()[g]) for s in singles]))
        batch.clear_dead()
        for s in singles:
            s.clear_dead()
    c1 = batch.get_counters()
    d = [b - a for a, b in zip(c0, c1)]
    assert d[0] == agent_steps, "agent_steps counter %d, host count %d" % (d[0], agent_steps)
    assert d[3] + d[4] == deaths, "kills %d + starved %d != deaths %d" % (d[3], d[4], deaths)
    assert d[7] == steps, "steps counter %d" % d[7]          # counted once per env_step (step_phases.h: arena 0)
    assert d[5] + d[6] > 0 and d[1] >= d[2] >= d[3]
    return d


def group_reward_across_reset(lib):
    """two agents of group 0 next to one of group 1; every attack of group 0 pays 1.0 to the whole group 0
    (receiver index 'all' = group reward).  Returns [rewards after the step, rewards of the fresh episode before and
    after its first clear_dead]."""
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": 12, "map_height": 12})
    t = cfg.register_agent_type("t", dict(width=1, length=1, hp=10, speed=1, view_range=gw.CircleRange(3),
                                          attack_range=gw.CircleRange(1), damage=1, step_recover=0, step_reward=0.25))
    g0, g1 = cfg.add_group(t), cfg.add_group(t)
    a, b = gw.AgentSymbol(g0, index='any'), gw.AgentSymbol(g1, index='any')
    cfg.add_reward_rule(gw.Event(a, 'attack', b), receiver=gw.AgentSymbol(g0, index='all'), value=1.0)
    env = magent.GridWorld(cfg, _lib=lib)
    env.reset()
    h0, h1 = env.get_handles()
    env.add_agents(h0, method="custom", pos=[[5, 5], [8, 8]])
    env.add_agents(h1, method="custom", pos=[[6, 5]])
    base, v2a = env.get_view2attack(h0)
    hit = base + int(v2a[v2a.shape[0] // 2, v2a.shape[1] // 2 + 1])          # attack the cell to the east
    env.set_action(h0, np.array([hit, 0], dtype=np.int32))
    env.set_action(h1, np.array([0], dtype=np.int32))
    env.step()
    out = [env.get_reward(h0).copy()]
    env.reset()                                                               # no clear_dead before the new episode
    env.add_agents(h0, method="custom", pos=[[2, 2], [3, 3], [4, 4]])
    env.add_agents(h1, method="custom", pos=[[9, 9]])
    out.append(env.get_reward(h0).copy())
    env.clear_dead()
    out.append(env.get_reward(h0).copy())
    return out


def self_kill_frames(lib, render_dir, action=None):
    """a 1x2 body whose type may attack its own group aims at one of its own cells and kills itself; Map::do_attack
    then feeds the (dead) killer its victim's kill_supply (Map.cc:265-273), which the replay dump shows as the hp of
    the un-culled corpse.  With action=None: returns the first attack action that makes the lone agent die."""
    import magent_b200 as magent
    gw = magent.gridworld

    def make():
        cfg = gw.Config()
        cfg.set({"map_width": 10, "map_height": 10})
        t = cfg.register_agent_type("t", dict(width=1, length=2, hp=1.0, speed=0, view_range=gw.CircleRange(2),
                                              attack_range=gw.CircleRange(1.5), damage=2.0, step_recover=0.0,
                                              kill_supply=1.5, attack_in_group=1, kill_reward=3.0, dead_penalty=-0.5))
        cfg.add_group(t)
        env = magent.GridWorld(cfg, _lib=lib)
        env.reset()
        env.add_agents(env.get_handles()[0], method="custom", pos=[[4, 4], [7, 2]])
        return env
    if action is None:
        n_act = make().get_action_space(make().get_handles()[0])[0]
        for a in range(n_act):
            env = make()
            h = env.get_handles()[0]
            env.set_action(h, np.array([a, 0], dtype=np.int32))
            env.step()
            if not env.get_alive(h)[0]:
                return a
        raise AssertionError("no attack action makes the agent kill itself")
    os.makedirs(render_dir, exist_ok=True)
    env = make()
    env.set_render_dir(render_dir)
    h = env.get_handles()[0]
    env.set_action(h, np.array([action, 0], dtype=np.int32))
    env.step()
    rew = env.get_reward(h).copy()
    env.render()                                            # before clear_dead: the corpse is still listed
    env.clear_dead()
    env.render()
    return rew, {n: open(os.path.join(render_dir, n), "rb").read() for n in sorted(os.listdir(render_dir))}
