"""The oracle side, on CPU: the compiled reference (when present) and the C restatement reproduce the
committed golden vectors through this repository's host wrapper; known-answer micro-scenarios from
SURVEY.md App. B.2 hold."""
import os

import numpy as np
import pytest

import golden_common as gc
import parity_common as pc


def oracle_libs():
    libs = [p for p in (pc.REF_LIB, pc.PORT_LIB) if os.path.exists(p)]
    return libs


@pytest.mark.parametrize("name", sorted(gc.SCENARIOS))
def test_oracles_reproduce_golden(name):
    libs = oracle_libs()
    if not libs:
        pytest.skip("no oracle library built")
    for lib in libs:
        gc.check_against_golden(name, lib)


def test_golden_files_present():
    for name in gc.SCENARIOS:
        assert os.path.exists(os.path.join(gc.GOLDEN_DIR, name + ".npz")), name


@pytest.fixture(params=["ref", "port"])
def olib(request):
    p = pc.REF_LIB if request.param == "ref" else pc.PORT_LIB
    if not os.path.exists(p):
        pytest.skip(request.param + " oracle not built")
    return p


def _battle20(lib, pos0, pos1):
    import magent_b200 as magent
    env = magent.GridWorld("battle", map_size=20, _lib=lib)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[0], method="custom", pos=pos0)
    if pos1:
        env.add_agents(h[1], method="custom", pos=pos1)
    return env, h


def test_kat_spaces(olib):
    import magent_b200 as magent
    env = magent.GridWorld("battle", map_size=40, _lib=olib)
    assert env.view_space[0] == (13, 13, 7) and env.feature_space[0] == (34,) and env.action_space[0] == (21,)
    env = magent.GridWorld("pursuit", map_size=40, _lib=olib)
    assert env.view_space == {0: (10, 10, 5), 1: (9, 9, 5)}
    assert env.feature_space == {0: (14,), 1: (10,)} and env.action_space == {0: (13,), 1: (9,)}
    env = magent.GridWorld(pc.gather_config(40), _lib=olib)
    assert env.view_space == {0: (3, 3, 7), 1: (15, 15, 7)}
    assert env.feature_space == {0: (4,), 1: (36,)} and env.action_space == {0: (1,), 1: (33,)}


def test_kat_first_random_placements(olib):
    """minstd_rand0 from state 1 (SURVEY.md App. B)"""
    env = pc.make_battle(olib, 200, 5, 0)
    np.testing.assert_array_equal(env.get_pos(env.get_handles()[0]),
                                  [[91, 122], [93, 123], [21, 142], [20, 161], [65, 130]])


def test_kat_six_hits_kill(olib):
    """hp 10, damage 2, +0.1 regen: the 6th hit kills (SURVEY.md App. B.2 row 1)"""
    env, h = _battle20(olib, [[5, 5]], [[6, 5]])
    seen, rewards = [], []
    for t in range(6):
        v, f = env.get_observation(h[0])
        seen.append(v[0, 6, 7, 5].copy())
        env.get_observation(h[1])
        env.set_action(h[0], np.array([17], dtype=np.int32))
        env.set_action(h[1], np.array([6], dtype=np.int32))
        done = env.step()
        rewards.append((env.get_reward(h[0])[0], env.get_reward(h[1])[0]))
        alive = env.get_alive(h[1])[0]
        env.clear_dead()
    want_hp = np.array([0x3f800000, 0x3f4f5c2a, 0x3f1eb852, 0x3edc28f6, 0x3e75c290, 0x3d4cccd0], dtype=np.uint32)
    np.testing.assert_array_equal(np.array(seen, dtype=np.float32).view(np.uint32), want_hp)
    for r0, r1 in rewards[:5]:
        assert abs(r0 - 0.0949999988) < 1e-7 and abs(r1 + 0.00499999989) < 1e-9
    assert abs(rewards[5][0] - 4.89499998) < 1e-6 and abs(rewards[5][1] + 0.100000001) < 1e-8
    assert done and not alive


def test_kat_move_contention_and_chains(olib):
    def play(pos0, acts, pos1=None, acts1=None, order=(0, 1)):
        env, h = _battle20(olib, pos0, pos1)
        a = {0: np.array(acts, dtype=np.int32), 1: None if acts1 is None else np.array(acts1, dtype=np.int32)}
        for g in order:
            if a[g] is not None:
                env.set_action(h[g], a[g])
        env.step()
        return env.get_pos(h[0]).tolist(), (env.get_pos(h[1]).tolist() if pos1 else None)
    assert play([[5, 5], [7, 5]], [7, 5])[0] == [[6, 5], [7, 5]]           # lower index wins the cell
    assert play([[5, 5], [6, 5]], [7, 7])[0] == [[5, 5], [7, 5]]           # follower first: blocked
    assert play([[6, 5], [5, 5]], [7, 7])[0] == [[7, 5], [6, 5]]           # leader first: both move
    p0, p1 = play([[5, 5]], [7], [[7, 5]], [5], order=(0, 1))
    assert p0 == [[6, 5]] and p1 == [[7, 5]]
    p0, p1 = play([[5, 5]], [7], [[7, 5]], [5], order=(1, 0))
    assert p0 == [[5, 5]] and p1 == [[6, 5]]


def test_kat_band_order_on_large_map(olib):
    """100x100 => 8 bands of 13: the interior agent moves before the boundary-zone agent"""
    import magent_b200 as magent
    env = magent.GridWorld("battle", map_size=100, _lib=olib)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[0], method="custom", pos=[[14, 50], [18, 50]])
    env.set_action(h[0], np.array([8, 4], dtype=np.int32))
    env.step()
    assert env.get_pos(h[0]).tolist() == [[14, 50], [16, 50]]


def test_kat_shuffle_decides_mutual_kill(olib):
    """two gather agents attack each other with lethal damage; who strikes first follows minstd_rand0
    (SURVEY.md App. B.2: alive = [T,F], [F,T], [F,T], [F,T] over four episodes of one env)"""
    import magent_b200 as magent
    env = magent.GridWorld(pc.gather_config(30), _lib=olib)
    h = env.get_handles()
    got = []
    for _ in range(4):
        env.reset()
        env.add_agents(h[1], method="custom", pos=[[10, 10], [11, 10]])
        env.add_agents(h[0], method="custom", pos=[[20, 20]])
        env.set_action(h[1], np.array([29 + 2, 29 + 1], dtype=np.int32))
        env.step()
        got.append(env.get_alive(h[1]).tolist())
        r = env.get_reward(h[1])
        np.testing.assert_allclose(sorted(r.tolist()), [-1.0, -0.11], atol=1e-6)
    assert got == [[True, False], [False, True], [False, True], [False, True]]


@pytest.mark.parametrize("game", ["forest", "double_attack"])
def test_port_matches_reference_beyond_golden(game):
    """the restatement's general rule evaluator (two free symbols in double_attack) vs the compiled reference"""
    import magent_b200 as magent

    def make(lib):
        env = magent.GridWorld(game, map_size=30, _lib=lib)
        env.set_seed(3)
        env.reset()
        h = env.get_handles()
        env.add_agents(h[0], method="random", n=120)
        env.add_agents(h[1], method="random", n=60)
        return env
    gc.check_reference_result("port_beyond_golden/" + game, lambda lib: pc.run_trace(make(lib), 60, 3, keep_obs=True),
                              pc.PORT_LIB)


@pytest.mark.parametrize("which", ["battle", "pursuit", "mixed", "arrange"])
def test_port_serves_the_cold_info_getters_like_the_reference(which):
    """view2attack / attack_base / groups_info / walls_info / global_minimap / mean_info (GridWorld.cc:717-894)"""
    make = {"battle": lambda lib: pc.make_battle(lib, 30, 120, 1), "pursuit": lambda lib: pc.make_pursuit(lib, 40, 2),
            "mixed": lambda lib: pc.make_mixed(lib), "arrange": lambda lib: pc.make_arrange(lib)}[which]
    gc.check_reference_result("cold_info/" + which, lambda lib: pc.info_log(make, lib), pc.PORT_LIB)


def test_port_reproduces_the_golden_edge_cases():
    """tests/golden/edge_cases.npz (recorded from the compiled reference): a group reward that survives reset(), the
    replay frames after a self-kill"""
    import tempfile
    gc.check_edge_cases(pc.PORT_LIB, tempfile.mkdtemp())


@pytest.mark.parametrize("which", ["battle", "arrange", "turn", "food"])
def test_port_writes_the_replay_dump_of_the_reference(tmp_path, which):
    """env_render: config.json + video_N.txt frames incl. attack events, render_window_info / attack_event
    (RenderGenerator.cc:56-185, GridWorld.cc:797-842)"""
    import tempfile
    from test_emu_parity_cpu import _render_episode
    scen = {"battle": lambda lib: pc.make_battle(lib, 30, 200, 3), "arrange": lambda lib: pc.make_arrange(lib, 30, 12),
            "turn": lambda lib: pc.make_turn(lib, 30, 5), "food": lambda lib: pc.make_food(lib, 30, 3)}[which]
    gc.check_reference_result("replay_dump/" + which, lambda lib: _render_episode(lib, tempfile.mkdtemp(dir=str(tmp_path)), scen),
                              pc.PORT_LIB)
