"""Algorithm checks on CPU: the *same phase functions the CUDA kernels run* (step_phases.h, obs_phases.h),
executed by the test-only single-thread emulation backend (tests/emu/), against the committed golden
vectors recorded from the compiled reference.  This validates the parallel formulations (shuffle replay,
attack/move relaxation, rule programs, compaction) and the whole host engine where no GPU exists; the
`-m gpu` tests then validate the CUDA execution of the same functions."""
import os
import subprocess

import numpy as np
import pytest

import golden_common as gc
import parity_common as pc


@pytest.fixture(scope="module")
def emu():
    src_dir = os.path.join(pc.REPO, "magent_b200", "csrc")
    newest = max(os.path.getmtime(os.path.join(src_dir, f)) for f in os.listdir(src_dir))
    newest = max(newest, os.path.getmtime(os.path.join(pc.REPO, "tests", "emu", "backend_emu.cc")))
    if not os.path.exists(pc.EMU_LIB) or os.path.getmtime(pc.EMU_LIB) < newest:
        subprocess.run([os.path.join(pc.REPO, "tests", "emu", "build.sh")], check=True, capture_output=True)
    return pc.EMU_LIB


@pytest.mark.parametrize("name", sorted(gc.SCENARIOS))
def test_phase_functions_reproduce_golden(emu, name):
    gc.check_against_golden(name, emu)


def test_arena_batch_matches_single_arenas(emu):
    """A arenas behind one handle == A single-arena engines seeded seed+a (host logic of the batching)"""
    import magent_b200 as magent
    A, n, size = 3, 80, 30
    env = magent.GridWorld("battle", map_size=size, _lib=emu, _num_arenas=A)
    env.set_seed(5)
    env.reset()
    for h in env.get_handles():
        env.add_agents(h, method="random", n=n)
    singles = []
    for a in range(A):
        s = magent.GridWorld("battle", map_size=size, _lib=emu)
        s.set_seed(5 + a)
        s.reset()
        for h in s.get_handles():
            s.add_agents(h, method="random", n=n)
        singles.append(s)
    rs = np.random.RandomState(1)
    hs = env.get_handles()
    for t in range(25):
        nums = [env.get_arena_nums(h) for h in hs]
        acts = [rs.randint(0, 21, size=int(nums[g].sum())).astype(np.int32) for g in range(2)]
        for g, h in enumerate(hs):
            v, f = env.get_observation(h)
            off = np.concatenate([[0], np.cumsum(nums[g])])
            for a, s in enumerate(singles):
                sv, sf = s.get_observation(s.get_handles()[g])
                np.testing.assert_array_equal(v[off[a]:off[a + 1]], sv)
                np.testing.assert_array_equal(f[off[a]:off[a + 1]], sf)
                s.set_action(s.get_handles()[g], np.ascontiguousarray(acts[g][off[a]:off[a + 1]]))
            env.set_action(h, acts[g])
        env.step()
        for s in singles:
            s.step()
        for g, h in enumerate(hs):
            off = np.concatenate([[0], np.cumsum(nums[g])])
            rew, pos = env.get_reward(h), env.get_pos(h)
            for a, s in enumerate(singles):
                np.testing.assert_array_equal(rew[off[a]:off[a + 1]], s.get_reward(s.get_handles()[g]))
                np.testing.assert_array_equal(pos[off[a]:off[a + 1]], s.get_pos(s.get_handles()[g]))
        env.clear_dead()
        for s in singles:
            s.clear_dead()


def test_mid_episode_add_agents_roundtrip(emu):
    """add_agents after stepping: device image -> host image -> mutate -> device image"""
    def run(lib):
        env = pc.make_battle(lib, 30, 60, 2)
        hs = env.get_handles()
        rs = np.random.RandomState(2)
        out = []
        for t in range(20):
            if t == 8:
                env.add_agents(hs[0], method="random", n=15)
                env.add_agents(hs[1], method="custom", pos=[[3, 3], [4, 9], [12, 12]])
            for h in hs:
                v, f = env.get_observation(h)
                out.append(pc.sha(v) + pc.sha(f))
            for h in hs:
                env.set_action(h, rs.randint(0, 21, size=env.get_num(h)).astype(np.int32))
            env.step()
            out.append([env.get_reward(h).tolist() for h in hs])
            out.append([env.get_agent_id(h).tolist() for h in hs])
            env.clear_dead()
        return out
    gc.check_reference_result("mid_episode_add_agents", run, emu)


def test_forty_rules(emu):
    gc.check_reference_result("forty_rules", lambda lib: pc.run_trace(pc.make_many_rules(lib), 25, 5, keep_obs=True), emu)


def test_unsupported_rule_shapes_fail_loudly(emu):
    """'align' reads counters the reference never allocates (a null dereference there): the engine must abort with a
    message naming the rule, not diverge silently; same for a receiver the trigger does not bind"""
    import sys
    for rule, msg in (("gw.Event(gw.AgentSymbol(0, 'any'), 'align'), receiver=gw.AgentSymbol(1, 'all')", "'align'"),
                      ("gw.Event(gw.AgentSymbol(0, 'any'), 'die'), receiver=gw.AgentSymbol(1, 'any')", "not bound")):
        code = ("import magent_b200 as m; gw = m.gridworld; c = m.builtin.config.battle.get_config(30); "
                "c.add_reward_rule(%s, value=1); e = m.GridWorld(c, _lib=%r); e.reset()" % (rule, emu))
        out = subprocess.run([sys.executable, "-c", code], cwd=pc.REPO, capture_output=True, text=True)
        assert out.returncode != 0 and msg in out.stderr, out.stderr


@pytest.mark.parametrize("seed", [13, 14, 15])
def test_absorb_contention_matches_reference(emu, seed):
    """dense absorbers: several movers reach the same goal in one step; only the first in move order is absorbed"""
    kw = dict(act_groups=[1], keep_obs=True, stop_on_done=False)
    gc.check_reference_result("absorb_contention/%d" % seed,
                              lambda lib: pc.run_trace(pc.make_arrange(lib, 20, seed, n_goal=40, n_agent=200), 40, seed, **kw), emu)


def _render_episode(lib, tmpdir, scenario):
    os.makedirs(tmpdir, exist_ok=True)
    env = scenario(lib)
    env.set_render_dir(tmpdir)
    hs = env.get_handles()
    rs = np.random.RandomState(3)
    for t in range(12):
        for h in hs:
            env.set_action(h, rs.randint(0, env.get_action_space(h)[0], size=env.get_num(h)).astype(np.int32))
        env.step()
        env.render()
        env.clear_dead()
    info = env._get_render_info((0, 20), (0, 20))
    files = {}
    for name in sorted(os.listdir(tmpdir)):
        files[name] = open(os.path.join(tmpdir, name), "rb").read()
    return files, sorted((k, tuple(v)) for k, v in info[0].items()), info[1].tolist()


@pytest.mark.parametrize("which", ["battle", "arrange", "turn", "food"])
def test_render_dump_is_byte_identical(emu, tmp_path, which):
    """env_render: config.json + video_N.txt frames incl. attack events (RenderGenerator.cc:63-185)"""
    scen = {"battle": lambda lib: pc.make_battle(lib, 30, 200, 3), "arrange": lambda lib: pc.make_arrange(lib, 30, 12),
            "turn": lambda lib: pc.make_turn(lib, 30, 5), "food": lambda lib: pc.make_food(lib, 30, 3)}[which]
    a = _render_episode(pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB, str(tmp_path / "ref"), scen)
    b = _render_episode(emu, str(tmp_path / "emu"), scen)
    assert sorted(a[0]) == sorted(b[0]) and "config.json" in a[0]
    for name in a[0]:
        assert a[0][name] == b[0][name], name
    assert any(line.startswith(b"0 ") for line in a[0]["video_1.txt"].splitlines()) or which != "battle"
    assert a[1] == b[1] and a[2] == b[2]


def _f16_trace(lib, mk, steps, seed):
    """per step: ((view, feature) float32, (view, feature) float16) of every group, random actions in between"""
    env = mk(lib)
    handles = env.get_handles()
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(steps):
        rec = []
        for h in handles:
            if env.get_num(h) == 0:
                continue
            v32, f32 = [x.copy() for x in env.get_observation(h)]
            v16, f16 = [x.copy() for x in env.get_observation_f16(h)]
            rec.append((v32, f32, v16, f16))
        out.append(rec)
        for h in handles:
            env.set_action(h, rs.randint(0, env.get_action_space(h)[0], size=env.get_num(h)).astype(np.int32))
        env.step()
        env.clear_dead()
    return out


@pytest.mark.parametrize("which", ["battle", "pursuit", "arrange"])
def test_f16_observation_is_the_rounded_f32_observation(emu, which):
    """magent_b200_get_observation_f16 (include/magent_b200_ext.h): every element equals the float32 observation
    of the same state rounded to nearest-even (numpy astype), NaN payloads included; interleaving the two calls
    does not disturb the state."""
    mk = {"battle": lambda lib: pc.make_battle(lib, 40, 60, seed=3),
          "pursuit": lambda lib: pc.make_pursuit(lib),
          "arrange": lambda lib: pc.make_arrange(lib, 24, 14, n_goal=60, n_agent=150)}[which]
    for rec in _f16_trace(emu, mk, 12 if which != "arrange" else 40, 5):
        for v32, f32, v16, f16 in rec:
            assert v16.dtype == np.float16 and v16.shape == v32.shape and f16.shape == f32.shape
            with np.errstate(all="ignore"):
                np.testing.assert_array_equal(v16.view(np.uint16), v32.astype(np.float16).view(np.uint16))
                np.testing.assert_array_equal(f16.view(np.uint16), f32.astype(np.float16).view(np.uint16))


def _goal_trace(lib):
    """goal_mode (deprecated in the reference, GridWorld.cc:137,667-679,929): two extra, never-written feature
    slots; set_goal('random') only advances the engine RNG by two draws per agent"""
    import magent_b200 as magent
    cfg = magent.builtin.config.battle.get_config(30)
    cfg.set({"goal_mode": True})
    env = magent.GridWorld(cfg, _lib=lib)
    env.set_seed(5)
    env.reset()
    h = env.get_handles()
    env.add_agents(h[0], method="random", n=40)
    env.set_goal(h[0], "random")
    env.add_agents(h[1], method="random", n=40)      # placement after the goal draws: the RNG stream must agree
    out = [env.get_feature_space(h[0]), env.get_pos(h[1]).copy()]
    rs = np.random.RandomState(1)
    for _ in range(5):
        for g in h:
            v, f = env.get_observation(g)
            out += [v.copy(), f.copy()]
        for g in h:
            env.set_action(g, rs.randint(0, 21, size=env.get_num(g)).astype(np.int32))
        env.step()
        env.set_goal(h[1], "random")                 # mid-episode: moves the attack shuffle of the next step
        out.append(env.get_reward(h[0]).copy())
        env.clear_dead()
    return out


def test_goal_mode_feature_slots_and_rng_draws(emu):
    want, got = _goal_trace(pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB), _goal_trace(emu)
    assert want[0] == got[0] == (34 + 2,)
    for a, b in zip(want[1:], got[1:]):
        if a.dtype == np.float32 and a.ndim == 1:
            np.testing.assert_allclose(a, b, atol=pc.REWARD_TOL, rtol=0)
        else:
            np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("which", ["battle", "pursuit", "mixed", "arrange"])
def test_cold_info_getters_match_the_reference(emu, which):
    """view2attack / attack_base / groups_info / walls_info / global_minimap / mean_info (GridWorld.cc:717-894)"""
    make = {"battle": lambda lib: pc.make_battle(lib, 30, 120, 1), "pursuit": lambda lib: pc.make_pursuit(lib, 40, 2),
            "mixed": lambda lib: pc.make_mixed(lib), "arrange": lambda lib: pc.make_arrange(lib)}[which]
    pc.play_and_compare_info(make, pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB, emu)


def test_select_arena_and_event_counters(emu):
    """per-arena setup through magent_b200_select_arena; counters of the batch against host-side counts"""
    checker = pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB
    d = pc.play_selected_arenas(emu, checker)
    assert d[3] + d[4] > 0, "the scenario is supposed to see deaths"


def test_uncollected_group_reward_survives_reset(emu):
    """Group::clear (GridWorld.h:277-280) keeps the group's next_reward: a group reward earned in the last step of an
    episode that ends without clear_dead is still added to every get_reward of the next episode until clear_dead"""
    checker = pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB
    outs = []
    for lib in (checker, emu):
        outs.append(pc.group_reward_across_reset(lib))
    assert outs[0][0].max() > 0.5, "the scenario is supposed to earn a group reward"
    for a, b in zip(*outs):
        np.testing.assert_allclose(a, b, rtol=0, atol=pc.REWARD_TOL)


def test_self_kill_feeds_the_corpse(emu, tmp_path):
    """found by the chaotic fuzz: hp of an un-culled corpse in the replay dump after a self-aimed in-group attack"""
    checker = pc.REF_LIB if os.path.exists(pc.REF_LIB) else pc.PORT_LIB
    act = pc.self_kill_frames(checker, None)
    want = pc.self_kill_frames(checker, str(tmp_path / "ref"), act)
    got = pc.self_kill_frames(emu, str(tmp_path / "emu"), act)
    np.testing.assert_allclose(want[0], got[0], rtol=0, atol=pc.REWARD_TOL)
    assert want[1] == got[1]
    frame = want[1]["video_1.txt"].decode().splitlines()
    assert any(l.split()[:2] == ["0", "50"] for l in frame), frame       # corpse: hp = -1 + 1.5 = 0.5 of 1.0 -> "50"


def test_golden_edge_cases(emu, tmp_path):
    """tests/golden/edge_cases.npz: group reward across reset, replay frames after a self-kill"""
    gc.check_edge_cases(emu, str(tmp_path / "frames"))
