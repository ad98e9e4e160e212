"""Parity of the CUDA engine against the oracle, through the C ABI, on a real GPU.

Checker = the compiled reference (oracle/_ref/libmagent.so, built from /root/reference by
oracle/Makefile and shipped to the GPU box) or, when absent, the C restatement (oracle/_build).
Both engines are driven by the same host code (magent_b200.gridworld) with the same seeds and the same
pre-generated action streams; integer state and observations must match bit-exactly, rewards within 1e-6.
"""
import os

import numpy as np
import pytest

import parity_common as pc

pytestmark = pytest.mark.gpu


def checker_lib():
    for p in (pc.REF_LIB, pc.PORT_LIB):
        if os.path.exists(p):
            return p
    pytest.skip("no oracle library available (oracle/_ref or oracle/_build)")


def both(make, steps, seed, **kw):
    want = pc.run_trace(make(checker_lib()), steps, seed, keep_obs=True, **kw)
    got = pc.run_trace(make(pc.CUDA_LIB), steps, seed, keep_obs=True, **kw)
    pc.compare_traces(want, got)
    return want


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_battle_small(seed):
    both(lambda lib: pc.make_battle(lib, 40, 150, seed), 60, seed)


def test_battle_dense_blocks():
    both(lambda lib: pc.make_battle_blocks(lib, 40), 80, 5)


def test_battle_kills_happen():
    """dense enough that agents die, get culled and re-indexed"""
    want = both(lambda lib: pc.make_battle(lib, 30, 300, 3), 80, 3)
    assert want[-1]["num"][0] < 300 and want[-1]["num"][1] < 300


def test_battle_large_map_bands():
    """w*h > 99*99 switches the reference to banded move buffers (GridWorld.cc:75-85,411-438)"""
    both(lambda lib: pc.make_battle(lib, 120, 2000, 7), 25, 7)


def test_battle_config2_200x200():
    """BASELINE.json configs[1]: battle 200x200, 2x1000 agents"""
    both(lambda lib: pc.make_battle(lib, 200, 1000, 0), 20, 0)


def test_set_action_order_decides_contention():
    """the group whose set_action is called first moves first (SURVEY.md App. B.2)"""
    both(lambda lib: pc.make_battle(lib, 30, 250, 11), 30, 11, order=[1, 0])


@pytest.mark.parametrize("seed", [0, 1])
def test_pursuit_2x2_bodies(seed):
    """BASELINE.json configs[0] geometry: 40x40, walls, 2x2 predators"""
    both(lambda lib: pc.make_pursuit(lib, 40, seed), 100, seed)


@pytest.mark.parametrize("seed", [0, 1])
def test_gather_attack_in_group(seed):
    both(lambda lib: pc.make_gather(lib, 40, seed), 100, seed, act_groups=[1])


def test_gather_dense_infighting():
    """agents kill each other (hp 3, damage 6): exercises shuffle order + skip-dead-attacker"""
    want = both(lambda lib: pc.make_gather(lib, 24, 2, n_agent=150, n_food=60), 40, 2, act_groups=[1])
    assert want[-1]["num"][1] < 150


def test_forest_kill_supply_heals():
    """tigers eat deer: kill_supply heals the killer inside the attack timeline (Map.cc:274)"""
    want = both(lambda lib: pc.make_builtin(lib, "forest", 30, 3), 80, 3)
    assert want[-1]["num"][0] < 120


def test_double_attack_two_subject_rule():
    """`e1 & e2` with two free tiger symbols: the pair-scan rule kernel vs the reference DFS"""
    want = both(lambda lib: pc.make_builtin(lib, "double_attack", 30, 4, n0=150, n1=120), 60, 4)
    assert any((r["reward"][1] > 0.5).any() for r in want), "no cooperative reward ever fired: test too weak"


def test_mixed_three_groups_big_view_rules():
    """3 groups, 2x2 + 1x1 bodies, 19x19 view (> 256 cells), starvation, kill_supply, in-group attacks,
    rules with kill/collide/in/die/not/or and agent / object / whole-group receivers"""
    both(lambda lib: pc.make_mixed(lib, 36, 6), 60, 6, order=[2, 0, 1])


def test_four_groups_sixteen_rules():
    """the examples/train_multi.py game: 2 unit types x 2 armies, 13 channels, 16 attack/kill rules"""
    both(lambda lib: pc.make_multi4(lib), 50, 8, order=[3, 1, 0, 2])


def test_general_rule_shapes():
    """'all' subjects (attack / in_a_line / die / at), fixed-index subjects and objects (Agent::index is refreshed by
    clear_dead only), three free symbols, a rule that can never fire, a terminal group rule (RewardEngine.cc:216-443)"""
    want = both(lambda lib: pc.make_general_rules(lib), 70, 21, stop_on_done=False)
    assert any(r["done"] for r in want) and want[-1]["num"][2] == 0


def test_forty_rules():
    # more rules than the C restatement holds: against the reference's recorded result
    import golden_common as gc
    gc.check_reference_result("forty_rules", lambda lib: pc.run_trace(pc.make_many_rules(lib), 25, 5, keep_obs=True),
                              pc.CUDA_LIB)


@pytest.mark.parametrize("seed", [12, 13])
def test_absorbing_goals(seed):
    """can_absorb types (train_arrange): the first mover (in move order) that bumps into a free goal dies into it"""
    want = both(lambda lib: pc.make_arrange(lib, 30, seed), 60, seed, act_groups=[1], stop_on_done=False)
    assert want[-1]["num"][1] < 160


def test_sector_view_and_attack_ranges():
    """SectorRange (angle < 180) views and attacks, 1x1 and 2x2 bodies (Range.h:104-144)"""
    both(lambda lib: pc.make_sector(lib), 50, 9, order=[1, 0])


@pytest.mark.parametrize("seed,order", [(3, [1, 2, 0]), (5, [2, 0, 1])])
def test_turn_mode_headings_long_bodies(seed, order):
    """turn_mode: headings, [moves][turn L,R][attacks], rotated views / attacks / moves, pivoting 1x3 and 2x1 bodies"""
    both(lambda lib: pc.make_turn(lib, 30, seed), 80, seed, order=order, stop_on_done=False)


@pytest.mark.parametrize("seed,order", [(3, [1, 2, 0]), (5, [2, 0, 1]), (9, [0, 1, 2])])
def test_food_mode_kills_leave_food_that_is_eaten(seed, order):
    """food_mode: food on the attacked cell of a kill, eaten by later attackers (any group), blocks moves, own channel"""
    both(lambda lib: pc.make_food(lib, 30, seed), 80, seed, order=order, stop_on_done=False)


def test_absorbing_goals_that_move_themselves():
    """goals receive actions too: a goal bumping into a goal is absorbed by it, and an absorber that swallowed somebody
    earlier in the move phase skips its own move (GridWorld.cc:581 evaluated at its turn)"""
    both(lambda lib: pc.make_arrange(lib, 24, 14, n_goal=60, n_agent=150), 40, 14, stop_on_done=False)


def test_render_dump_matches_reference(tmp_path):
    """env_render through the CUDA engine: config.json + video_N.txt byte-identical, attack events included"""
    from test_emu_parity_cpu import _render_episode
    scen = lambda lib: pc.make_battle(lib, 30, 200, 3)
    a = _render_episode(checker_lib(), str(tmp_path / "ref"), scen)
    b = _render_episode(pc.CUDA_LIB, str(tmp_path / "gpu"), scen)
    assert a[0] == b[0] and a[1] == b[1] and a[2] == b[2]


def test_two_engines_interleaved_in_one_process():
    """two CUDA environments of different games stepping alternately: per-engine state must not leak through the
    backend's shared scratch (hp_norm plane, template tiles, header table)"""
    ea, eb = pc.make_battle(pc.CUDA_LIB, 40, 150, 0), pc.make_pursuit(pc.CUDA_LIB, 40, 0)
    ra, rb = pc.make_battle(checker_lib(), 40, 150, 0), pc.make_pursuit(checker_lib(), 40, 0)
    rs = np.random.RandomState(0)
    for t in range(15):
        for env, ref in ((ea, ra), (eb, rb)):
            hs, hr = env.get_handles(), ref.get_handles()
            for h, k in zip(hs, hr):
                v, f = env.get_observation(h)
                rv, rf = ref.get_observation(k)
                np.testing.assert_array_equal(v.view(np.uint32), rv.view(np.uint32), err_msg="view t%d" % t)
                np.testing.assert_array_equal(f.view(np.uint32), rf.view(np.uint32), err_msg="feat t%d" % t)
        for env, ref in ((ea, ra), (eb, rb)):
            for h, k in zip(env.get_handles(), ref.get_handles()):
                a = rs.randint(0, env.get_action_space(h)[0], size=env.get_num(h)).astype(np.int32)
                env.set_action(h, a)
                ref.set_action(k, a)
            assert env.step() == ref.step()
            for h, k in zip(env.get_handles(), ref.get_handles()):
                np.testing.assert_array_equal(env.get_pos(h), ref.get_pos(k))
            env.clear_dead()
            ref.clear_dead()


def test_non_square_map():
    both(lambda lib: pc.make_battle_rect(lib), 40, 2)


def test_episodes_share_one_rng_stream():
    """reset() keeps the engine RNG running (GridWorld.cc:29,72-118): three episodes on one env, device -> host ->
    device round trips included"""
    import magent_b200 as magent

    def run(lib):
        env = magent.GridWorld("battle", map_size=30, _lib=lib)
        env.set_seed(9)
        hs = env.get_handles()
        rs = np.random.RandomState(9)
        out = []
        for ep in range(3):
            env.reset()
            for h in hs:
                env.add_agents(h, method="random", n=100 + 20 * ep)
            for t in range(12):
                for h in hs:
                    v, f = env.get_observation(h)
                    out.append(pc.sha(v) + pc.sha(f))
                for h in hs:
                    env.set_action(h, rs.randint(0, 21, size=env.get_num(h)).astype(np.int32))
                out.append(env.step())
                out.append([env.get_reward(h).round(6).tolist() for h in hs])
                out.append([env.get_pos(h).tolist() for h in hs])
                env.clear_dead()
        return out
    assert run(checker_lib()) == run(pc.CUDA_LIB)


def test_empty_group_observation_and_actions():
    """a group with no agents: its calls are no-ops, the other group still observes (its minimap channel for the
    empty group is 0/0 = NaN in the reference; the engine emits the x86 default-NaN payload, so even that is bit-exact)"""
    import magent_b200 as magent

    def run(lib):
        env = magent.GridWorld("battle", map_size=30, _lib=lib)
        env.reset()
        h = env.get_handles()
        env.add_agents(h[0], method="custom", pos=[[5, 5], [8, 9], [20, 11]])
        assert env.get_num(h[1]) == 0
        v, f = env.get_observation(h[0])
        v, f = v.copy(), f.copy()
        env.set_action(h[0], np.array([3, 4, 15], dtype=np.int32))
        env.set_action(h[1], np.zeros((0,), dtype=np.int32))
        done = env.step()
        r = env.get_reward(h[0]).copy()
        assert env.get_reward(h[1]).shape == (0,) and env.get_alive(h[1]).shape == (0,)
        env.clear_dead()
        return v, f, done, r, env.get_pos(h[0]).copy()
    a, b = run(checker_lib()), run(pc.CUDA_LIB)
    assert a[2] == b[2] is True
    assert np.isnan(a[0]).any()
    np.testing.assert_array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    np.testing.assert_array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    np.testing.assert_allclose(a[3], b[3], atol=pc.REWARD_TOL, rtol=0)
    np.testing.assert_array_equal(a[4], b[4])


def test_unculled_dead_agents_keep_their_slots():
    """no clear_dead between steps: dead agents stay in the vectors, still get actions, are skipped"""
    import magent_b200  # noqa: F401

    def run(lib):
        env = pc.make_battle(lib, 24, 150, 4)
        hs = env.get_handles()
        rs = np.random.RandomState(4)
        out = []
        for t in range(30):
            obs = [tuple(x.copy() for x in env.get_observation(h)) for h in hs]
            acts = [rs.randint(0, 21, size=env.get_num(h)).astype(np.int32) for h in hs]
            for h, a in zip(hs, acts):
                env.set_action(h, a)
            done = env.step()
            out.append((obs, [env.get_reward(h).copy() for h in hs], [env.get_alive(h).copy() for h in hs],
                        [env.get_pos(h).copy() for h in hs], done))
            if t % 5 == 4:
                env.clear_dead()
        return out
    a, b = run(checker_lib()), run(pc.CUDA_LIB)
    for t, (ra, rb) in enumerate(zip(a, b)):
        for g in range(2):
            np.testing.assert_array_equal(ra[0][g][0].view(np.uint32), rb[0][g][0].view(np.uint32), err_msg="view t%d" % t)
            np.testing.assert_array_equal(ra[0][g][1].view(np.uint32), rb[0][g][1].view(np.uint32), err_msg="feat t%d" % t)
            np.testing.assert_allclose(ra[1][g], rb[1][g], atol=pc.REWARD_TOL, rtol=0)
            np.testing.assert_array_equal(ra[2][g], rb[2][g])
            np.testing.assert_array_equal(ra[3][g], rb[3][g])
        assert ra[4] == rb[4]


def test_arena_batch_equals_independent_references():
    """4 arenas behind one handle == 4 reference environments seeded seed+a"""
    import magent_b200 as magent
    A, n, size, steps = 4, 120, 36, 40
    env = magent.GridWorld("battle", map_size=size, _lib=pc.CUDA_LIB, _num_arenas=A)
    env.set_seed(20)
    env.reset()
    hs = env.get_handles()
    for h in hs:
        env.add_agents(h, method="random", n=n)
    refs = []
    for a in range(A):
        r = magent.GridWorld("battle", map_size=size, _lib=checker_lib())
        r.set_seed(20 + a)
        r.reset()
        for h in r.get_handles():
            r.add_agents(h, method="random", n=n)
        refs.append(r)
    rs = np.random.RandomState(9)
    for t in range(steps):
        nums = [env.get_arena_nums(h) for h in hs]
        for g, h in enumerate(hs):
            v, f = env.get_observation(h)
            off = np.concatenate([[0], np.cumsum(nums[g])])
            for a, r in enumerate(refs):
                rv, rf = r.get_observation(r.get_handles()[g])
                assert rv.shape[0] == nums[g][a]
                np.testing.assert_array_equal(v[off[a]:off[a + 1]].view(np.uint32), rv.view(np.uint32), err_msg="view t%d a%d" % (t, a))
                np.testing.assert_array_equal(f[off[a]:off[a + 1]].view(np.uint32), rf.view(np.uint32), err_msg="feat t%d a%d" % (t, a))
        acts = [rs.randint(0, 21, size=int(nums[g].sum())).astype(np.int32) for g in range(2)]
        for g, h in enumerate(hs):
            env.set_action(h, acts[g])
            off = np.concatenate([[0], np.cumsum(nums[g])])
            for a, r in enumerate(refs):
                r.set_action(r.get_handles()[g], np.ascontiguousarray(acts[g][off[a]:off[a + 1]]))
        env.step()
        dones = [r.step() for r in refs]
        np.testing.assert_array_equal(env.get_arena_done() != 0, np.array(dones))
        for g, h in enumerate(hs):
            rew, pos, alive = env.get_reward(h), env.get_pos(h), env.get_alive(h)
            off = np.concatenate([[0], np.cumsum(nums[g])])
            for a, r in enumerate(refs):
                rh = r.get_handles()[g]
                np.testing.assert_allclose(rew[off[a]:off[a + 1]], r.get_reward(rh), atol=pc.REWARD_TOL, rtol=0)
                np.testing.assert_array_equal(pos[off[a]:off[a + 1]], r.get_pos(rh))
                np.testing.assert_array_equal(alive[off[a]:off[a + 1]], r.get_alive(rh))
        env.clear_dead()
        for r in refs:
            r.clear_dead()


def test_huge_arena_grid_mode():
    """> 32768 agents in one arena: the cooperative whole-grid kernels (grid.sync between phases)"""
    both(lambda lib: pc.make_battle(lib, 320, 20000, 1), 6, 1)


def test_device_pointer_observation_matches_host_pointer():
    import torch
    env = pc.make_battle(pc.CUDA_LIB, 40, 150, 0)
    h = env.get_handles()[0]
    v, f = env.get_observation(h)
    tv, tf = env.get_observation_torch(h)
    np.testing.assert_array_equal(tv.cpu().numpy().view(np.uint32), v.view(np.uint32))
    np.testing.assert_array_equal(tf.cpu().numpy().view(np.uint32), f.view(np.uint32))


@pytest.mark.parametrize("which", ["battle", "pursuit", "arrange", "batch"])
def test_f16_observation_is_the_rounded_reference_observation(which):
    """compact hand-off (magent_b200_get_observation_f16): every element == the REFERENCE float32 observation of
    the same state rounded to nearest-even, bit for bit (NaN payloads included); tiles of 8 agents, ragged tails
    and arena-straddling tiles are covered by the 3-arena batch with odd group sizes"""
    import magent_b200 as magent
    if which == "batch":
        A, size = 3, 30
        env = magent.GridWorld("battle", map_size=size, _lib=pc.CUDA_LIB, _num_arenas=A)
        env.set_seed(7)
        env.reset()
        for k, h in enumerate(env.get_handles()):
            env.add_agents(h, method="random", n=37 + 6 * k)
        refs = []
        for a in range(A):
            r = magent.GridWorld("battle", map_size=size, _lib=checker_lib())
            r.set_seed(7 + a)
            r.reset()
            for k, h in enumerate(r.get_handles()):
                r.add_agents(h, method="random", n=37 + 6 * k)
            refs.append(r)
        for g, h in enumerate(env.get_handles()):
            v16, f16 = env.get_observation_f16(h)
            rv = np.concatenate([r.get_observation(r.get_handles()[g])[0] for r in refs])
            rf = np.concatenate([r.get_observation(r.get_handles()[g])[1] for r in refs])
            np.testing.assert_array_equal(v16.view(np.uint16), rv.astype(np.float16).view(np.uint16))
            np.testing.assert_array_equal(f16.view(np.uint16), rf.astype(np.float16).view(np.uint16))
        return
    mk = {"battle": lambda lib: pc.make_battle(lib, 40, 61, seed=3),
          "pursuit": lambda lib: pc.make_pursuit(lib),
          "arrange": lambda lib: pc.make_arrange(lib, 24, 14, n_goal=60, n_agent=150)}[which]
    ref, env = mk(checker_lib()), mk(pc.CUDA_LIB)
    rs = np.random.RandomState(14)
    saw_nan = False
    for _ in range(40 if which == "arrange" else 10):
        for hr, he in zip(ref.get_handles(), env.get_handles()):
            if ref.get_num(hr) == 0:
                continue
            rv, rf = ref.get_observation(hr)
            v16, f16 = env.get_observation_f16(he)
            saw_nan |= bool(np.isnan(rv).any())
            with np.errstate(all="ignore"):
                np.testing.assert_array_equal(v16.view(np.uint16), rv.astype(np.float16).view(np.uint16))
                np.testing.assert_array_equal(f16.view(np.uint16), rf.astype(np.float16).view(np.uint16))
        for hr, he in zip(ref.get_handles(), env.get_handles()):
            act = rs.randint(0, ref.get_action_space(hr)[0], size=ref.get_num(hr)).astype(np.int32)
            ref.set_action(hr, act)
            env.set_action(he, act)
        ref.step(), env.step()
        ref.clear_dead(), env.clear_dead()


def test_f16_device_pointer_observation():
    import torch
    env = pc.make_battle(pc.CUDA_LIB, 40, 150, 0)
    h = env.get_handles()[1]
    v, f = env.get_observation(h)
    tv, tf = env.get_observation_torch(h, dtype=torch.float16)
    assert tv.dtype == torch.float16 and tuple(tv.shape) == v.shape
    np.testing.assert_array_equal(tv.cpu().numpy().view(np.uint16), v.astype(np.float16).view(np.uint16))
    np.testing.assert_array_equal(tf.cpu().numpy().view(np.uint16), f.astype(np.float16).view(np.uint16))


@pytest.mark.parametrize("seed", list(range(0, 36)) + list(range(1000, 1024)))
def test_random_games_match_checker(seed):
    """randomised differential test (tests/fuzz_common.py): random configs (2-4 groups, long bodies, sector ranges,
    turn / food / goal / minimap modes, absorbers, random rule sets incl. two-subject rules), random placements, call
    order and acting subsets -- CUDA engine vs the checker, step by step, bit-exact observations"""
    import fuzz_common as fz
    fz.play(seed, checker_lib(), pc.CUDA_LIB, steps=20)


@pytest.mark.parametrize("seed", list(range(300, 312)) + list(range(1300, 1308)))
def test_random_games_with_an_irregular_caller(seed):
    """fuzz_common.play_irregular: skipped clear_dead, agents added mid-episode (host <-> device round trips of the
    whole state incl. kind / food planes), observations not fetched every step"""
    import fuzz_common as fz
    fz.play_irregular(seed, checker_lib(), pc.CUDA_LIB, steps=20)


@pytest.mark.parametrize("seed", list(range(500, 516)))
def test_random_arena_batches_match_independent_checkers(seed):
    """`_num_arenas` batches of random games vs independent checker environments (tiles straddling arenas, ragged
    tails, empty groups in some arenas)"""
    import fuzz_common as fz
    fz.play_batch(seed, checker_lib(), pc.CUDA_LIB, n_arenas=2 + seed % 5, steps=12)


# ---- host-buffer observations: wire records from the CUDA kernels + host expansion (tests/test_host_expand_cpu.py
# runs the same checks with the emulated producer)
import test_host_expand_cpu as hx  # noqa: E402


@pytest.mark.parametrize("threads", [1, 5])
@pytest.mark.parametrize("game", sorted(hx.MAKERS))
def test_wire_records_from_the_gpu_expand_to_the_reference_bytes(game, threads):
    hx.test_wire_expansion_matches_the_reference(pc.CUDA_LIB, game, threads)


def test_wire_path_many_chunks_many_arenas():
    hx.test_many_chunks_many_arenas(pc.CUDA_LIB)


@pytest.mark.parametrize("shift", [4, 36])
def test_wire_path_into_pageable_unaligned_caller_buffers(shift):
    """plain numpy memory (what the reference's own wrapper hands over), any alignment"""
    hx.test_caller_buffers_of_any_alignment(pc.CUDA_LIB, shift)


def test_wire_and_dense_host_paths_agree_at_scale():
    """64 arenas x 2x1000 agents: every record of both groups through both host paths, bit for bit"""
    import magent_b200 as magent
    envs = []
    for path in ("wire", "dense"):
        env = magent.GridWorld("battle", map_size=200, _lib=pc.CUDA_LIB, _num_arenas=64, _host_path=path)
        env.set_seed(3)
        env.reset()
        for h in env.get_handles():
            env.add_agents(h, method="random", n=1000)
        envs.append(env)
    rs = np.random.RandomState(0)
    for t in range(4):
        acts = [rs.randint(0, 21, size=envs[0].get_num(h)).astype(np.int32) for h in envs[0].get_handles()]
        obs = []
        for env in envs:
            hs = env.get_handles()
            obs.append([tuple(x.copy() for x in env.get_observation(h)) for h in hs])
            for h, a in zip(hs, acts):
                env.set_action(h, a)
            env.step()
            env.clear_dead()
        for (v0, f0), (v1, f1) in zip(obs[0], obs[1]):
            assert np.array_equal(v0.view(np.uint32), v1.view(np.uint32))
            assert np.array_equal(f0.view(np.uint32), f1.view(np.uint32))


def test_device_done_and_deferred_counts():
    """env_step with a device pointer for `done`, clear_dead without waiting: the host's counts catch up when asked"""
    import ctypes
    torch = pytest.importorskip("torch")
    import magent_b200 as magent
    from magent_b200.c_lib import load_library
    L = load_library(pc.CUDA_LIB)
    env = pc.make_battle(pc.CUDA_LIB, 30, 300, 3)
    ref = pc.make_battle(checker_lib(), 30, 300, 3)
    hs, rhs = env.get_handles(), ref.get_handles()
    done_dev = torch.zeros((1,), dtype=torch.int32, device="cuda")
    rs = np.random.RandomState(3)
    for t in range(60):
        acts = [rs.randint(0, 21, size=ref.get_num(h)).astype(np.int32) for h in rhs]
        for e, hh in ((env, hs), (ref, rhs)):
            for h, a in zip(hh, acts):
                if e is env:
                    # device-pointer actions: the host may hold pre-cull (larger) counts at this point
                    ta = torch.from_numpy(a).cuda()
                    L.env_set_action(e.game, e._hv(h), ta.data_ptr())
                else:
                    e.set_action(h, a)
        env.step_device_done(done_dev.data_ptr())
        rdone = ref.step()
        env.clear_dead()
        ref.clear_dead()
        assert bool(done_dev.item()) == rdone
        if t % 7 == 6:                                  # now ask: exact numbers, ids, positions
            for h, rh in zip(hs, rhs):
                assert env.get_num(h) == ref.get_num(rh)
                np.testing.assert_array_equal(env.get_agent_id(h), ref.get_agent_id(rh))
                np.testing.assert_array_equal(env.get_pos(h), ref.get_pos(rh))
    assert ref.get_num(rhs[0]) < 300
    for h, rh in zip(hs, rhs):
        v, f = env.get_observation(h)
        rv, rf = ref.get_observation(rh)
        np.testing.assert_array_equal(v.view(np.uint32), rv.view(np.uint32))
        np.testing.assert_array_equal(f.view(np.uint32), rf.view(np.uint32))


def test_replayed_cuda_graph_of_two_steps_matches_the_reference():
    """magent_b200_graph_*: two whole steps (observations, actions, step, rewards, clear_dead; device buffers only) recorded
    once and replayed; the caller refills its action buffers between replays.  State after every replay == the reference."""
    import ctypes
    torch = pytest.importorskip("torch")
    from magent_b200.c_lib import load_library
    L = load_library(pc.CUDA_LIB)
    env = pc.make_battle(pc.CUDA_LIB, 30, 300, 3)
    ref = pc.make_battle(checker_lib(), 30, 300, 3)
    hs, rhs = env.get_handles(), ref.get_handles()
    dev = "cuda"
    n0 = [env.get_num(h) for h in hs]
    obs = [(torch.empty((n,) + env.get_view_space(h), dtype=torch.float32, device=dev),
            torch.empty((n,) + env.get_feature_space(h), dtype=torch.float32, device=dev)) for h, n in zip(hs, n0)]
    acts = [[torch.zeros((n,), dtype=torch.int32, device=dev) for n in n0] for _ in range(2)]     # even / odd step
    rew = [[torch.zeros((n,), dtype=torch.float32, device=dev) for n in n0] for _ in range(2)]
    done = torch.zeros((2,), dtype=torch.int32, device=dev)

    def one(k):
        for h, (v, f) in zip(hs, obs):
            L.env_get_observation(env.game, env._hv(h), (ctypes.c_void_p * 2)(v.data_ptr(), f.data_ptr()))
        for h, a in zip(hs, acts[k]):
            L.env_set_action(env.game, env._hv(h), a.data_ptr())
        env.step_device_done(done.data_ptr() + 4 * k)
        for h, r in zip(hs, rew[k]):
            L.env_get_reward(env.game, env._hv(h), r.data_ptr())
        env.clear_dead()

    rs = np.random.RandomState(7)

    def draw():
        return [[rs.randint(0, 21, size=n).astype(np.int32) for n in n0] for _ in range(2)]

    a = draw()
    for k in range(2):                                   # one un-captured pair first: every buffer gets its size
        for g in range(2):
            acts[k][g].copy_(torch.from_numpy(a[k][g]))

    def ref_pair(a):
        out = []
        for k in range(2):
            nums = [ref.get_num(h) for h in rhs]
            for h, x, n in zip(rhs, a[k], nums):
                ref.set_action(h, np.ascontiguousarray(x[:n]))
            d = ref.step()
            out.append((d, [ref.get_reward(h).copy() for h in rhs], nums))
            ref.clear_dead()
        return out

    one(0); one(1)
    want = ref_pair(a)
    gid = env.capture_graph(lambda: (one(0), one(1)))
    for rep_i in range(25):
        a = draw()
        for k in range(2):
            for g in range(2):
                acts[k][g].copy_(torch.from_numpy(a[k][g]))
        env.launch_graph(gid, 1)
        want = ref_pair(a)
        torch.cuda.synchronize()
        for k in range(2):
            assert bool(done[k].item()) == want[k][0]
            for g in range(2):
                n = want[k][2][g]
                np.testing.assert_allclose(rew[k][g].cpu().numpy()[:n], want[k][1][g], rtol=0, atol=pc.REWARD_TOL)
        if rep_i % 6 == 5:
            for h, rh in zip(hs, rhs):
                assert env.get_num(h) == ref.get_num(rh)
                np.testing.assert_array_equal(env.get_agent_id(h), ref.get_agent_id(rh))
                np.testing.assert_array_equal(env.get_pos(h), ref.get_pos(rh))
    assert ref.get_num(rhs[0]) < 300                    # agents died and were culled inside the replays
    for h, rh in zip(hs, rhs):
        v, f = env.get_observation(h)
        rv, rf = ref.get_observation(rh)
        np.testing.assert_array_equal(v.view(np.uint32), rv.view(np.uint32))
        np.testing.assert_array_equal(f.view(np.uint32), rf.view(np.uint32))


def test_pinned_divergences_on_the_gpu():
    """set_action twice in a step: the second call wins; out-of-range action ids: ignored (DESIGN.md section 9)"""
    import divergence_common as dv
    dv.second_set_action_wins(pc.CUDA_LIB, checker_lib())
    dv.invalid_actions_are_ignored(pc.CUDA_LIB, checker_lib())


@pytest.mark.parametrize("seed", list(range(40000, 40012)) + [47002, 47170, 70003, 72001, 110000, 113018])
def test_chaotic_caller_with_wire_records_forced(seed, monkeypatch):
    """every host-buffer observation of the chaotic caller through the wire kernels + host expansion, whatever its size"""
    import fuzz_common as fz
    monkeypatch.setenv("MAGENT_B200_HOST_PATH", "wire")
    fz.play_chaotic(seed, checker_lib(), pc.CUDA_LIB)


@pytest.mark.parametrize("seed", [60000, 60003, 60007, 115000])
def test_chaotic_arena_batch_with_wire_records_forced(seed, monkeypatch):
    import fuzz_common as fz
    monkeypatch.setenv("MAGENT_B200_HOST_PATH", "wire")
    fz.play_batch_chaotic(seed, checker_lib(), pc.CUDA_LIB, n_arenas=1 + seed % 4)
