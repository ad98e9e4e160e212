"""bench.py's timed loop (device-drawn actions, `done` to a device int, a replayed CUDA graph of two steps) step for step
against the checker, and the step / observation / reduction kernels at the sizes where they switch code paths.

The actions of the device loop are never seen by the host.  They are read back from the engine itself: after a step and
before clear_dead, every agent's feature row shows that step's action as a one-hot (GridWorld.h:182), dead agents
included.  Each row must hold exactly one 1 in its action slice (which also proves the draw was in [0, n_action)); its
argmax is handed to an independent checker environment, and everything the step produced is compared with what the
checker computed from those actions.
"""
import ctypes
import os

import numpy as np
import pytest

import fullsize_common as fs
import parity_common as pc

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1200)]      # (pytest-timeout: a stuck test fails instead of hanging the suite)

ENGINE = os.environ.get("MAGENT_FULLSIZE_ENGINE", pc.CUDA_LIB)      # (tests/_emu library for a dry run on the CPU)
ON_GPU = ENGINE == pc.CUDA_LIB
ARENAS = int(os.environ.get("MAGENT_FULLSIZE_SOAK_ARENAS", "512"))   # (smaller for a dry run on the CPU)
GRID_MODE_THRESHOLD = 32768          # agents per arena above which one step runs as the cooperative grid kernel
CNT_AGENT_STEPS, CNT_KILLS, CNT_STARVED, CNT_STEPS = 0, 3, 4, 7


def checker_lib():
    for p in (pc.REF_LIB, pc.PORT_LIB):
        if os.path.exists(p):
            return p
    pytest.skip("no oracle library available (oracle/_ref or oracle/_build)")


def device():
    import torch
    return torch.device("cuda") if ON_GPU else torch.device("cpu")     # (CPU tensors in the dry run: host pointers)


def empty(shape, dtype):
    import torch
    return torch.empty(shape, dtype=dtype, device=device())


def observe(env, h, dtype=None):
    """(view, feature) torch tensors on the device (host tensors in the dry run)"""
    import torch
    if ON_GPU:
        return env.get_observation_torch(h, dtype=dtype)
    v, f = env.get_observation_f16(h) if dtype == torch.float16 else env.get_observation(h)
    return torch.from_numpy(v.copy()), torch.from_numpy(f.copy())


def actions_from_features(feat, n_action, what):
    """the action of every row of a feature block read between step and clear_dead (numpy int32)"""
    emb = feat.shape[1] - n_action - 3
    hot = feat[:, emb:emb + n_action]
    assert bool(((hot == 0) | (hot == 1)).all()), "%s: action slots hold something else than 0 / 1" % what
    assert bool((hot.sum(dim=1) == 1).all()), "%s: action slots are not a one-hot (or the action is out of range)" % what
    return hot.argmax(dim=1).cpu().numpy().astype(np.int32)


def offsets(nums):
    return np.concatenate([[0], np.cumsum(nums)]).astype(np.int64)


def assert_f16_is_rounded_f32(v16, v32, what, chunk=1 << 16):
    """f16 observation == numpy's astype(float16) of the f32 one, bit for bit (NaN payloads included; torch's CUDA cast
    would canonicalise them)"""
    assert v16.shape == v32.shape
    for s in range(0, v32.shape[0], chunk):
        want = v32[s:s + chunk].cpu().numpy().astype(np.float16).view(np.uint16)
        got = v16[s:s + chunk].cpu().numpy().view(np.uint16)
        if not np.array_equal(got, want):
            bad = np.argwhere(got != want)[0]
            raise AssertionError("%s: f16 differs from the rounded f32 observation at record %d, %s: %#06x vs %#06x" % (
                what, s + bad[0], tuple(bad[1:]), got[tuple(bad)], want[tuple(bad)]))


# ---------------------------------------------------------------------------------------------- 1. the timed loop
def play_device_loop(workload, seed0, steps, obs_every=10):
    """bench.dev_step without the graph at the workload's own size: observation into device buffers,
    set_random_actions, step_device_done, device rewards, clear_dead.  Arenas 0, A/2-1 and A-1 against independent
    checkers at every step; the whole batch through fs.check_state and the PyTorch restatement every `obs_every` steps,
    where the f16 observation is also checked against the f32 one rounded by numpy.  Returns the recovered actions of
    the first step (all groups) for the draw-distribution check."""
    import torch
    import bench
    wl = bench.WORKLOADS[workload]
    env, hs = bench.build_env(wl, ENGINE, ARENAS, seed0=seed0)
    L = env._lib
    A, size = ARENAS, wl["map_size"]
    samples = sorted({0, A // 2 - 1, A - 1})
    refs = {a: bench.build_env(wl, checker_lib(), 1, seed0=seed0 + a)[0] for a in samples}
    G = len(hs)
    n_action = env.get_action_space(hs[0])[0]
    done_dev = torch.full((1,), -1, dtype=torch.int32, device=device())
    nums = [env.get_arena_nums(h).astype(np.int64) for h in hs]
    last_action = [np.full(int(n.sum()), n_action, dtype=np.int64) for n in nums]
    last_reward = [np.zeros(int(n.sum()), dtype=np.float32) for n in nums]
    c0 = env.get_counters()
    agent_steps = deaths = 0
    prev = None
    first_actions = None
    for t in range(steps):
        off = [offsets(n) for n in nums]
        pos = [env.get_pos(h).copy() for h in hs]
        ids = [env.get_agent_id(h).copy() for h in hs]
        fs.check_state(pos, ids, nums, size, size, prev=prev, speed=2)
        for a, r in refs.items():
            for g, rh in enumerate(r.get_handles()):
                sl = slice(int(off[g][a]), int(off[g][a + 1]))
                np.testing.assert_array_equal(pos[g][sl], r.get_pos(rh), err_msg="pos t%d arena %d g%d" % (t, a, g))
                np.testing.assert_array_equal(ids[g][sl], r.get_agent_id(rh), err_msg="id t%d arena %d g%d" % (t, a, g))
        if t % obs_every == 0 or t == steps - 1:
            obs = [observe(env, h) for h in hs]
            views, feats = [o[0] for o in obs], [o[1] for o in obs]
            fs.check_battle_observation(views, feats, pos, ids, nums, last_action, last_reward, size, size)
            for a, r in refs.items():
                for g, rh in enumerate(r.get_handles()):
                    rv, rf = r.get_observation(rh)
                    sl = slice(int(off[g][a]), int(off[g][a + 1]))
                    np.testing.assert_array_equal(views[g][sl].cpu().numpy().view(np.uint32), rv.view(np.uint32))
                    np.testing.assert_array_equal(feats[g][sl].cpu().numpy().view(np.uint32), rf.view(np.uint32))
            if t % obs_every == 0:
                for g, h in enumerate(hs):
                    v16, f16 = observe(env, h, torch.float16)
                    assert_f16_is_rounded_f32(v16, views[g], "view t%d g%d" % (t, g))
                    assert_f16_is_rounded_f32(f16, feats[g], "feature t%d g%d" % (t, g))
                    del v16, f16
            del obs, views, feats
        for h in hs:
            env.set_random_actions(h, seed0 * 1000 + t)
        agent_steps += int(sum(n.sum() for n in nums))
        done_dev.fill_(-1)
        env.step_device_done(done_dev.data_ptr())
        acts = [actions_from_features(observe(env, h)[1], n_action, "t%d g%d" % (t, g)) for g, h in enumerate(hs)]
        if first_actions is None:
            first_actions = np.concatenate(acts)
        rew = []
        for g, h in enumerate(hs):
            d_rew = torch.full((int(nums[g].sum()),), -7.0, dtype=torch.float32, device=device())
            L.env_get_reward(env.game, env._hv(h), ctypes.c_void_p(d_rew.data_ptr()))
            rew.append(d_rew.cpu().numpy())
        alive = [env.get_alive(h).astype(bool) for h in hs]
        pos_after = [env.get_pos(h).copy() for h in hs]
        done = env.get_arena_done()
        done_word = int(done_dev.item())
        for a, r in refs.items():
            for g, rh in enumerate(r.get_handles()):
                r.set_action(rh, np.ascontiguousarray(acts[g][off[g][a]:off[g][a + 1]]))
            d = bool(r.step())
            assert bool(done[a]) == d, "done flag of arena %d at t%d" % (a, t)
            if not d:
                assert done_word == 0, "device done word %d with arena %d not done" % (done_word, a)
            for g, rh in enumerate(r.get_handles()):
                sl = slice(int(off[g][a]), int(off[g][a + 1]))
                np.testing.assert_allclose(rew[g][sl], r.get_reward(rh), atol=pc.REWARD_TOL, rtol=0,
                                           err_msg="reward t%d arena %d g%d" % (t, a, g))
                np.testing.assert_array_equal(alive[g][sl], r.get_alive(rh).astype(bool))
                np.testing.assert_array_equal(pos_after[g][sl], r.get_pos(rh))
            r.clear_dead()
        assert done_word in (0, 1)
        env.clear_dead()
        new_nums = [env.get_arena_nums(h).astype(np.int64) for h in hs]
        for g in range(G):
            ar = np.repeat(np.arange(A), nums[g])
            np.testing.assert_array_equal(np.bincount(ar[alive[g]], minlength=A), new_nums[g],
                                          err_msg="clear_dead kept a different number of agents than were alive")
            deaths += int((~alive[g]).sum())
        prev = (ids, pos, nums)
        last_action = [acts[g][alive[g]].astype(np.int64) for g in range(G)]
        last_reward = [rew[g][alive[g]] for g in range(G)]
        nums = new_nums
    c1 = env.get_counters()
    d = [y - x for x, y in zip(c0, c1)]
    assert d[CNT_AGENT_STEPS] == agent_steps, "agent_steps counter %d, agents acting %d" % (d[CNT_AGENT_STEPS], agent_steps)
    assert d[CNT_STEPS] == steps, "steps counter %d" % d[CNT_STEPS]
    assert d[CNT_KILLS] + d[CNT_STARVED] == deaths, "kills %d + starved %d != deaths %d" % (d[CNT_KILLS], d[CNT_STARVED], deaths)
    return first_actions, n_action


@pytest.mark.parametrize("workload", ["battle512", "battle512_blocks"])
def test_device_action_loop_against_the_checker(workload):
    """30 steps of bench.py's loop without the graph: sampled arenas step for step against checkers, the whole batch
    against the restatement, the event counters against the host's counts, and the first step's draw (1.024 M actions
    at 512 arenas of 2x1000) against the uniform distribution"""
    from scipy.stats import chisquare
    acts, n_action = play_device_loop(workload, 91, 30)
    if workload == "battle512" and ON_GPU:
        cnt = np.bincount(acts, minlength=n_action)
        assert cnt.size == n_action and acts.size == 2 * 1000 * ARENAS
        p = chisquare(cnt).pvalue            # the draws are deterministic: this is a fixed number, not a flaky one
        assert p > 1e-6, "device-drawn actions are not uniform: chi2 p = %g, counts %s" % (p, cnt.tolist())


def test_two_engines_draw_the_same_actions():
    """set_random_actions depends on the seed, the call count and the device step counter only"""
    if not ON_GPU:
        pytest.skip("the dry run's emulation draws its own stream")
    import torch
    got = []
    for _ in range(2):
        env = pc.make_battle(ENGINE, 40, 150, 3, _num_arenas=4)
        done = torch.zeros((1,), dtype=torch.int32, device="cuda")
        acts = []
        for t in range(3):
            for h in env.get_handles():
                env.set_random_actions(h, 17)
            env.step_device_done(done.data_ptr())
            acts.append(np.concatenate([actions_from_features(env.get_observation_torch(h)[1], 21, "t%d" % t)
                                        for h in env.get_handles()]))
            env.clear_dead()
        got.append(np.concatenate(acts))
    np.testing.assert_array_equal(got[0], got[1])


def test_graph_replays_against_the_checker():
    """bench.py's graph: two device steps captured once and replayed; after every replay the actions of both steps are
    read back, replayed on one checker per arena, and rewards, per-step done words and (every few replays) the state
    compared.  The counters follow the replays, and a step slot draws fresh actions in every replay (the seed rides on
    the device step counter): an agent keeps its action from one replay to the next with probability 1/21."""
    if not ON_GPU:
        pytest.skip("CUDA graphs need the CUDA engine")
    import torch
    import bench
    wl = dict(game="battle", map_size=40, n=300)
    A, seed0, replays = 8, 500, 24
    env, hs = bench.build_env(wl, ENGINE, A, seed0=seed0)
    refs = [bench.build_env(wl, checker_lib(), 1, seed0=seed0 + a)[0] for a in range(A)]
    L = env._lib
    n_action = env.get_action_space(hs[0])[0]
    n0 = [env.get_num(h) for h in hs]
    spaces = [(env.get_view_space(h), env.get_feature_space(h)) for h in hs]
    mk = lambda g: (torch.empty((n0[g],) + spaces[g][0], device="cuda"), torch.empty((n0[g],) + spaces[g][1], device="cuda"))
    obs_in = [mk(g) for g in range(len(hs))]                       # what bench observes before each step
    obs_after = [[mk(g) for g in range(len(hs))] for _ in range(2)]  # per step slot: read after the step, before clear_dead
    rew = [[torch.empty((n0[g],), device="cuda") for g in range(len(hs))] for _ in range(2)]
    done = [torch.full((1,), -1, dtype=torch.int32, device="cuda") for _ in range(2)]

    def dev_step(k):
        for g, h in enumerate(hs):
            L.env_get_observation(env.game, env._hv(h), (ctypes.c_void_p * 2)(obs_in[g][0].data_ptr(), obs_in[g][1].data_ptr()))
        for h in hs:
            env.set_random_actions(h, k)
        env.step_device_done(done[k].data_ptr())
        for g, h in enumerate(hs):
            v, f = obs_after[k][g]
            L.env_get_observation(env.game, env._hv(h), (ctypes.c_void_p * 2)(v.data_ptr(), f.data_ptr()))
            L.env_get_reward(env.game, env._hv(h), ctypes.c_void_p(rew[k][g].data_ptr()))
        env.clear_dead()

    tally = {"agent_steps": 0, "deaths": 0, "steps": 0}

    def check_step(k, what):
        """replay step slot k on the checkers and compare; returns {(arena, group, id): action}"""
        drawn, got_rew = {}, []
        for g in range(len(hs)):
            nums = np.array([r.get_num(r.get_handles()[g]) for r in refs], dtype=np.int64)
            n = int(nums.sum())
            acts = actions_from_features(obs_after[k][g][1][:n], n_action, "%s g%d" % (what, g))
            off = offsets(nums)
            got_rew.append([rew[k][g][:n].cpu().numpy()[off[a]:off[a + 1]] for a in range(A)])
            for a, r in enumerate(refs):
                rh = r.get_handles()[g]
                a_act = np.ascontiguousarray(acts[off[a]:off[a + 1]])
                r.set_action(rh, a_act)
                drawn.update(((a, g, int(i)), int(x)) for i, x in zip(r.get_agent_id(rh), a_act))
            tally["agent_steps"] += n
        flags = [bool(r.step()) for r in refs]
        assert int(done[k].item()) == int(all(flags)), "%s: device done word %d, checkers %s" % (what, int(done[k].item()), flags)
        for g in range(len(hs)):
            for a, r in enumerate(refs):
                rh = r.get_handles()[g]
                np.testing.assert_allclose(got_rew[g][a], r.get_reward(rh), atol=pc.REWARD_TOL, rtol=0,
                                           err_msg="%s reward arena %d g%d" % (what, a, g))
                tally["deaths"] += int((~r.get_alive(rh).astype(bool)).sum())
        for r in refs:
            r.clear_dead()
        tally["steps"] += 1
        return drawn

    def check_state(what):
        for g, h in enumerate(hs):
            np.testing.assert_array_equal(env.get_pos(h), np.concatenate([r.get_pos(r.get_handles()[g]) for r in refs]),
                                          err_msg=what + " pos g%d" % g)
            np.testing.assert_array_equal(env.get_agent_id(h), np.concatenate([r.get_agent_id(r.get_handles()[g]) for r in refs]),
                                          err_msg=what + " id g%d" % g)

    c0 = env.get_counters()
    for k in range(2):                          # un-captured first: the same calls, read right away
        dev_step(k)
        torch.cuda.synchronize()
        check_step(k, "plain step %d" % k)
    check_state("before capture")
    gid = env.capture_graph(lambda: (dev_step(0), dev_step(1)))
    same = total = 0
    prev_slot0 = None
    for rep in range(replays):
        env.launch_graph(gid, 1)
        torch.cuda.synchronize()
        slot0 = check_step(0, "replay %d step 0" % rep)
        check_step(1, "replay %d step 1" % rep)
        if prev_slot0 is not None:
            common = prev_slot0.keys() & slot0.keys()
            same += sum(prev_slot0[key] == slot0[key] for key in common)
            total += len(common)
        prev_slot0 = slot0
        if rep % 5 == 4 or rep == replays - 1:
            check_state("after replay %d" % rep)
    c1 = env.get_counters()
    d = [y - x for x, y in zip(c0, c1)]
    assert d[CNT_AGENT_STEPS] == tally["agent_steps"], "agent_steps counter %d, agents acting %d" % (d[CNT_AGENT_STEPS], tally["agent_steps"])
    assert d[CNT_STEPS] == tally["steps"] == 2 + 2 * replays
    assert d[CNT_KILLS] + d[CNT_STARVED] == tally["deaths"]
    assert total > 10000
    share = same / total
    assert abs(share - 1.0 / n_action) < 0.015, "%d of %d agents drew the same action in consecutive replays" % (same, total)


def test_counters_in_grid_mode():
    """2 arenas of 2x20000 agents (each stepped by the cooperative grid kernel), host actions: the event counters
    against the host's counts"""
    env = pc.make_battle(ENGINE, 320, 20000, 61, _num_arenas=2)
    hs = env.get_handles()
    rs = np.random.RandomState(4)
    c0 = env.get_counters()
    agent_steps = deaths = 0
    steps = 4
    for _ in range(steps):
        assert (env.get_arena_nums(hs[0]) + env.get_arena_nums(hs[1]) > GRID_MODE_THRESHOLD).all()
        for h in hs:
            n = env.get_num(h)
            env.set_action(h, rs.randint(0, 21, size=n).astype(np.int32))
            agent_steps += n
        env.step()
        deaths += sum(int((~env.get_alive(h).astype(bool)).sum()) for h in hs)
        env.clear_dead()
    d = [y - x for x, y in zip(c0, env.get_counters())]
    assert d[CNT_AGENT_STEPS] == agent_steps and d[CNT_STEPS] == steps
    assert d[CNT_KILLS] + d[CNT_STARVED] == deaths


# ---------------------------------------------------------------------------------------------- 2. arena counts
def tiny_arenas(lib, A, live, seed, batch):
    """A 12x12 battle arenas with 0-6 agents per group, set up per arena; `live[a]` False gives arena a an empty group
    (done from the first step, minimap 0/0 = NaN).  batch=True: one engine behind select_arena, else A checkers."""
    import magent_b200 as magent
    rs = np.random.RandomState(seed)
    cells = np.array([(x, y) for x in range(1, 11) for y in range(1, 11)], dtype=np.int32)
    if batch:
        env = magent.GridWorld("battle", map_size=12, _lib=lib, _num_arenas=A)
        env.reset()
        out = env
    else:
        out = []
    for a in range(A):
        ns = [int(rs.randint(1, 7)), int(rs.randint(1, 7))]
        if not live[a]:
            ns[int(rs.randint(0, 2))] = 0
        pick = cells[rs.choice(len(cells), sum(ns), replace=False)]
        pos = [pick[:ns[0]], pick[ns[0]:]]
        if batch:
            env.select_arena(a)
            env.set_seed(seed + a)
        else:
            env = magent.GridWorld("battle", map_size=12, _lib=lib)
            env.set_seed(seed + a)
            env.reset()
            out.append(env)
        for g, h in enumerate(env.get_handles()):
            if ns[g]:
                env.add_agents(h, method="custom", pos=pos[g].tolist())
    if batch:
        env.select_arena(-1)
    return out


def checker_observation(r, h):
    """the reference cannot observe an empty group: zero records of the right shape"""
    if r.get_num(h) == 0:
        return (np.zeros((0,) + r.get_view_space(h), np.float32), np.zeros((0,) + r.get_feature_space(h), np.float32))
    v, f = r.get_observation(h)
    return v.copy(), f.copy()


ARENA_CASES =[(257, o, True) for o in (0, 255, 256)] + [(257, 100, False)] + \
              [(1025, o, True) for o in (0, 255, 256, 1023, 1024)] + [(1025, 1024, False)] + \
              [(4096, 1024, True), (4096, 255, False)]


@pytest.mark.parametrize("A,odd,odd_live", ARENA_CASES)
def test_arena_count_boundaries(A, odd, odd_live):
    """every arena against its own checker: observations f32 and f16, positions, ids, rewards, per-arena done flags,
    env.step()'s value and the device done word.  The one arena that differs (the only live one, or the only done one)
    sits on either side of the 256-arena stride of the done reduction and the 1024-arena tile of the offset scan;
    4096 arenas is one GPU's share of the strong-scaling configuration (more arenas than resident step CTAs)."""
    import torch
    live = [(a == odd) == odd_live for a in range(A)]
    seed = 7 * A + odd
    env = tiny_arenas(ENGINE, A, live, seed, batch=True)
    refs = tiny_arenas(checker_lib(), A, live, seed, batch=False)
    hs = env.get_handles()
    rs = np.random.RandomState(seed)
    done_dev = torch.full((1,), -1, dtype=torch.int32, device=device())
    for t in range(8):
        nums = [env.get_arena_nums(h).astype(np.int64) for h in hs]
        for g, h in enumerate(hs):
            rh = [r.get_handles()[g] for r in refs]
            np.testing.assert_array_equal(nums[g], [r.get_num(x) for r, x in zip(refs, rh)], err_msg="t%d nums g%d" % (t, g))
            obs = [checker_observation(r, x) for r, x in zip(refs, rh)]
            rv, rf = np.concatenate([o[0] for o in obs]), np.concatenate([o[1] for o in obs])
            del obs
            v, f = observe(env, h)
            np.testing.assert_array_equal(v.cpu().numpy().view(np.uint32), rv.view(np.uint32), err_msg="t%d view g%d" % (t, g))
            np.testing.assert_array_equal(f.cpu().numpy().view(np.uint32), rf.view(np.uint32), err_msg="t%d feature g%d" % (t, g))
            v, f = observe(env, h, torch.float16)
            np.testing.assert_array_equal(v.cpu().numpy().view(np.uint16), rv.astype(np.float16).view(np.uint16),
                                          err_msg="t%d f16 view g%d" % (t, g))
            np.testing.assert_array_equal(f.cpu().numpy().view(np.uint16), rf.astype(np.float16).view(np.uint16),
                                          err_msg="t%d f16 feature g%d" % (t, g))
            np.testing.assert_array_equal(env.get_pos(h), np.concatenate([r.get_pos(x) for r, x in zip(refs, rh)]))
            np.testing.assert_array_equal(env.get_agent_id(h), np.concatenate([r.get_agent_id(x) for r, x in zip(refs, rh)]))
            act = rs.randint(0, 21, size=int(nums[g].sum())).astype(np.int32)
            env.set_action(h, act)
            off = offsets(nums[g])
            for a, (r, x) in enumerate(zip(refs, rh)):
                r.set_action(x, np.ascontiguousarray(act[off[a]:off[a + 1]]))
        flags = np.array([bool(r.step()) for r in refs])
        if t % 2 == 0:
            assert env.step() == bool(flags.all()), "t%d: env.step()" % t
        else:
            done_dev.fill_(-1)
            env.step_device_done(done_dev.data_ptr())
            assert int(done_dev.item()) == int(flags.all()), "t%d: device done word" % t
        np.testing.assert_array_equal(env.get_arena_done() != 0, flags, err_msg="t%d arena done" % t)
        if t == 0:
            assert flags.sum() == (A - 1 if odd_live else 1) and flags[odd] != odd_live, "arena %d is not the odd one out" % odd
        for g, h in enumerate(hs):
            rh = [r.get_handles()[g] for r in refs]
            np.testing.assert_allclose(env.get_reward(h), np.concatenate([r.get_reward(x) for r, x in zip(refs, rh)]),
                                       atol=pc.REWARD_TOL, rtol=0, err_msg="t%d reward g%d" % (t, g))
            np.testing.assert_array_equal(env.get_alive(h), np.concatenate([r.get_alive(x) for r, x in zip(refs, rh)]))
            np.testing.assert_array_equal(env.get_pos(h), np.concatenate([r.get_pos(x) for r, x in zip(refs, rh)]))
        env.clear_dead()
        for r in refs:
            r.clear_dead()


# ---------------------------------------------------------------------------------------------- 3. size boundaries
def circle_cells(radius):
    """in-range cells of CircleRange(radius) (Range.h: distance from the centre < radius + 1e-8)"""
    r = int(np.floor(radius))
    d = np.arange(-r, r + 1)
    return int((np.sqrt(d[:, None] ** 2 + d[None, :] ** 2) < radius + 1e-8).sum())


class DeviceObservations:
    """an engine whose get_observation goes through device buffers (f32, or f16 as raw bits)"""

    def __init__(self, env, half=False):
        self.env, self.half = env, half

    def __getattr__(self, name):
        return getattr(self.env, name)

    def get_observation(self, h):
        import torch
        v, f = self.env.get_observation_torch(h, dtype=torch.float16 if self.half else torch.float32)
        v, f = v.cpu().numpy(), f.cpu().numpy()
        return (v.view(np.uint16), f.view(np.uint16)) if self.half else (v, f)


class RoundedObservations:
    """a checker whose observations are rounded to f16 by numpy (raw bits)"""

    def __init__(self, env):
        self.env = env

    def __getattr__(self, name):
        return getattr(self.env, name)

    def get_observation(self, h):
        v, f = self.env.get_observation(h)
        return v.astype(np.float16).view(np.uint16), f.astype(np.float16).view(np.uint16)


def test_step_kernel_switches_from_grid_to_cta_mid_episode():
    """one arena of 2x16500 agents on 200x200: the cooperative grid kernel steps it until the culls bring it to at most
    32768 agents, then the CTA kernel; every step against the checker, several steps past the crossing"""
    want = pc.run_trace(pc.make_battle(checker_lib(), 200, 16500, 11), 14, 5)
    got = pc.run_trace(pc.make_battle(ENGINE, 200, 16500, 11), 14, 5)
    pc.compare_traces(want, got)
    total = [sum(rec["num"]) for rec in got]
    assert total[0] > GRID_MODE_THRESHOLD
    cross = next(t for t, n in enumerate(total) if n <= GRID_MODE_THRESHOLD)
    assert cross <= len(total) - 4, "only %d steps after the crossing" % (len(total) - cross)


@pytest.mark.parametrize("n", [8192, 8193])
def test_minimap_kernel_choice_at_8192_agents(n):
    """a group of 8192 agents (capacity 8192: the shared-memory minimap kernel) and of 8193 (capacity 8256: the chunked
    histogram + normalisation kernels)"""
    def make(lib):
        import magent_b200 as magent
        env = magent.GridWorld("battle", map_size=110, _lib=lib)
        env.set_seed(n)
        env.reset()
        h = env.get_handles()
        env.add_agents(h[0], method="random", n=n)
        env.add_agents(h[1], method="random", n=300)
        return env
    want = pc.run_trace(make(checker_lib()), 4, 1, keep_obs=True)
    got = pc.run_trace(make(ENGINE), 4, 1, keep_obs=True)
    pc.compare_traces(want, got)


def view_config(size, radius, turn):
    import magent_b200 as magent
    gw = magent.gridworld
    cfg = gw.Config()
    cfg.set({"map_width": size, "map_height": size, "minimap_mode": True, "turn_mode": turn, "embedding_size": 10})
    t = cfg.register_agent_type("scout", dict(
        width=1, length=1, hp=5, speed=2, damage=2, step_recover=0.1, view_range=gw.CircleRange(radius),
        attack_range=gw.CircleRange(1.5), step_reward=-0.01, kill_reward=1, dead_penalty=-0.5, attack_penalty=-0.02))
    g0, g1 = cfg.add_group(t), cfg.add_group(t)
    a, b = gw.AgentSymbol(g0, "any"), gw.AgentSymbol(g1, "any")
    cfg.add_reward_rule(gw.Event(a, "attack", b), receiver=a, value=0.2)
    return cfg


@pytest.mark.parametrize("radius,cells", [(6.2, 121), (6.4, 129), (9, 253), (9.1, 261)])
@pytest.mark.parametrize("turn", [False, True])
@pytest.mark.parametrize("half", [False, True])
def test_view_sizes_around_the_render_paths(radius, cells, turn, half):
    """in-range view cells just below / above 128 (4 or 8 cells per lane in registers) and 256 (beyond: the tail loop
    and its own undo); groups of 37 and 13 observers leave ragged 4- and 8-agent tiles"""
    if not ON_GPU:
        pytest.skip("device buffers")
    assert circle_cells(radius) == cells
    assert (cells <= 128) == (radius < 6.3) and (cells <= 256) == (radius < 9.05)

    def make(lib):
        import magent_b200 as magent
        env = magent.GridWorld(view_config(30, radius, turn), _lib=lib)
        env.set_seed(int(radius * 10))
        env.reset()
        h = env.get_handles()
        env.add_agents(h[0], method="random", n=37)
        env.add_agents(h[1], method="random", n=13)
        return env
    engine = make(ENGINE)
    r = int(np.floor(radius))
    assert engine.get_view_space(engine.get_handles()[0])[:2] == (2 * r + 1, 2 * r + 1)
    checker = make(checker_lib())
    want = pc.run_trace(RoundedObservations(checker) if half else checker, 10, 2, keep_obs=not half)
    got = pc.run_trace(DeviceObservations(engine, half), 10, 2, keep_obs=not half)
    pc.compare_traces(want, got)


@pytest.mark.parametrize("path", ["device", "dense", "wire"])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 8, 9, 255, 256, 257, 1023, 1024, 1025])
def test_group_sizes_around_tiles_and_chunks(n, path):
    """render tiles of 4 (f32) agents, header CTAs of 256 observers, wire chunks of 1024 observers: group sizes on both
    sides of each, through device buffers and both host paths"""
    if path == "device" and not ON_GPU:
        pytest.skip("device buffers")
    size = max(16, int(np.sqrt(6 * n)) + 2)
    kw = {} if path == "device" else {"_host_path": path}
    want = pc.run_trace(pc.make_battle(checker_lib(), size, n, n), 4, n, keep_obs=True)
    env = pc.make_battle(ENGINE, size, n, n, **kw)
    got = pc.run_trace(DeviceObservations(env) if path == "device" else env, 4, n, keep_obs=True)
    pc.compare_traces(want, got)


# ---------------------------------------------------------------------------------------------- 4. unaligned buffers
SENTINEL32 = np.uint32(0x7FBADBAD)           # a NaN nobody writes
SENTINEL16 = np.uint16(0x7DAD)


def test_unaligned_observation_destinations():
    """get_observation_torch(out=...) into views that start 4, 8 or 12 bytes (f32) / 2 to 14 bytes (f16) into a larger
    tensor: bit-equal to the aligned call, nothing written outside"""
    import torch
    env = pc.make_battle(ENGINE, 36, 123, 14)
    ref = pc.make_battle(checker_lib(), 36, 123, 14)
    rs = np.random.RandomState(9)
    for t in range(3):
        for g, h in enumerate(env.get_handles()):
            rh = ref.get_handles()[g]
            n = env.get_num(h)
            vs, fsp = env.get_view_space(h), env.get_feature_space(h)
            rv, rf = ref.get_observation(rh)
            for dtype, shifts, sentinel, idt in ((torch.float32, (0, 1, 2, 3), SENTINEL32, torch.int32),
                                                 (torch.float16, range(8), SENTINEL16, torch.int16)):
                wv = rv.astype(np.float16) if dtype == torch.float16 else rv
                wf = rf.astype(np.float16) if dtype == torch.float16 else rf
                bits = np.uint16 if dtype == torch.float16 else np.uint32
                for s in shifts:
                    out = []
                    for shape in (vs, fsp):
                        k = n * int(np.prod(shape))
                        big = torch.full((k + 16,), int(sentinel), dtype=idt, device=device()).view(dtype)
                        out.append((big, big[s:s + k].view((n,) + shape)))
                    env.get_observation_torch(h, out=(out[0][1], out[1][1]))
                    env.sync()
                    what = "t%d g%d %s +%d elements" % (t, g, dtype, s)
                    np.testing.assert_array_equal(out[0][1].cpu().numpy().view(bits), wv.view(bits), err_msg=what + " view")
                    np.testing.assert_array_equal(out[1][1].cpu().numpy().view(bits), wf.view(bits), err_msg=what + " feature")
                    for big, part in out:
                        raw = big.cpu().numpy().view(bits)
                        k = part.numel()
                        assert (raw[:s] == sentinel).all() and (raw[s + k:] == sentinel).all(), what + ": wrote outside its buffer"
            act = rs.randint(0, 21, size=n).astype(np.int32)
            env.set_action(h, act)
            ref.set_action(rh, act)
        env.step()
        ref.step()
        check_unaligned_info(env, ref, "after step %d" % t)
        env.clear_dead()
        ref.clear_dead()


def check_unaligned_info(env, ref, what):
    """reward / id / alive / pos into device buffers at odd element offsets (pos at 4 mod 8 bytes: int[n][2] need not be
    8-byte aligned)"""
    import torch
    L = env._lib
    for g, h in enumerate(env.get_handles()):
        rh = ref.get_handles()[g]
        n = env.get_num(h)
        want = {"reward": ref.get_reward(rh).view(np.uint32), "id": ref.get_agent_id(rh).view(np.uint32),
                "alive": ref.get_alive(rh).astype(np.uint8), "pos": ref.get_pos(rh).reshape(-1).view(np.uint32)}
        for name, shifts in (("reward", (1, 3)), ("id", (1, 3)), ("alive", (1, 3, 5, 7)), ("pos", (1, 3))):
            for s in shifts:
                if name == "alive":
                    big = torch.full((n + 16,), 0xA5, dtype=torch.uint8, device=device())
                    k, sentinel, view = n, 0xA5, np.uint8
                else:
                    k = 2 * n if name == "pos" else n
                    big = torch.full((k + 16,), int(SENTINEL32), dtype=torch.int32, device=device())
                    sentinel, view = SENTINEL32, np.uint32
                ptr = ctypes.c_void_p(big[s:s + k].data_ptr())
                if name == "reward":
                    L.env_get_reward(env.game, env._hv(h), ptr)
                else:
                    L.env_get_info(env.game, env._hv(h), name.encode(), ptr)
                env.sync()
                raw = big.cpu().numpy().view(view)
                tag = "%s %s g%d +%d elements" % (what, name, g, s)
                if name == "alive":
                    np.testing.assert_array_equal(raw[s:s + k] != 0, want[name] != 0, err_msg=tag)
                else:
                    np.testing.assert_array_equal(raw[s:s + k], want[name], err_msg=tag)
                assert (raw[:s] == sentinel).all() and (raw[s + k:] == sentinel).all(), tag + ": wrote outside its buffer"


# ---------------------------------------------------------------------------------------------- 5. f16 at full size
def test_f16_observation_of_one_arena_of_2x400k():
    """the f16 hand-off of the 2x400k arena (whole-grid kernels) against numpy's rounding of the f32 observation,
    before and after a device-drawn step"""
    import torch
    env = pc.make_battle(ENGINE, 1000, 400000, 3)
    for t in range(2):
        for g, h in enumerate(env.get_handles()):
            v32, f32 = observe(env, h)
            v16, f16 = observe(env, h, torch.float16)
            assert_f16_is_rounded_f32(v16, v32, "view t%d g%d" % (t, g))
            assert_f16_is_rounded_f32(f16, f32, "feature t%d g%d" % (t, g))
            del v32, f32, v16, f16
        for h in env.get_handles():
            env.set_random_actions(h, 5 + t)
        env.step()
        env.clear_dead()
