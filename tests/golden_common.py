"""Golden fixtures: traces recorded from the UNMODIFIED compiled reference (oracle/_ref, built from
/root/reference by oracle/Makefile) with tests/golden/make_golden.py, committed as small .npz files so the
parity suite has pinned vectors even where neither /root/reference nor oracle/_ref exists."""
import hashlib
import os

import numpy as np

import parity_common as pc

GOLDEN_DIR = os.path.join(pc.REPO, "tests", "golden")

# name -> (factory(lib) -> env, steps, seed, run_trace kwargs)
SCENARIOS = {
    "battle_small": (lambda lib: pc.make_battle(lib, 40, 150, 0), 40, 0, {}),
    "battle_blocks": (lambda lib: pc.make_battle_blocks(lib, 40), 40, 5, {}),
    "battle_kills": (lambda lib: pc.make_battle(lib, 30, 300, 3), 60, 3, {}),
    "battle_bands": (lambda lib: pc.make_battle(lib, 120, 1500, 7), 12, 7, {}),
    "battle_order10": (lambda lib: pc.make_battle(lib, 30, 250, 11), 25, 11, {"order": [1, 0]}),
    "pursuit_40": (lambda lib: pc.make_pursuit(lib, 40, 0), 120, 0, {}),
    "gather_40": (lambda lib: pc.make_gather(lib, 40, 0), 80, 0, {"act_groups": [1]}),
    "forest_30": (lambda lib: pc.make_builtin(lib, "forest", 30, 3), 60, 3, {}),
    "double_attack_30": (lambda lib: pc.make_builtin(lib, "double_attack", 30, 4, n0=150, n1=120), 60, 4, {}),
    "mixed_3groups": (lambda lib: pc.make_mixed(lib, 36, 6), 60, 6, {"order": [2, 0, 1]}),
    "battle_rect": (lambda lib: pc.make_battle_rect(lib), 40, 2, {}),
    "multi4": (lambda lib: pc.make_multi4(lib), 50, 8, {"order": [3, 1, 0, 2]}),
    "arrange_absorb": (lambda lib: pc.make_arrange(lib), 60, 12, {"act_groups": [1], "stop_on_done": False}),
    "arrange_goals_move": (lambda lib: pc.make_arrange(lib, 24, 14, n_goal=60, n_agent=150), 40, 14, {"stop_on_done": False}),
    "sector_ranges": (lambda lib: pc.make_sector(lib), 50, 9, {"order": [1, 0]}),
    "turn_mode": (lambda lib: pc.make_turn(lib, 30, 5), 60, 5, {"order": [2, 0, 1], "stop_on_done": False}),
    "food_mode": (lambda lib: pc.make_food(lib, 30, 3), 70, 3, {"order": [1, 2, 0], "stop_on_done": False}),
    "general_rules": (lambda lib: pc.make_general_rules(lib), 70, 21, {"stop_on_done": False}),
    "gather_infight": (lambda lib: pc.make_gather(lib, 24, 2, n_agent=150, n_food=60), 40, 2, {"act_groups": [1]}),
}
FULL_OBS_STEPS = (0, 7)      # steps whose observation tensors are stored in full (others: sha256)


def record(name, lib):
    make, steps, seed, kw = SCENARIOS[name]
    return pc.run_trace(make(lib), steps, seed, keep_obs=True, **kw)


def pack(trace):
    out = {"n_steps": np.array(len(trace))}
    for t, rec in enumerate(trace):
        out["s%d_num" % t] = np.array(rec["num"], dtype=np.int32)
        out["s%d_done" % t] = np.array(int(rec["done"]))
        for g in range(len(rec["num"])):
            out["s%d_id%d" % (t, g)] = rec["id"][g]
            out["s%d_pos%d" % (t, g)] = rec["pos"][g].astype(np.int16)
            out["s%d_posafter%d" % (t, g)] = rec["pos_after"][g].astype(np.int16)
            out["s%d_alive%d" % (t, g)] = rec["alive"][g]
            out["s%d_reward%d" % (t, g)] = rec["reward"][g]
        for g, (v, f) in rec["obs"].items():
            out["s%d_viewsha%d" % (t, g)] = np.frombuffer(bytes.fromhex(pc.sha(v)), dtype=np.uint8)
            out["s%d_featsha%d" % (t, g)] = np.frombuffer(bytes.fromhex(pc.sha(f)), dtype=np.uint8)
            if t in FULL_OBS_STEPS and sum(rec["num"]) <= 400:
                out["s%d_view%d" % (t, g)] = v
                out["s%d_feat%d" % (t, g)] = f
    return out


def compare_to_golden(name, trace):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    assert int(z["n_steps"]) == len(trace), "%s: %d steps vs golden %d" % (name, len(trace), int(z["n_steps"]))
    for t, rec in enumerate(trace):
        tag = "%s step %d" % (name, t)
        np.testing.assert_array_equal(z["s%d_num" % t], np.array(rec["num"]), err_msg=tag + " num")
        assert int(z["s%d_done" % t]) == int(rec["done"]), tag + " done"
        for g in range(len(rec["num"])):
            np.testing.assert_array_equal(z["s%d_id%d" % (t, g)], rec["id"][g], err_msg=tag + " id")
            np.testing.assert_array_equal(z["s%d_pos%d" % (t, g)], rec["pos"][g], err_msg=tag + " pos")
            np.testing.assert_array_equal(z["s%d_posafter%d" % (t, g)], rec["pos_after"][g], err_msg=tag + " pos_after")
            np.testing.assert_array_equal(z["s%d_alive%d" % (t, g)], rec["alive"][g], err_msg=tag + " alive")
            np.testing.assert_allclose(z["s%d_reward%d" % (t, g)], rec["reward"][g], rtol=0, atol=pc.REWARD_TOL,
                                       err_msg=tag + " reward")
        for g, (v, f) in rec["obs"].items():
            if ("s%d_view%d" % (t, g)) in z.files:
                np.testing.assert_array_equal(z["s%d_feat%d" % (t, g)].view(np.uint32), f.view(np.uint32), err_msg=tag + " feature")
                np.testing.assert_array_equal(z["s%d_view%d" % (t, g)].view(np.uint32), v.view(np.uint32), err_msg=tag + " view")
            assert bytes(z["s%d_featsha%d" % (t, g)]).hex() == pc.sha(f), tag + " feature sha256"
            assert bytes(z["s%d_viewsha%d" % (t, g)]).hex() == pc.sha(v), tag + " view sha256"


def check_against_golden(name, lib):
    compare_to_golden(name, record(name, lib))


# ------------------------------------------------------------------ edge cases found by the chaotic-caller fuzz
EDGE_FILE = os.path.join(GOLDEN_DIR, "edge_cases.npz")


def record_edge_cases(lib, tmpdir):
    """group reward across reset (parity_common.group_reward_across_reset) and the self-kill replay frames
    (parity_common.self_kill_frames) as a flat dict of arrays"""
    out = {}
    for i, r in enumerate(pc.group_reward_across_reset(lib)):
        out["group_reward_%d" % i] = r
    act = pc.self_kill_frames(lib, None)
    rew, files = pc.self_kill_frames(lib, tmpdir, act)
    out["self_kill_action"] = np.array([act])
    out["self_kill_reward"] = rew
    for name, data in files.items():
        out["self_kill_file_" + name] = np.frombuffer(data, dtype=np.uint8)
    return out



# ------------------------------------------------------------------ recorded results of the reference, one per test case
# Differential tests that used to run the compiled reference next to the library under test compare with these instead,
# so they run where the reference cannot be built.  A result (nested dicts / lists / tuples of arrays, numbers, strings,
# bytes) is stored as a fingerprint: the sha256 of every value that is compared exactly, and the rewards, which are
# compared within REWARD_TOL as in compare_traces, in full.
RESULTS_FILE = os.path.join(GOLDEN_DIR, "reference_results.npz")
RECORD_ENV = "MAGENT_B200_RECORD_REFERENCE"     # =1: check_reference_result records the reference's result instead


def fingerprint(result):
    """(sha256 hex of the exactly compared part, float32 array of the rewards) of a nested result.  Rewards are the
    'reward' entry of a run_trace record and the float32 arrays of a fuzz_common log record labelled '... reward ...'."""
    h = hashlib.sha256()
    rewards = []

    def walk(x, reward=False):
        if isinstance(x, dict):
            h.update(b"{%d" % len(x))
            for k in sorted(x, key=repr):
                h.update(repr(k).encode())
                walk(x[k], reward or k == "reward")
        elif isinstance(x, (list, tuple)):
            h.update(b"[%d" % len(x))
            labelled = len(x) > 0 and isinstance(x[0], str) and " reward" in x[0]
            for i, v in enumerate(x):
                walk(v, reward or (labelled and i > 0 and getattr(v, "dtype", None) == np.float32))
        elif isinstance(x, str):
            h.update(b"s" + x.encode())
        elif isinstance(x, bytes):
            h.update(b"b%d:" % len(x) + x)
        else:
            a = np.asarray(x)
            h.update(("%s%s" % (a.dtype, a.shape)).encode())
            if reward:
                rewards.append(a.astype(np.float32).ravel())
            else:
                h.update(np.ascontiguousarray(a).tobytes())
    walk(result)
    return h.hexdigest(), (np.concatenate(rewards) if rewards else np.zeros((0,), np.float32))


def check_reference_result(key, run, lib):
    """run(lib) must give the result run(oracle/_ref) gave when tests/golden/reference_results.npz was recorded
    (tests/golden/make_golden.py)"""
    if os.environ.get(RECORD_ENV) == "1":
        a, b = fingerprint(run(pc.REF_LIB)), fingerprint(run(pc.REF_LIB))
        assert a[0] == b[0] and np.array_equal(a[1], b[1]), key + ": reference not deterministic"
        stored = dict(np.load(RESULTS_FILE)) if os.path.exists(RESULTS_FILE) else {}
        stored[key + "/sha"] = np.frombuffer(bytes.fromhex(a[0]), dtype=np.uint8)
        stored[key + "/reward"] = a[1]
        np.savez_compressed(RESULTS_FILE, **stored)
    z = np.load(RESULTS_FILE)
    assert key + "/sha" in z.files, key + ": no recorded reference result"
    sha, rewards = fingerprint(run(lib))
    want = z[key + "/reward"]
    assert rewards.shape == want.shape, "%s: %d rewards vs %d recorded from the reference" % (key, rewards.size, want.size)
    np.testing.assert_allclose(rewards, want, rtol=0, atol=pc.REWARD_TOL, err_msg=key + " rewards")
    assert sha == bytes(z[key + "/sha"]).hex(), key + ": differs from the result recorded from the reference"


def check_edge_cases(lib, tmpdir, with_render=True):
    want = np.load(EDGE_FILE)
    for i, r in enumerate(pc.group_reward_across_reset(lib)):
        np.testing.assert_allclose(r, want["group_reward_%d" % i], rtol=0, atol=pc.REWARD_TOL)
    if with_render:
        rew, files = pc.self_kill_frames(lib, tmpdir, int(want["self_kill_action"][0]))
        np.testing.assert_allclose(rew, want["self_kill_reward"], rtol=0, atol=pc.REWARD_TOL)
        for name, data in files.items():
            assert data == want["self_kill_file_" + name].tobytes(), "replay file %s differs from the golden" % name
