#!/usr/bin/env python
"""bench.py -- agent-steps/s of the GridWorld step path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference]

A "step" is one pass of the hot path over one batch of synthetic input, through the C ABI:
    for every acting group: env_get_observation;  set_action (uniform random);  env_step;
    env_get_reward;  gridworld_clear_dead.
`value`   = whole-job agent-steps/s with every buffer resident in HBM (device pointers through the same
            ABI calls, random actions generated on the device), timed with CUDA events, max over ranks.
`e2e`     = the same loop through HOST buffers (page-locked numpy arrays): observation and reward D2H and
            action H2D copies are inside the timed region.
`roofline`= the observation-render kernel: algorithmic bytes per launch / mean launch duration (CUDA events
            around every launch inside the timed region) against the measured HBM copy bandwidth.
`cpu_baseline` / `--impl reference` = the UNMODIFIED reference C++ engine (oracle/_ref/libmagent.so, built
            by oracle/Makefile where the reference sources exist) driven by the same host code on the host cores;
            without it, the plain-C restatement (oracle/_build), reported as `cpu_baseline.kind` = "port".
`--dump-outputs DIR` writes what the device-resident loop computed in its last timed step (see dump_outputs).

Workloads (BASELINE.json configs; the default is the per-GPU share of configs[4], weak scaling):
    battle512  battle 200x200, 2x1000 agents, 512 independent arenas per GPU          [default]
    battle1    battle 200x200, 2x1000 agents, 1 arena                     (configs[1])
    battle512_blocks  the dense two-block layout of examples/train_battle.py (2x1600), 512 arenas per GPU
    gather64   gather 200x200, 495 agents + 1847 food, 64 arenas          (configs[2])
    battle1m   battle 1000x1000, 2x400k agents, 1 arena (obs-render roofline; configs[3] as placeable)
    battle1m_sparse  battle 4472x4472, 2x500k agents, 1 arena (configs[3] in the reference's own 1 M geometry)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "agent-steps/sec on battle map at 1/2/4/8 B200 vs ref C++ on host cores"
UNIT = "agent-steps/s"
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libmagent.so")
PORT_LIB = os.path.join(ROOT, "oracle", "_build", "libmagent_oracle.so")

WORKLOADS = {
    "battle512": dict(desc="battle 200x200, 2x1000 agents random placement, 512 independent arenas per GPU "
                           "(per-GPU share of BASELINE configs[4]), uniform random actions",
                      game="battle", map_size=200, arenas=512, n=1000),
    "battle512_blocks": dict(desc="battle 200x200, 2x1600 agents in the two facing blocks of examples/train_battle.py:15-40 "
                                  "(dense fighting; SURVEY 8d 'dense variant'), 512 independent arenas per GPU",
                             game="battle_blocks", map_size=200, arenas=512),
    "battle1": dict(desc="battle 200x200, 2x1000 agents, 1 arena (BASELINE configs[1]), uniform random actions",
                    game="battle", map_size=200, arenas=1, n=1000),
    "gather64": dict(desc="gather 200x200, 495 agents + 1847 food (examples/train_gather.py layout), 64 arenas "
                          "(BASELINE configs[2]); only the agent group observes/acts",
                     game="gather", map_size=200, arenas=64),
    "battle1m": dict(desc="battle 1000x1000, 2x400k agents (80% fill; BASELINE configs[3] as placeable), 1 arena",
                     game="battle", map_size=1000, arenas=1, n=400000),
    "battle1m_sparse": dict(desc="battle 4472x4472, 2x500k agents (the reference's own 1 M geometry, "
                                 "scripts/test/test_1m.py:66-74: map = sqrt(20 N)), 1 arena",
                            game="battle", map_size=4472, arenas=1, n=500000),
}


def build_env(wl, lib, arenas, seed0=0):
    import magent_b200 as magent
    kw = {}
    if arenas != 1:
        kw["_num_arenas"] = arenas
    if wl.get("host_path"):
        kw["_host_path"] = wl["host_path"]
    if wl["game"] == "battle":
        env = magent.GridWorld("battle", map_size=wl["map_size"], _lib=lib, **kw)
        env.set_seed(seed0)
        env.reset()
        hs = env.get_handles()
        for h in hs:
            env.add_agents(h, method="random", n=wl["n"])
        return env, list(hs)
    if wl["game"] == "battle_blocks":
        import math
        size = wl["map_size"]
        env = magent.GridWorld("battle", map_size=size, _lib=lib, **kw)
        env.set_seed(seed0)
        env.reset()
        hs = env.get_handles()
        gap, side = 3, int(math.sqrt(size * size * 0.04)) * 2
        ys = range((size - side) // 2, (size - side) // 2 + side, 2)
        env.add_agents(hs[0], method="custom", pos=[[x, y, 0] for x in range(size // 2 - gap - side, size // 2 - gap, 2) for y in ys])
        env.add_agents(hs[1], method="custom", pos=[[x, y, 0] for x in range(size // 2 + gap, size // 2 + gap + side, 2) for y in ys])
        return env, list(hs)
    if wl["game"] == "gather":
        env = magent.GridWorld("gather", map_size=wl["map_size"], _lib=lib, **kw)
        env.set_seed(seed0)
        env.reset()
        hs = env.get_handles()
        gather_map(env, wl["map_size"], hs[0], hs[1])
        return env, [hs[1]]
    raise ValueError(wl["game"])


def gather_map(env, map_size, food_handle, agent_handle):
    """square rings of agents and food as in examples/train_gather.py:46-77 (legend omitted)"""
    cx = cy = map_size // 2

    def add_square(pos, side, gap):
        side = int(side)
        for x in range(cx - side // 2, cx + side // 2 + 1, gap):
            pos.append([x, cy - side // 2]); pos.append([x, cy + side // 2])
        for y in range(cy - side // 2, cy + side // 2 + 1, gap):
            pos.append([cx - side // 2, y]); pos.append([cx + side // 2, y])
    pos = []
    for frac, gap in ((0.9, 3), (0.8, 4), (0.7, 6)):
        add_square(pos, map_size * frac, gap)
    env.add_agents(agent_handle, method="custom", pos=pos)
    pos = []
    for frac, gap in ((0.65, 10), (0.6, 10), (0.55, 10), (0.5, 4), (0.45, 3), (0.4, 1), (0.3, 1)):
        add_square(pos, map_size * frac, gap)
    for d in (2, 4, 6):
        add_square(pos, map_size * 0.3 - d, 1)
    env.add_agents(food_handle, method="custom", pos=pos)


# ---------------------------------------------------------------------------------------------- CPU arm
def cpu_worker(args):
    """child process: run the reference (or the C restatement) for --cpu-steps and print agent-steps, seconds"""
    import numpy as np
    wl = WORKLOADS[args.workload]
    lib = REF_LIB if os.path.exists(REF_LIB) else PORT_LIB
    env, act = build_env(wl, lib, 1, seed0=args.cpu_seed)
    rs = np.random.RandomState(args.cpu_seed)

    def one():
        n = 0
        for h in act:
            env.get_observation(h)
        for h in act:
            k = env.get_num(h)
            env.set_action(h, rs.randint(0, env.get_action_space(h)[0], size=k).astype(np.int32))
            n += k
        env.step()
        for h in act:
            env.get_reward(h)
        env.clear_dead()
        return n
    for _ in range(args.cpu_warmup):
        one()
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.cpu_steps):
        total += one()
    dt = time.perf_counter() - t0
    print(json.dumps({"agent_steps": total, "seconds": dt}))


def usable_cores():
    """host threads this process may really use: affinity mask, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except (OSError, ValueError, IndexError):
            pass
    return n


def run_cpu_baseline(workload, budget_steps=None):
    """time the reference engine on the host cores: best of {P single-thread processes, 1 process x all
    OpenMP threads} (SURVEY.md §8d); every process simulates its own arena of the workload."""
    cores = usable_cores()
    kind = "reference" if os.path.exists(REF_LIB) else "port"
    if kind == "port" and not os.path.exists(PORT_LIB):
        return None
    wl = WORKLOADS[workload]
    agents = 2 * wl.get("n", 500)
    steps = budget_steps or max(3, min(400, int(3.0e6 / max(agents, 1))))
    warm = max(1, min(20, steps // 5))

    def launch(nproc, omp):
        env = dict(os.environ, OMP_NUM_THREADS=str(omp))
        procs = [subprocess.Popen([sys.executable, os.path.abspath(__file__), "--_cpu-worker", "--workload", workload,
                                   "--cpu-steps", str(steps), "--cpu-warmup", str(warm), "--cpu-seed", str(i)],
                                  env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                 for i in range(nproc)]
        outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in procs]
        slowest = max(o["seconds"] for o in outs)
        return sum(o["agent_steps"] for o in outs) / slowest, 1e3 * slowest / steps
    tried = {}
    if wl["arenas"] > 1:      # independent arenas: the CPU can run one per process
        for p in sorted({cores, max(1, cores // 2), max(1, cores // 4)}, reverse=True):
            tried["%d procs x 1 thread" % p] = launch(p, 1) + (p,)
    else:                     # a single arena cannot be split across processes: one process, 1..N OpenMP threads
        tried["1 proc x 1 thread"] = launch(1, 1) + (1,)
    omp = min(cores, 16)                      # the reference's own harness uses 8-16 OpenMP threads (scripts/test/test_fps.py:22-36)
    tried["1 proc x %d OpenMP threads" % omp] = launch(1, omp) + (omp,)
    how = max(tried, key=lambda k: tried[k][0])
    best, ms_per_sample_step, used = tried[how]
    return {"value": best, "unit": UNIT, "cores": used, "kind": kind, "cores_usable": cores,
            "ms_per_sample_step": ms_per_sample_step,
            "sample": "%s: one arena per process, %d timed steps after %d warm-up; tried %s -> best: %s"
                      % (wl["desc"].split(",")[0], steps, warm,
                         ", ".join("%s: %.3g" % (k, v[0]) for k, v in tried.items()), how)}


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"],     # the recipe's interval (B200_PROFILING.md):
                                         # at 20 ms a query landing inside a 25 ms timed window cost rank 0 up to 0.2 ms/step
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def sample_now(self):
        pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 7:
                    continue
                try:
                    sm.append(float(p[0])); mx.append(float(p[1]))
                except ValueError:
                    continue
                for nm, v in zip(names, p[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
            out["sm_max_mhz"] = max(mx)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and the engine's host threads, which inherit the mask) to the CPUs of the NUMA node its GPU hangs
    off, BEFORE any page-locked buffer is allocated: the 5 GB of observations per step are then written to local
    memory.  Returns a short description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out                   # 00000000:9c:00.0 -> 0000:9c:00.0
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return "GPU reports no NUMA node"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "node %d has no CPU in the affinity mask" % node
        os.sched_setaffinity(0, cpus)
        return "rank bound to NUMA node %d (%d cpus) of GPU %s" % (node, len(cpus), bus)
    except Exception as e:                                           # noqa: BLE001  (binding is best effort)
        return "not bound (%s)" % type(e).__name__


class NvmlClockSampler:
    """SM clock and throttle reasons of one GPU, polled from a thread of this process through NVML (nvidia-ml-py): two
    cheap queries per sample.  The nvidia-smi poller above asks for more (power draw among it) and was seen to stall
    the GPU for several milliseconds when a query landed inside the 25 ms timed window (profiles/README.md, round 2)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index, interval=0.05, pci_bus_id=None):
        import threading
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        # NVML numbers the physical GPUs, CUDA the visible ones (CUDA_VISIBLE_DEVICES): go by PCI bus id when it is known
        self.h = pynvml.nvmlDeviceGetHandleByPciBusId(pci_bus_id.encode()) if pci_bus_id else pynvml.nvmlDeviceGetHandleByIndex(index)
        self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        self.get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        self.sm, self.bits, self.interval = [], 0, interval
        self._stop = threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def sample_now(self):
        try:
            self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            self.bits |= int(self.get_reasons(self.h))
        except Exception:                                            # noqa: BLE001
            pass

    def _run(self):
        while not self._stop.is_set():
            self.sample_now()
            self._stop.wait(self.interval)

    def stop(self):
        self._stop.set()
        self.t.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": sorted(n for b, n in self.REASONS.items() if self.bits & b),
               "samples": len(self.sm), "how": "NVML from a thread of the bench process, every %d ms" % int(self.interval * 1e3)}
        if self.sm:
            sm = sorted(self.sm)
            out["sm_mhz"] = sm[len(sm) // 2]
        return out


def make_clock_sampler(index, pci_bus_id=None):
    if os.environ.get("MAGENT_B200_BENCH_SAMPLER") != "smi":
        try:
            return NvmlClockSampler(index, pci_bus_id=pci_bus_id)
        except Exception:                                            # noqa: BLE001  (no nvidia-ml-py: fall back to nvidia-smi)
            pass
    return ClockSampler(pci_bus_id or index)


DUMP_BYTES = 64 * 10 ** 6 - 64 * 1024      # 64 MB with room for the .npy headers


def dump_outputs(out_dir, bufs, nums, done, prefix=""):
    """Write what the last timed step handed its caller, in float32: per acting group g the observation views
    g<g>_view (n, H, W, C), the feature rows g<g>_feature (n, F) and the rewards g<g>_reward (n,) of the n agents it
    observed, and the done flag.  Where that is more than 64 MB, every group keeps an equal share of its rows, drawn
    with a fixed seed (g as the seed); g<g>_rows (float64) lists the rows kept."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // max(1, len(bufs))
    for g, (v, f, r) in sorted(bufs.items()):
        n = nums[g]
        row_bytes = 4 * (int(np.prod(v.shape[1:])) + int(np.prod(f.shape[1:])) + 1) + 8
        keep = min(n, budget // row_bytes)
        rows = np.arange(n) if keep == n else np.sort(np.random.RandomState(g).choice(n, keep, replace=False))
        idx = torch.from_numpy(rows).to(v.device)
        for name, t in (("view", v), ("feature", f), ("reward", r)):
            np.save(os.path.join(out_dir, "%sg%d_%s.npy" % (prefix, g, name)), t.index_select(0, idx).float().cpu().numpy())
        np.save(os.path.join(out_dir, "%sg%d_rows.npy" % (prefix, g)), rows.astype(np.float64))
    np.save(os.path.join(out_dir, prefix + "done.npy"), done.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="battle512", choices=sorted(WORKLOADS) + ["all"],
                    help="'all': one JSON line per BASELINE config (battle1, gather64, battle1m, battle1m_sparse, battle512), N=1 only")
    ap.add_argument("--arenas", type=int, default=None, help="override arenas per GPU")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's arenas PER GPU (default); strong: BASELINE configs[4] literally -- 4096 arenas "
                         "in total (or --arenas), sharded over the ranks (magent_b200.sharding.shard_arenas)")
    ap.add_argument("--obs-dtype", default="f32", choices=["f32", "f16"],
                    help="f32 = the reference ABI (headline); f16 = the compact hand-off extension (reported separately)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-seconds", type=float, default=1.5, help="the e2e loop runs at least this long (and >= 3 steps)")
    ap.add_argument("--host-path", default=None, choices=["wire", "dense"],
                    help="env_get_observation into host memory: wire records + host expansion (default) or the round-1 dense DMA")
    ap.add_argument("--numa-bind", action="store_true",
                    help="pin the rank to the NUMA node of its GPU (default: off -- the engine spreads its host threads and the "
                         "wrapper's big receive buffers over all nodes, which doubles the host write bandwidth on two sockets)")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="device-resident loop as a replayed CUDA graph of two steps (magent_b200_graph_*): auto = for "
                         "launch-bound workloads (fewer than 250k agents per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the observations, rewards and done flag of the last timed step to DIR/<name>.npy")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--_cpu-worker", dest="cpu_worker", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=100)
    ap.add_argument("--cpu-warmup", type=int, default=5)
    ap.add_argument("--cpu-seed", type=int, default=0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cpu_worker:
        return cpu_worker(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "all":
        # one child per workload (a fresh CUDA context each): every BASELINE config in one call
        for w in ("battle1", "gather64", "battle1m", "battle1m_sparse", "battle512"):
            cmd = [sys.executable, os.path.abspath(__file__), "--workload", w, "--steps", str(args.steps), "--warmup", str(args.warmup),
                   "--e2e-seconds", str(args.e2e_seconds)] + (["--no-cpu"] if args.no_cpu or w != "battle512" else []) + \
                  (["--no-e2e"] if args.no_e2e else []) + \
                  (["--dump-outputs", os.path.join(args.dump_outputs, w)] if args.dump_outputs else [])
            r = subprocess.run(cmd, capture_output=True, text=True)
            sys.stdout.write(r.stdout if r.returncode == 0 else json.dumps({"workload": w, "failed": r.stderr[-400:]}) + "\n")
            sys.stdout.flush()
        return
    wl = dict(WORKLOADS[args.workload])
    if args.arenas:
        wl["arenas"] = args.arenas
    first_arena = None
    if args.scaling == "strong":
        from magent_b200.sharding import shard_arenas
        total_arenas = args.arenas or 4096
        first_arena, wl["arenas"] = shard_arenas(total_arenas, rank, world)
        wl["desc"] = wl["desc"].replace("512 independent arenas per GPU (per-GPU share of BASELINE configs[4])",
                                        "%d independent arenas in total (BASELINE configs[4]) sharded over %d GPU(s)" % (total_arenas, world))

    if args.impl == "reference":
        if rank != 0:
            return
        if args.dump_outputs:
            sys.exit("bench.py: --dump-outputs dumps the B200 arm's outputs; it does not apply to --impl reference")
        if not os.path.exists(REF_LIB):
            # never silently the C restatement: the JSON line says cpu_baseline.kind = "port"
            sys.stderr.write("bench.py --impl reference: oracle/_ref/libmagent.so is missing (`make -C oracle ref` builds it "
                             "from the reference sources); timing the plain-C restatement instead\n")
        cb = run_cpu_baseline(args.workload, budget_steps=None)
        if cb is None:
            sys.exit("bench.py --impl reference: no CPU engine built (run __graft_entry__.build())")
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_sample_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "note": "CPU engine: rate of a bounded sample (one arena per process); ms_per_step = wall time of one "
                                                    "loop iteration of that sample (all its processes in parallel)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
    # ... and make sure of it: libraries (NCCL prints its version banner with printf) get stderr as their fd 1; the JSON
    # line goes to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    numa = bind_to_gpu_numa_node(local_rank) if args.numa_bind else None
    import numpy as np
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import magent_b200 as magent  # noqa: F401
    from magent_b200.c_lib import load_library
    lib = load_library()
    A = wl["arenas"]
    t_setup = time.time()
    if args.host_path:
        wl["host_path"] = args.host_path
    env, act = build_env(wl, lib.path, A, seed0=first_arena if first_arena is not None else rank * A)
    handles = env.get_handles()
    spaces = {env._hv(h): (env.get_view_space(h), env.get_feature_space(h)) for h in handles}

    # device-resident receive buffers, sized for the initial population (it only shrinks)
    dev = torch.device("cuda", local_rank)
    half = args.obs_dtype == "f16"
    obs_torch_dtype, obs_esz = (torch.float16, 2) if half else (torch.float32, 4)
    obs_call = lib.magent_b200_get_observation_f16 if half else lib.env_get_observation
    bufs = {}
    for h in act:
        g = env._hv(h)
        n0 = env.get_num(h)
        bufs[g] = (torch.empty((n0,) + spaces[g][0], dtype=obs_torch_dtype, device=dev),
                   torch.empty((n0,) + spaces[g][1], dtype=obs_torch_dtype, device=dev),
                   torch.empty((n0,), dtype=torch.float32, device=dev))

    import ctypes
    done_dev = torch.zeros((1,), dtype=torch.int32, device=dev)

    def dev_step(seed):
        for h in act:
            g = env._hv(h)
            v, f, _r = bufs[g]
            ptrs = (ctypes.c_void_p * 2)(v.data_ptr(), f.data_ptr())
            obs_call(env.game, g, ptrs)
        for h in act:
            env.set_random_actions(h, seed)
        env.step_device_done(done_dev.data_ptr())      # `done` to a device int: no read-back, no host wait
        for h in act:
            g = env._hv(h)
            lib.env_get_reward(env.game, g, bufs[g][2].data_ptr())
        env.clear_dead()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock sampler starts before the warm-up, so that its own start-up (and first query) is over by the time the
    # timed region begins; it keeps sampling through the timed region and the e2e loop
    bus = None
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:                                                # noqa: BLE001
        pass
    sampler = make_clock_sampler(local_rank, bus) if rank == 0 else None
    for w in range(args.warmup):
        dev_step(1000 + w)
    setup_s = time.time() - t_setup

    # per-launch algorithmic bytes of the obs-render kernel at the start of the timed region
    obs_bytes = 0          # everything get_observation writes per step (views + feature rows)
    render_bytes = 0       # what obs_render_kernel itself moves: the views it writes + one pass over the 1-byte kind plane
    for h in act:
        g = env._hv(h)
        (vh, vw, vc), (fs,) = spaces[g]
        obs_bytes += env.get_num(h) * obs_esz * (vh * vw * vc + fs)
        render_bytes += env.get_num(h) * obs_esz * (vh * vw * vc) + A * wl["map_size"] ** 2 * 1
    obs_bytes_per_launch = render_bytes / len(act)

    n_agents_now = sum(env.get_num(h) for h in handles)
    use_graph = args.graph == "on" or (args.graph == "auto" and n_agents_now < 250000)
    graph_note = None
    steps_timed = args.steps
    last_nums = {}

    def last_step(s):
        # the group sizes the last step observes; the engine settles them with a host wait, so only when dumping
        if args.dump_outputs:
            last_nums.update({env._hv(h): env.get_num(h) for h in act})
        dev_step(s)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if use_graph:
        # launch-bound workload: two steps (the ping-pong buffers come back after two culls) recorded once, replayed
        # steps/2 times -- one launch per replay.  The random-action seed rides on the device-side step counter, so every
        # replayed step still draws fresh actions.  The render kernel's duration is taken from a few un-captured steps
        # just before (CUDA events cannot bracket a node of a replayed graph).
        env.set_profiling(True)
        for s in range(4):
            dev_step(2000 + s)
        torch.cuda.synchronize()
        obs_ms, obs_launches = env.get_profile()
        env.set_profiling(False)
        l_cap = env.launch_count()
        gid = env.capture_graph(lambda: (dev_step(0), dev_step(1)))
        per_replay = env.launch_count() - l_cap
        # an odd last step (and, when dumping, the last step, whose group sizes are read first) runs un-captured
        replays = (args.steps - 1) // 2 if args.dump_outputs else args.steps // 2
        tail = args.steps - 2 * replays
        env.launch_graph(gid, 2)                        # warm the instantiated graph
        barrier()
        c0 = env.get_counters()
        ev0.record()
        if replays:
            env.launch_graph(gid, replays)
        l_tail = env.launch_count()
        for s in range(tail):
            (last_step if s == tail - 1 else dev_step)(2 * replays + s)
        ev1.record()
        if sampler:
            sampler.sample_now()                        # the host is ahead of the GPU here: a sample inside the timed region
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        barrier()
        c1 = env.get_counters()
        launches = per_replay * replays + env.launch_count() - l_tail
        graph_note = "CUDA graph of 2 steps (%d kernels) replayed %d times" % (per_replay, replays) + \
            (", then %d un-captured step(s)" % tail if tail else "")
    else:
        c0 = env.get_counters()
        l0 = env.launch_count()
        env.set_profiling(True)
        ev0.record()
        for s in range(args.steps):
            (last_step if s == args.steps - 1 else dev_step)(s)
        ev1.record()
        if sampler:
            sampler.sample_now()                        # everything is queued, the GPU is mid-way: a sample inside the timed region
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        obs_ms, obs_launches = env.get_profile()
        env.set_profiling(False)
        barrier()
        c1 = env.get_counters()
        launches = env.launch_count() - l0
    agent_steps = c1[0] - c0[0]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bufs, last_nums, done_dev, "rank%d_" % rank if world > 1 else "")

    if os.environ.get("MAGENT_B200_BENCH_RANK_REPORT"):
        sys.stderr.write("rank %d: %.4f ms/step device time, render %.4f ms/launch, %d launches\n"
                         % (rank, ms / steps_timed, (obs_ms / obs_launches) if obs_launches else 0.0, launches))
    from magent_b200.sharding import reduce_window
    # NCCL over NVLink: SUM of the throughput counters, MAX over ranks of the device time -- the only collective of the job
    (total_steps, total_launches), ms_max = reduce_window([agent_steps, launches], ms, device=dev)
    value = total_steps / (ms_max * 1e-3)

    # ---- end-to-end: host (pinned) buffers through the public API, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        pools = {}
        rs = np.random.RandomState(rank)
        for h in act:
            pools[env._hv(h)] = rs.randint(0, env.get_action_space(h)[0], size=env.get_num(h)).astype(np.int32)

        def host_step():
            for h in act:
                env.get_observation_f16(h) if half else env.get_observation(h)
            for h in act:
                env.set_action(h, pools[env._hv(h)][:env.get_num(h)])
            env.step()
            for h in act:
                env.get_reward(h)
            env.clear_dead()
        for _ in range(3):                              # allocates the pinned receive buffers, starts the host threads
            host_step()
        barrier()
        t0 = time.perf_counter()
        host_step()
        one = time.perf_counter() - t0
        e2e_steps = max(3, int(args.e2e_seconds / max(one, 1e-6)) + 1)
        if world > 1:                                   # every rank must run the same number of steps
            ts = torch.tensor([e2e_steps], dtype=torch.int64, device=dev)
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            e2e_steps = int(ts.item())
        barrier()
        c0 = env.get_counters()
        io0 = env.get_io_stats()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        c1 = env.get_counters()
        io1 = env.get_io_stats()
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        cnt = torch.tensor([c1[0] - c0[0], io1["h2d"] - io0["h2d"], io1["d2h"] - io0["d2h"],
                            io1["host_written"] - io0["host_written"]], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        e2e = {"value": int(cnt[0].item()) / float(t.item()), "unit": UNIT, "steps": e2e_steps, "seconds": float(t.item()),
               "h2d_bytes_per_step": int(cnt[1].item()) // e2e_steps, "d2h_bytes_per_step": int(cnt[2].item()) // e2e_steps,
               "host_bytes_written_per_step": int(cnt[3].item()) // e2e_steps,
               "host_threads": int(lib.magent_b200_host_threads()),
               "ms_per_step_by_phase": {"wire_records_until_first_copy": (io1["us_wire"] - io0["us_wire"]) / 1e3 / e2e_steps,
                                        "host_expansion": (io1["us_expand"] - io0["us_expand"]) / 1e3 / e2e_steps,
                                        "feature_rows": (io1["us_feature"] - io0["us_feature"]) / 1e3 / e2e_steps,
                                        "whole_step": 1e3 * dt / e2e_steps},
               "path": "observations cross PCIe as compact wire records (headers + marks) and are expanded into the caller's "
                       "float32 buffers by the engine's host threads; feature rows, rewards and actions are plain copies"
                       if (args.host_path or "wire") == "wire" and not half else "dense records over PCIe",
               "bytes_counted": "by the engine (magent_b200_get_io_stats): every byte it copies across PCIe / writes into caller buffers",
               "timing": "host wall clock around the API loop (includes PCIe copies, host expansion and syncs), max over ranks",
               "host_buffers": "page-locked numpy arrays owned by the wrapper",
               "numa": numa or "%d node(s): receive buffers split over the nodes, host threads pinned per node" % int(lib.magent_b200_numa_nodes())}

    clocks = sampler.stop() if sampler else None      # sampled across the device-timed and the e2e timed regions
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    achieved = (obs_bytes_per_launch / (obs_ms / obs_launches * 1e-3)) / 1e9 if obs_launches and obs_ms > 0 else None
    # DRAM bytes per launch of the roofline kernel from the ncu --set full capture (profiles/obs_render_traffic.json); the
    # capture is tied to the kernel source it was taken from: a changed backend_cuda.cu makes it stale -> null
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "obs_render_traffic.json")
    if os.path.exists(tpath):
        import hashlib
        tj = json.load(open(tpath))
        src_sha = hashlib.sha256(open(os.path.join(ROOT, "magent_b200", "csrc", "backend_cuda.cu"), "rb").read()).hexdigest()[:16]
        if tj.get("workload") == args.workload and not half and tj.get("kernel_source_sha16") == src_sha:
            traffic = tj.get("dram_bytes_per_launch")
    roofline = {"bound": "hbm", "kernel": "obs_render_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": obs_bytes_per_launch,
                "algorithmic_bytes": "views written by this kernel (sizeof(elem) * H_v * W_v * C per observer) + one read of the "
                                     "1-byte kind plane per arena; the feature rows (F elements per observer) are written by "
                                     "obs_headers_kernel and not counted here",
                "mean_launch_ms": (obs_ms / obs_launches) if obs_launches else None, "launches_timed": obs_launches,
                "kernel_share_of_step": (obs_ms / ms) if ms > 0 and not use_graph else None}

    cpu = None
    if args.gpus == 1 and world == 1 and not args.no_cpu:
        cpu = run_cpu_baseline(args.workload)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps_timed, "warmup": args.warmup,
        "ms_per_step": ms_max / steps_timed, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32" if not half else "f32 state, f16 observation hand-off (extension, not the reference ABI)",
        "data": "synthetic",
        "config": {"workload": wl["desc"], "arenas_per_gpu": A, "agents_per_arena_at_start": 2 * wl.get("n", 0) or None,
                   "observation": "float16 via magent_b200_get_observation_f16 (extension)" if half
                                  else "float32 via env_get_observation (reference ABI)",
                   "buffers": "device-resident (CUDA pointers through the C ABI)", "actions": "uniform random, generated on device",
                   "l2": "per-step observation output (%.0f MB) exceeds the 126 MB L2" % (obs_bytes / 1e6) if obs_bytes > 126e6
                         else "per-step output %.1f MB fits L2 (latency-bound workload)" % (obs_bytes / 1e6),
                   "parallelism": "arena-sharded x%d, no data-path collective" % world, "setup_seconds": round(setup_s, 2),
                   "launch": graph_note or "one kernel launch per engine kernel (no graph)"},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": total_launches, "clocks": clocks,
        "agent_steps_timed": total_steps,
    }
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
