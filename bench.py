#!/usr/bin/env python
"""bench.py - headline measurement of the self-play hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA path through libkgb200's C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path timed on this box's host cores

A "step" is one pass of the hot path over one batch: one playout wave for `games` concurrent 19x19 games - for every
game one PUCT descent on its device-resident tree and bitboard, leaf featurisation, one b18c384nbt evaluation, policy /
value post-processing and backup (kgb_selfplay_run; stages in config["stages"]).  One visit per game per step; games
that reach maxVisits play their move and clear the tree inside the same kernels, so the loop never returns to the host.

value  : whole-job visits/s of that device-resident loop (boards, trees and NN rows live in HBM), CUDA events on the
         launching stream, max over ranks.  Per-step working set (tree arrays ~1 GB, activations ~0.5 GB) >> L2.
e2e    : visits/s through the reference-facing evaluator boundary (NeuralNet::getOutput -> kgb_forward) with HOST
         buffers: one evaluation = one visit, H2D of the feature rows and D2H of policy/value/ownership inside the timed
         region, every step, rotating over more distinct input batches than fit in L2.
N > 1  : one process per GPU (torchrun), games shard across ranks with no data-path collective ("weak" scaling);
         NCCL carries only the model-weight broadcast from rank 0 before the timed region (SURVEY.md §8e).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only: bench.py writes nothing into it

METRIC = "visits/sec 19x19 b18c384nbt selfplay"
UNIT = "visits/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="b18c384nbt")
    ap.add_argument("--games", type=int, default=256, help="concurrent games (= NN batch) per GPU")
    ap.add_argument("--fp32", action="store_true", help="use the fp32-equivalent (3-term split) mode instead of fp16 operands")
    ap.add_argument("--max-playouts-per-wave", type=int, default=0,
                    help="playouts a game may finish inside one select launch without needing the evaluator (cache hits, graph-search catch-ups) before it "
                         "skips the wave; bounds the slowest block of the launch, results are identical for every value")
    ap.add_argument("--ladder-nodes-per-wave", type=int, default=256,
                    help="ladder-reader moves per warp per wave before a game's unfinished searches are carried into the next wave "
                         "(0 = finish inside the wave); results are identical, only the schedule changes")
    ap.add_argument("--opening-max", type=int, default=150, help="games start from their own random legal play-out of 0..N moves "
                    "(a self-play server holds games at all stages; SURVEY.md 8d), then search")
    ap.add_argument("--settle-waves", type=int, default=700, help="untimed waves after the openings, so that every game has finished a move "
                    "and the evaluation cache holds what a running server's cache would hold")
    ap.add_argument("--nn-cache-pow2", type=int, default=20, help="evaluation cache entries per GPU = 2^N (nnCacheSizePowerOfTwo; 0 = off)")
    ap.add_argument("--mixed-sizes", action="store_true", help="BASELINE.json configs[3]: every game draws its board from 9x9 / 13x13 / 19x19 (equal "
                    "probabilities, like bSizes = 9,13,19) inside the 19x19 evaluator frame; a finished game's slot draws again")
    ap.add_argument("--visits", type=int, default=600, help="maxVisits per move (BASELINE.json configs[1]: 600)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the device loop's last wave left for its caller (roots, boards, leaf rows) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def model_file(name: str, rank: int):
    """Every rank synthesises a net of the architecture (no network: random init): rank 0 THE net (seed 0), the others a different
    one (seed 1, their "previous" net) which the weight broadcast below replaces."""
    from katago_b200 import modelgen
    path = os.path.join(tempfile.mkdtemp(prefix=f"kgb_rank{rank}_"), f"{name}.bin")
    return modelgen.write_model(path, name, seed=0 if rank == 0 else 1)


def broadcast_weights(handle, model, rank: int, world: int, device):
    """NCCL - the only collective on this path: rank 0 stages its net, the library's ncclBroadcast moves the packed weight arena
    into every other rank's device memory, all commit (katago_b200/dist_weights.py; include/kgb200.h; reference analogue: every
    process polls the models directory and loads the file itself, selfplay.cpp:142-231).  Device time per broadcast, max over
    ranks; the first call includes NCCL's connection set-up.  Afterwards every rank must evaluate a fixed batch bit-identically."""
    import hashlib
    import torch
    import torch.distributed as dist
    from katago_b200 import NeuralNet, modelgen
    from katago_b200.dist_weights import WeightBroadcaster
    wb = WeightBroadcaster(handle, 0, device)
    times = []
    for _ in range(4):
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([wb.update(model if rank == 0 else None)], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
    sp, gl = modelgen.synthetic_inputs(2, 19, 19, seed=4242)
    out = NeuralNet.getOutput(handle, sp.reshape(2, -1), gl)
    sha = hashlib.sha256(np.ascontiguousarray(out["policy"]).tobytes() + np.ascontiguousarray(out["value"]).tobytes()).digest()
    mine = torch.from_numpy(np.frombuffer(sha, np.uint8).copy()).to(device)
    everyone = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(everyone, mine)
    if not all(bool((x == everyone[0]).all()) for x in everyone):
        raise RuntimeError("bench.py: after the weight broadcast the ranks do not evaluate identically")
    steady = sorted(times[1:])[len(times[1:]) // 2]
    return {"ms": steady, "first_ms": times[0], "bytes": handle.weights_bytes, "GBps_per_receiver": handle.weights_bytes / (steady * 1e-3) / 1e9,
            "how": "kgb_handle_stage_weights on rank 0 -> ncclBroadcast of the packed arena (device to device) -> kgb_handle_commit_weights on every rank; "
                   "ranks > 0 started from a different net and evaluate bit-identically to rank 0 afterwards"}


CPU_SELFPLAY = os.path.join(ROOT, "oracle", "_ref", "kgref_cpu_selfplay")


def host_cores() -> int:
    """CPUs this process may actually use: the affinity mask, cut down to the cgroup's CPU quota when there is one (a container can
    see 128 CPUs in its mask and still be throttled to a few CPUs' worth of time - running 128 busy threads there measures the
    throttle, not the cores)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.999)))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, (q + per - 1) // per))
        except (OSError, ValueError):
            pass
    return n


def cpu_selfplay(model_name: str, seconds: float, warmup_seconds: float, visits: int = 600, cores: int = 0):
    """The CPU arm: the reference's own self-play hot path on the host cores - the unmodified reference Search / Board / NNEvaluator
    (linked from oracle/_ref/libkgref.a) around the restated CPU NN backend (oracle/cpubackend.cpp: the Eigen backend's algorithm in
    C++ - Winograd F(4x4,3x3) + GEMM, AVX-512; Eigen3 itself is not in this image), oracle/ref_cpu_selfplay.cpp.  One NN server thread
    per host core (single-threaded handles, batch <= 2, as the reference's CPU build runs), two game threads per core, 600-visit
    searches on cleared trees, games starting from random legal play-outs like the GPU arm's.  Returns the driver's JSON."""
    from katago_b200 import modelgen
    if not os.path.exists(CPU_SELFPLAY):
        raise RuntimeError("oracle/_ref/kgref_cpu_selfplay is not built (python -c 'import __graft_entry__ as g; g.build()' where /root/reference exists)")
    cores = cores or host_cores()
    path = os.path.join(tempfile.mkdtemp(prefix="kgb_cpuarm_"), f"{model_name}.bin")
    modelgen.write_model(path, model_name, seed=0)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([CPU_SELFPLAY, path, f"{seconds:.1f}", str(2 * cores), str(cores), str(visits), "19", f"{warmup_seconds:.1f}", "150"],
                         capture_output=True, text=True, env=env, timeout=seconds + warmup_seconds + 900)
    if out.returncode != 0:
        raise RuntimeError("kgref_cpu_selfplay failed: " + out.stderr[-500:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def cpu_baseline_object(r, model_name):
    return {"value": r["visits_per_s"], "unit": UNIT, "cores": r["nn_server_threads"], "kind": "reference", "detail": "restated Eigen path (C++), full selfplay",
            "nn_backend": "port: oracle/cpubackend.cpp behind the reference's nninterface.h (its Eigen backend needs Eigen3, absent here)",
            "sample": (f"{r['visits']} visits ({r['nn_rows']} evaluated rows) of {model_name} 19x19 self-play in {r['seconds']:.1f} s: reference Search + Board + NNEvaluator "
                       f"with oracle/cpubackend.cpp, {r['nn_server_threads']} single-threaded NN server threads + {r['game_threads']} game threads, maxVisits {r['max_visits']}")}


def run_reference(args, rank: int):
    """--impl reference: the CPU arm (cpu_selfplay above), rank 0 only.  One process plays for warmup + steps x (seconds per step); a step
    is a bounded sample of the workload."""
    if rank != 0:
        return
    steps = max(1, args.steps)
    per_step = max(1.0, min(6.0, 90.0 / steps))
    r = cpu_selfplay(args.model, steps * per_step, max(2.0, args.warmup * 1.0), args.visits)
    value = r["visits_per_s"]
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["seconds"] / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"19x19 {args.model} self-play on the host CPU, maxVisits {args.visits}: the reference's Search / Board / NNEvaluator with the restated "
                               f"Eigen-path NN backend (Winograd F(4x4,3x3) + AVX-512 GEMM), {r['nn_server_threads']} NN server threads + {r['game_threads']} game threads, "
                               f"{per_step:.1f} s per step (bounded sample)",
                   "stages": ["board", "puct_select", "featurize", "nn_eval", "postprocess", "backup"],
                   "search_params": "the search block of selfplay8mainb18.cfg incl. rootEndingBonusPoints and rootPruneUselessMoves (oracle/ref_cpu_selfplay.cpp)",
                   "driver_output": r},
        "cpu_baseline": cpu_baseline_object(r, args.model),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


class CountingSlots:
    """The SelfPlay readers the recorder calls, counting the bytes each call brings back from (or sends to) the device."""

    def __init__(self, sp):
        self._sp, self.d2h, self.h2d = sp, 0, 0

    def __getattr__(self, name):
        attr = getattr(self._sp, name)
        if name in ("game", "root_value_stats", "root_visits", "root_extra", "last_move", "play_selection_values", "root_children", "root_row", "komi_values", "game_setups", "root_raw_policy_entropy"):
            def counted(*a, **k):
                out = attr(*a, **k)
                self.d2h += _nbytes(out)
                return out
            return counted
        if name == "release":
            def released(mask=None):
                self.h2d += 0 if mask is None else int(np.asarray(mask).nbytes)
                return attr(mask)
            return released
        return attr


def _nbytes(x):
    if isinstance(x, np.ndarray):
        return int(x.nbytes)
    if isinstance(x, dict):
        return sum(_nbytes(v) for v in x.values())
    if isinstance(x, (tuple, list)):
        return sum(_nbytes(v) for v in x)
    return 8 if isinstance(x, (int, float, bool)) else 0


DUMP_MAX_GAMES = 256


def dump_outputs(sp, out_dir, world):
    """What a caller of the device loop reads back after its last wave: per game the root's children (visits, prior policy, utility),
    their value statistics, the root's own, the board and game state, and the NN row the wave evaluated; plus the loop's counters.
    Integer and float32 arrays are written as float32 (exact: every count stays below 2^24), the loop's doubles as float64.  More than
    DUMP_MAX_GAMES games over all ranks: a fixed sample of each rank's games (seed 0), listed in games.npy, keeps the files of all
    ranks together near 14 MB."""
    n, keep = sp.num_games, max(1, DUMP_MAX_GAMES // world)
    games = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    cols = {k: [] for k in ("child_visits", "child_policy", "child_utility", "child_value_stats", "root_value_stats", "board", "game_info",
                            "nn_row_spatial", "nn_row_global")}
    for g in games:
        visits, policy, util = sp.root_children(int(g))
        ch, rt = sp.root_value_stats(int(g))
        colors, info = sp.game(int(g))
        spatial, glob = sp.nn_row(int(g))
        for k, v in (("child_visits", visits), ("child_policy", policy), ("child_utility", util), ("child_value_stats", ch), ("root_value_stats", rt),
                     ("board", colors), ("game_info", list(info.values())), ("nn_row_spatial", spatial), ("nn_row_global", glob)):
            cols[k].append(v)
    out = {k: np.asarray(v, np.float64 if k in ("child_utility", "child_value_stats", "root_value_stats") else np.float32) for k, v in cols.items()}
    out["games"] = games.astype(np.float32)
    out["root_visits"] = sp.root_visits()[games].astype(np.float32)
    out["nn_symmetries"] = sp.nn_symmetries()[games].astype(np.float32)
    out["stats"] = np.array(list(sp.stats().values()), np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from katago_b200 import NeuralNet, SelfPlay, load_library, modelgen

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    path = model_file(args.model, rank)
    lib = load_library()
    model = NeuralNet.loadModelFile(path)
    ctx = NeuralNet.createComputeContext([local_rank], 19, 19, not args.fp32, model)
    n = args.games
    handle = NeuralNet.createComputeHandle(ctx, model, n, False, True, local_rank)
    bcast = broadcast_weights(handle, model, rank, world, device) if world > 1 else None
    bcast_ms = bcast["ms"] if bcast else 0.0
    macs = model.desc["conv_macs_per_position"]
    flop_per_eval = 2.0 * macs * 361

    # distinct input batches: 16 x 8.1 MB = 130 MB of feature rows > 126 MB L2, rotated every step
    NBUF = 16
    host_sp, host_gl = [], []
    for b in range(NBUF):
        sp, gl = modelgen.synthetic_inputs(n, 19, 19, seed=1000 * rank + b)
        host_sp.append(torch.from_numpy(sp.reshape(n, -1)).pin_memory())
        host_gl.append(torch.from_numpy(gl).pin_memory())
    dev_sp = [t.to(device) for t in host_sp]
    dev_gl = [t.to(device) for t in host_gl]
    sym = torch.from_numpy((np.arange(n) % 8).astype(np.int32))
    opt = torch.zeros(n, dtype=torch.float32)
    dsym, dopt = sym.to(device), opt.to(device)
    dpol = torch.empty((n, 362), device=device); dval = torch.empty((n, 3), device=device)
    dsc = torch.empty((n, 6), device=device); down = torch.empty((n, 361), device=device)
    hpol = np.empty((n, 362), np.float32); hval = np.empty((n, 3), np.float32); hsc = np.empty((n, 6), np.float32); hown = np.empty((n, 361), np.float32)
    stream = torch.cuda.ExternalStream(handle.stream, device=device)

    def step_device(i):
        b = i % NBUF
        rc = lib.kgb_forward_device(handle._p, n, dev_sp[b].data_ptr(), dev_gl[b].data_ptr(), dsym.data_ptr(), dopt.data_ptr(),
                                    dpol.data_ptr(), dval.data_ptr(), dsc.data_ptr(), down.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.kgb_last_error().decode())

    def step_host(i):
        b = i % NBUF
        rc = lib.kgb_forward(handle._p, n, host_sp[b].data_ptr(), host_gl[b].data_ptr(), sym.data_ptr(), opt.data_ptr(),
                             hpol.ctypes.data, hval.ctypes.data, hsc.ctypes.data, hown.ctypes.data)
        if rc != 0:
            raise RuntimeError(lib.kgb_last_error().decode())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        handle.sync()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    W, K = max(3, args.warmup), args.steps
    # device-resident self-play loop: selfplay8mainb18.cfg search parameters that the loop implements (DESIGN.md §8)
    sp_kwargs = dict(komi=7.5, multi_stone_suicide_legal=True, early_temperature_moves=30,
                  cpuct_exploration=1.05, cpuct_exploration_log=0.28, cpuct_exploration_base=500.0, fpu_reduction_max=0.2,
                  root_fpu_reduction_max=0.0, value_weight_exponent=0.5, fpu_parent_weight_by_visited_policy=True,
                  fpu_parent_weight_by_visited_policy_pow=2.0, root_desired_per_child_visits_coeff=2.0,
                  subtree_value_bias_factor=0.30, subtree_value_bias_weight_exponent=0.8, use_graph_search=True, graph_search_rep_bound=11,
                  root_noise_enabled=True, root_dirichlet_noise_total_concentration=10.83, root_dirichlet_noise_weight=0.25,
                  root_policy_temperature=1.1, root_policy_temperature_early=1.5, chosen_move_temperature_halflife=19.0,
                  nn_cache_size_power_of_two=args.nn_cache_pow2, root_num_symmetries_to_sample=4, root_ending_bonus_points=0.5, root_prune_useless_moves=True, ko_rule=0, full_history_rules=True,
                  use_play_selection=True, use_lcb_for_selection=True, use_non_buggy_lcb=True, lcb_stdevs=5.0, min_visit_prop_for_lcb=0.15,
                  chosen_move_temperature=0.15, chosen_move_temperature_early=0.75, chosen_move_subtract=0.0, chosen_move_prune=1.0,
                  seed=1234 + rank, ladder_nodes_per_wave=args.ladder_nodes_per_wave, max_playouts_per_wave=args.max_playouts_per_wave,
                  static_score_utility_factor=0.05, dynamic_score_utility_factor=0.30, dynamic_score_center_zero_weight=0.25,
                  dynamic_score_center_scale=0.50, draw_equivalent_wins_for_white=0.5)
    sp = SelfPlay(handle, n, args.visits, **sp_kwargs)
    mixed_rng = np.random.default_rng(99 + rank)

    def mixed_setups(loop):
        """--mixed-sizes: what GameInitializer draws with bSizes = 9,13,19 and equal bSizeRelProbs; the slots' next games get a second draw."""
        if not args.mixed_sizes:
            return None
        def draw():
            e = mixed_rng.choice([9, 13, 19], size=n)
            return np.stack([e, e, np.zeros(n, np.int64), np.ones(n, np.int64)], 1).astype(np.int32)
        first = draw()
        loop.set_game_setup(first, also_current_games=True)
        loop.set_game_setup(draw())
        return {int(e): int((first[:, 0] == e).sum()) for e in (9, 13, 19)}
    mixed_counts = mixed_setups(sp)
    # steady state before timing: games at different stages, trees hundreds of nodes deep, cache filled by the previous moves
    sp.random_openings(args.opening_max)
    sp.run(W + args.settle_waves)
    handle.sync()
    before = sp.stats()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev = timed(lambda i: sp.run(1), K)
    clocks = sampler.stop() if rank == 0 else None
    after = sp.stats()
    if args.dump_outputs:
        dump_outputs(sp, os.path.join(args.dump_outputs, f"rank{rank}") if world > 1 else args.dump_outputs, world)
    # a wave delivers one evaluated leaf per game, except for games whose ladder searches are still running (stalled_waves);
    # under graph search a game can also finish extra playouts inside the wave on edges that only need to catch up
    done = after["total_visits"] - before["total_visits"]
    instant = after["instant_playouts"] - before["instant_playouts"]
    cache_hits = after["nn_cache_hits"] - before["nn_cache_hits"]
    assert (done - instant - cache_hits) + (after["stalled_waves"] - before["stalled_waves"]) == n * K, (before, after)
    visits_done = torch.tensor([float(done)], device=device)
    if world > 1:
        dist.all_reduce(visits_done, op=dist.ReduceOp.SUM)
    visits_done = float(visits_done.item())
    ms_nn = timed(step_device, K)
    s0 = sp.stats()
    ms_select, ms_backup = sp.time_tree_kernels(20)
    s1 = sp.stats()
    tree_depth = (s1["sum_leaf_depth"] - s0["sum_leaf_depth"]) / max(1, s1["total_visits"] - s0["total_visits"])
    for i in range(W):
        step_host(i)
    ms_e2e_nn = timed(step_host, K)
    assert np.isfinite(hpol).all() and np.isfinite(hval).all()
    launches_per_step = sp.launches_per_step
    sp.free()

    # ---- e2e: the repo's own data-producing path (what `python -m katago_b200.selfplay_cli -per-game-release` runs): the device loop in
    # hold mode + katago_b200.game_recorder.GameRecorder (every game is read back and released as soon as ITS search is finished) +
    # katago_b200.npz_writer.TrainingDataWriter writing .npz training files.  Host readbacks, target computation and file writing are
    # inside the timed region; a step is still one playout wave.
    from katago_b200.game_recorder import GameRecorder
    from katago_b200.npz_writer import RowRand, TrainingDataWriter
    sp_kwargs["debug_hold_at_max_visits"] = True
    sp2 = SelfPlay(handle, n, args.visits, **sp_kwargs)
    mixed_setups(sp2)
    sp2.random_openings(args.opening_max)
    slots = CountingSlots(sp2)
    out_dir = tempfile.mkdtemp(prefix=f"kgb_bench_tdata_rank{rank}_")
    writer = TrainingDataWriter(out_dir, 20000, 1.0, 19, f"bench:rank{rank}")
    rec = GameRecorder(slots, writer, 7.5, draw_equivalent_wins_for_white=0.5, policy_surprise_data_weight=0.5, value_surprise_data_weight=0.1,
                       weight_rand=RowRand(f"bench:rank{rank}:weights"))
    PUMP = 8
    settle = 0
    while settle < W + args.settle_waves:        # games at all stages of their searches, recorder warm
        rec.pump(PUMP)
        settle += PUMP
    handle.sync()
    rb0, moves0, games0, rows0 = sp2.stats(), rec.moves_recorded, rec.games_written, writer.row_count
    slots.d2h = slots.h2d = 0
    if rank == 0:
        sampler2 = ClockSampler(local_rank)
        sampler2.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for first in range(0, K, PUMP):
        rec.pump(min(PUMP, K - first))
    e1.record(stream)
    handle.sync()
    barrier()
    clocks_e2e = sampler2.stop() if rank == 0 else None
    ms_rec = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(ms_rec, op=dist.ReduceOp.MAX)
    ms_rec = float(ms_rec.item())
    rb1 = sp2.stats()
    rec_visits = torch.tensor([float(rb1["total_visits"] - rb0["total_visits"])], device=device)
    if world > 1:
        dist.all_reduce(rec_visits, op=dist.ReduceOp.SUM)
    rec_visits = float(rec_visits.item())
    rec_moves, rec_games, rec_rows = rec.moves_recorded - moves0, rec.games_written - games0, writer.row_count - rows0
    writer.flush_if_nonempty()
    rec_files = len([f for f in os.listdir(out_dir) if f.endswith(".npz")])
    sp2.free()

    # ---- the precision-compliant mode (north_star: logits within 1e-3 of fp32): the same loop on an fp32-equivalent handle (3-term split
    # fp16 on the tensor pipe, fp32 streams); N = 1 only, shorter settling (the wave time is dominated by the evaluator)
    value_fp32 = None
    if world == 1 and not args.fp32:
        ctx32 = NeuralNet.createComputeContext([local_rank], 19, 19, False, model)
        h32 = NeuralNet.createComputeHandle(ctx32, model, n, False, True, local_rank)
        kw32 = dict(sp_kwargs); kw32["debug_hold_at_max_visits"] = False
        sp32 = SelfPlay(h32, n, args.visits, **kw32)
        sp32.random_openings(args.opening_max)
        sp32.run(W + 60); h32.sync()
        s32a = sp32.stats()
        stream32 = torch.cuda.ExternalStream(h32.stream, device=device)
        a32, b32 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a32.record(stream32); sp32.run(K); b32.record(stream32); h32.sync()
        s32b = sp32.stats()
        value_fp32 = {"value": (s32b["total_visits"] - s32a["total_visits"]) / (a32.elapsed_time(b32) * 1e-3), "unit": UNIT, "ms_per_step": a32.elapsed_time(b32) / K,
                      "dtype": "f32-split3 (fp16 tensor pipe, fp32 accumulate and streams)", "tolerance": "logits within 1e-3 of the fp32 oracle (tests/test_gpu_nn_parity.py FP32_TOL)"}
        sp32.free(); h32.free(); ctx32.free()

    # ---- same-box GPU competitor (SURVEY.md 8d): the reference's own CUDA/cuDNN backend against libkgb200 through the same caller
    # (oracle/ref_nnloop_driver.cpp: NeuralNet::getOutput in a loop, host buffers, batch = games); N = 1, rank 0, if the binaries travelled
    competitor = None
    if world == 1 and rank == 0:
        competitor = {}
        for key, exe in (("reference_cuda_cudnn_backend", "kgref_nnloop_cuda"), ("libkgb200", "kgref_nnloop_b200")):
            binp = os.path.join(ROOT, "oracle", "_ref", exe)
            if not os.path.exists(binp):
                competitor[key] = "binary not built"
                continue
            try:
                r = subprocess.run([binp, path, str(n), "12", "0" if args.fp32 else "1", "1", "1"], capture_output=True, text=True, timeout=240)
                competitor[key] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else "failed: " + (r.stderr or r.stdout)[-200:]
            except Exception as e:       # the competitor is context, not the measurement
                competitor[key] = "failed: " + str(e)[:200]
        competitor["what"] = "ms per NeuralNet::getOutput at batch = games, host buffers in and out, identical caller code linked against either backend"

    total_games = n * world
    value = visits_done / (ms_dev * 1e-3)      # playouts actually completed by all ranks / max-over-ranks device time
    e2e_nn_value = total_games * K / (ms_e2e_nn * 1e-3)
    h2d_nn = n * (22 * 361 + 19 + 2) * 4
    d2h_nn = n * (362 + 3 + 6 + 361) * 4
    e2e_value = rec_visits / (ms_rec * 1e-3)

    if rank == 0:
        peaks = load_peaks()
        # roofline of the dominant kernel: the 3x3 trunk convolution (mid x mid channels, M = games*(19+1)^2 padded rows),
        # timed alone with CUDA events inside the library on its launching stream.
        mid = {"b18c384nbt": 192, "b28c512nbt": 256}.get(args.model, 192)
        ms_conv = (np.zeros(1, np.float32))
        import ctypes as C
        # epilogue kind 1 = the first conv of a residual unit (BN + mish + mask -> fp16); 4 rotating buffer sets (4 x 79 MB in + out > L2)
        rc = lib.kgb_bench_conv_ex(3, 3, mid, mid, n, 19, 19, 0 if args.fp32 else 1, 1, 4, 5, 48, ms_conv.ctypes.data_as(C.POINTER(C.c_float)))
        if rc != 0:
            raise RuntimeError(lib.kgb_last_error().decode())
        conv_flop = 2.0 * 9 * mid * mid * 361 * n  # algorithmic: direct convolution over the 361 real board points
        achieved = conv_flop / (float(ms_conv[0]) * 1e-3) / 1e12
        whole = flop_per_eval * n * K / (ms_nn * 1e-3) / 1e12
        cpu_obj = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "measured at N=1 only"}
        if world == 1 and not os.path.exists(CPU_SELFPLAY):       # the CPU arm links the reference's sources: built only where they are present
            cpu_obj["sample"] = "not measured: oracle/_ref/kgref_cpu_selfplay is not built"
        elif world == 1:      # the CPU baseline is a property of the box: measured at N=1 only
            cpu_obj = cpu_baseline_object(cpu_selfplay(args.model, 15.0, 5.0, args.visits), args.model)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32-split3(fp16 tensor pipe)" if args.fp32 else "f16 (fp32 accumulate)", "data": "synthetic",
            "config": {"workload": (f"mixed 9x9 / 13x13 / 19x19 boards ({mixed_counts} games at the start) in a 19x19 evaluator frame, per-board masking, "
                                    if args.mixed_sizes else "19x19 ") +
                                   f"{args.model}, {n} concurrent games per GPU, maxVisits {args.visits}, one playout (visit) per game per step, device-resident loop",
                       "stages": ["root_move+tree_reset", "puct_select", "board_playmove(bitboard)", "featurize(all 22 V7 planes incl. ladders 14-17 and pass-alive area 18-19, 19 globals)",
                                  "nn_eval", "policy/value/score postprocess", "utility (win/loss + static/dynamic score utility)",
                                  "backup = recomputeNodeStats per path node (value weighting, exponent 0.5)"],
                       "search_params": "selfplay8mainb18.cfg: cpuct 1.05/0.28/500, fpu 0.2 (root 0), fpuParentWeightByVisitedPolicy^2, valueWeightExponent 0.5, "
                                        "score utility 0.05/0.30/0.25/0.50, rootDesiredPerChildVisitsCoeff 2, subtreeValueBias 0.30/0.8, useGraphSearch (repBound 11), root Dirichlet noise 10.83/0.25, root policy temperature 1.1 (early 1.5), move choice by play selection values with LCB 5.0/0.15 and chosenMoveTemperature 0.75->0.15; rootNumSymmetriesToSample 4; rootEndingBonusPoints 0.5, rootPruneUselessMoves",
                       "rules": "area scoring, simple ko with BoardHistory's game-end rules (two passes, spight-like ending pass, third repetition = no result), multi-stone suicide legal, komi 7.5 (positional / situational / spight superko available via ko_rule; territory scoring and encore not built)",
                       "games_per_gpu": n, "parallelism": f"games sharded over {world} GPU(s), no data-path collective",
                       "weights": "random init, real architecture (katago_b200/modelgen.py)",
                       "positions": f"every game starts from its own random legal play-out of 0..{args.opening_max} moves, then {W + args.settle_waves} untimed waves",
                       "l2": "per-step working set (tree arrays ~1 GB + activations ~0.5 GB) far larger than the 126 MB L2; "
                             f"e2e rotates {NBUF} distinct feature batches ({NBUF * n * 22 * 361 * 4 / 1e6:.0f} MB)",
                       "avg_leaf_depth": (after["sum_leaf_depth"] - before["sum_leaf_depth"]) / max(1, after["total_visits"] - before["total_visits"]),
                       "nn_only_ms_per_step": ms_nn / K,
                       "max_playouts_per_wave": args.max_playouts_per_wave,
                       "ladder": {"nodes_per_warp_per_wave": args.ladder_nodes_per_wave,
                                  "searches": after["ladder_searches"] - before["ladder_searches"],
                                  "search_moves": after["ladder_nodes"] - before["ladder_nodes"],
                                  "game_waves_without_leaf": after["stalled_waves"] - before["stalled_waves"],
                                  "playouts_without_evaluation(graph search catch-up)": instant,
                                  "playouts_served_by_nn_cache": cache_hits, "nn_cache_entries": (1 << args.nn_cache_pow2) if args.nn_cache_pow2 > 0 else 0,
                                  "game_waves": n * K},
                       "weight_broadcast_ms": bcast_ms, "weight_broadcast": bcast, "gpu_competitor": competitor},
            "value_fp32_equivalent": value_fp32,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": slots.h2d / K, "d2h_bytes_per_step": slots.d2h / K,
                    "ms_per_step": ms_rec / K,
                    "what": "device loop in hold mode + GameRecorder.pump (per-game release every 8 waves: root readback, training targets) + TrainingDataWriter "
                            ".npz files; host work inside the timed region; a step = one playout wave (the wave in which released games move is extra)",
                    "moves_recorded": rec_moves, "games_finished": rec_games, "rows_written": rec_rows, "npz_files": rec_files, "frac_of_value": e2e_value / value,
                    "clocks": clocks_e2e},
            "e2e_nn_boundary": {"value": e2e_nn_value, "unit": UNIT, "h2d_bytes_per_step": h2d_nn, "d2h_bytes_per_step": d2h_nn, "ms_per_step": ms_e2e_nn / K,
                                "what": "NeuralNet::getOutput -> kgb_forward with host buffers (boundary 1): one evaluated row = one visit of a host-side search"},
            "gpu_launches": launches_per_step * K,
            "roofline": {"bound": "tensor", "kernel": f"{'kgb_conv_tc_kernel (3-term split)' if args.fp32 else 'kgb_conv_tc3_kernel'} 3x3 {mid}->{mid}, batch {n}, 4 rotating buffer sets", "achieved": achieved,
                         "peak": peaks["tflops_burst"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops_burst"],
                         "traffic": 42.4e6 if args.model == "b18c384nbt" and n == 256 and not args.fp32 else None,   # dram read 40.45 MB + write 1.93 MB per launch (profiles/r02_conv_ncu_raw.md)
                         "peak_source": peaks["source"] + " (burst cuBLAS bf16, kernel timed alone)",
                         "ms_per_launch": float(ms_conv[0]),
                         "whole_forward_tflops": whole, "whole_forward_frac_of_sustained": whole / peaks["tflops_sustained"]},
            # tree / board kernels: HBM-bound byte work.  Algorithmic bytes per playout (DESIGN.md §4): every node on the descent
            # path reads its policy/childNode/childVisits/childUtilSum arrays (362 x 20 B); the leaf initialises its arrays
            # (362 x 20 B written), writes the NN row (22*361+19 floats, zero-fill + ones) and the legality mask; the backup reads
            # 362 logits, writes 362 policy floats and updates 2 x 12 B + 2 x 12 B per path node.
            "roofline_tree": (lambda bytes_sel, bytes_bak: {
                "bound": "hbm", "kernel": "spSelectKernel (one 8-warp block per game) + spBackupKernel (one warp per game)",
                "achieved": (bytes_sel + bytes_bak) * n / ((ms_select + ms_backup) * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": (bytes_sel + bytes_bak) * n / ((ms_select + ms_backup) * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "ms_select": ms_select, "ms_backup": ms_backup, "avg_depth": tree_depth,
                "bytes_per_playout": bytes_sel + bytes_bak,
                "traffic": 13.2e6 if args.model == "b18c384nbt" and n == 256 and not args.mixed_sizes else None,   # DRAM bytes per wave, both kernels: ncu dram__bytes_read + write (profiles/r02_tree_kernels_ncu_summary.md)
                "note": "latency-bound at 256 warps per launch (1.7 warps per SM); see DESIGN.md §6"})(
                    tree_depth * 362 * 20 + 362 * 20 + (22 * 361 + 19) * 4 * 2 + 128, 362 * 8 + tree_depth * 48 + 64),
            "cpu_baseline": cpu_obj,
            "clocks": clocks,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
