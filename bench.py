#!/usr/bin/env python
"""bench.py — MCTS simulations/s of the B200 self-play hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference ...                      CPU arm: the reference's OWN `run.py self` plumbing on host cores

A "step" is one move of self-play for every concurrent game: a full PUCT search (sims/move simulations per game,
tree walk + leaf evaluation by the residual network + backup, all on the device) followed by the on-device move
selection / adjudication.  Workload = BASELINE.json configs[2] (the one the metric is quoted on: 1024 concurrent
games per GPU, 800 sims/move, 20x256 resnet, random-init weights, games from INIT_STATE; weak scaling: every rank
runs its own 1024 games).  Prints ONE JSON line on rank 0; at N = 1 that line also carries `secondary` (short runs of
BASELINE configs[1] and configs[4], each with its own roofline) and `cpu_baseline`.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (games per GPU, sims/move, filters, blocks)
    "c3": (1024, 800, 256, 20),     # BASELINE.json configs[2]/[3] (per GPU)
    "c2": (256, 200, 128, 7),       # BASELINE.json configs[1]
    "c5": (800, 1600, 256, 20),     # BASELINE.json configs[4]: arena, 400 paired games = 800 player slots, two networks
    "tiny": (32, 40, 64, 2),        # plumbing check
}
CONFIG_INDEX = dict(c2=1, c3=2, c5=4)

# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) per launch of the dominant kernel from `ncu --set full` (None where no
# capture exists).  c3, 8192-board launches (profiles/r02i_conv_256_ncu_raw_subset.csv): conv1 (k_igemm3, fp16 in / out)
# 0.332 + 0.290 GB, conv2 (k_igemm2, + fp32 skip in / fp32 copy out) 1.399 + 0.943 GB; mean of the two = one launch of the
# tower on average.  Algorithmic bytes: 0.754 GB and 2.264 GB (conv1 reads part of its input from L2: 126 MB of the 377 MB
# the previous launch wrote).  c2, 2048-board launches (r02i_conv_128_*): 0.057 / 0.118 GB (activations are L2-resident).
NCU_TRAFFIC = {("c3", 1024, 8): 1.482e9, ("c2", 256, 8): 0.0875e9}


def net_flops(filters, blocks):
    return 2 * 90 * (350 * filters + blocks * 18 * filters * filters + 6 * filters) + 2 * (360 * 2086 + 180 * 256 + 256)


def workload_text(name, games, sims, filters, blocks):
    return (f"{name} = BASELINE.json configs[{CONFIG_INDEX.get(name, '-')}]: {games} concurrent "
            f"{'player slots (arena)' if name == 'c5' else 'games'}/GPU, {sims} sims/move, {filters}x{blocks} resnet")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1428.0))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
# The reference's own plumbing (oracle/ref_selfplay_bench.py: unmodified self_play.start -> SelfPlayWorker / CChessPlayer <->
# Pipe <-> CChessModelAPI thread, byte-compiled from /root/reference into oracle/_ref by __graft_entry__.build()).  The ONE
# prediction thread of the reference is its bottleneck on a CPU, so it gets half of the host threads as torch intra-op
# threads and the player processes a quarter (they mostly wait on their pipes); both numbers are reported.
def cpu_layout():
    cores = os.cpu_count() or 1
    procs = int(os.environ.get("CZ_BENCH_CPU_PROCS", max(1, cores // 4)))
    nn_threads = int(os.environ.get("CZ_BENCH_CPU_NN_THREADS", max(1, cores // 2)))
    return cores, procs, nn_threads


def ref_conf(sims, filters, blocks, k):
    play = {"simulation_num_per_move": sims, "search_threads": k, "c_puct": 1.5, "noise_eps": 0.15, "dirichlet_alpha": 0.2,
            "tau_decay_rate": 0.9, "virtual_loss": 3, "resign_threshold": -0.98, "enable_resign_rate": 0.5, "min_resign_turn": 40,
            "max_game_length": 100}
    model = {"cnn_filter_num": filters, "res_layer_num": blocks, "value_fc_size": 256}
    return play, model


def reference_windows(sims, filters, blocks, k, n_windows, window_s, warm_windows=0, free_nn=False, config_type="normal"):
    """Runs the reference self-play ONCE (persistent process pool) and samples it in windows.
    Returns (list of (sims, positions, batches, seconds), description, threads used, kind)."""
    from oracle import ref_selfplay_bench as rb
    cores, procs, nn_threads = cpu_layout()
    play, model = ref_conf(sims, filters, blocks, k)
    if not rb.available():
        return None, "oracle/_ref not built", 0, "port"
    run = rb.ReferenceSelfPlay(config_type, procs, 1 if free_nn else nn_threads, play=play, model=model, free_nn=free_nn)
    try:
        run.wait_started(timeout=600.0, min_sims=max(1, procs))
        run.window(float(os.environ.get("CZ_BENCH_CPU_SETTLE", 8.0)))      # every process past its first batches before anything counts
        for _ in range(warm_windows):
            run.window(window_s)
        wins = [run.window(window_s) for _ in range(n_windows)]
    finally:
        run.close()
    used = procs + (0 if free_nn else nn_threads)
    return wins, rb.describe(play, model, procs, nn_threads, free_nn), used, "reference"


def port_sample(filters, blocks, sims, k, budget_s):
    """Fallback when oracle/_ref is absent (a checkout that never saw /root/reference): the oracle port, one process per core."""
    from oracle import cpu_baseline
    cores = os.cpu_count() or 1
    rate, n, dt, _ = cpu_baseline.run(filters, blocks, sims, k, budget_s, cores)
    return rate, n, dt, cores


def cpu_baseline_block(filters, blocks, sims, k, seconds):
    wins, desc, used, kind = reference_windows(sims, filters, blocks, k, 1, seconds)
    if wins is None:
        rate, n, dt, cores = port_sample(filters, blocks, sims, k, seconds)
        return {"value": rate, "unit": "sims/s", "cores": cores, "kind": "port",
                "sample": f"oracle/_ref missing -> oracle port (agent/player.py + static_env.py restated), {cores} single-threaded "
                          f"processes, {n} simulations in a {dt:.1f} s window"}
    s, p, b, dt = wins[0]
    return {"value": s / dt, "unit": "sims/s", "cores": used, "kind": kind, "positions_per_s": p / dt, "mean_batch": p / max(1, b),
            "sample": f"{desc}; one {dt:.0f} s window after start-up ({s} simulations)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    games, sims, filters, blocks = WORKLOADS[args.workload]
    K = args.leaves
    cores, procs, nn_threads = cpu_layout()
    # total timed span >= 60 s (BASELINE.md §3.4) split into `steps` windows; the whole run stays within a few minutes
    window = float(os.environ.get("CZ_BENCH_CPU_WINDOW", max(3.0, 60.0 / max(1, args.steps))))
    load0 = os.getloadavg()[0]          # runnable tasks on the box BEFORE this arm starts: the boxes of the pool are shared, and the
                                        # rates of the same plumbing differed 4x between boxes (56 ... 221 sims/s, profiles/README.md)
    wins, desc, used, kind = reference_windows(sims, filters, blocks, K, args.steps, window, warm_windows=args.warmup)
    load1 = os.getloadavg()[0]
    extra = {}
    if wins is None:
        vals = [port_sample(filters, blocks, sims, K, window) for _ in range(max(1, min(args.steps, 4)))]
        tot_n, tot_t = sum(v[1] for v in vals), sum(v[2] for v in vals)
        value, used, kind = sum(v[0] for v in vals) / len(vals), vals[0][3], "port"
        desc = "oracle/_ref missing -> oracle port (agent/player.py + static_env.py restated), one single-threaded process per core"
        per_window = [v[0] for v in vals]
    else:
        tot_n, tot_t = sum(w[0] for w in wins), sum(w[3] for w in wins)
        value = tot_n / tot_t
        per_window = [w[0] / w[3] for w in wins]
        extra["nn_positions_per_sec"] = sum(w[1] for w in wins) / tot_t
        extra["mean_batch"] = sum(w[1] for w in wins) / max(1, sum(w[2] for w in wins))
        if not args.no_secondary:
            # BASELINE.json configs[0]: `run.py self --type mini --new` as shipped (1 process, 10 threads, 100 sims, 256x7)
            # one player process whose batches are <= 10 positions: more than one intra-op thread only oversubscribes (BASELINE.md
            # section 4: 70.9 sims/s with OMP_NUM_THREADS=1 vs 9.2 with 8 threads on the survey box)
            saved = {k: os.environ.get(k) for k in ("CZ_BENCH_CPU_PROCS", "CZ_BENCH_CPU_NN_THREADS")}
            os.environ["CZ_BENCH_CPU_PROCS"], os.environ["CZ_BENCH_CPU_NN_THREADS"] = "1", "1"
            w1, d1, u1, _ = reference_windows(100, 256, 7, 10, 1, 30.0, config_type="mini")
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
            extra["c1_mini"] = {"value": w1[0][0] / w1[0][3], "unit": "sims/s", "cores": u1, "positions_per_s": w1[0][1] / w1[0][3],
                                "mean_batch": w1[0][1] / max(1, w1[0][2]), "sample": d1 + f"; one {w1[0][3]:.0f} s window"}
            # tree-code ceiling: the same plumbing with a constant-output network (BASELINE.md §3.5)
            w2, d2, u2, _ = reference_windows(sims, filters, blocks, K, 1, 20.0, free_nn=True)
            extra["free_nn_ceiling"] = {"value": w2[0][0] / w2[0][3], "unit": "sims/s", "cores": u2,
                                        "sample": d2 + f"; one {w2[0][3]:.0f} s window of a separate run of the plumbing (on a shared box its rate moves with the host load, like the main windows)"}
    sample = f"{desc}; {len(per_window)} windows of {window:.1f} s after {args.warmup} warm-up windows ({tot_n} simulations in {tot_t:.0f} s)"
    line = {
        "impl": "reference", "metric": "mcts_sims_per_sec", "value": value, "unit": "sims/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, len(per_window)), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init Keras-equivalent weights, games from INIT_STATE)",
        "config": bench_config(args.workload, games, sims, filters, blocks, K, args.gpus, args.skip_stream),
        "cpu_baseline": {"value": value, "unit": "sims/s", "cores": used, "kind": kind, "sample": sample,
                         "host_cores": cores, "max_processes": procs, "nn_threads": nn_threads,
                         "window_rates": [round(v, 2) for v in per_window],
                         "host_loadavg_1min": {"before": round(load0, 1), "at_end_of_windows": round(load1, 1)}},
        "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    line.update(extra)
    print(json.dumps(line))
    return 0


def conv_kernel_names(filters):
    """The residual-conv kernels cz_nn.cu's launch selection runs at this width (use_tma_epilogue_for): all-TMA-epilogue pair kernel,
    two M-tiles per CTA at C <= 128; the fp32-skip conv2 of the 256-wide tower keeps the round-1 pair kernel."""
    if filters <= 128:
        return f"igemm::k_igemm3<{filters}, 2> (3x3 residual conv, tcgen05 cta_group::2, two M-tiles per CTA)"
    if filters >= 256:
        return (f"igemm::k_igemm3<{filters}, 1> (conv1) + igemm::k_igemm2<{filters}> (conv2, fp32 skip stream): 3x3 residual conv, "
                "tcgen05 cta_group::2")
    return f"igemm::k_igemm3<{filters}, 1> (3x3 residual conv, tcgen05 cta_group::2)"


def bench_config(workload, games, sims, filters, blocks, K, world=1, skip_stream="auto"):
    """The `config` object BOTH arms print — identical, key for key, so that the driver's same-config check can compare them
    (what differs between runs — games finished, records gathered, gather time — is in `run_info`)."""
    act_mb = games * K * 90 * filters * 2 * 3 / 1e6
    return {"workload": workload_text(workload, games, sims, filters, blocks), "games_per_gpu": games, "sims_per_move": sims,
            "leaves_per_round": K, "net": f"{filters}x{blocks}", "skip_stream": skip_stream,
            "parallelism": f"dp{world} (games sharded, no data-path collective; finished-game rings all_gathered every step)",
            "l2": (f"GPU arm: activations {act_mb:.0f} MB per round + tree pools stream through HBM (> 126 MB L2, no flush needed)"
                   if act_mb > 2 * 126 else
                   f"GPU arm: activations {act_mb:.0f} MB per round fit the 126 MB L2 and are NOT flushed between steps (secondary "
                   f"workload; the headline workload c3 streams 1.1 GB per round)")}


# ------------------------------------------------------------------------------------------------ our arm
def make_worker(workload, games, sims, filters, blocks, K, rank, seed, skip_stream, nodes, data_dir, lib, max_game_length=100):
    """The drop-in SelfPlayWorker (cczero_b200/self_play.py) on this rank's GPU: it owns the engine the bench times."""
    from types import SimpleNamespace
    from cczero_b200.model import CChessModel
    from cczero_b200.self_play import SelfPlayWorker
    play = SimpleNamespace(max_processes=1, simulation_num_per_move=sims, search_threads=K, virtual_loss=3, c_puct=1.5, noise_eps=0.15,
                           dirichlet_alpha=0.2, tau_decay_rate=0.9, resign_threshold=-0.98, enable_resign_rate=0.5, min_resign_turn=40,
                           max_game_length=max_game_length)
    mc = SimpleNamespace(cnn_filter_num=filters, res_layer_num=blocks, value_fc_size=256, cnn_first_filter_size=5, cnn_filter_size=3,
                         input_depth=14)
    cfg = SimpleNamespace(play=play, model=mc, play_data=SimpleNamespace(nb_game_in_file=1),
                          resource=SimpleNamespace(play_data_dir=data_dir, play_data_filename_tmpl="play_%s.json"))
    model = CChessModel(cfg)
    model.build(seed=0)                      # random-init, Keras-equivalent (agent/model.py:32-66 defaults)
    w = SelfPlayWorker(cfg, pid=rank, model=model, concurrent_games=games, lib=lib, seed=seed, rank=rank,
                       engine_kwargs=dict(max_nodes_per_game=nodes or max(4096, 24 * sims), arena=workload == "c5",
                                          nn_fp32_skip={"auto": None, "fp32": True, "fp16": False}[skip_stream]))
    if workload == "c5":                     # the arena's second network (next generation): another random init
        model2 = CChessModel(cfg)
        model2.build(seed=1)
        w.engine.set_weights(model2.torch_weights(), net=1)
        w.engine.reset()
    return w


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 128          # np.save's header for these arrays (format 1.0, padded to 64 bytes; shapes of <= 3 numbers)


def dump_outputs(eng, out_dir, last_step, records, seed=0):
    """Writes what a caller of the timed path (Engine.selfplay, one move of every game) holds after its last step, as
    float64 .npy files: the step's (simulations, games finished); the games that step finished (finished_games: game
    index, plies, value for red, flags; finished_moves: their moves as cz move codes, -1 past the last ply); and per game
    the root position the move led to, the simulations its search ran, and the visit counts of the new root's moves.
    Everything stays within DUMP_LIMIT_BYTES: beyond it a seeded sample of the games (indices in game_index.npy) and of the
    finished games is written."""
    import numpy as np
    from cczero_b200 import records as rec
    from cczero_b200.env import move_to_u16
    rng = np.random.default_rng(seed)
    stage = rec.RootStage(eng)
    visits, moves, counts = eng.download_root_stats(stage)
    per_game = {"root_boards": eng.download_roots(stage), "root_visits": visits, "root_moves": moves, "root_move_counts": counts,
                "sims_run": stage.sims, "active": eng.active_flags()}
    per_game = {k: np.asarray(v, dtype=np.float64).reshape(eng.n_games, -1) for k, v in per_game.items()}
    plies = eng.cfg.max_plies
    records = sorted(records, key=lambda r: r["game_index"])   # the ring's order follows the warps' finishing race
    fin = np.array([[r["game_index"], r["n_plies"], r["value_red"], r["flags"]] for r in records], dtype=np.float64).reshape(-1, 4)
    fin_moves = np.full((len(records), plies), -1.0)
    for i, r in enumerate(records):
        fin_moves[i, :len(r["moves"])] = [move_to_u16(m) for m in r["moves"]]
    budget = DUMP_LIMIT_BYTES - (len(per_game) + 4) * NPY_HEADER_BYTES - 2 * 8
    rec_bytes = (4 + plies) * 8
    if len(records) * rec_bytes > budget // 2:                 # finished games get at most half of the budget
        keep = np.sort(rng.choice(len(records), budget // 2 // rec_bytes, replace=False))
        fin, fin_moves = fin[keep], fin_moves[keep]
    budget -= fin.nbytes + fin_moves.nbytes
    game_bytes = sum(v[0].nbytes for v in per_game.values()) + 8  # + its entry in game_index
    idx = np.arange(eng.n_games)
    if eng.n_games * game_bytes > budget:
        idx = np.sort(rng.choice(eng.n_games, budget // game_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    out = {"last_step": np.asarray(last_step, dtype=np.float64), "finished_games": fin, "finished_moves": fin_moves,
           "game_index": idx.astype(np.float64)}
    out.update({k: v[idx] for k, v in per_game.items()})
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def measure(args, workload, steps, warmup, world, rank, local, dist, want_e2e=True, sample_clocks=True, dump_dir=None):
    """Device-resident timing (+ optional end-to-end timing) of one workload; returns a dict (rank 0) or None.
    dump_dir: where rank 0 writes the outputs of the last timed step (dump_outputs)."""
    import torch
    from cczero_b200 import records as rec
    from cczero_b200.lib import get_lib

    lib = get_lib()
    games, sims, filters, blocks = WORKLOADS[workload]
    if args.games and workload == args.workload:
        games = args.games
    if args.sims and workload == args.workload:
        sims = args.sims
    K = args.leaves
    data_dir = tempfile.mkdtemp(prefix=f"cz_bench_{workload}_")
    worker = make_worker(workload, games, sims, filters, blocks, K, rank, args.seed, args.skip_stream, args.nodes, data_dir, lib,
                         args.max_game_length)
    eng = worker.engine

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gather_ev = []
    last_records = []                   # the finished-game records of the latest step (rank 0)

    def step_device(warm=False):
        g, s = eng.selfplay(target_games=0, max_moves=1)
        n_rec = 0
        last_records.clear()
        if world > 1:          # the ONE collective of the path: finished-game rings -> rank 0, inside the timed region
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            recs, total = rec.gather_records(eng, dist, world, warm=warm)
            b.record()
            gather_ev.append((a, b))
            n_rec = total
            if recs:
                last_records.extend(rc for r, rc in recs)
                for r, rc in recs:
                    if not (rc["flags"] & 4):
                        worker.games_stored += 1
                        worker.save_play_data(worker.games_stored, rec.record_to_play_data(rc))
        elif g:
            # one GPU: nothing else empties the finished-game ring, and cz_selfplay plays no move while the ring could
            # overflow; draining it keeps every step one move of every game
            last_records.extend(eng.drain_records())
        return s, g, n_rec

    for _ in range(warmup):
        step_device(warm=True)
    gather_ev.clear()
    # ---- device-resident timing: the production path (cz_selfplay -> one WHILE-graph launch per search, no host in the loop)
    st0, c0 = eng.search_stats(), eng.counters()
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0 and sample_clocks:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sims_total, games_done, gathered = 0, 0, 0
    s = g = 0
    for _ in range(steps):
        s, g, nr = step_device()
        sims_total += s
        games_done += g
        gathered += nr
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - launches0
    st1, c1 = eng.search_stats(), eng.counters()
    if dump_dir and rank == 0:          # after the counters: its own kernel launches are not the timed path's
        dump_outputs(eng, dump_dir, (s, g), last_records, args.seed)
    gather_ms = sum(a.elapsed_time(b) for a, b in gather_ev)
    # ---- roofline region: the same steps with CUDA events bracketing every residual-tower launch group.  Events cannot live
    # inside the WHILE graph, so while cz_nn_profile is on the engine runs the same iteration as three sub-graphs (tree + first
    # conv | tower | heads) launched from the host with the event records in between: same kernels, same shapes, same stream.
    prof_steps = max(1, min(steps, 4))
    eng.nn_profile(True)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(prof_steps):
        step_device()
    p1.record()
    barrier()
    ms_prof = p0.elapsed_time(p1)
    clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
    conv_ms, conv_launches, conv_flops = eng.nn_profile(False)
    # ---- end-to-end timing through the drop-in worker with host buffers (SelfPlayWorker.host_step)
    ms_e2e, e2e_sims, h2d, d2h, files = 0.0, 0, 0, 0, 0
    if want_e2e:
        stage = rec.RootStage(eng)
        eng.download_roots(stage)                         # the host-held positions of the first e2e step
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stored0 = worker.games_stored
        e2.record()
        rec_bytes = 0
        for _ in range(steps):
            s, recs = worker.host_step(stage)
            e2e_sims += s
            rec_bytes += sum(16 + 2 * r["n_plies"] for r in recs)
        e3.record()
        barrier()
        ms_e2e = e2.elapsed_time(e3)
        h2d = stage.h2d_bytes
        d2h = stage.d2h_bytes + 4 * games + rec_bytes // max(1, steps)
        files = worker.games_stored - stored0

    t = torch.tensor([ms, ms_e2e, conv_ms, gather_ms, ms_prof], device="cuda", dtype=torch.float64)
    c = torch.tensor([sims_total, e2e_sims, launches, conv_launches, games_done, conv_flops], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    ms, ms_e2e, conv_ms, gather_ms, ms_prof = [float(x) for x in t.tolist()]
    sims_total, e2e_sims, launches, conv_launches, games_done, conv_flops = [float(x) for x in c.tolist()]
    out = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        achieved = (conv_flops / world) / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0   # conv_ms: max over ranks, flops: sum
        d_sims = max(1, st1["sims"] - st0["sims"])
        depth = (st1["path_edges"] - st0["path_edges"]) / d_sims
        legal = st1["edges_stored"] / max(1, st1["nodes_stored"])
        expand = (st1["nodes_created"] - st0["nodes_created"]) / d_sims
        live = games // 2 if workload == "c5" else games
        out = {
            "value": sims_total / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
            "config": bench_config(workload, games, sims, filters, blocks, K, world, args.skip_stream),
            "run_info": {"games_finished": int(games_done), "records_gathered": int(gathered), "gather_ms_per_step": gather_ms / steps,
                         "search_loop": os.environ.get("CZ_SEARCH_LOOP", "while (one graph launch per search)")},
            "nn_positions_per_sec": (st1["nodes_created"] - st0["nodes_created"]) * world / (ms * 1e-3),
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": NCU_TRAFFIC.get((workload, games, K)),
                         "kernel": conv_kernel_names(filters),
                         "launches": int(conv_launches), "avg_launch_ms": conv_ms / max(1.0, conv_launches / world),
                         "peak_source": peak_src, "share_of_step": conv_ms / ms_prof,
                         "measured_over": f"{prof_steps} further steps right after the {steps} timed ones, CUDA events around every tower "
                                          f"launch group on the engine's stream ({ms_prof / prof_steps:.1f} ms per step in this region)",
                         "whole_net_frac_of_step": (st1["nodes_created"] - st0["nodes_created"]) * net_flops(filters, blocks)
                                                   / (ms * 1e-3) / 1e12 / peak},
            "search_stats": {
                "mean_path_edges": depth, "mean_legal_moves": legal, "no_network_rate": (st1["no_network"] - st0["no_network"]) / d_sims,
                "expansions_per_sim": expand,
                "waves_per_move": float(c1[2] - c0[2]) / steps,
                "mean_reused_sims_per_move": sims - (st1["sims"] - st0["sims"]) / (steps * live),
                "compactions": int(c1[5] - c0[5]), "table_resets": int(c1[4] - c0[4]), "records_dropped": int(c1[3] - c0[3]),
                "error_flags": int(c1[6]),
                "tree_bytes_per_sim": depth * (32 + 14 * legal) + depth * 24 + depth * 90
                                      + expand * ((32 + 22 * legal) + 90 + 2 * legal + 96 + policy_bytes_per_leaf(legal)),
                "note": "algorithmic HBM bytes of the integer kernels per simulation (SURVEY.md section 8d): select reads + virtual-loss/"
                        "backup RMW + board replay per path edge; per expansion node+edge write, movegen, leaf record, and what k_apply "
                        "reads of the network output; compactions / table_resets / records_dropped counted over rank 0's timed region"},
            "clocks": clocks,
        }
        if want_e2e:
            out["e2e"] = {"value": e2e_sims / (ms_e2e * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                          "ms_per_step": ms_e2e / steps, "play_data_files_written": int(files),
                          "path": "SelfPlayWorker.host_step: pinned root upload -> cz_search -> visit counts down -> cz_play_move -> "
                                  "records drained + play-data JSON written -> new roots down"}
    worker.close()
    del worker, eng
    torch.cuda.empty_cache()
    return out


FUSED_POLICY = True      # flipped when the integrated search gathers legal logits itself (no [B][2086] f32 policy row)


def policy_bytes_per_leaf(legal):
    """What k_apply reads of the network output per expanded leaf: the 2086-entry f32 policy row k_softmax wrote, or — fused
    path — the legal logits (4 bytes each) plus the 9 per-tile softmax statistics (72 bytes)."""
    return (4 * legal + 72) if FUSED_POLICY else 4 * 2086


def uci_latency_block():
    """Single-game latency path (SURVEY §8f rank 4): `go depth 8` (800 simulations, search_threads 10) through the drop-in
    `CChessPlayer(uci=True)` on the reference's trained 192x10 weights (as the committed fixture rebuilds them), wall clock around `action()`, with the
    nps figure the REFERENCE's formula gives (agent/player.py:446-447).  tools/bench_uci.py is the measurement."""
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location("bench_uci", os.path.join(ROOT, "tools", "bench_uci.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        if not os.path.exists(os.path.join(ROOT, "tests", "golden", "model_best_192x10_compact.npz")):
            return {"error": "tests/golden/model_best_192x10_compact.npz missing"}
        weights, src = mod.load_weights(192, 10)
        keep = os.environ.get("CZ_SEARCH_LOOP")
        try:
            runs, info = mod.run(keep or "while", 192, 10, 8, 10, weights)
        finally:
            if keep is not None:
                os.environ["CZ_SEARCH_LOOP"] = keep
        best = min(runs[1:], key=lambda r: r["seconds"])
        return {"go": "depth 8 = 800 simulations, search_threads 10, one game", "net": "192x10", "weights": src,
                "ms": best["seconds"] * 1e3, "sims_per_s": best["sims_per_s"], "waves": best["waves"],
                "nps_reference_formula": best["nps_reference_formula"], "runs_ms": [r["seconds"] * 1e3 for r in runs],
                "last_info_line": info}
    except Exception as e:
        return {"error": repr(e)}


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    main = measure(args, args.workload, args.steps, args.warmup, world, rank, local, dist, dump_dir=args.dump_outputs)
    secondary = {}
    if world == 1 and not args.no_secondary and args.workload == "c3":
        # BASELINE.json configs[1] and configs[4], short, each with its own roofline (driver-visible; VERDICT r1 item 4)
        for name, st, wu in (("c2", 12, 4), ("c5", 2, 3)):
            try:
                m = measure(args, name, st, wu, world, rank, local, dist, want_e2e=False, sample_clocks=False)
                secondary[name] = {k: m[k] for k in ("value", "ms_per_step", "steps", "warmup", "config", "run_info", "nn_positions_per_sec",
                                                     "roofline", "search_stats", "gpu_launches")}
                secondary[name]["unit"] = "sims/s"
            except Exception as e:        # a secondary workload must never take the headline down with it
                secondary[name] = {"error": repr(e)}
        secondary["uci"] = uci_latency_block()
    if rank == 0:
        games, sims, filters, blocks = WORKLOADS[args.workload]
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline_block(filters, blocks, sims, args.leaves, args.cpu_seconds)
        line = {"metric": "mcts_sims_per_sec", "value": main["value"], "unit": "sims/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16", "data": "synthetic (random-init Keras-equivalent weights, games from INIT_STATE)",
                "config": main["config"], "run_info": main["run_info"], "nn_positions_per_sec": main["nn_positions_per_sec"], "e2e": main["e2e"],
                "gpu_launches": main["gpu_launches"], "roofline": main["roofline"], "cpu_baseline": cpu, "clocks": main["clocks"],
                "search_stats": main["search_stats"]}
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--leaves", type=int, default=8, help="simulations per game per round (reference search_threads)")
    ap.add_argument("--games", type=int, default=0)
    ap.add_argument("--sims", type=int, default=0)
    ap.add_argument("--nodes", type=int, default=0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--max-game-length", type=int, default=100, help="play_config.max_game_length (configs/normal.py: 100); smaller "
                    "values make games finish inside a short run so that the record gather / file writes carry data")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short c2 / c5 runs (and the c1 / free-NN legs of the CPU arm)")
    ap.add_argument("--skip-stream", default="auto", choices=["auto", "fp32", "fp16"],
                    help="precision of the residual skip stream (auto = fp32 beyond 10 blocks: keeps the 1e-3 parity bound)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB) for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
