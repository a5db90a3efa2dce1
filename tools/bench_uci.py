"""Single-game latency path: one `CChessPlayer(uci=True)` on the built-in network answering `go depth 8` (= 800 simulations,
uci.py:293-327 -> player.py:160-161), the way the reference's UCI front end drives its player.  Prints the wall time of the
search, simulations/s and the `nps` figure computed with the REFERENCE'S formula, nps = int(depth * 100 / duration) * 1000
(agent/player.py:446-447), for the device-driven loop in both forms (CZ_SEARCH_LOOP=while, the default: one graph launch per
slice of the search; =graph: three sub-graphs per iteration and a polled flag) and the round-1 host-driven loop (=host).

    python tools/bench_uci.py [filters blocks] [depth] [search_threads]
Weights: the reference's trained 192x10 network as tests/golden/model_best_192x10_compact.npz rebuilds it (real batch-norm
statistics and biases, kernels of the real per-channel scale) by default."""
import io
import json
import os
import sys
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np   # noqa: E402
import torch         # noqa: E402


def run(loop, filters, blocks, depth, k, weights):
    os.environ["CZ_SEARCH_LOOP"] = loop
    from cczero_b200.player import CChessPlayer
    from cczero_b200.env import INIT_STATE
    play = SimpleNamespace(simulation_num_per_move=800, search_threads=k, c_puct=1.5, noise_eps=0.15, dirichlet_alpha=0.2,
                           tau_decay_rate=0.9, virtual_loss=3, resign_threshold=-0.98, min_resign_turn=40, max_game_length=100)
    cfg = SimpleNamespace(play=play, model=SimpleNamespace(cnn_filter_num=filters, res_layer_num=blocks, value_fc_size=256, input_depth=14))
    p = CChessPlayer(cfg, uci=True, weights=weights, exact_noise=False, infinite_capacity=20000)
    os.environ.pop("CZ_SEARCH_LOOP", None)
    p.info_stream = io.StringIO()
    out = []
    state = INIT_STATE
    for rep in range(3):                                   # first call warms the kernels and captures the graphs
        p.engine.reset([state])
        p._fresh = False
        torch.cuda.synchronize()
        w0 = int(p.engine.counters()[2])
        t0 = time.perf_counter()
        action, _ = p.action(state, 0, depth=depth * 100)
        dt = time.perf_counter() - t0
        waves = int(p.engine.counters()[2]) - w0
        out.append({"seconds": dt, "sims": depth * 100, "sims_per_s": depth * 100 / dt, "waves": waves, "us_per_wave": 1e6 * dt / max(1, waves),
                    "nps_reference_formula": int(depth * 100 / dt) * 1000, "bestmove": action})
    last_info = p.info_stream.getvalue().strip().splitlines()[-1]
    p.close()
    return out, last_info


def load_weights(filters, blocks):
    from oracle import model as om
    npz = os.path.join(ROOT, "tests", "golden", "model_best_192x10_compact.npz")
    if (filters, blocks) == (192, 10) and os.path.exists(npz):
        return ({key: torch.as_tensor(v) for key, v in om.load_compact(npz).items()},
                "reference's trained 192x10 weights, rebuilt from tests/golden/model_best_192x10_compact.npz")
    return {key: torch.as_tensor(v) for key, v in om.init_weights(filters, blocks, 256, seed=0).items()}, "random-init weights"


def main():
    filters = int(sys.argv[1]) if len(sys.argv) > 2 else 192
    blocks = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    depth = int(sys.argv[3]) if len(sys.argv) > 3 else 8
    k = int(sys.argv[4]) if len(sys.argv) > 4 else 10      # configs/distribute.py: search_threads = 10
    weights, src = load_weights(filters, blocks)
    res = {"net": f"{filters}x{blocks}", "weights": src, "go": f"depth {depth} ({depth * 100} simulations), search_threads {k}"}
    for loop in os.environ.get("UCI_LOOPS", "while,graph,host").split(","):      # one WHILE-graph launch per slice (default) | three sub-graphs per iteration | round-1 host loop
        runs, info = run(loop, filters, blocks, depth, k, weights)
        res[loop] = {"best": min(runs[1:], key=lambda r: r["seconds"]), "runs": runs, "last_info_line": info}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
