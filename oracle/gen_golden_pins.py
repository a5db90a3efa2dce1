"""Fixture generator (needs the reference tree): what tests/test_oracle_vs_reference.py compares the oracle restatements
against, recorded from the REAL reference so that those comparisons run on any checkout.

  tests/golden/reference_pins.json.gz   rules answers of the real static_env on the test's playouts and arbitrary boards,
                                        FEN helpers, real-player searches (K = 1), real self-play / arena games, and the
                                        real EvaluateWorker's tally
  tests/golden/reference_pins.npz       the real trainer's expanding_data on one golden game (14 and 28 planes) and the
                                        outputs of the layer graph Keras wrote for the shipped networks

Inputs are generated exactly as the tests generate them (same seeds, same helpers), so each test replays its own inputs
and checks the oracle's answers against the recorded ones.  Planes are recorded as the SHA-1 of their float32 bytes.

    python -m oracle.gen_golden_pins
"""
import gzip
import hashlib
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
JSON_OUT = os.path.join(GOLD, "reference_pins.json.gz")
NPZ_OUT = os.path.join(GOLD, "reference_pins.npz")

# test_player_restatement_equals_real_player_k1
K1_CASES = ((80, 1), (150, 2))
# test_game_loop_restatements_replay_live_reference_games
LOOP_PLAY = dict(max_game_length=20, tau_decay_rate=0.98, noise_eps=0.25, enable_resign_rate=0.1, resign_threshold=-0.5, min_resign_turn=4)
LOOP_SELFPLAY_SEEDS = (41, 42)
LOOP_ARENA = ((43, 0), (44, 1))
LOOP_SIMS = 16
# test_evaluator_tally_matches_the_real_worker
TALLY_RESULTS = [1, -1, 0, 1, 1, -1, 0, 0, -1, 1, 1, -1]
FEN_CASES_STATE = '4s4/9/4e4/p8/2e2R2p/P5E2/8P/9/9/4S1E2'


def planes_digest(planes):
    return hashlib.sha1(np.ascontiguousarray(planes, dtype=np.float32).tobytes()).hexdigest()


def rules_row(r, s):
    """Every answer of the real static_env the rules pins compare, for one position."""
    return {"state": s, "legal": r.get_legal_moves(s), "done": list(r.done(s)), "done_check": list(r.done(s, need_check=True)),
            "planes": planes_digest(r.state_to_planes(s)), "attack": r.has_attack_chessman(s), "flipped": r.fliped_state(s)}


def move_row(r, s, m):
    return {"move": m, "new_step": r.new_step(s, m), "check_or_catch": r.will_check_or_catch(s, m), "catched": r.be_catched(s, m)}


def playouts(r):
    """test_env_restatement_on_random_playouts: 25 seeded random playouts of up to 200 plies."""
    rng = random.Random(7)
    games = []
    for g in range(25):
        s, rows = r.INIT_STATE, []
        for ply in range(200):
            row = rules_row(r, s)
            rows.append(row)
            if r.done(s)[0]:
                break
            m = rng.choice(row["legal"])
            row["move"] = m
            row["new_step"] = r.new_step(s, m)
            if ply % 2 == 0:
                row["check_or_catch"] = r.will_check_or_catch(s, m)
                row["catched"] = r.be_catched(s, m)
            s = r.step(s, m)
        games.append(rows)
    return games


def arbitrary_boards(r):
    """test_env_restatement_on_arbitrary_boards."""
    from tests.env_checks import EXTREME_STATES, random_boards
    rows = []
    for s in random_boards(600, 5) + [x for x in EXTREME_STATES if 's' in x and 'S' in x]:
        row = rules_row(r, s)
        lm = row["legal"]
        if lm and not r.done(s)[0]:
            row.update(move_row(r, s, lm[len(s) % len(lm)]))
        rows.append(row)
    return rows


def fen_rows(r, o):
    out = []
    for st, t in ((o.INIT_STATE, 0), (o.step(o.INIT_STATE, '0001'), 1), (FEN_CASES_STATE, 7), (FEN_CASES_STATE, 10)):
        fen = r.state_to_fen(st, t)
        out.append({"state": st, "turns": t, "fen": fen, "state_of_fen": r.fen_to_state(fen)})
    return out


def k1_searches(o):
    from .ref_player_harness import real_player_moves
    out = []
    for sims, seed in K1_CASES:
        a, edges, sum_n = real_player_moves([(o.INIT_STATE, 0, None, False)], sims, seed)[0]
        out.append({"sims": sims, "seed": seed, "action": a, "edges": {m: list(v) for m, v in edges.items()}, "sum_n": sum_n})
    return out


def loop_games():
    from . import ref_worker_harness as h
    sp = [dict(seed=s, **h.real_selfplay_game(s, LOOP_SIMS, **LOOP_PLAY)) for s in LOOP_SELFPLAY_SEEDS]
    ar = [dict(seed=s, idx=i, **h.real_arena_game(s, i, LOOP_SIMS, **LOOP_PLAY)) for s, i in LOOP_ARENA]
    return {"sims": LOOP_SIMS, "play": LOOP_PLAY, "selfplay": sp, "arena": ar}


def evaluator_tally():
    from . import ref_import
    from . import ref_worker_harness as h
    _, ev = h.worker_modules()
    cfg = ref_import.config("mini")
    cfg.eval.game_num = len(TALLY_RESULTS)
    w = ev.EvaluateWorker(cfg, pid=0)
    w.start_game = lambda idx: (TALLY_RESULTS[idx], 40)
    sleep = ev.sleep
    ev.sleep = lambda s: None
    try:
        want = w.start()
    finally:
        ev.sleep = sleep
    return {"results": TALLY_RESULTS, "tally": list(want)}


def expanding_data_arrays():
    """The real trainer's expanding_data (worker/optimize.py) on the first decisive golden self-play game."""
    from . import ref_worker_harness as h
    from cczero_b200.records import record_to_play_data
    from tests.test_oracle_vs_reference import expanding_data_game
    h.worker_modules()
    import cchess_alphazero.worker.optimize as ropt
    data = record_to_play_data(expanding_data_game())
    out = {}
    for tag, use_history in (("14", False), ("28", True)):
        rs, rp, rv = ropt.expanding_data(data, use_history)
        assert set(np.unique(rs)) <= {0.0, 1.0}
        out[f"expand{tag}_states_bits"] = np.packbits(np.asarray(rs) != 0)
        out[f"expand{tag}_states_shape"] = np.array(np.asarray(rs).shape)
        out[f"expand{tag}_policy"] = np.asarray(rp, dtype=np.float32)
        out[f"expand{tag}_value"] = np.asarray(rv, dtype=np.float32)
    return out


def keras_graph_arrays():
    """oracle/keras_graph.py executing the configs Keras wrote for the shipped networks, on the test's inputs."""
    from . import keras_graph, ref_import
    from tests.test_oracle_vs_reference import keras_graph_inputs
    mdir = os.path.join(ref_import.REF_ROOT, "data", "model")
    w, planes, w28, p28 = keras_graph_inputs()
    gp, gv = keras_graph.run(os.path.join(mdir, "model_best_config.json"), w, planes)
    gp28, gv28 = keras_graph.run(os.path.join(mdir, "model_128_l1_config.json"), w28, p28)
    return {"graph_policy": gp, "graph_value": gv, "graph28_policy": gp28, "graph28_value": gv28}


def main():
    sys.path.insert(0, ROOT)
    from . import ref_import
    from . import senv as o
    if not ref_import.source_available():
        raise SystemExit("reference tree not present at " + ref_import.REF_ROOT)
    r = ref_import.senv()
    lt = ref_import.lookup_tables()
    labels = {"red": lt.ActionLabelsRed, "flipped_first_50": [lt.flip_move(m) for m in lt.ActionLabelsRed[:50]]}
    doc = {"generator": "oracle/gen_golden_pins.py", "labels": labels, "playouts": playouts(r), "arbitrary_boards": arbitrary_boards(r),
           "fen": fen_rows(r, o), "k1_searches": k1_searches(o), "loop_games": loop_games(), "evaluator": evaluator_tally()}
    with gzip.open(JSON_OUT, "wt") as f:
        json.dump(doc, f, separators=(",", ":"))
    arrays = expanding_data_arrays()
    arrays.update(keras_graph_arrays())
    np.savez_compressed(NPZ_OUT, **arrays)
    for p in (JSON_OUT, NPZ_OUT):
        print(p, os.path.getsize(p), "bytes")


if __name__ == "__main__":
    main()
