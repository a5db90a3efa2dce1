"""Pin the oracle restatements to the REAL reference.  The reference's answers on the inputs below were recorded by
oracle/gen_golden_pins.py into tests/golden/reference_pins.json.gz / .npz, so every comparison runs on any checkout.  The
tests that execute the reference's own code around the drop-in (its model API, game loops, UCI front end and player) import
it from its tree or from the byte-compiled modules build() leaves in oracle/_ref, and skip only where neither exists."""
import gzip
import json
import os
import random

import numpy as np
import pytest

from oracle import gen_golden_pins as gen_pins
from oracle import player as op
from oracle import ref_import
from oracle import senv as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not ref_import.available(), reason="runs the reference's own code: neither its tree nor "
                                     "oracle/_ref (built by build() where the tree is present)")


@pytest.fixture(scope="module")
def pins():
    with gzip.open(os.path.join(ROOT, "tests", "golden", "reference_pins.json.gz"), "rt") as f:
        return json.load(f)


@pytest.fixture(scope="module")
def pin_arrays():
    with np.load(os.path.join(ROOT, "tests", "golden", "reference_pins.npz")) as z:
        return {k: z[k] for k in z.files}


def _check_rules(row):
    s = row["state"]
    assert o.get_legal_moves(s) == row["legal"], s
    assert list(o.done(s)) == row["done"] and list(o.done(s, need_check=True)) == row["done_check"], s
    assert gen_pins.planes_digest(o.state_to_planes(s)) == row["planes"], s
    assert o.has_attack_chessman(s) == row["attack"] and o.fliped_state(s) == row["flipped"], s


def test_env_restatement_on_random_playouts(pins):
    assert o.ActionLabelsRed == pins["labels"]["red"]
    assert [o.flip_move(m) for m in o.ActionLabelsRed[:50]] == pins["labels"]["flipped_first_50"]
    n = 0
    for game in pins["playouts"]:
        s = o.INIT_STATE
        for ply, row in enumerate(game):
            assert s == row["state"]
            _check_rules(row)
            if row["done"][0]:
                break
            m = row["move"]
            assert m in row["legal"]
            if ply % 2 == 0:
                assert o.will_check_or_catch(s, m) == row["check_or_catch"]
                assert o.be_catched(s, m) == row["catched"]
            assert list(o.new_step(s, m)) == row["new_step"]
            s = o.step(s, m)
            n += 1
    assert n > 500


def test_reference_smoke_vectors():
    """The print-and-eyeball vectors of the reference's test.py (SURVEY.md §4), as assertions on the oracle."""
    assert o.done('4s4/9/4e4/p8/2e2R2p/P5E2/8P/9/9/4S1E2') == (False, 0, None)
    assert o.get_legal_moves('4s4/9/9/9/9/9/9/9/9/4S4') == ['4050', '4049', '4041', '4049', '4030', '4049']
    s1 = o.step(o.INIT_STATE, '0001')
    assert s1 == 'rkemsmek1/8r/1c5c1/p1p1p1p1p/9/9/P1P1P1P1P/1C5C1/9/RKEMSMEKR'
    assert o.step(s1, o.flip_move('7770')) == 'rkemsmekr/9/1c7/p1p1p1p1p/9/9/P1P1P1P1P/1C5C1/R8/1KEMSMEcR'
    assert len(o.get_legal_moves(o.INIT_STATE)) == 44


def test_fen_helpers_match_reference(pins):
    from cczero_b200 import env as penv
    assert len(pins["fen"]) == 4
    for row in pins["fen"]:
        st, t = row["state"], row["turns"]
        assert o.state_to_fen(st, t) == row["fen"] == penv.state_to_fen(st, t)
        assert o.fen_to_state(row["fen"]) == row["state_of_fen"]


def _oracle_root(state, sims, k, seed):
    pc = op.PlayConfig(simulation_num_per_move=sims, search_threads=k, c_puct=1.5, noise_eps=0.25, dirichlet_alpha=0.2,
                       tau_decay_rate=0.98, virtual_loss=3, resign_threshold=-0.92, min_resign_turn=20)
    np.random.seed(seed)
    pl = op.OraclePlayer(pc, op.fake_evaluate_states)
    a, _ = pl.action(state, 0)
    return a, pl.tree[state]


def test_player_restatement_equals_real_player_k1(pins):
    assert [(c["sims"], c["seed"]) for c in pins["k1_searches"]] == list(gen_pins.K1_CASES)
    for real in pins["k1_searches"]:
        a, node = _oracle_root(o.INIT_STATE, real["sims"], 1, real["seed"])
        got = {m: [int(e.n), float(e.w), float(e.q), float(e.p)] for m, e in node.a.items()}
        assert a == real["action"] and got == real["edges"] and node.sum_n == real["sum_n"]


def test_canonical_schedule_is_statistically_the_threaded_player_k10():
    """search_threads = 10: the real player is a racy thread pool (not reproducible); the canonical schedule must be
    statistically indistinguishable from it.  Total-variation distance between root visit distributions: oracle-vs-real
    must not exceed the real player's own run-to-run spread, and the seed-averaged distributions must agree.  The real
    player's distributions are the INIT_STATE row of tests/golden/mcts_k10_threaded.json.gz (oracle/gen_golden_k10.py)."""
    with gzip.open(os.path.join(ROOT, "tests", "golden", "mcts_k10_threaded.json.gz"), "rt") as f:
        gold = json.load(f)
    row = next(r for r in gold["rows"] if r["state"] == o.INIT_STATE)
    sims, k, seeds = gold["sims"], gold["search_threads"], range(5)
    assert (sims, k) == (300, 10)
    lm = o.get_legal_moves(o.INIT_STATE)
    assert row["moves"] == lm

    def mine(seed):
        _, node = _oracle_root(o.INIT_STATE, sims, k, seed)
        return np.array([node.a[m].n if m in node.a else 0 for m in lm], float)

    def tv(a, b):
        return 0.5 * np.abs(a / a.sum() - b / b.sum()).sum()

    R, O = [np.array(row["visits"][s], float) for s in seeds], [mine(s) for s in seeds]
    assert all(x.sum() == sims - 1 for x in R + O)
    spread_real = np.mean([tv(R[i], R[j]) for i in seeds for j in seeds if i < j])
    cross = np.mean([tv(R[i], O[j]) for i in seeds for j in seeds])
    assert cross <= 1.5 * spread_real + 0.02, (cross, spread_real)
    assert tv(sum(R), sum(O)) < 0.05


def test_game_loop_restatements_replay_live_reference_games(pins):
    """The unmodified SelfPlayWorker.start_game / EvaluateWorker.start_game (Keras/TensorFlow imports satisfied by empty
    stand-ins, oracle/ref_worker_harness.py; recorded by oracle/gen_golden_pins.py) against oracle/selfplay.py and
    oracle/arena.py, seeds of their own."""
    from oracle import arena as oarena
    from oracle import ref_worker_harness as h
    from oracle import selfplay as osp
    games = pins["loop_games"]
    assert games["play"] == gen_pins.LOOP_PLAY and games["sims"] == 16
    pc = op.PlayConfig(simulation_num_per_move=16, search_threads=1, c_puct=1.5, noise_eps=0.25, dirichlet_alpha=0.2,
                       tau_decay_rate=0.98, virtual_loss=3, resign_threshold=-0.5, min_resign_turn=4)
    assert [g["seed"] for g in games["selfplay"]] == [41, 42]
    for g in games["selfplay"]:
        random.seed(g["seed"])
        np.random.seed(g["seed"])
        r = osp.play_game(pc, op.fake_evaluate_states, h.ReferenceDraws(), max_game_length=20, enable_resign_rate=0.1)
        assert (r["turns"], r["value_red"], r["store"], r["final_state"]) == (g["turns"], g["value_red"], g["store"], g["final_state"])
        assert g["moves"] is None or g["moves"] == r["moves"]
    assert [(g["seed"], g["idx"]) for g in games["arena"]] == [(43, 0), (44, 1)]
    for g in games["arena"]:
        random.seed(g["seed"])
        np.random.seed(g["seed"])
        d = h.ReferenceDraws()
        r = oarena.play_arena_game(pc, op.fake_evaluate_states, op.fake_evaluate_states, g["idx"], lambda slot: d, 1, max_game_length=20)
        assert (r["turns"], r["value_red"]) == (g["turns"], g["value_red"]) and r["moves"][:len(g["moves"])] == g["moves"]


@needs_reference
@pytest.mark.filterwarnings("ignore::DeprecationWarning")          # api.py:68 float(array) under numpy 2
def test_drop_in_player_searches_through_the_real_model_api(emul_lib):
    """The reference's own CChessModelAPI (agent/api.py:16-74, unmodified; a stand-in object plays the Keras model) serves
    the drop-in CChessPlayer over its Pipe: the wire protocol of player.py:118-140 <-> api.py:48-74 is what the product
    speaks.  Result == the oracle search with the same evaluator."""
    from contextlib import nullcontext
    from types import SimpleNamespace
    from oracle import ref_worker_harness as h
    from cczero_b200.player import CChessPlayer
    from tests import search_checks as sc
    h.worker_modules()                                   # installs the Keras / TensorFlow import stand-ins
    from cchess_alphazero.agent.api import CChessModelAPI

    class FakeKeras:
        def predict_on_batch(self, data):
            out = [op.fake_eval_from_planes(p) for p in data]
            return np.stack([o[0] for o in out]), np.array([[o[1]] for o in out], dtype=np.float32)
    agent_model = SimpleNamespace(model=FakeKeras(), graph=SimpleNamespace(as_default=lambda: nullcontext()))
    cfg = ref_import.config("mini")
    cfg.internet.distributed = False
    api = CChessModelAPI(cfg, agent_model)
    api.start(need_reload=False)
    pipe = api.get_pipe(need_reload=False)
    sims, k, seed = 120, 4, 9
    np.random.seed(seed)
    player = CChessPlayer(sc.make_config(sims, k), pipes=pipe, lib=emul_lib, device="cpu")
    state = sc.midgame_states(1, 21)[0]
    action, policy = player.action(state, 33)
    root = player.engine.root(0)
    np.random.seed(seed)
    pl = op.OraclePlayer(op.PlayConfig(simulation_num_per_move=sims, search_threads=k, c_puct=1.5, noise_eps=0.25, dirichlet_alpha=0.2,
                                       tau_decay_rate=0.98, virtual_loss=3), op.fake_evaluate_states)
    a2, pol2 = pl.action(state, 33)
    node = pl.tree[state]
    assert action == a2 and list(policy) == list(pol2)
    assert root["n"] == [node.a[m].n if m in node.a else 0 for m in root["moves"]]
    api.done = True                                      # stop the reference's server thread before its pipe goes away
    import time
    time.sleep(0.05)
    player.close()


def expanding_data_game():
    """The first decisive self-play game of tests/golden/games_k1.json.gz, as the record record_to_play_data takes."""
    with gzip.open(os.path.join(ROOT, "tests", "golden", "games_k1.json.gz"), "rt") as f:
        game = next(g for g in json.load(f)["games"] if g["kind"] == "selfplay" and g["result"]["moves"] and g["result"]["value_red"] != 0)
    return {"moves": game["result"]["moves"], "value_red": game["result"]["value_red"]}


def test_expanding_data_matches_the_real_trainer_side(emul_env, pin_arrays):
    """records.expanding_data vs the reference's worker/optimize.py:234-281 (unmodified; Keras imports stubbed; recorded by
    oracle/gen_golden_pins.py) on one golden game record, 14 and 28 planes."""
    from cczero_b200.records import expanding_data, record_to_play_data
    data = record_to_play_data(expanding_data_game())
    for tag, use_history in (("14", False), ("28", True)):
        shape = tuple(pin_arrays[f"expand{tag}_states_shape"])
        rs = np.unpackbits(pin_arrays[f"expand{tag}_states_bits"], count=int(np.prod(shape))).reshape(shape)
        rp, rv = pin_arrays[f"expand{tag}_policy"], pin_arrays[f"expand{tag}_value"]
        s, p, v = expanding_data(data, emul_env, use_history=use_history)
        assert s.shape == rs.shape and (s == rs).all() and (p == rp).all() and (v == rv).all()


def keras_graph_inputs():
    """(192x10 weights, planes, 28-plane weights, 28-plane history planes) the Keras-graph pin runs on."""
    from oracle import model as om
    from tests.search_checks import game_history, midgame_states
    w = om.load_compact(os.path.join(ROOT, "tests", "golden", "model_best_192x10_compact.npz"))
    states = [o.INIT_STATE] + midgame_states(11, 4, lo=2, hi=110)
    planes = np.stack([o.state_to_planes(s) for s in states])
    # the 28-plane variant (Input (28,10,9), 7 blocks x 128): random weights under the names of that config
    # (that legacy file keeps the head widths of an earlier model version: 32 policy / 4 value channels)
    w28 = om.init_weights(128, 7, 256, seed=2, trained_like=True, spread=0.5, in_planes=28, policy_filters=32, value_filters=4)
    hists = [game_history(n, 30 + n) for n in (2, 5, 17, 40)]
    p28 = np.stack([o.state_history_to_planes(h[-1], h) for h in hists])
    return w, planes, w28, p28


def test_network_restatement_matches_the_shipped_keras_graph(pin_arrays):
    """oracle/model.py (restated from agent/model.py) vs the layer graph Keras itself wrote for the shipped networks
    (data/model/model_best_config.json with the shipped weights as tests/golden/model_best_192x10_compact.npz rebuilds
    them; model_128_l1_config.json = the 28-plane variant), executed by oracle/keras_graph.py and recorded by
    oracle/gen_golden_pins.py."""
    from oracle import model as om
    w, planes, w28, p28 = keras_graph_inputs()
    gp, gv = pin_arrays["graph_policy"], pin_arrays["graph_value"]
    rp, rv = om.forward(w, planes, 10)
    assert gp.shape == (12, 2086) and np.abs(gp - rp).max() < 2e-6 and np.abs(gv[:, 0] - rv).max() < 2e-6
    assert gp.max() > 50 / 2086                                  # a peaked policy - not a degenerate comparison
    gp, gv = pin_arrays["graph28_policy"], pin_arrays["graph28_value"]
    rp, rv = om.forward(w28, p28, 7)
    assert gp.shape == (4, 2086) and np.abs(gp - rp).max() < 2e-6 and np.abs(gv[:, 0] - rv).max() < 2e-6


def test_evaluator_tally_matches_the_real_worker(pins):
    """EvaluateWorker.start's win / draw / fail bookkeeping and score (evaluator.py:93-145, unmodified; recorded by
    oracle/gen_golden_pins.py) over canned game results vs cczero_b200.evaluator.tally_games."""
    from cczero_b200.evaluator import tally_games
    results = pins["evaluator"]["results"]
    assert results == gen_pins.TALLY_RESULTS
    assert list(tally_games(list(enumerate(results)))) == pins["evaluator"]["tally"]


@needs_reference
def test_reference_game_loops_drive_the_drop_in_player(emul_lib):
    """INTEGRATION.md §3, literally: the name `CChessPlayer` inside the reference's worker modules is rebound to
    cczero_b200.player.CChessPlayer and the UNMODIFIED SelfPlayWorker.start_game / EvaluateWorker.start_game play whole
    games with it.  Since the drop-in consumes np.random exactly like the reference player, every golden game - sampled
    moves, resignations, repetition bans included - must come out identical."""
    import gzip
    import json
    import os
    from functools import partial
    from oracle import ref_worker_harness as h
    from cczero_b200.player import CChessPlayer
    factory = partial(CChessPlayer, lib=emul_lib, device="cpu")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with gzip.open(os.path.join(root, "tests", "golden", "games_k1.json.gz"), "rt") as f:
        games = json.load(f)["games"]
    done = 0
    for g in games:
        want = g["result"]
        if want["turns"] > 60:                           # keep the CPU tier short: the long games are covered elsewhere
            continue
        if g["kind"] == "selfplay":
            r = h.real_selfplay_game(g["seed"], g["sims"], use_history=bool(g.get("use_history")), player_factory=factory, **g["play"])
            assert (r["moves"], r["value_red"], r["turns"], r["store"], r["final_state"]) == \
                   (want["moves"], want["value_red"], want["turns"], want["store"], want["final_state"]), (g["seed"], g["sims"])
        else:
            r = h.real_arena_game(g["seed"], g["idx"], g["sims"], player_factory=factory, **g["play"])
            assert (r["moves"], r["value_red"], r["turns"]) == (want["moves"], want["value_red"], want["turns"])
        done += 1
    assert done >= 8


@needs_reference
def test_reference_uci_front_end_drives_the_drop_in_player(emul_lib):
    """The REAL uci.UCI class with `CChessPlayer` rebound to the drop-in: the golden session (recorded with the real
    player) must come out line for line."""
    import contextlib
    import gzip
    import io
    import json
    import os
    import sys
    import time
    from functools import partial
    from oracle import gen_golden_uci as gu
    from oracle import ref_worker_harness as h
    from oracle.ref_player_harness import FakeNetServer
    from cczero_b200.player import CChessPlayer
    h.worker_modules()
    err = sys.stderr
    import cchess_alphazero.uci as ruci
    sys.stderr = err
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with gzip.open(os.path.join(root, "tests", "golden", "uci_session_k1.json.gz"), "rt") as f:
        gold = json.load(f)
    cfg = ruci.config
    for k, v in gold["play"].items():
        setattr(cfg.play, k, v)
    servers = []

    class FakeModel:
        def get_pipes(self, need_reload=True):
            servers.append(FakeNetServer())
            return servers[-1].you

        def close_pipes(self):
            pass
    u = ruci.UCI(cfg)
    u.load_model = lambda config_file=None: (setattr(u, "model", FakeModel()) or False)
    real_player, real_ssc = ruci.CChessPlayer, ruci.set_session_config
    ruci.set_session_config = lambda **k: None
    ruci.CChessPlayer = partial(CChessPlayer, lib=emul_lib, device="cpu", infinite_capacity=4000)
    try:
        for step in gold["steps"]:
            buf = io.StringIO()
            parts = step["cmd"].split(" ")
            u.args = parts[1:]
            if step["seed"] is not None:
                np.random.seed(step["seed"])
            with contextlib.redirect_stdout(buf):
                getattr(u, "cmd_" + parts[0])()
                if parts[0] == "go":
                    t0 = time.time()
                    while "bestmove" not in buf.getvalue() and time.time() - t0 < 120:
                        time.sleep(0.02)
                    time.sleep(0.1)
            assert [gu.strip_clock(x) for x in buf.getvalue().splitlines()] == step["out"], step["cmd"]
    finally:
        ruci.CChessPlayer, ruci.set_session_config = real_player, real_ssc
        for s in servers:
            s.close()


@needs_reference
def test_reference_player_runs_on_the_drop_in_rules_engine(emul_env):
    """The other import swap of INTEGRATION.md §3: `senv` inside the reference's agent/player.py rebound to
    cczero_b200.env.StaticEnv - the REAL player must search exactly as it does on its own static_env."""
    from oracle.ref_player_harness import real_player_moves
    from tests.search_checks import load_mcts_golden
    pm = ref_import.player_module()
    gold = {c["name"]: c for c in load_mcts_golden()["cases"]}
    hist = {c["name"]: c for c in load_mcts_golden("mcts_k1_hist.json.gz")["cases"]}
    own = pm.senv
    pm.senv = emul_env
    try:
        for case, use_history in ((gold["init_60"], False), (gold["mid2_no_act"], False), (hist["hist_mid30_150"], True)):
            calls = [(c["state"], c["turns"], c["no_act"], c["increase_temp"], c.get("hist")) for c in case["calls"]]
            res = real_player_moves(calls, case["sims"], case["seed"], use_history=use_history)
            for (a, edges, sum_n), c in zip(res, case["calls"]):
                assert a == c["action"] and sum_n == c["sum_n"]
                assert {m: list(v) for m, v in edges.items()} == c["edges"]
    finally:
        pm.senv = own


def test_env_restatement_on_arbitrary_boards(pins):
    """Unreachable positions (random pieces on random squares, piece counts no game can have): oracle == real static_env."""
    from tests.env_checks import EXTREME_STATES, random_boards
    states = random_boards(600, 5) + [x for x in EXTREME_STATES if 's' in x and 'S' in x]
    assert [row["state"] for row in pins["arbitrary_boards"]] == states
    for row in pins["arbitrary_boards"]:
        s = row["state"]
        _check_rules(row)
        if "move" in row:
            m = row["move"]
            assert list(o.new_step(s, m)) == row["new_step"], (s, m)
            assert o.will_check_or_catch(s, m) == row["check_or_catch"], (s, m)
            assert o.be_catched(s, m) == row["catched"], (s, m)
