"""Keras .h5 import (SURVEY.md §8f row 3): the pure-Python HDF5 subset reader on the reference's shipped weights, and the
engine against the fp32 restatement on those REAL trained weights."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import model as om
from oracle import senv as osenv
from tests.search_checks import midgame_states

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the shipped data/model/model_best_weight.h5 with every tensor cut to its first 16 values (the rest zeroed), written by
# `python -m oracle.gen_golden_weights sampled`: the real file layout at a fixture size
SAMPLED_H5 = os.path.join(GOLDEN, "model_best_weight_sampled.h5.gz")
SAMPLED = 16
# the shipped network at a fixture size (oracle/gen_golden_weights.py, rebuilt by oracle.model.load_compact): real
# batch-norm statistics and biases, kernels of the real per-channel scale with the real first values; and the real
# network's output on the opening position
COMPACT = os.path.join(GOLDEN, "model_best_192x10_compact.npz")


def _cfg():
    return SimpleNamespace(model=SimpleNamespace(cnn_filter_num=0, res_layer_num=0, value_fc_size=0, cnn_first_filter_size=5,
                                                 cnn_filter_size=3, input_depth=14))


def test_reads_shipped_keras_weights(tmp_path):
    import gzip
    import shutil
    from cczero_b200.model import CChessModel
    h5 = str(tmp_path / "model_best_weight.h5")
    with gzip.open(SAMPLED_H5, "rb") as src, open(h5, "wb") as dst:
        shutil.copyfileobj(src, dst)
    m = CChessModel(_cfg())
    assert m.load("unused.json", h5)
    mc = m.config.model
    assert (mc.cnn_filter_num, mc.res_layer_num, mc.value_fc_size) == (192, 10, 256)
    assert len(m.weights) == 121 and sum(v.size for v in m.weights.values()) == 7519663
    assert set(m.weights) == set(om.keras_names(192, 10))
    assert m.weights["res7_conv2-3-192/kernel"].shape == (3, 3, 192, 192) and m.weights["policy_out/kernel"].shape == (360, 2086)
    assert m.digest == m.fetch_digest(h5)
    rebuilt = om.load_compact(COMPACT)
    assert len(rebuilt) == 121
    for k, v in m.weights.items():
        want = rebuilt[k].ravel()
        got = v.ravel()
        assert v.shape == rebuilt[k].shape and (got[:SAMPLED] == want[:SAMPLED]).all() and not got[SAMPLED:].any(), k
    # the trained net knows an opening: its favourite first moves are the classical ones (central cannon, knights, pawns).
    # This checks the fixture's record of the REAL network's output (computed by oracle/gen_golden_weights.py through the
    # fp32 restatement from the full weights), not the reader: the fixture keeps too little of the weights to rerun it.
    with np.load(COMPACT) as z:
        p, v = z["real.opening_policy"], z["real.opening_value"]
    top = [osenv.ActionLabelsRed[i] for i in np.argsort(-p)[:4]]
    assert abs(p.sum() - 1) < 1e-4 and abs(v) < 0.5
    assert set(top) & {"7242", "1242", "7062", "1022", "2324", "6364", "7747", "1747"}, top


@pytest.mark.gpu
def test_real_trained_weights_within_1e3(cuda_lib, cuda_env):
    """The reference's trained 192x10 network as the fixture rebuilds it (real batch-norm statistics and biases, kernels of
    the real per-channel scale): tensor-core forward vs the fp32 restatement, tolerance 1e-3."""
    import torch
    from cczero_b200.engine import Engine
    w = om.load_compact(COMPACT)
    states = [osenv.INIT_STATE] + midgame_states(47, 11, lo=1, hi=100)
    ref_p, ref_v = om.forward(w, np.stack([osenv.state_to_planes(s) for s in states]), 10)
    eng = Engine(cuda_lib, "cuda", n_games=64, sims_per_move=8, leaves_per_round=1, nn_filters=192, nn_blocks=10, nn_value_fc=256)
    eng.set_weights({k: torch.as_tensor(v) for k, v in w.items()})
    pol, val = eng.nn_forward_boards(cuda_env.boards_from_states(states))
    pol, val = pol.cpu().numpy(), val.cpu().numpy()
    dp, dv = np.abs(pol - ref_p).max(), np.abs(val - ref_v).max()
    print(f"rebuilt 192x10 weights: max|dp|={dp:.2e} max|dv|={dv:.2e} max p={ref_p.max():.3f} |v|max={np.abs(ref_v).max():.3f}")
    assert dp < 1e-3 and dv < 1e-3, (dp, dv)
    assert (pol.argmax(1) == ref_p.argmax(1)).mean() > 0.95
    eng.close()
