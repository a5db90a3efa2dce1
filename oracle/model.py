"""oracle/model.py — PyTorch fp32 restatement of the reference network.  TEST INFRASTRUCTURE.

Restates cchess_alphazero/agent/model.py:32-83 (CChessModel.build / _build_residual_block) with the Keras
defaults recorded in data/model/model_best_config.json: Conv2D channels_first, padding "same", no bias;
BatchNormalization(axis=1, epsilon=1e-3) in inference mode; Flatten over (C,H,W); Dense kernels (in,out);
softmax policy, tanh value.  TensorFlow/Keras are not installable here, so NN parity is pinned only by
this restatement ("parity unpinned" by any reference test, SURVEY.md §8c) with tolerance 1e-3.

Weights are exchanged as a dict of Keras-style names -> float32 arrays in Keras layouts
(conv HWIO, dense (in,out)), the same dict the product's `cz_nn_set_weights` consumes.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = 1e-3
N_LABELS = 2086


def keras_names(filters, blocks):
    names = [f"input_conv-5-{filters}/kernel"] + [f"input_batchnorm/{w}" for w in ("gamma", "beta", "moving_mean", "moving_variance")]
    for i in range(1, blocks + 1):
        for j in (1, 2):
            names.append(f"res{i}_conv{j}-3-{filters}/kernel")
            names += [f"res{i}_batchnorm{j}/{w}" for w in ("gamma", "beta", "moving_mean", "moving_variance")]
    names += ["policy_conv-1-2/kernel"] + [f"policy_batchnorm/{w}" for w in ("gamma", "beta", "moving_mean", "moving_variance")]
    names += ["policy_out/kernel", "policy_out/bias"]
    names += ["value_conv-1-4/kernel"] + [f"value_batchnorm/{w}" for w in ("gamma", "beta", "moving_mean", "moving_variance")]
    names += ["value_dense/kernel", "value_dense/bias", "value_out/kernel", "value_out/bias"]
    return names


def load_compact(path):
    """The network a compact weight file describes (written by oracle/gen_golden_weights.py): tensors stored whole
    ("exact.<name>") are returned as they are; the large ones are regenerated from their per-output-channel mean and
    standard deviation ("mean.", "std.", "shape.<name>") with a generator seeded by the tensor's name, and carry their
    real first values ("head.<name>").  Names use '__' for '/'."""
    import zlib
    with np.load(path) as z:
        d = {k: z[k] for k in z.files}
    w = {}
    for key, v in d.items():
        kind, name = key.split(".", 1)
        if kind == "exact":
            w[name.replace("__", "/")] = v.astype(np.float32)
        elif kind == "shape":
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            a = rng.standard_normal(tuple(int(x) for x in v), dtype=np.float32) * d["std." + name] + d["mean." + name]
            head = d["head." + name]
            a.reshape(-1)[:head.size] = head
            w[name.replace("__", "/")] = a.astype(np.float32)
    return w


def _glorot(rng, shape, fan_in, fan_out):
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def init_weights(filters, blocks, value_fc=256, seed=0, trained_like=False, spread=1.0, in_planes=14, policy_filters=4,
                 value_filters=2):
    """Keras-equivalent initialisation (glorot-uniform kernels, zero biases, BN gamma=1 beta=0 mean=0 var=1).
    trained_like=True perturbs the BN statistics and biases so that folding bugs cannot hide; `spread` scales the
    perturbation (1.0: gamma in [0.5,1.5], variance in [0.5,2] - a deep random net in that regime amplifies any
    perturbation of its inputs several-fold per 10 blocks; 0.3 keeps the conditioning close to a Keras-initialised net)."""
    rng = np.random.RandomState(seed)
    w = {}

    def conv(name, k, cin, cout):
        w[name + "/kernel"] = _glorot(rng, (k, k, cin, cout), k * k * cin, k * k * cout)

    def bn(name, c):
        if trained_like:
            w[name + "/gamma"] = rng.uniform(1 - 0.5 * spread, 1 + 0.5 * spread, c).astype(np.float32)
            w[name + "/beta"] = rng.uniform(-0.3 * spread, 0.3 * spread, c).astype(np.float32)
            w[name + "/moving_mean"] = rng.uniform(-0.2 * spread, 0.2 * spread, c).astype(np.float32)
            w[name + "/moving_variance"] = np.exp(rng.uniform(-0.7 * spread, 0.7 * spread, c)).astype(np.float32)
        else:
            w[name + "/gamma"] = np.ones(c, np.float32)
            w[name + "/beta"] = np.zeros(c, np.float32)
            w[name + "/moving_mean"] = np.zeros(c, np.float32)
            w[name + "/moving_variance"] = np.ones(c, np.float32)

    def dense(name, cin, cout):
        w[name + "/kernel"] = _glorot(rng, (cin, cout), cin, cout)
        w[name + "/bias"] = (rng.uniform(-0.1, 0.1, cout) if trained_like else np.zeros(cout)).astype(np.float32)

    conv(f"input_conv-5-{filters}", 5, in_planes, filters)     # 28 = the use_history variant (model_128_l1_config.json)
    bn("input_batchnorm", filters)
    for i in range(1, blocks + 1):
        for j in (1, 2):
            conv(f"res{i}_conv{j}-3-{filters}", 3, filters, filters)
            bn(f"res{i}_batchnorm{j}", filters)
    # agent/model.py:47-61 builds 4 policy and 2 value channels; the older JSON configs under data/model/ (128f, 256f,
    # 128_l1) still carry the head widths of earlier versions (policy 2 or 32, value 4) under the same layer names
    conv("policy_conv-1-2", 1, filters, policy_filters)
    bn("policy_batchnorm", policy_filters)
    dense("policy_out", 90 * policy_filters, N_LABELS)
    conv("value_conv-1-4", 1, filters, value_filters)
    bn("value_batchnorm", value_filters)
    dense("value_dense", 90 * value_filters, value_fc)
    dense("value_out", value_fc, 1)
    return w


def _find(w, layer, weight):
    for k, v in w.items():
        l, ww = k.split("/", 1)
        if ww.split(":")[0] == weight and (l == layer or l.startswith(layer + "-")):
            return torch.as_tensor(np.asarray(v), dtype=torch.float32)
    raise KeyError((layer, weight))


def _conv(x, w, layer, pad):
    k = _find(w, layer, "kernel").permute(3, 2, 0, 1).contiguous()      # HWIO -> OIHW
    return F.conv2d(x, k, padding=pad)


def _bn(x, w, layer):
    g, b = _find(w, layer, "gamma"), _find(w, layer, "beta")
    m, v = _find(w, layer, "moving_mean"), _find(w, layer, "moving_variance")
    sh = (1, -1, 1, 1)
    return (x - m.view(sh)) / torch.sqrt(v.view(sh) + BN_EPS) * g.view(sh) + b.view(sh)


def forward(w, planes, blocks):
    """planes: float32 [B,14,10,9] -> (policy [B,2086] softmax, value [B]) in fp32 on the CPU."""
    x = torch.as_tensor(np.asarray(planes), dtype=torch.float32)
    with torch.no_grad():
        x = F.relu(_bn(_conv(x, w, "input_conv", 2), w, "input_batchnorm"))
        for i in range(1, blocks + 1):
            y = F.relu(_bn(_conv(x, w, f"res{i}_conv1", 1), w, f"res{i}_batchnorm1"))
            y = _bn(_conv(y, w, f"res{i}_conv2", 1), w, f"res{i}_batchnorm2")
            x = F.relu(x + y)
        p = F.relu(_bn(_conv(x, w, "policy_conv", 0), w, "policy_batchnorm")).flatten(1)
        p = torch.softmax(p @ _find(w, "policy_out", "kernel") + _find(w, "policy_out", "bias"), dim=1)
        v = F.relu(_bn(_conv(x, w, "value_conv", 0), w, "value_batchnorm")).flatten(1)
        v = F.relu(v @ _find(w, "value_dense", "kernel") + _find(w, "value_dense", "bias"))
        v = torch.tanh(v @ _find(w, "value_out", "kernel") + _find(w, "value_out", "bias"))
    return p.numpy(), v.numpy()[:, 0]


class TorchNet:
    """predict_on_batch-compatible wrapper (what api.py:63-64 calls on the Keras model)."""

    def __init__(self, weights, blocks):
        self.w, self.blocks = weights, blocks

    def predict_on_batch(self, data):
        p, v = forward(self.w, data, self.blocks)
        return p, v[:, None]
