"""Fixture generator (needs the reference tree): the reference's shipped, trained 192x10 network
(data/model/model_best_weight.h5, loaded by agent/model.py:95-107 through Keras) in two small files.

  tests/golden/model_best_192x10_compact.npz   the network as oracle.model.load_compact rebuilds it: every tensor of at
                                               most EXACT_MAX values stored whole (batch-norm statistics, biases, heads'
                                               1x1 convs), the large kernels as per-output-channel mean / standard
                                               deviation plus their first SAMPLED values; and the REAL network's output on
                                               the opening position ("real.opening_policy", "real.opening_value")
  tests/golden/model_best_weight_sampled.h5.gz the shipped .h5 byte for byte except that every tensor keeps only its first
                                               SAMPLED values and the rest of its data is zeroed: the real file layout
                                               for the reader test (tests/test_keras_h5.py)

The whole network (7.5 M values) cannot be stored at a fixture size, so the tests that run a 192x10 network run the
rebuilt one: the real batch-norm statistics and biases, and kernels of the real per-channel scale.

TEST INFRASTRUCTURE: nothing in the product package or bench.py's GPU arm reads these files.

    python -m oracle.gen_golden_weights
"""
import gzip
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPACT_OUT = os.path.join(ROOT, "tests", "golden", "model_best_192x10_compact.npz")
SAMPLED_OUT = os.path.join(ROOT, "tests", "golden", "model_best_weight_sampled.h5.gz")
SAMPLED = 16
EXACT_MAX = 20000


def sampled_h5(data, weights):
    """The bytes of the .h5 file `data` with every tensor's data zeroed past its first SAMPLED float32 values.  Each
    tensor's data is found by its bytes (the files Keras writes store them contiguous, little-endian float32)."""
    out = bytearray(data)
    for name, arr in weights.items():
        raw = np.ascontiguousarray(arr, dtype="<f4").tobytes()
        off = data.find(raw)
        assert off >= 0, name
        out[off + 4 * SAMPLED:off + len(raw)] = bytes(max(0, len(raw) - 4 * SAMPLED))
    return bytes(out)


def compact(weights):
    out = {}
    for name, a in weights.items():
        key = name.replace("/", "__")
        if a.size <= EXACT_MAX:
            out["exact." + key] = a
            continue
        flat = a.reshape(-1, a.shape[-1])                            # Keras layouts: output channels last
        out["shape." + key] = np.array(a.shape, dtype=np.int64)
        out["mean." + key] = flat.mean(axis=0).astype(np.float32)
        out["std." + key] = flat.std(axis=0).astype(np.float32)
        out["head." + key] = a.reshape(-1)[:SAMPLED].copy()
    return out


def main():
    sys.path.insert(0, ROOT)
    from oracle import model as om
    from oracle import ref_import
    from oracle import senv as osenv
    from cczero_b200.keras_h5 import read_keras_weights
    h5 = os.path.join(ref_import.REF_ROOT, "data", "model", "model_best_weight.h5")
    if not os.path.exists(h5):
        raise SystemExit("reference weights not present: " + h5)
    w = read_keras_weights(h5)
    assert len(w) == 121 and sum(v.size for v in w.values()) == 7519663
    arrays = compact(w)
    p, v = om.forward(w, osenv.state_to_planes(osenv.INIT_STATE)[None], 10)
    arrays["real.opening_policy"], arrays["real.opening_value"] = p[0].astype(np.float32), np.float32(v[0])
    np.savez_compressed(COMPACT_OUT, **arrays)
    with open(h5, "rb") as f:
        data = f.read()
    with gzip.GzipFile(SAMPLED_OUT, "wb", mtime=0) as f:
        f.write(sampled_h5(data, w))
    check = read_keras_weights_bytes(gzip.decompress(open(SAMPLED_OUT, "rb").read()))
    for name, a in w.items():
        got = check[name].reshape(-1)
        assert (got[:SAMPLED] == a.reshape(-1)[:SAMPLED]).all() and not got[SAMPLED:].any(), name
    for path in (COMPACT_OUT, SAMPLED_OUT):
        print(path, os.path.getsize(path), "bytes")


def read_keras_weights_bytes(data):
    import tempfile
    from cczero_b200.keras_h5 import read_keras_weights
    with tempfile.NamedTemporaryFile(suffix=".h5") as f:
        f.write(data)
        f.flush()
        return read_keras_weights(f.name)


if __name__ == "__main__":
    main()
