"""Loader for tests/golden/*.npz (vectors dumped from the unmodified reference on a B200, see tests/golden/make_golden.sh)."""
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# case -> (config file, n_in, n_out, batch, probe file with the device-evaluated level scales)
CASES = {
    "hash3d_small": ("hash3d_small.json", 3, 3, 512, "probe_s1.5_b16.json"),
    "dense_mix3d": ("dense_mix3d.json", 3, 2, 256, "probe_s1.5_b4.json"),
    "image2d": ("image2d.json", 2, 3, 512, "probe_s1.5_b16.json"),
    # Tanh hidden / Sigmoid output / 32 neurons / 3 hidden layers: pins the activation set and the narrow-network path
    "tanh_w32": ("tanh_w32.json", 3, 3, 512, "probe_s1.5_b16.json"),
}


def load_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: z[k] for k in z.files if k != "meta"}
    d["meta"] = json.loads(bytes(z["meta"]).decode())
    return d


def load_config(name):
    return json.load(open(os.path.join(GOLDEN, "configs", CASES[name][0])))


def device_scales(name, n_levels):
    """grid_scale() as the REFERENCE's device code evaluates it (fast-math ex2.approx), from its probe kernel."""
    probe = json.load(open(os.path.join(GOLDEN, CASES[name][4])))
    bits = np.array([l["dev_bits"] for l in probe["levels"][:n_levels]], np.uint32)
    return bits.view(np.float32).tolist(), probe


def init_params_match(g, params):
    """Initial fp32 parameters bit for bit against the reference's: the stored array, or its SHA-256 where the fixture keeps only
    the digest to stay small (tests/golden/pack_golden.py)."""
    params = np.ascontiguousarray(params, np.float32)
    if "params_init_f32" in g:
        return np.array_equal(params.view(np.uint32), g["params_init_f32"].view(np.uint32))
    return hashlib.sha256(params.tobytes()).hexdigest() == g["meta"]["params_init_sha256"]


def rae(a, b, percentile=100.0):
    """tests/test_common.h:59-117 of the reference: symmetric relative absolute error, best-p% trimmed mean."""
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    eps = 1e-2 * 0.5 * (np.abs(a).mean() + np.abs(b).mean()) + 1e-30
    e = np.abs(a - b) / (0.5 * (np.abs(a) + np.abs(b)) + eps)
    if percentile < 100.0:
        e = np.sort(e)[: max(1, int(len(e) * percentile / 100.0))]
    return float(e.mean())


def mlp_gradients_agree(a, b, rae_bar):
    """Weight-gradient agreement with the reference. Normally the reference's own bar (mean RAE on the best 99.9 %,
    tests/test_common.h:218). When the gradients themselves sit at the bottom of fp16 (loss-scaled values of a few dozen
    subnormal quanta, 2^-24), the reference's fp16 split-K partial sums (cutlass_matmul.h:67) are quantisation noise of a few
    quanta and a relative measure is meaningless: then the bar is absolute, mean <= 2.5 quanta and max <= 16 quanta."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if rae(a, b, 99.9) < rae_bar:
        return True
    q = 2.0 ** -24
    if np.abs(b).mean() < 64 * q:
        d = np.abs(a - b)
        return d.mean() <= 2.5 * q and d.max() <= 16 * q
    return False
