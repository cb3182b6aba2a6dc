"""GPU parity tests: every stage of the fused sm_100a kernel against the CPU oracle on identical seeded inputs, through
the C ABI (libtcnn_b200.so). Integer work (cells, hash indices => which table entries are blended) must be bit-exact,
which shows up as bit-exact encoded features; floating-point stages are checked stage-by-stage (each oracle stage is fed
the DEVICE's previous stage) within stated fp16 tolerances, using the reference's own vocabulary (tests/test_common.h:59-117:
symmetric relative absolute error, percentile trimming).
"""
import json
import os

import numpy as np
import pytest

import oracle_binding as ob

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG_DIR = os.path.join(ROOT, "tests", "golden", "configs")


def load_cfg(name):
    return json.load(open(os.path.join(CFG_DIR, name + ".json")))


def rae(a, b, percentile=100.0):
    """tests/test_common.h:59-117: |a-b| / (|a|+|b|)/2 + eps with eps scaled by the mean magnitude, best-p% trimmed mean."""
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    eps = 1e-2 * 0.5 * (np.abs(a).mean() + np.abs(b).mean()) + 1e-30
    e = np.abs(a - b) / (0.5 * (np.abs(a) + np.abs(b)) + eps)
    if percentile < 100.0:
        e = np.sort(e)[: max(1, int(len(e) * percentile / 100.0))]
    return float(e.mean())


def f16(t):
    return t.cpu().numpy().view(np.uint16)


CASES = [
    ("hash3d_small", 3, 3, 512),
    ("dense_mix3d", 3, 2, 256),
    ("image2d", 2, 3, 512),
]




def make_batch(n_in, n_out, B, seed=1337):
    rng = ob.default_rng(seed)
    x = ob.generate_random_uniform(rng, B * n_in).reshape(B, n_in)
    return x, ob.make_targets(x, n_out)


@pytest.mark.parametrize("name,n_in,n_out,B", CASES)
def test_stagewise_parity(torch_cuda, name, n_in, n_out, B):
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg(name)
    model = tcnn_b200.create_from_config(n_in, n_out, cfg)
    levels = model.grid_levels()
    orc = ob.OracleModel(n_in, n_out, cfg, scales=levels["scales"])
    NH = cfg["network"]["n_hidden_layers"]

    # ---- sizing and initial parameters: bit-exact
    assert model.n_params == orc.n_params and model.n_mlp_params == orc.n_mlp
    assert levels["offsets"] == list(orc.grid.offsets[: orc.grid.n_levels + 1])
    p0 = model.trainer.params_full_precision().cpu().numpy()
    assert np.array_equal(p0.view(np.uint32), orc.params_fp32.view(np.uint32))
    assert np.array_equal(f16(model.trainer.params()), orc.params_fp16)

    x, y = make_batch(n_in, n_out, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    taps = dict(
        encoded=torch.zeros(B, 64, dtype=torch.float16, device="cuda"),
        hidden=torch.zeros(NH, B, 64, dtype=torch.float16, device="cuda"),
        output=torch.zeros(B, 16, dtype=torch.float16, device="cuda"),
        dL_doutput=torch.zeros(B, 16, dtype=torch.float16, device="cuda"),
        grad_hidden=torch.zeros(NH, B, 64, dtype=torch.float16, device="cuda"),
        dL_dencoded=torch.zeros(B, 64, dtype=torch.float16, device="cuda"),
        loss_values=torch.zeros(B, n_out, dtype=torch.float32, device="cuda"),
    )
    model.set_debug_taps(**taps)
    model.trainer.training_step(xd, yd, run_optimizer=False)
    loss = model.trainer.loss()
    torch.cuda.synchronize()
    W = orc.grid.padded_width

    # ---- stage 1: hash-grid gather + blend: BIT-EXACT (integer indices + deterministic fp16 fma chain)
    enc_dev = f16(taps["encoded"])  # [B][64]
    enc_ref = orc.encode(x)  # SoA [W][B]
    assert np.array_equal(enc_dev[:, :W].T, enc_ref), "encoded features differ"
    assert (enc_dev[:, W:] == 0).all()

    # ---- stage 2: MLP forward on the device's encoding (oracle with fp32 accumulation like tcgen05)
    hid_ref, out_ref = orc.mlp_forward(np.ascontiguousarray(enc_dev[:, :W].T))
    hid_dev = f16(taps["hidden"])
    a, b = ob.half_bits_to_float(hid_dev), ob.half_bits_to_float(hid_ref)
    # fp32-accumulated dot products rounded once to fp16: at most 1 fp16 ulp apart (summation order), rarely
    assert np.abs(a - b).max() <= 2.0 ** -10 * max(1.0, np.abs(b).max())
    assert (hid_dev != hid_ref).mean() < 0.02
    out_dev = f16(taps["output"])
    a, b = ob.half_bits_to_float(out_dev), ob.half_bits_to_float(out_ref)
    # feed-forward from identical hidden values only where the last hidden layer agrees bitwise; compare all with tolerance
    assert rae(a, b) < 1e-3
    assert np.abs(a - b).max() <= 4e-3 * max(1.0, np.abs(b).max())

    # ---- stage 3: loss on the device's output
    lv_ref, dy_ref = orc.loss(out_dev, y)
    lv_dev = taps["loss_values"].cpu().numpy()
    assert rae(lv_dev, lv_ref[:, :n_out]) < 1e-3  # tests/test_jit_losses.cu:109-110 bar
    dy_dev = f16(taps["dL_doutput"])
    assert rae(ob.half_bits_to_float(dy_dev), ob.half_bits_to_float(dy_ref)) < 1e-3
    assert (dy_dev[:, n_out:] == 0).all()
    assert abs(loss - float(lv_dev.sum(dtype=np.float64))) <= 1e-4 * abs(loss) + 1e-7

    # ---- stage 4: MLP backward on the device's activations and loss gradients
    dW_ref, denc_ref = orc.mlp_backward(np.ascontiguousarray(enc_dev[:, :W].T), hid_dev, dy_dev)
    denc_dev = f16(taps["dL_dencoded"])[:, :W].T
    a, b = ob.half_bits_to_float(denc_dev), ob.half_bits_to_float(denc_ref)
    assert rae(a, b, 99.0) < 1e-2  # tests/test_common.h:216 bar (input gradients)
    assert rae(a, b) < 2e-2
    grads = ob.half_bits_to_float(f16(model.trainer.param_gradients()))
    dW_dev = grads[: orc.n_mlp].astype(np.float64)
    dW16 = dW_ref.astype(np.float16).astype(np.float64)
    assert rae(dW_dev, dW16, 99.9) < 1.2e-2  # tests/test_common.h:218 bar (parameter gradients)
    assert rae(dW_dev, dW16) < 1.2e-2

    # ---- stage 5: grid gradient scatter of the device's dL/d(encoded): fp16 atomics vs exact sums
    g_ref = orc.grid_backward(x, np.ascontiguousarray(np.pad(denc_dev, ((0, 0), (0, 0)))))
    g_dev = grads[orc.n_mlp :].astype(np.float64)
    touched = g_ref != 0
    assert ((g_dev != 0) <= touched | (np.abs(g_ref) < 1e-12)).all(), "gradient written to an entry no sample touches"
    assert rae(g_dev, g_ref.astype(np.float16).astype(np.float64), 99.9) < 1.2e-2
    # untouched entries stay exactly zero (GradientMode::Overwrite + Adam's zero-gradient skip depend on it)
    assert (g_dev[~touched] == 0).all()


@pytest.mark.parametrize("name,n_in,n_out,B", CASES)
def test_training_trajectory_matches_oracle(torch_cuda, name, n_in, n_out, B):
    """10 optimiser steps on one batch: loss curve and final parameters track the oracle (Adam amplifies the sign of tiny
    gradients, so parameters are compared on the mean, losses to 2%)."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg(name)
    model = tcnn_b200.create_from_config(n_in, n_out, cfg)
    orc = ob.OracleModel(n_in, n_out, cfg, scales=model.grid_levels()["scales"])
    x, y = make_batch(n_in, n_out, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    dev_losses, ref_losses = [], []
    for _ in range(10):
        model.trainer.training_step(xd, yd)
        dev_losses.append(model.trainer.loss())
        ref_losses.append(orc.training_step(x, y))
    assert dev_losses[-1] < dev_losses[0]
    for a, b in zip(dev_losses, ref_losses):
        assert abs(a - b) <= 2e-2 * abs(b) + 1e-6, (dev_losses, ref_losses)
    p = model.trainer.params_full_precision().cpu().numpy()
    lr = cfg["optimizer"]["learning_rate"]
    assert np.abs(p - orc.params_fp32).mean() < 0.05 * lr * 10
    # step counters / zero-gradient skip: the set of grid parameters that moved is identical
    p0 = ob.OracleModel(n_in, n_out, cfg).params_fp32
    moved_dev = p[orc.n_mlp :] != p0[orc.n_mlp :]
    moved_ref = orc.params_fp32[orc.n_mlp :] != p0[orc.n_mlp :]
    assert (moved_dev != moved_ref).mean() < 1e-3
    out_dev = model.network.inference(xd).cpu().numpy()
    out_ref = orc.inference(x)
    assert rae(out_dev, out_ref, 99.0) < 5e-2


def test_inference_matches_forward(torch_cuda):
    """tests/test_common.h:153-166: inference vs the training forward of the same implementation, RAE < 1e-4."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    B = 1024
    model = tcnn_b200.create_from_config(3, 3, cfg)
    x, y = make_batch(3, 3, B, seed=99)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    out_tap = torch.zeros(B, 16, dtype=torch.float16, device="cuda")
    model.set_debug_taps(output=out_tap)
    inf = model.network.inference(xd).cpu().numpy()
    model.trainer.training_step(xd, yd, run_optimizer=False)
    torch.cuda.synchronize()
    fwd = out_tap.float().cpu().numpy()[:, :3]
    assert rae(inf, fwd) < 1e-4
    host = np.zeros((B, 3), np.float32)
    model.inference_host(x, host)
    assert np.array_equal(host, inf)


def test_full_size_properties(torch_cuda):
    """BASELINE.json configs[1] at its full size (T=2^19, batch 2^18): size-independent properties.
    (1) batch linearity: gradients of a batch == sum of the gradients of its two halves normalised over the full batch;
    (2) untouched table entries keep zero gradient and are skipped by Adam; (3) the loss decreases; (4) host == device path."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("headline")
    B = 1 << 18
    model = tcnn_b200.create_from_config(3, 3, cfg)
    assert model.n_params == 13026992 + 7168
    x, y = make_batch(3, 3, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()

    model.trainer.training_step(xd, yd, run_optimizer=False)
    full_loss = model.trainer.loss()
    g_full = model.trainer.param_gradients().float().clone()
    h = B // 2
    model.trainer.training_step_shard(xd[:h], yd[:h], B)
    la = model.trainer.loss()
    ga = model.trainer.param_gradients().float().clone()
    model.trainer.training_step_shard(xd[h:], yd[h:], B)
    lb = model.trainer.loss()
    gb = model.trainer.param_gradients().float().clone()
    assert abs((la + lb) - full_loss) <= 1e-3 * full_loss
    gsum = ga + gb
    nz = g_full != 0
    assert ((gsum != 0) == nz).float().mean() > 0.999
    err = rae(gsum[nz].cpu().numpy()[:2000000], g_full[nz].cpu().numpy()[:2000000], 99.0)
    assert err < 2e-2, err

    p_before = model.trainer.params_full_precision().clone()
    model.trainer.training_step(xd, yd)
    losses = [model.trainer.loss()]
    p_after = model.trainer.params_full_precision().clone()
    g_step = model.trainer.param_gradients().float()
    # adam.h:79-82: grid entries whose gradient of THIS step is exactly zero are skipped; every other one moved by ~lr
    zero = g_step[7168:] == 0
    assert zero.any() and (~zero).any()
    assert torch.equal(p_before[7168:][zero], p_after[7168:][zero])
    moved = (p_before[7168:][~zero] != p_after[7168:][~zero]).float().mean().item()
    assert moved > 0.999
    for _ in range(4):
        model.trainer.training_step(xd, yd)
        losses.append(model.trainer.loss())
    assert losses[-1] < losses[0]
    assert torch.isfinite(model.trainer.params_full_precision()).all()

    l_host = model.training_step_host(x, y)
    assert np.isfinite(l_host) and l_host < losses[0]


def test_serialize_roundtrip(torch_cuda):
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    a = tcnn_b200.create_from_config(3, 3, cfg)
    x, y = make_batch(3, 3, 512)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    for _ in range(3):
        a.trainer.training_step(xd, yd)
    blob = a.trainer.serialize(with_optimizer=True)
    b = tcnn_b200.create_from_config(3, 3, cfg, seed=7)
    b.trainer.deserialize(blob)
    assert torch.equal(a.trainer.params(), b.trainer.params())
    assert torch.equal(a.network.inference(xd), b.network.inference(xd))


def test_errors_fail_loudly(torch_cuda):
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    m = tcnn_b200.create_from_config(3, 3, cfg)
    torch = torch_cuda
    x = torch.zeros(100, 3, device="cuda")
    with pytest.raises(tcnn_b200.TcnnError):
        m.network.inference(x)  # batch not a multiple of 256 (object.h:217)
    bad = json.loads(json.dumps(cfg))
    bad["encoding"]["hash"] = "Prime"
    with pytest.raises(tcnn_b200.TcnnError, match="compiled without Prime"):
        tcnn_b200.create_from_config(3, 3, bad)
    bad = json.loads(json.dumps(cfg))
    bad["network"]["n_neurons"] = 48
    with pytest.raises(tcnn_b200.TcnnError, match="only supports 16, 32, 64, and 128"):
        tcnn_b200.create_from_config(3, 3, bad)


# ------------------------------------------------------------------------------------------------------------------
# Against the reference itself: tests/golden/*.npz were dumped by the UNMODIFIED reference (sm_100 build) on a B200.
# ------------------------------------------------------------------------------------------------------------------
from golden_util import CASES as GOLDEN_CASES, init_params_match, load_case, load_config, mlp_gradients_agree  # noqa: E402


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_against_reference_golden_vectors(torch_cuda, name):
    torch = torch_cuda
    import tcnn_b200

    _, n_in, n_out, B, _ = GOLDEN_CASES[name]
    g = load_case(name)
    cfg = load_config(name)
    model = tcnn_b200.create_from_config(n_in, n_out, cfg)
    x, y = g["x_f32"].reshape(B, n_in), g["y_f32"].reshape(B, n_out)
    xd, yd = torch.from_numpy(x.copy()).cuda(), torch.from_numpy(y.copy()).cuda()

    # initial parameters: bit-exact with the reference's Trainer (same pcg32 streams, same fp32 expressions)
    p0 = model.trainer.params_full_precision().cpu().numpy()
    assert init_params_match(g, p0)

    enc_tap = torch.zeros(B, 64, dtype=torch.float16, device="cuda")
    out_tap = torch.zeros(B, 16, dtype=torch.float16, device="cuda")
    lv_tap = torch.zeros(B, n_out, dtype=torch.float32, device="cuda")
    model.set_debug_taps(encoded=enc_tap, output=out_tap, loss_values=lv_tap)

    inf = model.network.inference(xd).cpu().numpy()
    assert rae(inf, g["inference_f32"].reshape(B, n_out), 99.0) < 1e-2  # tests/test_common.h:177

    model.trainer.training_step(xd, yd, run_optimizer=False)
    loss0 = model.trainer.loss()
    torch.cuda.synchronize()
    # encoded features == the reference's kernel_grid output, bit for bit (hash indices, cell selection, fp16 blend)
    W = g["meta"]["encoded_width"]
    assert np.array_equal(f16(enc_tap)[:, :W].T, g["encoded_f16"].reshape(W, B))
    a = ob.half_bits_to_float(f16(out_tap))[:, :n_out]
    b = ob.half_bits_to_float(g["output_f16"].reshape(B, 16))[:, :n_out]
    assert rae(a, b, 99.0) < 1e-2
    assert np.abs(a - b).max() <= 4 * 2.0 ** -24 + 4e-3 * np.abs(b).max()
    assert abs(loss0 - g["meta"]["losses"][0]) <= 1e-3 * g["meta"]["losses"][0]
    assert rae(lv_tap.cpu().numpy(), g["loss_values_f32"].reshape(B, 16)[:, :n_out], 99.0) < 1e-2

    # parameter gradients: tests/test_common.h:218 (mean RAE < 1.2e-2 on the best 99.9 %)
    grads = ob.half_bits_to_float(f16(model.trainer.param_gradients()))
    ref = ob.half_bits_to_float(g["grads_step0_f16"])
    n_mlp = model.n_mlp_params
    # The MLP weight gradients are where the accumulator model matters: the reference accumulates 512..2^18 products in
    # fp16 (CUTLASS split-K, cutlass_matmul.h:67), this kernel in fp32 (tcgen05). The reference's own two implementations
    # (offline vs JIT) differ by 1.17e-2 on this vector, the fp32-accumulating oracle sits 1.23e-2 / 1.34e-2 from them and
    # the fp16-accumulating oracle 7e-4 from the offline kernels (tests/test_oracle_golden.py): bar = 2e-2 for the MLP part.
    assert mlp_gradients_agree(grads[:n_mlp], ref[:n_mlp], 2e-2)
    assert rae(grads[n_mlp:], ref[n_mlp:], 99.9) < 1.2e-2
    assert ((grads[n_mlp:] != 0) != (ref[n_mlp:] != 0)).mean() < 2e-3

    # Adam: one step, then the whole 10-step trajectory
    lr = cfg["optimizer"]["learning_rate"]
    model.trainer.training_step(xd, yd)
    losses = [loss0, model.trainer.loss()]
    p1 = model.trainer.params_full_precision().cpu().numpy()
    d = np.abs(p1 - g["params_step1_f32"])
    assert np.percentile(d, 99) < 2e-2 * lr and d.mean() < 1e-2 * lr
    assert ((p1 != p0) != (g["params_step1_f32"] != p0)).mean() < 2e-3
    for _ in range(g["meta"]["n_steps"] - 1):
        model.trainer.training_step(xd, yd)
        losses.append(model.trainer.loss())
    for mine, theirs in zip(losses, g["meta"]["losses"]):
        assert abs(mine - theirs) <= 3e-2 * abs(theirs), (losses, g["meta"]["losses"])
    out = model.network.inference(xd).cpu().numpy()
    assert rae(out, g["inference_final_f32"].reshape(B, n_out), 99.0) < 5e-2
    pf = ob.half_bits_to_float(f16(model.trainer.params()))
    assert np.abs(pf - ob.half_bits_to_float(g["params_final_f16"])).mean() < 0.05 * lr * g["meta"]["n_steps"]


@pytest.mark.parametrize("activation,output_activation", [("LeakyReLU", "None"), ("Sigmoid", "None"), ("Tanh", "Sigmoid"), ("Squareplus", "None"), ("Softplus", "Exponential"), ("None", "None")])
def test_other_activations_match_oracle(torch_cuda, activation, output_activation):
    """FullyFusedMLP's activation set (fully_fused_mlp.cu:689-699), hidden and output, against the oracle's restatement of
    warp_activation / warp_activation_backward (common_device.h:110-215, 354-420)."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    cfg["network"]["activation"] = activation
    cfg["network"]["output_activation"] = output_activation
    cfg["loss"] = {"otype": "L2"}
    B = 512
    model = tcnn_b200.create_from_config(3, 3, cfg)
    orc = ob.OracleModel(3, 3, cfg, scales=model.grid_levels()["scales"])
    x, y = make_batch(3, 3, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    out_tap = torch.zeros(B, 16, dtype=torch.float16, device="cuda")
    model.set_debug_taps(output=out_tap)
    model.trainer.training_step(xd, yd, run_optimizer=False)
    loss = model.trainer.loss()
    torch.cuda.synchronize()
    ref_loss = orc.training_step(x, y, run_optimizer=False)
    enc = orc.encode(x)
    _, out_ref = orc.mlp_forward(enc)
    a = ob.half_bits_to_float(f16(out_tap))[:, :3]
    b = ob.half_bits_to_float(out_ref)[:, :3]
    assert rae(a, b, 99.0) < 2e-3, (activation, output_activation)  # fast-math exp/tanh vs libm
    assert abs(loss - ref_loss) <= 2e-3 * abs(ref_loss) + 1e-7
    g_dev = ob.half_bits_to_float(f16(model.trainer.param_gradients()))
    g_ref = ob.half_bits_to_float(orc.grads_fp16)
    assert rae(g_dev[: orc.n_mlp], g_ref[: orc.n_mlp], 99.9) < 1.2e-2
    assert rae(g_dev[orc.n_mlp :], g_ref[orc.n_mlp :], 99.9) < 1.2e-2
    with pytest.raises(tcnn_b200.TcnnError, match="Unsupported activation"):
        bad = json.loads(json.dumps(cfg))
        bad["network"]["activation"] = "Sine"
        tcnn_b200.create_from_config(3, 3, bad)


@pytest.mark.parametrize("width,n_hidden", [(16, 2), (32, 1), (32, 3), (64, 3)])
def test_network_shapes_match_oracle(torch_cuda, width, n_hidden):
    """FullyFusedMLP widths 16 / 32 / 64 (src/network.cu:116-123) and 1-3 hidden layers: 10 training steps track the oracle."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    cfg["network"]["n_neurons"] = width
    cfg["network"]["n_hidden_layers"] = n_hidden
    B = 512
    model = tcnn_b200.create_from_config(3, 3, cfg)
    orc = ob.OracleModel(3, 3, cfg, scales=model.grid_levels()["scales"])
    assert model.n_params == orc.n_params and model.n_mlp_params == orc.n_mlp == width * 32 + (n_hidden - 1) * width * width + 16 * width
    assert np.array_equal(model.trainer.params_full_precision().cpu().numpy().view(np.uint32), orc.params_fp32.view(np.uint32))
    x, y = make_batch(3, 3, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    model.trainer.training_step(xd, yd, run_optimizer=False)
    orc.training_step(x, y, run_optimizer=False)
    g_dev = ob.half_bits_to_float(f16(model.trainer.param_gradients()))
    g_ref = ob.half_bits_to_float(orc.grads_fp16)
    assert rae(g_dev[: orc.n_mlp], g_ref[: orc.n_mlp], 99.9) < 1.2e-2
    assert rae(g_dev[orc.n_mlp :], g_ref[orc.n_mlp :], 99.9) < 1.2e-2
    dev_losses, ref_losses = [], []
    for _ in range(10):
        model.trainer.training_step(xd, yd)
        dev_losses.append(model.trainer.loss())
        ref_losses.append(orc.training_step(x, y))
    for a, b in zip(dev_losses, ref_losses):
        assert abs(a - b) <= 3e-2 * abs(b) + 1e-6, (dev_losses, ref_losses)
    assert rae(model.network.inference(xd).cpu().numpy(), orc.inference(x), 99.0) < 5e-2


@pytest.mark.parametrize("batch", [512, 32768])
def test_module_tier_matches_trainer_tier_and_oracle(torch_cuda, batch):
    """tcnn::cpp::Module semantics (src/cpp_api.cu:71-158): caller-owned fp16 parameters, padded fp16 outputs, dL_dparams from an
    external dL_doutput. Checked against (i) the oracle's restatement of initialize_params, (ii) the trainer tier run on the
    same parameters (which the golden tests tie to the reference), (iii) the oracle's forward / backward on a small batch."""
    torch = torch_cuda
    import ctypes

    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    mod = tcnn_b200.Module(3, 3, cfg["encoding"], cfg["network"])
    model = tcnn_b200.create_from_config(3, 3, cfg)
    assert mod.n_params == model.n_params and mod.n_output_dims == 16
    orc = ob.OracleModel(3, 3, cfg, scales=model.grid_levels()["scales"])

    # (i) initialize_params(seed, params_full_precision, scale): pcg32{seed}, network weights then grid table
    for seed, scale in ((42, 1.0), (7, 0.5)):
        rng = ob.default_rng(seed)
        expect = np.zeros(orc.n_params, np.float32)
        orc.lib.orc_initialize_params(ctypes.byref(orc.grid), ctypes.byref(orc.mlp), ctypes.byref(rng), expect.ctypes.data_as(ctypes.c_void_p))
        got = mod.initial_params(seed, scale).cpu().numpy()
        if scale == 1.0:
            assert np.array_equal(got.view(np.uint32), expect.view(np.uint32))
        else:
            assert np.allclose(got, expect * scale, rtol=1e-6, atol=0)

    # (ii) same parameters as the trainer -> same outputs (bit for bit) and the same gradients
    x, y = make_batch(3, 3, batch)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    p16 = model.trainer.params().clone()
    out_tap = torch.zeros(batch, 16, dtype=torch.float16, device="cuda")
    dy_tap = torch.zeros(batch, 16, dtype=torch.float16, device="cuda")
    model.set_debug_taps(output=out_tap, dL_doutput=dy_tap)
    model.trainer.training_step(xd, yd, run_optimizer=False)
    g_trainer = ob.half_bits_to_float(f16(model.trainer.param_gradients()))
    out = mod.fwd(xd, p16)
    out_inf = mod.fwd(xd, p16, inference=True)
    torch.cuda.synchronize()
    assert np.array_equal(f16(out), f16(out_tap)) and np.array_equal(f16(out), f16(out_inf))
    g_mod = ob.half_bits_to_float(f16(mod.bwd(xd, p16, dy_tap, output=out)))
    n_mlp = model.n_mlp_params
    assert rae(g_mod[:n_mlp], g_trainer[:n_mlp], 99.9) < 1e-3          # fp32 sums, different accumulation order only
    assert rae(g_mod[n_mlp:], g_trainer[n_mlp:], 99.9) < 5e-3          # fp16 atomics in a different order
    # same set of touched table entries, up to sums that cancel to exactly zero in one accumulation order only
    assert ((g_mod[n_mlp:] != 0) != (g_trainer[n_mlp:] != 0)).mean() < 2e-3
    # gradients are OVERWRITTEN, not accumulated: a second call gives the same result
    g_again = ob.half_bits_to_float(f16(mod.bwd(xd, p16, dy_tap)))
    assert rae(g_again, g_mod, 99.9) < 5e-3

    # (iii) the oracle, with an arbitrary dL_doutput (small batch only: the oracle is a scalar CPU port)
    if batch <= 512:
        rng = np.random.default_rng(5)
        dy = (rng.standard_normal((batch, 16)) * 1e-2).astype(np.float16)
        dy[:, 3:] = 0
        enc = orc.encode(x)
        hidden, out_ref = orc.mlp_forward(enc)
        assert np.array_equal(f16(out), out_ref.view(np.uint16).reshape(batch, 16)) or rae(ob.half_bits_to_float(f16(out)), ob.half_bits_to_float(out_ref), 99.0) < 2e-3
        g_ref = orc.backward_from_dy(x, dy.view(np.uint16))
        g_dev = ob.half_bits_to_float(f16(mod.bwd(xd, p16, torch.from_numpy(dy).cuda())))
        assert rae(g_dev[:n_mlp], g_ref[:n_mlp], 99.9) < 1.2e-2
        assert rae(g_dev[n_mlp:], g_ref[n_mlp:], 99.9) < 1.2e-2

    # the two tiers do not mix, and unsupported requests fail loudly
    with pytest.raises(tcnn_b200.TcnnError, match="tcnnb_module_"):
        tcnn_b200._check(tcnn_b200.load().tcnnb_training_step(mod._h, None, batch, xd.data_ptr(), yd.data_ptr(), 0))
    # prepare_input_gradients is accepted (nothing to prepare: backward recomputes the forward pass)
    tcnn_b200._check(tcnn_b200.load().tcnnb_module_forward(mod._h, None, batch, xd.data_ptr(), out.data_ptr(), p16.data_ptr(), 1))


def test_torch_autograd_layer_on_the_module_tier(torch_cuda):
    """tcnn_b200.torch_modules mirrors tinycudann's modules.py: fp32 nn.Parameter, fp16 compute, batch padding to 256,
    loss-scaled backward. The gradients autograd delivers must be the native module's, and a plain torch optimizer must train."""
    torch = torch_cuda
    import tcnn_b200
    import tcnn_b200.torch_modules as tcnn

    cfg = load_cfg("hash3d_small")
    torch.manual_seed(0)
    model = tcnn.NetworkWithInputEncoding(3, 3, cfg["encoding"], cfg["network"], seed=1337)
    assert model.params.dtype == torch.float32 and model.params.numel() == model.native_tcnn_module.n_params
    B = 1000  # not a multiple of 256: exercises the padding path (modules.py:222-226)
    x = torch.rand(B, 3, device="cuda")
    y = torch.stack([torch.sin(7 * x[:, 0]) * 0.5 + 0.5, x[:, 1] * x[:, 2], torch.cos(5 * x[:, 2]) * 0.5 + 0.5], 1)

    out = model(x)
    assert out.shape == (B, 3) and out.dtype == torch.float16
    ((out.float() - y) ** 2).sum().backward()  # O(1) output gradients: the fp16 parameter gradients stay well above the fp16 floor
    g_autograd = model.params.grad.clone()
    # the same thing by hand on the native module: pad, dL/dout = 2 (out - y) scaled by 128, native backward, unscale
    xp = torch.nn.functional.pad(x, [0, 0, 0, 1024 - B]).contiguous()
    p16 = model.params.detach().to(torch.float16).contiguous()
    full = model.native_tcnn_module.fwd(xp, p16)
    dy = torch.zeros_like(full)
    dy[:B, :3] = (2 * (full[:B, :3].float() - y) * model.loss_scale).to(torch.float16)
    g_native = model.native_tcnn_module.bwd(xp, p16, dy).float() / model.loss_scale
    torch.cuda.synchronize()
    a, b = g_autograd.cpu().numpy(), g_native.cpu().numpy()
    n_mlp = 7168
    assert rae(a[:n_mlp], b[:n_mlp], 99.9) < 2e-3 and rae(a[n_mlp:], b[n_mlp:], 99.9) < 5e-3

    opt = torch.optim.Adam(model.parameters(), lr=1e-2, eps=1e-15)
    losses = []
    for _ in range(60):
        opt.zero_grad()
        loss = ((model(x).float() - y) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert losses[-1] < 0.1 * losses[0], losses[::10]
    xg = x.clone().requires_grad_(True)
    model(xg).float().sum().backward()  # input gradients are delivered (tests/test_gpu_encoding.py checks their values)
    assert xg.grad is not None and torch.isfinite(xg.grad).all()


@pytest.mark.parametrize("loss", ["L1", "RelativeL1", "Mape", "Smape", "RelativeL2Luminance", "CrossEntropy", "Variance"])
def test_other_losses_match_oracle(torch_cuda, loss):
    """src/loss.cu:57-65: the element-wise losses beside L2 / RelativeL2 (losses/l1.h:68-73, relative_l1.h:71-76, mape.h:72-77,
    smape.h:72-77), fused into the output epilogue like them: loss values, loss gradients and everything downstream against the oracle."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    cfg["loss"] = {"otype": loss}
    if loss in ("CrossEntropy", "Variance"):  # log(prediction) / 1 / prediction (cross_entropy.h:66-75, variance_is.h:66-76): predictions in (0, 1)
        cfg["network"]["output_activation"] = "Sigmoid"
    B = 1024
    model = tcnn_b200.create_from_config(3, 3, cfg)
    assert model.hyperparams()["loss"]["otype"] == loss
    orc = ob.OracleModel(3, 3, cfg, scales=model.grid_levels()["scales"])
    x, y = make_batch(3, 3, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    out_tap = torch.zeros(B, 16, dtype=torch.float16, device="cuda")
    dy_tap = torch.zeros(B, 16, dtype=torch.float16, device="cuda")
    lv_tap = torch.zeros(B, 3, dtype=torch.float32, device="cuda")
    model.set_debug_taps(output=out_tap, dL_doutput=dy_tap, loss_values=lv_tap)
    model.trainer.training_step(xd, yd, run_optimizer=False)
    loss_dev = model.trainer.loss()
    torch.cuda.synchronize()
    lv_ref, dy_ref = orc.loss(f16(out_tap), y)  # the oracle's loss on the DEVICE's outputs: isolates the epilogue
    assert rae(lv_tap.cpu().numpy(), lv_ref[:, :3]) < 1e-3
    a, b = ob.half_bits_to_float(f16(dy_tap)), ob.half_bits_to_float(dy_ref)
    if cfg["network"].get("output_activation", "None") == "Sigmoid":
        # the device's tap sits behind the output activation's transfer (fully_fused_mlp.cu:755-762): grad * y (1 - y), fp16 products
        yv = ob.half_bits_to_float(f16(out_tap))
        b = (b.astype(np.float16) * (yv.astype(np.float16) * (1 - yv).astype(np.float16))).astype(np.float32)
    # sign(difference) flips where prediction == target to fp16 rounding; everywhere else the gradients agree to fp16 rounding
    assert (np.abs(a - b) > 2e-3 * np.abs(b).max()).mean() < 1e-3
    assert abs(loss_dev - float(lv_ref.sum(dtype=np.float64))) <= 1e-4 * abs(loss_dev)
    model.set_debug_taps()
    dev_losses, ref_losses = [], []
    for _ in range(8):
        model.trainer.training_step(xd, yd)
        dev_losses.append(model.trainer.loss())
        ref_losses.append(orc.training_step(x, y))
    assert dev_losses[-1] < dev_losses[0] or loss in ("CrossEntropy", "Variance")  # (those two are not distances to the target)
    for u, v in zip(dev_losses, ref_losses):
        assert abs(u - v) <= 5e-2 * abs(v) + 1e-6, (dev_losses, ref_losses)


def test_exponential_decay_wrapper_follows_the_schedule(torch_cuda):
    """optimizers/exponential_decay.h:60-70 around Adam: from decay_start on, every decay_interval steps the learning rate is
    multiplied by decay_base. The trajectory equals the oracle's Adam driven with the same per-step learning rates."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    adam = dict(cfg["optimizer"])
    cfg["optimizer"] = {"otype": "ExponentialDecay", "decay_start": 2, "decay_interval": 2, "decay_base": 0.5, "decay_end": 6, "nested": adam}
    B = 512
    model = tcnn_b200.create_from_config(3, 3, cfg)
    ocfg = load_cfg("hash3d_small")
    orc = ob.OracleModel(3, 3, ocfg, scales=model.grid_levels()["scales"])
    x, y = make_batch(3, 3, B)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    factor, base_lr = 1.0, adam["learning_rate"]
    for step in range(9):
        if step >= 2 and (step - 2) % 2 == 0 and step <= 6:
            factor *= 0.5
        orc.adam.learning_rate = base_lr * factor
        model.trainer.training_step(xd, yd)
        a, b = model.trainer.loss(), orc.training_step(x, y)
        assert abs(a - b) <= 3e-2 * abs(b) + 1e-6, (step, a, b)
    assert factor == 0.125
    p = model.trainer.params_full_precision().cpu().numpy()
    assert np.abs(p - orc.params_fp32).mean() < 0.05 * base_lr * 9
    # without the schedule the parameters would have moved further: the schedule is really applied
    plain = tcnn_b200.create_from_config(3, 3, ocfg)
    for _ in range(9):
        plain.trainer.training_step(xd, yd)
    p0 = ob.OracleModel(3, 3, ocfg).params_fp32
    assert np.abs(plain.trainer.params_full_precision().cpu().numpy() - p0).mean() > 1.3 * np.abs(p - p0).mean()
    with pytest.raises(tcnn_b200.TcnnError, match="outside the tcnn_b200 hot path"):
        bad = json.loads(json.dumps(ocfg))
        bad["optimizer"] = {"otype": "Shampoo"}
        tcnn_b200.create_from_config(3, 3, bad)


def test_ema_wrapper_averages_the_weights_inference_reads(torch_cuda):
    """optimizers/ema.h:46-132 around (ExponentialDecay around) Adam: after every step the debiased moving average of the fp16 working weights
    is updated; network->inference() reads the average (Trainer::params_inference, trainer.h:497-502), training keeps the raw weights."""
    torch = torch_cuda
    import tcnn_b200

    cfg = load_cfg("hash3d_small")
    decay = 0.9
    cfg["optimizer"] = {"otype": "Ema", "decay": decay, "nested": {"otype": "ExponentialDecay", "decay_start": 2, "decay_interval": 2, "decay_base": 0.5, "nested": cfg["optimizer"]}}
    model = tcnn_b200.create_from_config(3, 3, cfg)
    plain_cfg = json.loads(json.dumps(cfg))
    plain_cfg["optimizer"] = cfg["optimizer"]["nested"]
    plain = tcnn_b200.create_from_config(3, 3, plain_cfg)
    x, y = make_batch(3, 3, 512)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    assert torch.equal(model.trainer.params_inference(), model.trainer.params())  # starts as the initial parameters (trainer.h:415-419)
    ema = None
    for step in range(1, 7):
        model.trainer.training_step(xd, yd)
        plain.trainer.training_step(xd, yd)
        w = model.trainer.params().float().cpu().numpy()
        # ema.h:46-75 restated: fp16 storage of the average, fp32 arithmetic
        prev = np.zeros_like(w) if ema is None else ema
        ema = ((prev * np.float32(decay) * np.float32(1 - decay ** (step - 1)) + w * np.float32(1 - decay)) * np.float32(1.0 / (1 - decay ** step))).astype(np.float16).astype(np.float32)
        got = model.trainer.params_inference().float().cpu().numpy()
        assert np.abs(got - ema).max() <= 2.0 ** -10 * max(1e-3, np.abs(ema).max()), step
    # the wrapper does not touch training: the plain optimizer arrives at the same weights (up to the order of the fp16 atomics)
    pw, mw = plain.trainer.params().float(), model.trainer.params().float()
    assert float((pw - mw).abs().mean()) < 0.02 * float((mw - model.trainer.params_inference().float()).abs().mean()) + 1e-6
    # inference reads the averaged weights: equal to the plain model's inference once it is given them
    out = model.network.inference(xd)
    plain.trainer.set_params(model.trainer.params_inference())
    assert torch.equal(out, plain.network.inference(xd))
    assert not torch.equal(model.trainer.params_inference(), model.trainer.params())
