"""Pins oracle/oracle_cpu.cpp against the reference itself: vectors dumped by the UNMODIFIED reference (compiled from
/root/reference, run on a B200) and committed under tests/golden/. Integer/bit-level quantities must match exactly;
floating-point stages are held to the reference's own test tolerances (tests/test_common.h:153-219). CPU only."""
import numpy as np
import pytest

import oracle_binding as ob
from golden_util import CASES, device_scales, init_params_match, load_case, load_config, mlp_gradients_agree, rae

h2f = ob.half_bits_to_float


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    name = request.param
    cfg_file, n_in, n_out, B, _ = CASES[name]
    g = load_case(name)
    cfg = load_config(name)
    scales, probe = device_scales(name, cfg["encoding"]["n_levels"])
    return dict(name=name, n_in=n_in, n_out=n_out, B=B, g=g, cfg=cfg, scales=scales, probe=probe)


def test_probe_host_scale_matches_oracle(case):
    """The reference's HOST evaluation of grid_scale (sizing, grid.h:701) equals the oracle's; its DEVICE evaluation
    differs in the last bits at some levels (SURVEY.md §7 hard part) but never in the resolution."""
    m = ob.OracleModel(case["n_in"], case["n_out"], case["cfg"])
    for l, lv in enumerate(case["probe"]["levels"][: m.grid.n_levels]):
        assert np.float32(m.grid.scales[l]).view(np.uint32) == lv["host_bits"]
        assert m.grid.resolutions[l] == lv["host_res"] == lv["dev_res"]


def test_inputs_and_initial_parameters_bit_exact(case):
    g, n_in, n_out, B = case["g"], case["n_in"], case["n_out"], case["B"]
    rng = ob.default_rng(1337)
    x = ob.generate_random_uniform(rng, B * n_in)
    assert np.array_equal(x.view(np.uint32), g["x_f32"].view(np.uint32))
    y = ob.make_targets(x.reshape(B, n_in), n_out)
    assert np.abs(y.ravel() - g["y_f32"]).max() < 5e-7  # sinf: numpy vs glibc
    m = ob.OracleModel(n_in, n_out, case["cfg"])
    assert m.n_params == g["meta"]["n_params"]
    assert m.grid.n_params == g["meta"]["n_encoding_params"]
    assert init_params_match(g, m.params_fp32)


def test_encoded_features_bit_exact(case):
    """kernel_grid output of the reference == oracle restatement, bit for bit, once the oracle uses the device scales."""
    g, n_in, B = case["g"], case["n_in"], case["B"]
    m = ob.OracleModel(n_in, case["n_out"], case["cfg"], scales=case["scales"])
    x = g["x_f32"].reshape(B, n_in)
    enc = m.encode(x)
    ref = g["encoded_f16"].reshape(g["meta"]["encoded_width"], B)
    assert g["meta"]["encoded_layout"] == "SoA"
    assert np.array_equal(enc, ref)


def test_forward_loss_within_reference_tolerances(case):
    g, n_in, n_out, B = case["g"], case["n_in"], case["n_out"], case["B"]
    x, y = g["x_f32"].reshape(B, n_in), g["y_f32"].reshape(B, n_out)
    out_ref = g["output_f16"].reshape(B, 16)
    for mode in (ob.ACCUM_FP16_K16, ob.ACCUM_FP32):
        m = ob.OracleModel(n_in, n_out, case["cfg"], accum_mode=mode, scales=case["scales"])
        enc = m.encode(x)
        _, out = m.mlp_forward(enc)
        # At initialisation the outputs are ~1e-5, i.e. fp16 SUBNORMALS (quantum 6e-8 = 0.3 % of the value): the bar is
        # the reference's own JIT-vs-offline bar (tests/test_common.h:177: 1e-2 on the best 99 %) plus an absolute bound
        # of a few subnormal quanta.
        a, b = h2f(out[:, :n_out]), h2f(out_ref[:, :n_out])
        assert rae(a, b, 99.0) < 1e-2, mode
        assert np.abs(a - b).max() <= 4 * 2.0 ** -24 + 4e-3 * np.abs(b).max(), mode
        inf = m.inference(x)
        assert rae(inf, g["inference_f32"].reshape(B, n_out), 99.0) < 1e-2
    # loss kernel on the reference's own fp16 output: tests/test_jit_losses.cu:109-110 bar is 1e-3
    values, grads = m.loss(out_ref, y)
    lv_ref = g["loss_values_f32"].reshape(B, 16)
    assert rae(values, lv_ref) < 1e-5
    assert np.all(lv_ref[:, n_out:] == 0)
    assert abs(values.sum(dtype=np.float64) - g["meta"]["losses"][0]) < 1e-4 * g["meta"]["losses"][0]


def test_gradients_and_adam_within_reference_tolerances(case):
    g, n_in, n_out, B = case["g"], case["n_in"], case["n_out"], case["B"]
    x, y = g["x_f32"].reshape(B, n_in), g["y_f32"].reshape(B, n_out)
    m = ob.OracleModel(n_in, n_out, case["cfg"], accum_mode=ob.ACCUM_FP16_K16, scales=case["scales"])
    p0 = m.params_fp32.copy()
    assert init_params_match(g, p0)
    loss0 = m.training_step(x, y, run_optimizer=False)
    assert abs(loss0 - g["meta"]["losses"][0]) < 1e-3 * g["meta"]["losses"][0]
    grads = h2f(m.grads_fp16)
    ref = h2f(g["grads_step0_f16"])
    n_mlp = m.n_mlp
    # tests/test_common.h:218: parameter gradients, mean RAE < 1.2e-2 on the best 99.9 %
    assert mlp_gradients_agree(grads[:n_mlp], ref[:n_mlp], 1.2e-2)
    assert rae(grads[n_mlp:], ref[n_mlp:], 99.9) < 1.2e-2
    # the set of table entries that receive gradient is an integer property: identical
    assert np.array_equal(grads[n_mlp:] != 0, ref[n_mlp:] != 0) or ((grads[n_mlp:] != 0) != (ref[n_mlp:] != 0)).mean() < 2e-3
    # one Adam step
    loss1 = m.training_step(x, y)
    p1 = g["params_step1_f32"]
    lr = case["cfg"]["optimizer"]["learning_rate"]
    moved_ref = p1 != p0
    moved = m.params_fp32 != p0
    assert (moved != moved_ref).mean() < 2e-3  # zero-gradient skip (adam.h:79-82)
    # first Adam step = lr * sign(g) (bias-corrected m/sqrt(v)), so parameters agree to ~1e-3 * lr except where a tiny
    # gradient changes sign between implementations
    d = np.abs(m.params_fp32 - p1)
    assert np.percentile(d, 99) < 2e-2 * lr
    assert d.mean() < 1e-2 * lr


def test_training_trajectory(case):
    g, n_in, n_out, B = case["g"], case["n_in"], case["n_out"], case["B"]
    x, y = g["x_f32"].reshape(B, n_in), g["y_f32"].reshape(B, n_out)
    m = ob.OracleModel(n_in, n_out, case["cfg"], accum_mode=ob.ACCUM_FP16_K16, scales=case["scales"])
    ref_losses = g["meta"]["losses"]  # [fwd/bwd only, step 1, ..., step n]
    losses = [m.training_step(x, y, run_optimizer=False)] + [m.training_step(x, y) for _ in range(g["meta"]["n_steps"])]
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) <= 3e-2 * abs(b), (losses, ref_losses)
    out = m.inference(x)
    assert rae(out, g["inference_final_f32"].reshape(B, n_out), 99.0) < 5e-2


def test_jit_and_offline_reference_modes_agree_with_oracle():
    """The reference's two own implementations (offline kernels vs JIT-fused kernel) differ from each other by about as
    much as the oracle differs from either -- the tolerance budget of the parity tests is the reference's own spread."""
    a, b = load_case("hash3d_small"), load_case("hash3d_small_jit")
    ga, gb = h2f(a["grads_step0_f16"]), h2f(b["grads_step0_f16"])
    spread = rae(ga, gb, 99.9)
    assert spread < 1.2e-2
    cfg = load_config("hash3d_small")
    scales, _ = device_scales("hash3d_small", 16)
    m = ob.OracleModel(3, 3, cfg, accum_mode=ob.ACCUM_FP32, scales=scales)
    m.training_step(a["x_f32"].reshape(512, 3), a["y_f32"].reshape(512, 3), run_optimizer=False)
    go = h2f(m.grads_fp16)
    assert rae(go, ga, 99.9) < max(1.2e-2, 2 * spread)
    assert rae(go, gb, 99.9) < max(1.2e-2, 2 * spread)
