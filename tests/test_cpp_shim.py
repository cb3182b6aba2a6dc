"""The C++ source-compatibility headers (include/tiny-cuda-nn/*.h): an application written against tiny-cuda-nn's names
(tests/cpp/shim_sample.cu, modelled on the reference's samples/mlp_learning_an_image.cu) compiles against them, links
libtcnn_b200.so and trains. The binary is built by `__graft_entry__.build()` (nvcc cross-compiles without a GPU)."""
import json
import os
import subprocess

import numpy as np
import pytest

import oracle_binding as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "shim_sample")


def test_shim_headers_exist_and_cite_the_reference():
    inc = os.path.join(ROOT, "include", "tiny-cuda-nn")
    for h in ("common.h", "common_device.h", "config.h", "gpu_matrix.h", "gpu_memory.h", "random.h", "trainer.h", "network_with_input_encoding.h", "loss.h", "optimizer.h", "network.h", "encoding.h"):
        text = open(os.path.join(inc, h)).read()
        assert "#pragma once" in text
    assert "trainer.h:254-357" in open(os.path.join(inc, "config.h")).read()


@pytest.mark.gpu
def test_shim_sample_trains(torch_cuda):
    if not os.path.exists(BIN):
        pytest.skip("tests/cpp/shim_sample has not been built (python __graft_entry__.py build)")
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "tiny-cuda-nn_b200") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([BIN, "300"], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr
    r = json.loads(out.stdout.strip().splitlines()[-1])
    # HashGrid(2-D, L=16, F=2, T=2^15, base 16, s=1.5): 6 dense + 10 hashed levels = 354 184 entries (SURVEY.md appendix B) + 64x32+64x64+16x64 weights
    assert r["n_params"] == 354184 * 2 + 7168 and r["padded_output_width"] == 16
    assert r["last_loss"] < 0.05 * r["first_loss"], r
    assert r["inference_mse"] < 5e-3, r
    assert np.isfinite(r["create_from_config_loss"]) and abs(r["create_from_config_loss"] - r["first_loss"]) / r["first_loss"] < 0.5
    # default_rng_t{1337} + generate_random_uniform == the reference's generator (random.h:40-69), via the oracle restatement
    expect = ob.generate_random_uniform(ob.default_rng(1337), 8)
    assert np.array_equal(np.array(r["first_uniform"], np.float32), expect)


def test_shim_sample_compiles_without_a_gpu():
    """nvcc cross-compiles the application against the compatibility headers (compile only, no link, no GPU)."""
    import shutil
    import sys
    import tempfile

    sys.path.insert(0, ROOT)
    from __graft_entry__ import json_include_dir

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    inc = json_include_dir()
    if not os.path.exists(nvcc) or inc is None:
        pytest.skip("nvcc or nlohmann/json.hpp not available")
    with tempfile.TemporaryDirectory() as tmp:
        out = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", os.path.join(ROOT, "include"), "-I", inc, "-c",
                              os.path.join(ROOT, "tests", "cpp", "shim_sample.cu"), "-o", os.path.join(tmp, "shim_sample.o")], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]


# ------------------------------------------------------------------------------------------------------------------
# SURVEY.md section 8(b) acceptance test: the reference's OWN application sources, unmodified, against this library's headers.
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src", ["samples/mlp_learning_an_image.cu", "benchmarks/image/bench_ours.cu"])
def test_unmodified_reference_sources_compile_against_the_shim(src):
    import shutil
    import sys
    import tempfile

    if not os.path.exists(os.path.join("/root/reference", src)):
        pytest.skip("/root/reference is not mounted here (GPU box): the binaries were built in the build container")
    sys.path.insert(0, ROOT)
    from __graft_entry__ import reference_sample_command

    if not (shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc")):
        pytest.skip("nvcc not available")
    with tempfile.TemporaryDirectory() as tmp:
        out = subprocess.run(reference_sample_command(src, os.path.join(tmp, "a.o"), compile_only=True), capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]


@pytest.mark.gpu
def test_unmodified_reference_sample_trains(torch_cuda, tmp_path):
    """tests/cpp/ref_mlp_learning_an_image = the reference's samples/mlp_learning_an_image.cu, byte for byte, linked against
    libtcnn_b200: 300 training steps on a synthetic image with the reference's data/config_hash.json settings."""
    import re

    exe = os.path.join(ROOT, "tests", "cpp", "ref_mlp_learning_an_image")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/ref_mlp_learning_an_image has not been built (needs /root/reference at build time)")
    # a smooth 256 x 256 RGB test image as binary PPM (stb_image reads PNM)
    h = w = 256
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32) / h
    img = np.stack([0.5 + 0.5 * np.sin(9 * xx + 3 * yy), 0.5 + 0.5 * np.cos(7 * yy), xx * yy], -1)
    with open(tmp_path / "img.ppm", "wb") as f:
        f.write(b"P6\n%d %d\n255\n" % (w, h))
        f.write((np.clip(img, 0, 1) * 255).astype(np.uint8).tobytes())
    cfg = json.load(open(os.path.join(ROOT, "tests", "golden", "configs", "image2d.json")))
    json.dump(cfg, open(tmp_path / "config.json", "w"))
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "tiny-cuda-nn_b200") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    out = subprocess.run([exe, str(tmp_path / "img.ppm"), str(tmp_path / "config.json"), "300", str(tmp_path / "learned.jpg")], capture_output=True, text=True, timeout=600, env=env,
                         cwd=str(tmp_path))
    assert out.returncode == 0 and "Uncaught exception" not in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    losses = [float(m) for m in re.findall(r"Step#\d+: loss=([0-9.eE+-]+)", out.stdout)]
    assert len(losses) >= 3 and losses[-1] < 0.2 * losses[0], out.stdout[-1500:]
    assert os.path.getsize(tmp_path / "learned.jpg") > 1000 and os.path.exists(tmp_path / "reference.jpg")


def msgpack_decode(b):
    """The part of MessagePack that nlohmann::json::to_msgpack writes for a snapshot: maps, arrays, strings, binaries, numbers."""
    import struct

    def num(i, fmt):
        n = struct.calcsize(fmt)
        return struct.unpack(">" + fmt, b[i : i + n])[0], i + n

    def seq(n, i, pairs):
        out = {} if pairs else []
        for _ in range(n):
            if pairs:
                k, i = val(i)
                out[k], i = val(i)
            else:
                v, i = val(i)
                out.append(v)
        return out, i

    def val(i):
        t = b[i]
        i += 1
        if t <= 0x7F or t >= 0xE0:
            return (t if t <= 0x7F else t - 256), i
        if t <= 0x8F or 0x90 <= t <= 0x9F:
            return seq(t & 0x0F, i, t <= 0x8F)
        if 0xA0 <= t <= 0xBF:
            return b[i : i + (t & 0x1F)].decode(), i + (t & 0x1F)
        if t in (0xC0, 0xC2, 0xC3):
            return {0xC0: None, 0xC2: False, 0xC3: True}[t], i
        if t in (0xC4, 0xC5, 0xC6, 0xD9, 0xDA, 0xDB):
            n, i = num(i, {0xC4: "B", 0xC5: "H", 0xC6: "I", 0xD9: "B", 0xDA: "H", 0xDB: "I"}[t])
            return (bytes(b[i : i + n]) if t <= 0xC6 else b[i : i + n].decode()), i + n
        if t in (0xDC, 0xDD, 0xDE, 0xDF):
            n, i = num(i, "H" if t in (0xDC, 0xDE) else "I")
            return seq(n, i, t >= 0xDE)
        fmt = {0xCA: "f", 0xCB: "d", 0xCC: "B", 0xCD: "H", 0xCE: "I", 0xCF: "Q", 0xD0: "b", 0xD1: "h", 0xD2: "i", 0xD3: "q"}.get(t)
        if fmt is None:
            raise ValueError(f"msgpack type 0x{t:02x} is not part of a snapshot")
        return num(i, fmt)

    v, end = val(0)
    assert end == len(b)
    return v


def snapshot_schema(v):
    """Keys, value kinds and binary sizes of a decoded snapshot: what decides whether a reader accepts it."""
    if isinstance(v, dict):
        return {k: snapshot_schema(x) for k, x in v.items()}
    if isinstance(v, bytes):
        return ("bytes", len(v))
    return type(v if not isinstance(v, float) else 0.0).__name__


@pytest.mark.gpu
@pytest.mark.parametrize("with_optimizer", [0, 1])
def test_snapshots_interoperate_with_the_reference(torch_cuda, tmp_path, with_optimizer):
    """trainer->serialize() / deserialize() (trainer.h:442-482, optimizers/adam.h:303-325) exchange the reference's JSON schema.
    tests/golden/snapshot_small.npz holds snapshots the UNMODIFIED reference wrote (msgpack, as instant-ngp stores them) at
    initialisation and after 20 steps, and its inference after the 20 steps. The 20-step snapshot loads into this library and
    reproduces the reference's inference; the snapshot this library writes at initialisation decodes to exactly the reference's, and
    the one it writes after 20 steps has the reference's keys, value kinds and sizes and loads back into this library."""
    exe = os.path.join(ROOT, "tests", "cpp", "snapshot_interop")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/snapshot_interop has not been built")
    from golden_util import GOLDEN, rae

    g = np.load(os.path.join(GOLDEN, "snapshot_small.npz"))
    meta = json.loads(bytes(g["meta"]).decode())
    cfg = os.path.join(GOLDEN, "configs", "snapshot_small.json")
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "tiny-cuda-nn_b200") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    d = str(tmp_path)
    B = str(meta["batch"])
    g["x_f32"].tofile(os.path.join(d, "x.f32"))
    g["y_f32"].tofile(os.path.join(d, "y.f32"))
    ref0, ref20 = (g[f"snapshot_opt{with_optimizer}_step{n}"].tobytes() for n in (0, 20))
    open(os.path.join(d, "snapshot.msgpack"), "wb").write(ref20)

    def run(cmd):
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
        return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])

    # reference -> this library
    loaded = run([exe, "load", cfg, "3", "3", B, d, os.path.join(d, "snapshot.msgpack")])
    ref = g[f"inference_snapshot_opt{with_optimizer}_step20_f32"]
    ours = np.fromfile(os.path.join(d, "inference_loaded.f32"), np.float32)
    assert rae(ours, ref, 99.0) < 1e-2  # same parameters, the two forward kernels (tests/test_common.h:177)
    assert loaded["has_optimizer"] == bool(with_optimizer)
    # the step after loading continues the reference's trajectory (with its optimizer state: moments + per-parameter step counters)
    assert loaded["next_step_loss"] < 1.5 * meta["last_loss"][f"snapshot_opt{with_optimizer}_step20"] + 1e-6
    # this library -> reference: at initialisation the parameters are bit-exact with the reference's, so the whole snapshot must be
    run([exe, "save", cfg, "3", "3", B, d, "0", str(with_optimizer)])
    assert msgpack_decode(open(os.path.join(d, "snapshot_b200.msgpack"), "rb").read()) == msgpack_decode(ref0)
    run([exe, "save", cfg, "3", "3", B, d, "20", str(with_optimizer)])
    ours20 = open(os.path.join(d, "snapshot_b200.msgpack"), "rb").read()
    assert snapshot_schema(msgpack_decode(ours20)) == snapshot_schema(msgpack_decode(ref20))
    back = run([exe, "load", cfg, "3", "3", B, d, os.path.join(d, "snapshot_b200.msgpack")])
    ours2 = np.fromfile(os.path.join(d, "inference_b200.f32"), np.float32)
    back2 = np.fromfile(os.path.join(d, "inference_loaded.f32"), np.float32)
    assert rae(back2, ours2, 99.0) < 1e-2
    assert np.isfinite(back["next_step_loss"])


def test_unmodified_reference_torch_bindings_compile_against_cpp_api_h():
    """bindings/torch/tinycudann/bindings.cpp (the PyTorch extension's C++ half, which includes only <tiny-cuda-nn/cpp_api.h>) compiles
    UNCHANGED against this repo's include/tiny-cuda-nn/cpp_api.h: same tcnn::cpp::Module interface, factories and free functions."""
    import sysconfig
    import tempfile

    src = "/root/reference/bindings/torch/tinycudann/bindings.cpp"
    if not os.path.exists(src):
        pytest.skip("/root/reference is not mounted here")
    from torch.utils.cpp_extension import include_paths

    with tempfile.TemporaryDirectory() as tmp:
        cmd = ["g++", "-std=c++17", "-O0", "-w", "-c", src, "-o", os.path.join(tmp, "bindings.o"), "-I" + os.path.join(ROOT, "include"), "-I/root/reference/dependencies",
               "-I/usr/local/cuda/include", "-I" + sysconfig.get_paths()["include"], "-DTCNN_PARAMS_UNALIGNED", "-DTORCH_EXTENSION_NAME=_C"]
        for inc in include_paths():
            cmd += ["-I", inc]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
