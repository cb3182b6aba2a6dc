#!/usr/bin/env python3
"""Pack the raw dumps of oracle/ref_harness.cu (gpurun_out/golden/<case>/) into tests/golden/<case>.npz.

Usage: python tests/golden/pack_golden.py gpurun_out/golden tests/golden
The .npz files are the committed fixtures; they were produced by the unmodified reference (built from /root/reference by
oracle/Makefile) running on a B200 via tests/golden/make_golden.sh.
"""
import glob
import hashlib
import json
import os
import sys

import numpy as np

DT = {"f32": np.float32, "f16": np.uint16}
# the tests of the composite / parameter-free encoding cases check gradients and losses, not post-step parameters
NO_POST_STEP_PARAMS = ("composite_nrc", "composite_grid_sh", "frequency_top")
MAX_BYTES = 1_000_000


def save_case(path, name, arrays):
    """np.savez_compressed, kept under MAX_BYTES by leaving out what a case's tests can do without: first the post-step parameters of
    the cases in NO_POST_STEP_PARAMS, then the initial parameters, whose SHA-256 goes into meta instead (the tests compare the digest,
    which is as exact as the bits)."""
    np.savez_compressed(path, **arrays)
    if os.path.getsize(path) > MAX_BYTES and name in NO_POST_STEP_PARAMS:
        arrays = {k: v for k, v in arrays.items() if k not in ("params_step1_f32", "params_final_f16")}
        np.savez_compressed(path, **arrays)
    if os.path.getsize(path) > MAX_BYTES and "params_init_f32" in arrays:
        meta = json.loads(bytes(arrays["meta"]).decode())
        meta["params_init_sha256"] = hashlib.sha256(arrays["params_init_f32"].tobytes()).hexdigest()
        arrays = {k: v for k, v in arrays.items() if k != "params_init_f32"}
        arrays["meta"] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
        np.savez_compressed(path, **arrays)
    assert os.path.getsize(path) <= MAX_BYTES, path


def pack_snapshots(src, dst):
    """<src>/snapshot_opt<0|1>_step<n>/ (ref_harness snapshot save) -> <dst>/snapshot_small.npz: each msgpack file as uint8, the
    inference after it, the shared inputs / targets, and the last training loss per snapshot in meta."""
    dirs = sorted(glob.glob(os.path.join(src, "snapshot_opt*_step*")))
    if not dirs:
        return
    arrays = {"x_f32": np.fromfile(os.path.join(dirs[0], "x.f32"), np.float32), "y_f32": np.fromfile(os.path.join(dirs[0], "y.f32"), np.float32)}
    last_loss = {}
    for d in dirs:
        name = os.path.basename(d)
        arrays[name] = np.fromfile(os.path.join(d, "snapshot.msgpack"), np.uint8)
        arrays[f"inference_{name}_f32"] = np.fromfile(os.path.join(d, "inference.f32"), np.float32)
        last_loss[name] = json.load(open(os.path.join(d, "save.json")))["last_loss"]
    arrays["meta"] = np.frombuffer(json.dumps({"batch": 1024, "n_in": 3, "n_out": 3, "last_loss": last_loss}).encode(), np.uint8)
    save_case(os.path.join(dst, "snapshot_small.npz"), "snapshot_small", arrays)


src, dst = sys.argv[1], sys.argv[2]
for case in sorted(glob.glob(os.path.join(src, "*", "meta.json"))):
    d = os.path.dirname(case)
    name = os.path.basename(d)
    arrays = {"meta": np.frombuffer(open(case, "rb").read(), dtype=np.uint8)}
    jit = name.endswith("_jit")
    for f in sorted(os.listdir(d)):
        stem, ext = os.path.splitext(f)
        if ext[1:] not in DT:
            continue
        if stem == "params_final" and ext == ".f32":
            continue  # the fp16 copy is what the reference serialises (trainer.h:447)
        if jit and stem in ("x", "y", "params_init", "encoded", "params_step1"):
            continue  # identical to the non-JIT case by construction
        arrays[f"{stem}_{ext[1:]}"] = np.fromfile(os.path.join(d, f), dtype=DT[ext[1:]])
    save_case(os.path.join(dst, name + ".npz"), name, arrays)
    print(name, {k: v.shape for k, v in arrays.items() if k != "meta"})
pack_snapshots(src, dst)
for p in sorted(glob.glob(os.path.join(src, "probe_*.json"))):
    open(os.path.join(dst, os.path.basename(p)), "w").write(open(p).read())
