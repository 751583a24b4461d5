"""CPU-side checks of the pilots' path: the fp32 reference used as the checker (oracle/pilot_ref.py) against a naive restatement of
Conv2D / Dense, the weight container, and the loud failure without a GPU."""
import numpy as np
import pytest
import torch

from oracle import pilot_ref as ref


def naive_conv_valid(x, k, b, s):
    """x (H,W,Ci), k (kh,kw,Ci,Co) Keras layout, VALID padding, ReLU."""
    kh, kw, ci, co = k.shape
    ho, wo = (x.shape[0] - kh) // s + 1, (x.shape[1] - kw) // s + 1
    out = np.zeros((ho, wo, co), np.float64)
    for y in range(ho):
        for xx in range(wo):
            patch = x[y * s:y * s + kh, xx * s:xx * s + kw, :].astype(np.float64)
            out[y, xx] = np.tensordot(patch, k.astype(np.float64), axes=([0, 1, 2], [0, 1, 2])) + b
    return np.maximum(out, 0)


def test_reference_convolutions_follow_keras_layout():
    rng = np.random.default_rng(0)
    wts = ref.random_weights(ref.CNN_2D, 120, 160, seed=4)
    x = rng.uniform(0, 1, (1, 31, 37, 3)).astype(np.float32)
    a = ref.conv_stack(wts, torch.from_numpy(x), 0, 2)
    want1 = naive_conv_valid(x[0], wts["conv1/kernel"], wts["conv1/bias"], 2)
    assert a[0].shape[1:] == want1.shape and np.allclose(a[0][0].numpy(), want1, atol=1e-5)
    want2 = naive_conv_valid(want1, wts["conv2/kernel"], wts["conv2/bias"], 2)
    assert np.allclose(a[1][0].numpy(), want2, atol=1e-4)


def test_reference_shapes_and_head_wiring():
    assert ref.conv_out_hw(120, 160) == (4, 9)                       # Flatten -> 4 * 9 * 128 = 4608
    sh = ref.weight_shapes(ref.CNN_2D_FULL_HOUSE)
    assert sh["dense1/kernel"] == (4608 + 64, 100)                   # keras_train.py:215  x = Concatenate([x, y])
    assert sh["dense4/kernel"] == (4608 + 128, 100)                  # keras_train.py:231  s = Concatenate([x, s]) with that x
    assert ref.weight_shapes(ref.CNN_2D_SPD_FTR)["dense1/kernel"] == (4608 + 16, 100)
    assert ref.weight_shapes(ref.CNN_2D)["output_layer/kernel"] == (25, 2)
    # the full-house output row is (steering, speed): keras_train.py:239 Concatenate([out_steering, out_speed])
    wts = ref.random_weights(ref.CNN_2D_FULL_HOUSE, seed=2)
    frames = np.random.default_rng(1).integers(0, 256, (3, 120, 160, 3), dtype=np.uint8)
    spd, loc = np.array([.1, .5, .9], np.float32), np.array([1., 5., 9.], np.float32)
    base = ref.forward(wts, ref.CNN_2D_FULL_HOUSE, frames, spd, loc)
    w2 = dict(wts)
    w2["out_steering/bias"] = wts["out_steering/bias"] + 1
    assert np.allclose(ref.forward(w2, ref.CNN_2D_FULL_HOUSE, frames, spd, loc) - base, [[1, 0]] * 3, atol=1e-6)
    # the speed feature reaches only the steering head, the loc/segment feature both (it is part of x)
    d_spd = ref.forward(wts, ref.CNN_2D_FULL_HOUSE, frames, spd + 0.3, loc) - base
    assert np.abs(d_spd[:, 0]).max() > 0 and not d_spd[:, 1].any()
    d_loc = ref.forward(wts, ref.CNN_2D_FULL_HOUSE, frames, spd, loc + 2) - base
    assert np.abs(d_loc[:, 0]).max() > 0 and np.abs(d_loc[:, 1]).max() > 0


def naive_forward(wts, model_type, frame_u8, spd=None, loc=None):
    """One frame through the reference's layer list (keras_train.py:131-174 | 191-243) in float64 numpy, written independently of
    oracle/pilot_ref.py: explicit loops for Conv2D, C-order Flatten of the (H,W,C) tensor, np.concatenate in the reference's order."""
    relu = lambda v: np.maximum(v, 0)
    dense = lambda name, v, act=True: (relu if act else (lambda t: t))(v @ wts[f"{name}/kernel"].astype(np.float64) + wts[f"{name}/bias"])
    x = frame_u8.astype(np.float32) / np.float32(255)                    # keras_pilot.py:49-50
    for i, (k, s_, _) in enumerate(ref.CONVS):
        x = naive_conv_valid(x, wts[f"conv{i + 1}/kernel"], wts[f"conv{i + 1}/bias"], s_)
    x = x.reshape(-1)                                                     # Flatten (keras_train.py:153 | 211)
    if model_type == ref.CNN_2D_FULL_HOUSE:
        y = np.array([loc], np.float64)                                   # feature_vec_input <- loc/segment (keras_pilot.py:102-104)
        for n in ("feature1", "feature2", "feature3"):
            y = dense(n, y)
        x = np.concatenate([x, y])                                        # keras_train.py:215
        z = x
        for n in ("dense1", "dense2", "dense3"):
            z = dense(n, z)
        out_speed = dense("output_speed", z, act=False)
        s = np.array([spd], np.float64)                                   # current_spd_input <- speed / 20 (keras_pilot.py:100-101)
        for n in ("current_spd_1", "current_spd_2", "current_spd_3"):
            s = dense(n, s)
        s = np.concatenate([x, s])                                        # keras_train.py:231
        for n in ("dense4", "dense5", "dense6"):
            s = dense(n, s)
        out_steering = dense("out_steering", s, act=False)
        return np.concatenate([out_steering, out_speed])                  # keras_train.py:239
    z = x
    if model_type == ref.CNN_2D_SPD_FTR:
        y = np.array([spd], np.float64)
        for n in ("feature1", "feature2", "feature3"):
            y = dense(n, y)
        z = np.concatenate([x, y])                                        # keras_train.py:160
    for n in ("dense1", "dense2", "dense3"):
        z = dense(n, z)
    return dense("output_layer", z, act=False)


@pytest.mark.parametrize("model_type", [ref.CNN_2D, ref.CNN_2D_SPD_FTR, ref.CNN_2D_SPD_CTL, ref.CNN_2D_FULL_HOUSE])
def test_reference_network_against_an_independent_restatement(model_type):
    """The checker itself checked: the PyTorch restatement against explicit numpy loops over the reference's layer list."""
    h, w = 94, 96                                                         # the smallest frames the seven VALID convolutions accept
    rng = np.random.default_rng(model_type)
    wts = ref.random_weights(model_type, h, w, seed=20 + model_type)
    frames = rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    spd, loc = np.float32([0.35, 0.8]), np.float32([2.5, 9.0])
    got = ref.forward(wts, model_type, frames, spd, loc)
    for i in range(2):
        want = naive_forward(wts, model_type, frames[i], float(spd[i]), float(loc[i]))
        assert np.allclose(got[i], want, atol=2e-5), (got[i], want)


def test_weight_file_round_trip(tmp_path):
    from triton_racer_sim_b200.pilot import load_weights
    wts = ref.random_weights(ref.CNN_2D_SPD_FTR, seed=5)
    path = tmp_path / "model.npz"
    np.savez(path, **wts)
    back = load_weights(path)
    assert sorted(back) == sorted(wts) and all(np.array_equal(back[k], wts[k]) for k in wts)


def test_pilot_without_a_gpu_fails_loudly():
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that a machine with a GPU checks this too."""
    import os
    import subprocess
    import sys

    from tests.conftest import ROOT
    code = ("import pytest\nfrom oracle import pilot_ref as ref\nfrom triton_racer_sim_b200 import _native as nat\n"
            "from triton_racer_sim_b200.pilot import ModelType, PilotNet\n"
            "with pytest.raises((nat.NativeError, RuntimeError)):\n    PilotNet(ModelType.CNN_2D, ref.random_weights(ref.CNN_2D), device=0)\n")
    run = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True,
                         timeout=300)
    assert run.returncode == 0, run.stderr[-2000:]


# ---- the reference's own model-building and step code, executed over a numpy stand-in for the Keras primitives (tests/golden/pilot.npz) ----------
def _pilot_golden():
    import json
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pilot.npz"))
    return g, json.loads(bytes(g["meta_json"]).decode())


def test_checker_matches_the_graph_the_reference_code_builds():
    """tests/golden/make_golden_pilot.py imports keras_train.py / keras_pilot.py unmodified, lets the reference's `get_model` build its graphs and
    its `KerasPilot.step` feed them (the `/255`, the reshapes, the input tuple (img, spd, features), keras_pilot.py:49-104), with only Conv2D / Dense /
    Flatten / Concatenate supplied by a float64 numpy stand-in.  The fp32 checker the CUDA kernels are compared with (oracle/pilot_ref.py) must give
    those outputs: same layers, names, shapes, concatenation and input order, for all four model types at two frame sizes."""
    from triton_racer_sim_b200 import synth
    g, meta = _pilot_golden()
    assert len(meta["cases"]) == 8
    for case in meta["cases"]:
        mt, h, w, n = case["model_type"], case["h"], case["w"], case["n"]
        wts = ref.random_weights(mt, h, w, seed=case["weight_seed"])
        assert sorted({k.split("/")[0] for k in wts}) == case["layers"]                       # the reference's layer names, every trainable one
        frames = synth.frame_pool(n, h, w, seed=case["frame_seed"])
        speed, segment = g[f"speed/{mt}/{h}x{w}"], g[f"segment/{mt}/{h}x{w}"]
        spd_feature = (speed / 20).astype(np.float32)                                          # keras_pilot.py:68, :100
        got = ref.forward(wts, mt, frames, spd_feature=spd_feature, loc_feature=segment.astype(np.float32))
        for cname in meta["cfgs"]:
            want = g[f"model_out/{mt}/{h}x{w}/{cname}"]
            assert want.shape == (n, 2) and np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), (mt, h, w, np.abs(got - want).max())
    assert [c["inputs"] for c in meta["cases"] if c["model_type"] == ref.CNN_2D_FULL_HOUSE][0] == ["img_input", "current_spd_input", "feature_vec_input"]
    # the reference's cnn_2d / cnn_2d_speed_as_feature pilots raise on every frame: `__cap` gets the whole (steering, throttle) row
    assert sorted(meta["reference_raises"]) == [str(ref.CNN_2D), str(ref.CNN_2D_SPD_FTR)]


def test_speed_control_tail_matches_the_reference_step():
    """(steering, throttle, breaking) as the reference's KerasPilot.step returned them for the speed-control model types (keras_pilot.py:78-118:
    cap, x 20, calcThrottle / calcBreak, smoothing), against the oracle's speed controller fed the same model outputs."""
    import oracle
    from tests.helpers import cfg_for
    g, meta = _pilot_golden()
    checked = 0
    for case in meta["cases"]:
        mt, h, w = case["model_type"], case["h"], case["w"]
        if mt not in (ref.CNN_2D_SPD_CTL, ref.CNN_2D_FULL_HOUSE):
            continue
        for cname, over in meta["cfgs"].items():
            out, want = g[f"model_out/{mt}/{h}x{w}/{cname}"], g[f"ctl/{mt}/{h}x{w}/{cname}"]
            s, t, b, _ = oracle.speed_control(g[f"speed/{mt}/{h}x{w}"], out[:, 1], out[:, 0], cfg_for(over))
            assert np.array_equal(s, want[:, 0]), (mt, cname)
            assert np.allclose(t, want[:, 1], rtol=1e-5, atol=0) and np.allclose(b, want[:, 2], rtol=1e-5, atol=0), (mt, cname)
            checked += len(want)
    assert checked >= 40
