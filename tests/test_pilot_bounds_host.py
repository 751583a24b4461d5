"""The per-layer bounds of oracle/pilot_bounds.py, checked without a GPU.

* the fp16 packing: numpy's float16 rounding is the host __float2half_rn the library packs its weights with (ties, subnormals,
  overflow, 10^7 random floats), with and without conv1's fp32 division by 255;
* the fmaf emulation the bit-exact heads restatement rests on, against exact rational arithmetic;
* the checker has teeth: a numpy model of a correct layer (fp16 operands, fp32 accumulation in K = 16 blocks, RN16 epilogue) passes
  and each injected defect is rejected — including two that the older rule (max|err| <= 2e-3 * max|activation| against the fp32
  network) lets through.
"""
import ctypes as C
import os
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import pilot_bounds as pb
from oracle import pilot_ref as ref
from tests.conftest import ROOT
from triton_racer_sim_b200 import synth
from triton_racer_sim_b200.build import nvcc_path

OLD_LAYER_TOL = 2e-3                     # tests/test_pilot_gpu.py LAYER_TOL


def cuda_include():
    nvcc = nvcc_path()
    nvcc = nvcc if os.path.sep in nvcc else shutil.which(nvcc)
    return os.path.join(os.path.dirname(os.path.dirname(os.path.realpath(nvcc))), "include")


@pytest.fixture(scope="module")
def half_host(tmp_path_factory):
    out = tmp_path_factory.mktemp("half") / "libhalfpack.so"
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I", cuda_include(), "-o", str(out),
                           os.path.join(ROOT, "tests", "host_half_pack_check.cpp")])
    lib = C.CDLL(str(out))
    for fn in (lib.pack_rn, lib.pack_conv1):
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
        fn.restype = None
    return lib


def host_pack(fn, x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty(x.shape, np.uint16)
    fn(x.ctypes.data, out.ctypes.data, x.size)
    return out


def packing_inputs():
    """Every finite fp16 value, every midpoint between neighbours (ties; 65520 is the tie between 65504 and overflow, 2^-25 the one
    between 0 and the smallest subnormal) and the fp32 neighbours of both; the subnormal range; overflow; 10^7 random floats."""
    h = np.arange(0x7c00, dtype=np.uint16).view(np.float16).astype(np.float32)                  # 0 .. 65504, subnormals included
    up = np.append(h[1:], np.float32(65536))
    mids = (h.astype(np.float64) + up) / 2                                                       # exact in fp32 (12 significant bits)
    mids = mids.astype(np.float32)
    assert np.array_equal(mids.astype(np.float64), (h.astype(np.float64) + up) / 2)
    base = np.concatenate([h, mids])
    base = np.concatenate([base, np.nextafter(base, np.float32(np.inf)), np.nextafter(base, np.float32(0))])
    rng = np.random.default_rng(0)
    sub = rng.uniform(0, 2.0 ** -14, 200_000).astype(np.float32)
    over = np.concatenate([rng.uniform(65504, 65536, 50_000), [65519.996, 65520, 65520.004, 1e5, 3.4e38, np.inf]]).astype(np.float32)
    bits = rng.integers(0, 2 ** 32, 5_000_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    bits = bits[~np.isnan(bits)]
    logu = (2.0 ** rng.uniform(-30, 17, 5_000_000)).astype(np.float32)
    x = np.concatenate([base, sub, over, bits, logu])
    return np.concatenate([x, -x])


def test_numpy_float16_is_the_librarys_float2half_rn(half_host):
    x = packing_inputs()
    assert x.size > 10_000_000
    want = host_pack(half_host.pack_rn, x)
    with np.errstate(over="ignore"):                                                            # overflow to inf is a case
        got = x.astype(np.float16).view(np.uint16)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(float(x[i]), hex(got[i]), hex(want[i])) for i in bad[:8]]
    # the weights of a real layer, through pack_weights
    wts = ref.random_weights(ref.CNN_2D_FULL_HOUSE, 120, 160, seed=3)
    packed = pb.pack_weights(wts, ref.CNN_2D_FULL_HOUSE, 120, 160)
    for i in range(2, 8):
        k = wts[f"conv{i}/kernel"]
        assert np.array_equal(packed[f"conv{i}/kernel"].view(np.uint16), host_pack(half_host.pack_rn, k))
    assert np.array_equal(packed["dense4/image"].view(np.uint16), host_pack(half_host.pack_rn, wts["dense4/kernel"][:4608]))


def test_conv1_fold_is_the_fp32_division_then_float2half_rn(half_host):
    x = packing_inputs()
    x = np.concatenate([x, (x[np.abs(x) < 1e30] * np.float32(255)).astype(np.float32)])      # and the ties of the quotient
    want = host_pack(half_host.pack_conv1, x)
    with np.errstate(over="ignore"):
        got = (x / np.float32(255)).astype(np.float16).view(np.uint16)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(float(x[i]), hex(got[i]), hex(want[i])) for i in bad[:8]]
    wts = ref.random_weights(ref.CNN_2D, 120, 160, seed=3)
    packed = pb.pack_weights(wts, ref.CNN_2D, 120, 160)
    assert np.array_equal(packed["conv1/kernel"].view(np.uint16), host_pack(half_host.pack_conv1, wts["conv1/kernel"]))
    # and it is not the same as rounding twice: the double-rounding defect below is a real one
    twice = (wts["conv1/kernel"].astype(np.float16).astype(np.float32) / np.float32(255)).astype(np.float16)
    assert (twice != packed["conv1/kernel"]).mean() > 0.05


# ---- fmaf -------------------------------------------------------------------------------------------------------------------

def rn32_exact(q):
    """Fraction -> nearest float32, ties to even, by comparing the float32 neighbours of a close candidate exactly."""
    r = np.float32(float(q))
    cands = [np.nextafter(r, np.float32(-np.inf)), r, np.nextafter(r, np.float32(np.inf))]
    best = min(abs(Fraction(float(c)) - q) for c in cands)
    near = [c for c in cands if abs(Fraction(float(c)) - q) == best]
    return near[0] if len(near) == 1 else [c for c in near if int(np.array(c).view(np.uint32)) % 2 == 0][0]


def fma_cases():
    rng = np.random.default_rng(1)
    n = 6000
    mant = lambda k: rng.uniform(1, 2, k)
    a = (mant(n) * 2.0 ** rng.integers(-40, 40, n) * rng.choice([-1, 1], n)).astype(np.float32)
    b = (mant(n) * 2.0 ** rng.integers(-40, 40, n) * rng.choice([-1, 1], n)).astype(np.float32)
    c = (mant(n) * 2.0 ** rng.integers(-80, 80, n) * rng.choice([-1, 1], n)).astype(np.float32)
    cases = list(zip(a, b, c))
    # products of the same magnitude as c: cancellation
    for i in range(2000):
        x, y = np.float32(rng.uniform(-2, 2)), np.float32(rng.uniform(-2, 2))
        cases.append((x, y, np.float32(-(float(x) * float(y)) * rng.uniform(0.999, 1.001))))
    # exact values just off a float32 midpoint, closer than fp64 resolves: (2^32 + 1) = 641 * 6700417 and (2^32 - 1) = 65535 * 65537
    # put the product's leading bit on half a float32 unit of c, its last bit 2^-32 of that below; the fp64 sum then lands exactly
    # on the midpoint and rounding it again to float32 picks the wrong neighbour for half of the mantissas of c
    for i in range(2000):
        cm = int(rng.integers(2 ** 23, 2 ** 24))
        e = int(rng.integers(-60, 60))
        cv = np.float32(cm * 2.0 ** e)                            # float32 unit of c: 2^e
        f1, f2 = ((641, 6700417), (65535, 65537))[i % 2]
        sgn = (-1) ** (i // 2 % 2)
        sa = int(rng.integers(-10, 10))
        pa = np.float32(sgn * f1 * 2.0 ** sa)
        pb_ = np.float32(f2 * 2.0 ** (e - 1 - 32 - sa))             # f1 * f2 ~ 2^32: product ~ 2^(e - 1)
        cases.append((pa, pb_, cv if i % 3 else -cv))
    # subnormal results
    for i in range(1000):
        cases.append((np.float32(rng.uniform(-2, 2) * 2.0 ** -70), np.float32(rng.uniform(-2, 2) * 2.0 ** -70),
                      np.float32(rng.uniform(-2, 2) * 2.0 ** -130)))
    return cases


def test_fmaf_emulation_is_correctly_rounded():
    cases = fma_cases()
    a, b, c = (np.array(v, np.float32) for v in zip(*cases))
    got = pb.fmaf(a, b, c)
    want = np.array([rn32_exact(Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z))) for x, y, z in cases], np.float32)
    bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))[0]
    assert bad.size == 0, [(cases[i], got[i], want[i]) for i in bad[:5]]
    # the constructed midpoint cases are ones where rounding the fp64 sum again gives the wrong answer
    naive = (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)
    assert (naive.view(np.uint32) != want.view(np.uint32)).sum() >= 500


# ---- the checker has teeth ------------------------------------------------------------------------------------------------------

def im2col(x, k, s):
    n, h, w, c = x.shape
    ho, wo = (h - k) // s + 1, (w - k) // s + 1
    sn, sh, sw, sc = x.strides
    v = np.lib.stride_tricks.as_strided(x, (n, ho, wo, k, k, c), (sn, sh * s, sw * s, sh, sw, sc))
    return v.reshape(n, ho, wo, k * k * c)


def rtz16(v):
    """float64 -> fp16 rounded toward zero."""
    r = v.astype(np.float16)
    over = np.abs(r.astype(np.float64)) > np.abs(v)
    return np.where(over, np.nextafter(r, np.float16(0)), r)


def accumulate(cols, wmat, acc_type=np.float32, drop_last=0):
    """The accumulator of the MMAs: exact block sums added into an fp32 accumulator, one rounding per K = 16 step.  With
    acc_type=float16, an approximation of an fp16 accumulator (the D-format bit of the instruction descriptor): one rounding to fp16
    per 64-wide K block, the work of one pipeline stage.  (Rounding to fp16 after every K = 16 step is larger still, and the old
    rule catches it on some layers.)"""
    k = wmat.shape[0] - drop_last
    step = 16 if acc_type == np.float32 else 64
    acc = np.zeros(cols.shape[:-1] + (wmat.shape[1],), acc_type)
    for k0 in range(0, k, step):
        k1 = min(k0 + step, k)
        acc = (acc.astype(np.float64) + cols[..., k0:k1] @ wmat[k0:k1]).astype(acc_type)
    return acc.astype(np.float32)


def model_layer(x, kern16, bias, stride, acc_type=np.float32, epilogue="rn", drop_last_bias=False):
    """One convolution as the kernels compute it: fp16 (or u8) operands, accumulation, fl32(acc + b), ReLU, fp16."""
    k = kern16.shape[0]
    cols = im2col(np.ascontiguousarray(x, np.float64), k, stride)
    acc = accumulate(cols, kern16.astype(np.float64).reshape(-1, kern16.shape[-1]), acc_type)
    b = np.array(bias, np.float32)
    if drop_last_bias:
        b[-1] = 0
    if epilogue == "relu_first":
        return (np.maximum(acc, np.float32(0)) + b).astype(np.float16)
    v = np.maximum(acc + b, np.float32(0))                      # fp32 add: fl32(acc + b)
    return rtz16(v.astype(np.float64)) if epilogue == "rtz" else v.astype(np.float16)


@pytest.fixture(scope="module")
def net():
    """120x160 frames through the fp32 network with random_weights(seed=3): realistic inputs for each layer."""
    h, w, n = 120, 160, 3
    wts = ref.random_weights(ref.CNN_2D_FULL_HOUSE, h, w, seed=3)
    frames = synth.frame_pool(n, h, w, seed=11)
    _, acts = ref.forward(wts, ref.CNN_2D_FULL_HOUSE, frames, np.zeros(n, np.float32), np.zeros(n, np.float32), return_acts=True)
    return dict(h=h, w=w, wts=wts, frames=frames, acts=acts, packed=pb.pack_weights(wts, ref.CNN_2D_FULL_HOUSE, h, w))


def layer_input(net, layer):
    return net["frames"] if layer == 1 else net["acts"][layer - 2].astype(np.float16)


def check(net, layer, y):
    x = layer_input(net, layer)
    s, a = pb.conv_exact(x, net["packed"][f"conv{layer}/kernel"], ref.CONVS[layer - 1][1])
    return pb.fp16_layer(y, s, a, net["wts"][f"conv{layer}/bias"], pb.reduction_len(layer))


def rejected(rep):
    return rep["max_ratio"] > 1.0 or rep["mismatch"] > pb.MISMATCH_MAX


def old_rule_passes(net, layer, y):
    x = layer_input(net, layer)
    x = x.astype(np.float32) / np.float32(255) if layer == 1 else x.astype(np.float32)
    want = ref.conv_stack(net["wts"], torch.from_numpy(x), layer - 1, layer)[0].numpy()
    return np.abs(y.astype(np.float32) - want).max() <= OLD_LAYER_TOL * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("layer", [1, 2, 4, 7])
def test_a_correct_layer_passes(net, layer):
    k, s, _ = ref.CONVS[layer - 1]
    y = model_layer(layer_input(net, layer), net["packed"][f"conv{layer}/kernel"], net["wts"][f"conv{layer}/bias"], s)
    rep = check(net, layer, y)
    print(f"conv{layer}: max err/bound {rep['max_ratio']:.3f}, y != RN16(yhat) {rep['mismatch']:.2e}")
    assert rep["max_ratio"] <= 1.0 and rep["mismatch"] <= pb.MISMATCH_MAX / 10
    assert old_rule_passes(net, layer, y)


@pytest.mark.parametrize("layer", [2, 4, 7])
@pytest.mark.parametrize("defect", ["round_toward_zero", "fp16_accumulator"])
def test_subtle_defects_pass_the_old_rule_and_fail_the_bound(net, layer, defect):
    """The two defects a tensor-core kernel typically has: the old per-tensor rule lets both through, the per-element bound does not."""
    _, s, _ = ref.CONVS[layer - 1]
    kw = dict(epilogue="rtz") if defect == "round_toward_zero" else dict(acc_type=np.float16)
    y = model_layer(layer_input(net, layer), net["packed"][f"conv{layer}/kernel"], net["wts"][f"conv{layer}/bias"], s, **kw)
    assert old_rule_passes(net, layer, y)
    rep = check(net, layer, y)
    print(f"conv{layer} {defect}: max err/bound {rep['max_ratio']:.3f}, y != RN16(yhat) {rep['mismatch']:.3f}")
    assert rejected(rep)
    if defect == "round_toward_zero":
        assert rep["mismatch"] > pb.MISMATCH_MAX          # caught in aggregate too: about half of the elements are off by one unit


@pytest.mark.parametrize("defect", ["bias_dropped_for_last_filter", "relu_before_bias"])
def test_epilogue_defects_are_rejected(net, defect):
    layer = 4
    kw = dict(drop_last_bias=True) if defect == "bias_dropped_for_last_filter" else dict(epilogue="relu_first")
    y = model_layer(layer_input(net, layer), net["packed"]["conv4/kernel"], net["wts"]["conv4/bias"], 1, **kw)
    assert rejected(check(net, layer, y))


def test_conv1_weights_rounded_twice_are_rejected(net):
    twice = (net["wts"]["conv1/kernel"].astype(np.float16).astype(np.float32) / np.float32(255)).astype(np.float16)
    y = model_layer(net["frames"], twice, net["wts"]["conv1/bias"], 2)
    rep = check(net, 1, y)
    print(f"conv1 weights rounded twice: max err/bound {rep['max_ratio']:.3f}, y != RN16(yhat) {rep['mismatch']:.3f}")
    assert rejected(rep)


def test_a_box_edge_column_copied_from_its_neighbour_is_rejected(net):
    layer = 1
    kern, box = pb.layer_kernels(net["h"], net["w"])[layer]
    bx = box[0]
    y = model_layer(net["frames"], net["packed"]["conv1/kernel"], net["wts"]["conv1/bias"], 2)
    assert check(net, layer, y)["max_ratio"] <= 1.0
    assert bx < y.shape[2], (kern, box)
    y[:, :, bx, :] = y[:, :, bx - 1, :]
    rep = check(net, layer, y)
    assert rejected(rep)
    assert f"x%{bx}=0" in pb.worst(rep, box, 1)                  # the message points at the box edge


def layer8_inputs(net):
    flat = net["acts"][-1].astype(np.float16).reshape(net["frames"].shape[0], -1)
    w16 = net["packed"]["dense1/image"]
    return flat, w16, pb.dense_exact(flat, w16)


@pytest.mark.parametrize("defect", [None, "last_k_chunk_missing", "fp16_accumulator"])
def test_layer8_partial_sums(net, defect):
    flat, w16, (s, a) = layer8_inputs(net)
    p = accumulate(flat.astype(np.float64), w16.astype(np.float64), np.float16 if defect == "fp16_accumulator" else np.float32,
                   drop_last=64 if defect == "last_k_chunk_missing" else 0)
    rep = pb.partial_layer(p, s, a, flat.shape[1])
    print(f"layer 8 {defect}: max |p - S| / E_acc {rep['max_ratio']:.3g}, median |p - S| / A {rep['median']:.3g}")
    ok = rep["max_ratio"] <= 1.0 and rep["median"] <= pb.L8_MEDIAN_MAX
    assert ok == (defect is None)
    if defect == "fp16_accumulator":
        assert rep["median"] > pb.L8_MEDIAN_MAX                  # the median is the check that catches it


@pytest.mark.parametrize("mt", [ref.CNN_2D, ref.CNN_2D_SPD_FTR, ref.CNN_2D_SPD_CTL, ref.CNN_2D_FULL_HOUSE])
def test_heads_restatement_is_wired_like_the_graph(mt):
    """heads_exact on exact partial sums against the fp32 graph (oracle/pilot_ref.heads) with the same fp16 image weights: the two
    differ only in fp32 rounding, so every slot, feature branch and concatenation is where the graph has it."""
    h, w, n = 120, 160, 16
    wts = ref.random_weights(mt, h, w, seed=5)
    packed = pb.pack_weights(wts, mt, h, w)
    rng = np.random.default_rng(2)
    flat = rng.uniform(0, 1, (n, pb.flat_len(h, w))).astype(np.float16)
    spd, loc = rng.uniform(0, 1, n).astype(np.float32), rng.uniform(0, 10, n).astype(np.float32)
    full = mt == ref.CNN_2D_FULL_HOUSE
    ldp = 256 if full else 128
    part = np.zeros((n, ldp), np.float32)
    w16 = dict(wts)
    for hd, d in enumerate(("dense1", "dense4") if full else ("dense1",)):
        part[:, 128 * hd:128 * hd + 100] = pb.dense_exact(flat, packed[f"{d}/image"])[0]
        k = wts[f"{d}/kernel"].copy()
        k[:flat.shape[1]] = packed[f"{d}/image"]
        w16[f"{d}/kernel"] = k
    got = pb.heads_exact(wts, mt, part, ldp, spd, loc)
    want = ref.heads(w16, mt, torch.from_numpy(flat.astype(np.float32)), spd, loc).numpy()
    assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max()), np.abs(got - want).max()


def test_heads_with_two_fmaf_terms_swapped_are_rejected(net):
    """Two terms of dense2's chain swapped (two units of dense1 exchanged everywhere: the same products, summed in another order):
    the outputs move by an fp32 unit or so, and the bit-exact restatement sees it."""
    mt = ref.CNN_2D_FULL_HOUSE
    wts = net["wts"]
    flat, _, _ = layer8_inputs(net)
    n = flat.shape[0]
    rng = np.random.default_rng(3)
    reps = 64                                                     # more frames: perturbed copies of the three
    flat = np.concatenate([flat] * reps).astype(np.float64) * rng.uniform(0.5, 1.5, (n * reps, 1))
    flat = flat.astype(np.float16)
    part = np.zeros((flat.shape[0], 256), np.float32)
    part[:, :100] = accumulate(flat.astype(np.float64), net["packed"]["dense1/image"].astype(np.float64))
    part[:, 128:228] = accumulate(flat.astype(np.float64), net["packed"]["dense4/image"].astype(np.float64))
    spd, loc = rng.uniform(0, 1, flat.shape[0]).astype(np.float32), rng.uniform(0, 10, flat.shape[0]).astype(np.float32)
    good = pb.heads_exact(wts, mt, part, 256, spd, loc)
    sw = list(np.nonzero((part[:, :100] + wts["dense1/bias"] > 0).all(0))[0][:2])          # two units no ReLU zeroes
    bad_w = dict(wts)
    bad_w["dense1/kernel"] = wts["dense1/kernel"].copy()
    bad_w["dense1/kernel"][:, sw] = wts["dense1/kernel"][:, sw[::-1]]
    bad_w["dense1/bias"] = wts["dense1/bias"].copy()
    bad_w["dense1/bias"][sw] = wts["dense1/bias"][sw[::-1]]
    bad_w["dense2/kernel"] = wts["dense2/kernel"].copy()
    bad_w["dense2/kernel"][sw] = wts["dense2/kernel"][sw[::-1]]
    bad_p = part.copy()
    bad_p[:, sw] = part[:, sw[::-1]]
    bad = pb.heads_exact(bad_w, mt, bad_p, 256, spd, loc)
    assert np.abs(bad - good).max() <= 1e-5                      # subtle: a tolerance would pass it
    assert not np.array_equal(bad, good)
    assert np.array_equal(bad[:, 0], good[:, 0])                 # the steering head does not use dense2
