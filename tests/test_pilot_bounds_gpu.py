"""Every pilot kernel, layer by layer, within fp16 rounding plus a stated fp32 accumulation allowance of an fp64 evaluation of the
kernels' own operands (oracle/pilot_bounds.py), and the heads bit for bit.

tests/test_pilot_gpu.py compares with the fp32 network at one tolerance per tensor, which has to absorb the fp16 rounding of the weights;
here each layer is evaluated in fp64 on the weights as the library packs them and on the GPU's own fp16 input of that layer, so the
bound holds element by element.  The matrix reaches every kernel instantiation with partial tiles: both formulations of conv1..conv3,
the per-thread conv1 on ragged and misaligned frames, the smallest frame on the row path, all four model types (both Dense GEMMs, every
head layout), ragged frame stacking, and fp16-subnormal activations.  Run with -s to see the largest err / bound of each layer.

The speed-control tail of KerasPilot (trs_speed_control) is held to 8 float64 ulps of its golden vectors here as well.
"""
import numpy as np
import pytest
import torch

import oracle
from oracle import pilot_bounds as pb
from oracle import pilot_ref as ref
from tests.helpers import cfg_for, speed_cases
from triton_racer_sim_b200 import SpeedControl, synth
from triton_racer_sim_b200.pilot import ModelType, PilotNet

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

KIND = {ModelType.CNN_2D: ref.CNN_2D, ModelType.CNN_2D_SPD_FTR: ref.CNN_2D_SPD_FTR, ModelType.CNN_2D_SPD_CTL: ref.CNN_2D_SPD_CTL,
        ModelType.CNN_2D_FULL_HOUSE: ref.CNN_2D_FULL_HOUSE}
FULL = ModelType.CNN_2D_FULL_HOUSE

# name: (model, h, w, frames, max_batch, TRS_PILOT_ROWCONV, frames 4 bytes into their allocation, layer scaled by 2^-12)
CASES = {
    "120x160_rows": (FULL, 120, 160, 5, 8, "1", False, None),
    "120x160_per_output_row": (FULL, 120, 160, 5, 8, "0", False, None),
    "240x320_rows": (FULL, 240, 320, 3, 4, "1", False, None),
    "240x320_per_output_row": (FULL, 240, 320, 3, 4, "0", False, None),
    "93x96_smallest_row_path": (ModelType.CNN_2D, 93, 96, 4, 4, "1", False, None),
    "96x94_ragged": (ModelType.CNN_2D, 96, 94, 4, 4, "1", False, None),
    "122x166_ragged": (ModelType.CNN_2D_SPD_CTL, 122, 166, 3, 4, "1", False, None),
    "120x160_misaligned": (ModelType.CNN_2D, 120, 160, 4, 8, "1", True, None),
    "n1_speed_feature": (ModelType.CNN_2D_SPD_FTR, 120, 160, 1, 8, "1", False, None),
    "n13_speed_control": (ModelType.CNN_2D_SPD_CTL, 120, 160, 13, 16, "1", False, None),
    "n13_full_house_per_output_row": (FULL, 120, 160, 13, 13, "0", False, None),
    "subnormal_conv3": (FULL, 120, 160, 4, 4, "1", False, 3),
    "subnormal_conv5_per_output_row": (FULL, 120, 160, 4, 4, "0", False, 5),
}


@pytest.mark.parametrize("case", list(CASES))
def test_every_layer_within_the_bound_and_heads_bit_exact(monkeypatch, case):
    mt, h, w, n, cap, rowconv, misaligned, scaled = CASES[case]
    kind = KIND[mt]
    full = mt == FULL
    monkeypatch.setenv("TRS_PILOT_ROWCONV", rowconv)
    wts = ref.random_weights(kind, h, w, seed=3)
    if scaled:
        for t in ("kernel", "bias"):
            wts[f"conv{scaled}/{t}"] = (wts[f"conv{scaled}/{t}"] * np.float32(2.0 ** -12)).astype(np.float32)
    frames = synth.frame_pool(n, h, w, seed=h + w + n)
    rng = np.random.default_rng(n)
    spd, loc = rng.uniform(0, 1, n).astype(np.float32), rng.uniform(0, 10, n).astype(np.float32)
    net = PilotNet(mt, wts, h, w, device=0, max_batch=cap)
    dev = torch.from_numpy(frames).cuda()
    if misaligned:
        raw = torch.empty(frames.size + 64, dtype=torch.uint8, device="cuda")
        view = raw[4:4 + frames.size].view(n, h, w, 3)
        view.copy_(dev)
        assert view.data_ptr() % 16 == 4
        dev = view
    out = net.forward_device(dev, torch.from_numpy(spd).cuda(), torch.from_numpy(loc).cuda()).cpu().numpy()
    kernels = pb.layer_kernels(h, w, rowconv == "1", not misaligned, full)
    packed = pb.pack_weights(wts, kind, h, w)

    failures, lines = [], []
    prev = frames
    for layer in range(1, 8):
        kern, box = kernels[layer]
        y = net.activation(layer, n)
        s, a = pb.conv_exact(prev, packed[f"conv{layer}/kernel"], ref.CONVS[layer - 1][1])
        assert y.shape == s.shape, (layer, y.shape, s.shape)
        rep = pb.fp16_layer(y, s, a, wts[f"conv{layer}/bias"], pb.reduction_len(layer))
        sub = float(np.mean((y != 0) & (np.abs(y.astype(np.float32)) < 2.0 ** -14)))
        lines.append(f"conv{layer} {kern:26s} box {box}: max err/bound {rep['max_ratio']:.3f}  y != RN16(yhat) {rep['mismatch']:.2e}"
                     f"  subnormal {sub:.2e}")
        if rep["max_ratio"] > 1.0 or rep["mismatch"] > pb.MISMATCH_MAX:
            failures.append(f"conv{layer} ({kern}, box bx, by, bn = {box}): max err/bound {rep['max_ratio']:.3f}, "
                            f"y != RN16(yhat) in {rep['mismatch']:.2%}\n  {pb.worst(rep, box)}")
        if layer == scaled:                                           # out of this epilogue and into the next layer's MMA
            assert sub > 0.01, f"conv{layer}: only {sub:.2%} of the activations are fp16-subnormal"
        prev = y

    ldp = 256 if full else 128
    part = net.activation(8, n).reshape(n, ldp)
    flat = prev.reshape(n, -1)
    kern, box = kernels[8]
    for hd, d in enumerate(("dense1", "dense4") if full else ("dense1",)):
        s, a = pb.dense_exact(flat, packed[f"{d}/image"])
        rep = pb.partial_layer(part[:, 128 * hd:128 * hd + 100], s, a, flat.shape[1])
        lines.append(f"layer 8 {d} {kern:19s}: max |p - S| / E_acc {rep['max_ratio']:.3f}  median |p - S| / A {rep['median']:.2e}")
        if rep["max_ratio"] > 1.0 or rep["median"] > pb.L8_MEDIAN_MAX:
            r4 = {k: rep[k].reshape(n, 1, 1, -1) for k in ("ratio", "err", "bound")}
            failures.append(f"layer 8 {d} ({kern}): max |p - S| / E_acc {rep['max_ratio']:.3f}, median |p - S| / A {rep['median']:.3g}"
                            f"\n  {pb.worst(r4, box)}")

    want = pb.heads_exact(wts, kind, part, ldp, spd, loc)
    diff = np.nonzero((out != want).any(1))[0]
    lines.append(f"heads: {diff.size} of {n} frames differ from the bit-exact restatement")
    if diff.size:
        failures.append("k_pilot_heads: " + "; ".join(f"frame {f}: {out[f].tolist()} != {want[f].tolist()}" for f in diff[:5]))
    print(f"\n[{case}] {mt.value} {h}x{w} n={n} rowconv={rowconv}\n  " + "\n  ".join(lines))
    net.close()
    assert not failures, f"[{case}]\n" + "\n".join(failures)


def test_speed_control_within_8_ulps_of_the_goldens(golden_speed):
    """trs_speed_control (the tail of KerasPilot.step) against tests/golden/speed.npz: steering exact, throttle and brake within 8
    float64 ulps (CUDA's double atan is documented at 2 ulps, one multiply and one divide follow, and the golden's math.atan has its
    own last-ulp error).  States whose value lies within 8 ulps of a dead-band edge (-0.2 for throttle, 0.4 for brake) are excluded
    and counted: an ulp there can legitimately flip the zeroing."""
    cur, ms, st = golden_speed["cur"], golden_speed["model_spd"], golden_speed["model_steer"]
    half_pi = np.pi / 2
    for cname, over in speed_cases(golden_speed).items():
        for legacy in (False, True):
            cfg = dict(cfg_for(over), spd_ctl_numpy_legacy_promotion=legacy)
            p = oracle.spd_params_from_cfg(cfg)
            comp = SpeedControl(cfg, device=0)
            res = comp.control_device(torch.from_numpy(cur).cuda(), torch.from_numpy(st).cuda(), torch.from_numpy(ms).cuda())
            s, t, b = (v.cpu().numpy() for v in res[:3])
            comp.onShutdown()
            want = golden_speed[f"out_numpy1/{cname}" if legacy else f"out/{cname}"]
            assert np.array_equal(s, want[:, 0]), (cname, legacy)
            # the values before the dead-bands, in the promotion of this mode (oracle/trs_oracle.c orc_speed_control)
            if legacy:
                d = ms.astype(np.float64) * 20 * p.threshold - cur
                d2 = d * 2
            else:
                df = (ms.astype(np.float32) * np.float32(20)) * np.float32(p.threshold) - cur.astype(np.float32)
                d, d2 = df.astype(np.float64), (df * np.float32(2)).astype(np.float64)
            near = np.abs(p.reverse_multiplier * np.arctan(d2) / half_pi + 0.2) <= 8 * np.spacing(0.2) if not p.use_break \
                else np.abs(-p.break_multiplier * np.arctan(d) / half_pi - 0.4) <= 8 * np.spacing(0.4)
            for name, got, ref_ in (("throttle", t, want[:, 1]), ("brake", b, want[:, 2])):
                keep = ~near
                assert np.array_equal(got[keep] == 0, ref_[keep] == 0), f"{cname} {name}: dead-band decision differs"
                ulps = np.abs(got[keep] - ref_[keep]) / np.spacing(np.abs(ref_[keep]))
                print(f"[{cname}{' numpy1' if legacy else ''}] {name}: max {ulps.max():.1f} ulps; {int(near.sum())} states near a dead-band edge")
                assert ulps.max() <= 8, f"{cname}{' (numpy 1 promotion)' if legacy else ''} {name}: {ulps.max():.1f} ulps"
