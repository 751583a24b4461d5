"""Every pilot kernel, layer by layer, within fp16 rounding plus a stated fp32 accumulation allowance of an fp64 evaluation of the
kernels' own operands (oracle/pilot_bounds.py), and the heads bit for bit.

tests/test_pilot_gpu.py compares with the fp32 network at one tolerance per tensor, which has to absorb the fp16 rounding of the weights;
here each layer is evaluated in fp64 on the weights as the library packs them and on the GPU's own fp16 input of that layer, so the
bound holds element by element.  The matrix reaches every kernel instantiation with partial tiles: both formulations of conv1..conv3,
the per-thread conv1 on ragged and misaligned frames, the smallest frame on the row path, all four model types (both Dense GEMMs, every
head layout), ragged frame stacking, and fp16-subnormal activations.  The production-batch cases run every conv layer at three or
more tiles per persistent CTA, so the stage rings wrap and both TMEM accumulators alternate; there the fp64 evaluation runs on the GPU
in slices of frames.  Run with -s to see the largest err / bound of each layer.

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
from triton_racer_sim_b200 import _native as nat
from triton_racer_sim_b200.pilot import ModelType, PilotNet

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

KIND = {ModelType.CNN_2D: ref.CNN_2D, ModelType.CNN_2D_SPD_FTR: ref.CNN_2D_SPD_FTR, ModelType.CNN_2D_SPD_CTL: ref.CNN_2D_SPD_CTL,
        ModelType.CNN_2D_FULL_HOUSE: ref.CNN_2D_FULL_HOUSE}
FULL = ModelType.CNN_2D_FULL_HOUSE

# name: (model, h, w, frames, max_batch, TRS_PILOT_ROWCONV, frames 4 bytes into their allocation, layer scaled by 2^-12,
#        tiles every CTA of every conv layer must run)
CASES = {
    "120x160_rows": (FULL, 120, 160, 5, 8, "1", False, None, 0),
    "120x160_per_output_row": (FULL, 120, 160, 5, 8, "0", False, None, 0),
    "240x320_rows": (FULL, 240, 320, 3, 4, "1", False, None, 0),
    "240x320_per_output_row": (FULL, 240, 320, 3, 4, "0", False, None, 0),
    "93x96_smallest_row_path": (ModelType.CNN_2D, 93, 96, 4, 4, "1", False, None, 0),
    "96x94_ragged": (ModelType.CNN_2D, 96, 94, 4, 4, "1", False, None, 0),
    "122x166_ragged": (ModelType.CNN_2D_SPD_CTL, 122, 166, 3, 4, "1", False, None, 0),
    "120x160_misaligned": (ModelType.CNN_2D, 120, 160, 4, 8, "1", True, None, 0),
    "n1_speed_feature": (ModelType.CNN_2D_SPD_FTR, 120, 160, 1, 8, "1", False, None, 0),
    "n13_speed_control": (ModelType.CNN_2D_SPD_CTL, 120, 160, 13, 16, "1", False, None, 0),
    "n13_full_house_per_output_row": (FULL, 120, 160, 13, 13, "0", False, None, 0),
    "subnormal_conv3": (FULL, 120, 160, 4, 4, "1", False, 3, 0),
    "subnormal_conv5_per_output_row": (FULL, 120, 160, 4, 4, "0", False, 5, 0),
    # production batch: every persistent CTA walks several tiles, so the mbarrier rings wrap and both TMEM accumulators alternate
    "n3200_rows": (FULL, 120, 160, 3200, 3200, "1", False, None, 3),
    "n3200_per_output_row": (FULL, 120, 160, 3200, 3200, "0", False, None, 3),
    "n3200_misaligned_per_thread_conv1": (ModelType.CNN_2D, 120, 160, 3200, 3200, "1", True, None, 3),
    "n256_240x320_rows": (FULL, 240, 320, 256, 256, "1", False, None, 3),
}
SLICE = 256                  # frames per slice of the fp64 check: host memory stays bounded at production batch


def tiles_per_cta(kernels, h, w, n, sms):
    """conv layer -> (kernel, tiles, grid): tiles from the layer_kernels boxes, the grid from each launch in pilot_api.cu:
    k_pilot_gemm 2 SMs for NPAD <= 128, otherwise SMs (launch_gemm, line 141); k_pilot_rowconv SMs * 512 / (2 * ACC_COLS) with
    ACC_COLS = 256 (launch_rowconv, line 156); k_pilot_conv1r SMs (line 567); k_pilot_conv1 2 SMs, one frame per tile (line 580).
    The Dense GEMM (layer 8) tiles 128 frames and stays at one tile per CTA at any max_batch the workspace allows; its K loop wraps
    the stage ring within a tile."""
    out, hi, wi = {}, h, w
    for layer, (k, s, _) in enumerate(ref.CONVS, 1):
        ho, wo = (hi - k) // s + 1, (wi - k) // s + 1
        kern, (bx, by, bn) = kernels[layer]
        if kern == "k_pilot_conv1":
            tiles, cap = -(-wo // bx) * -(-ho // by) * n, 2 * sms
        else:
            tiles = -(-wo // bx) * -(-ho // by) * -(-n // bn)
            cap = sms if kern in ("k_pilot_conv1r",) or kern.startswith("k_pilot_rowconv") else \
                (2 * sms if int(kern.split("<")[1].split(",")[0]) <= 128 else sms)
        out[layer] = (kern, tiles, min(tiles, cap))
        hi, wi = ho, wo
    return out


@pytest.mark.parametrize("case", list(CASES))
def test_every_layer_within_the_bound_and_heads_bit_exact(monkeypatch, case):
    mt, h, w, n, cap, rowconv, misaligned, scaled, min_tiles = CASES[case]
    kind = KIND[mt]
    full = mt == FULL
    monkeypatch.setenv("TRS_PILOT_ROWCONV", rowconv)
    kernels = pb.layer_kernels(h, w, rowconv == "1", not misaligned, full)
    if min_tiles:
        assert cap == n, f"[{case}] max_batch {cap} < {n} frames: the layers run in several launches"
        ctx = nat.Context(0)
        sms = ctx.sm_count
        ctx.close()
        for layer, (kern, tiles, grid) in tiles_per_cta(kernels, h, w, n, sms).items():
            assert tiles // grid >= min_tiles, (f"[{case}] conv{layer} ({kern}): {tiles} tiles on {grid} CTAs leave a CTA "
                                                f"{tiles // grid} tiles, the case needs {min_tiles} on {sms} SMs")
    wts = ref.random_weights(kind, h, w, seed=3)
    if scaled:
        for t in ("kernel", "bias"):
            wts[f"conv{scaled}/{t}"] = (wts[f"conv{scaled}/{t}"] * np.float32(2.0 ** -12)).astype(np.float32)
    frames = synth.frame_pool(n, h, w, seed=h + w + n) if n <= 64 else synth.expand_numpy(synth.frame_pool(64, h, w, seed=h + w), n)
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
    del dev
    packed = pb.pack_weights(wts, kind, h, w)

    failures, lines = [], []
    prev = frames
    for layer in range(1, 8):
        kern, box = kernels[layer]
        y = net.activation(layer, n)
        # the worst element over frame slices; the mismatch fraction over all frames
        max_ratio, n_mismatch, n_sub, worst_rep, worst_f0 = -1.0, 0.0, 0, None, 0
        for f0 in range(0, n, SLICE):
            ys = y[f0:f0 + SLICE]
            s, a = pb.conv_exact(prev[f0:f0 + SLICE], packed[f"conv{layer}/kernel"], ref.CONVS[layer - 1][1], device="cuda")
            assert ys.shape == s.shape, (layer, ys.shape, s.shape)
            rep = pb.fp16_layer(ys, s, a, wts[f"conv{layer}/bias"], pb.reduction_len(layer))
            n_mismatch += rep["mismatch"] * ys.size
            n_sub += int(np.count_nonzero((ys != 0) & (np.abs(ys.astype(np.float32)) < 2.0 ** -14)))
            if rep["max_ratio"] > max_ratio:
                max_ratio, worst_rep, worst_f0 = rep["max_ratio"], rep, f0
            del s, a, rep
        mismatch, sub = n_mismatch / y.size, n_sub / y.size
        lines.append(f"conv{layer} {kern:26s} box {box}: max err/bound {max_ratio:.3f}  y != RN16(yhat) {mismatch:.2e}"
                     f"  subnormal {sub:.2e}")
        if max_ratio > 1.0 or mismatch > pb.MISMATCH_MAX:
            failures.append(f"conv{layer} ({kern}, box bx, by, bn = {box}): max err/bound {max_ratio:.3f}, "
                            f"y != RN16(yhat) in {mismatch:.2%}\n  {pb.worst(worst_rep, box, frame0=worst_f0)}")
        if layer == scaled:                                           # out of this epilogue and into the next layer's MMA
            assert sub > 0.01, f"conv{layer}: only {sub:.2%} of the activations are fp16-subnormal"
        worst_rep = None
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
