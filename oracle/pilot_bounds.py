"""Per-layer error bounds for the pilots' networks — TEST INFRASTRUCTURE ONLY (tests/test_pilot_bounds_*.py).

oracle/pilot_ref.py evaluates the reference's graph in fp32 with the fp32 weights, so a comparison with it has to absorb the fp16 rounding
of the weights, and one tolerance per tensor is all it can state.  This module evaluates each layer in fp64 on the operands the kernels
actually multiply — the weights packed to fp16 exactly as csrc/pilot_api.cu packs them, the GPU's own fp16 input of the layer — so the
only differences left are the fp32 accumulation inside the tensor cores and the rounding of the epilogue, and it states a bound for each
element:

    |y - yhat| <= 0.5 * ulp16(max(|y|, |yhat|)) + 2^-24 * |yhat| + E_acc,     E_acc = 2^-22 * (ceil(K / 16) + 16) * A

for an fp16 layer output y = RN16(max(0, fl32(acc + b))) (the epilogues of k_pilot_gemm, k_pilot_rowconv, k_pilot_conv1 and
k_pilot_conv1r), with S the exact dot product, A = sum |a_i * w_i| and yhat = max(0, S + b).  K is the real reduction length (padding
does not count).  E_acc is an ASSUMPTION about the MMA's fp32 accumulation, not a measurement: every K = 16 step loses at most two fp32
units of the running magnitude (bounded by A), plus 16 units for a truncating alignment inside a step.  DESIGN.md section 4.8 lists the
largest err / bound measured on a B200.

The heads (k_pilot_heads) are sequential fmaf chains in fp32 and are restated here bit for bit (heads_exact).
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from . import pilot_ref as ref

E_ACC_UNIT = 2.0 ** -22          # fp32 units of the running magnitude lost per K = 16 MMA step (assumed)
E_ACC_SLACK_STEPS = 16           # truncating alignment inside a step (assumed)
MISMATCH_MAX = 0.01              # fp16 layers: largest fraction of elements with y != RN16(yhat)
L8_MEDIAN_MAX = 2.0 ** -20       # layer 8: largest median of |p - S| / A


# ---- weights as the library packs them ------------------------------------------------------------------------------------------

def pack_weights(wts, model_type, h, w):
    """name -> the array the kernels multiply with.

    pilot_api.cu upload_weights (lines 233-256): conv2..7 and the image rows of dense1 / dense4 are __float2half_rn(w); conv1 is
    __float2half_rn(w / 255.0f), the fp32 division first (line 245, and line 378 for k_pilot_conv1r's copy).  Biases stay fp32
    (line 260), and so do all the weights k_pilot_heads reads (the blob, lines 427-453).  Returned as float16 arrays ("convN/kernel",
    "dense1/image", "dense4/image") and float32 arrays for everything else."""
    out = {k: np.asarray(v, np.float32) for k, v in wts.items()}
    out["conv1/kernel"] = (np.asarray(wts["conv1/kernel"], np.float32) / np.float32(255)).astype(np.float16)
    for i in range(2, 8):
        out[f"conv{i}/kernel"] = np.asarray(wts[f"conv{i}/kernel"], np.float32).astype(np.float16)
    flat = flat_len(h, w)
    for d in ("dense1", "dense4") if model_type == ref.CNN_2D_FULL_HOUSE else ("dense1",):
        out[f"{d}/image"] = np.asarray(wts[f"{d}/kernel"], np.float32)[:flat].astype(np.float16)
    return out


def flat_len(h, w):
    ho, wo = ref.conv_out_hw(h, w)
    return ho * wo * ref.CONVS[-1][2]


def reduction_len(layer):
    """Real K of conv `layer` (1..7): kh * kw * Cin."""
    k, _, _ = ref.CONVS[layer - 1]
    cin = 3 if layer == 1 else ref.CONVS[layer - 2][2]
    return k * k * cin


# ---- fp64 evaluation on the kernels' operands ----------------------------------------------------------------------------------

def conv_exact(x_nhwc, kern16, stride, device="cpu"):
    """S and A of a VALID convolution, NHWC float64.  x: the layer's input as the kernel sees it (u8 bytes for conv1, the fp16
    activation otherwise); kern16: (kh, kw, Cin, Cout) fp16.  fp16 x fp16 and u8 x fp16 products are exact in fp64; the fp64 sums
    are within ~K * 2^-53 * A of the exact ones in any summation order, 2^-25 below the smallest E_acc, so `device` may be a GPU
    (float64 convolutions there sum in another order than on the CPU)."""
    x = torch.from_numpy(np.asarray(x_nhwc).astype(np.float64)).to(device).permute(0, 3, 1, 2)
    k = torch.from_numpy(np.asarray(kern16).astype(np.float64)).to(device).permute(3, 2, 0, 1).contiguous()
    s = F.conv2d(x, k, stride=stride).permute(0, 2, 3, 1).cpu().numpy()
    a = F.conv2d(x.abs(), k.abs(), stride=stride).permute(0, 2, 3, 1).cpu().numpy()
    return s, a


def dense_exact(x_flat, w16):
    """S and A of the image part of the first Dense layers: (N, flat) fp16 features times (flat, units) fp16 weights."""
    x = np.asarray(x_flat).astype(np.float64)
    w = np.asarray(w16).astype(np.float64)
    return x @ w, np.abs(x) @ np.abs(w)


def e_acc(a, k):
    return E_ACC_UNIT * (math.ceil(k / 16) + E_ACC_SLACK_STEPS) * a


def ulp16(v):
    """Spacing of the fp16 grid at |v| (np.spacing on float16: subnormals included)."""
    return np.spacing(np.abs(np.asarray(v, np.float64)).astype(np.float16)).astype(np.float64)


def fp16_layer(y, s, a, bias, k):
    """Check one fp16 layer output y (NHWC float16) against S, A (NHWC float64).  Returns a dict:
    ratio (err / bound per element), max_ratio, mismatch (fraction of y != RN16(yhat)), yhat."""
    y64 = np.asarray(y).astype(np.float64)
    yhat = np.maximum(s + np.asarray(bias, np.float64), 0.0)
    bound = 0.5 * ulp16(np.maximum(np.abs(y64), yhat)) + 2.0 ** -24 * yhat + e_acc(a, k)
    err = np.abs(y64 - yhat)
    ratio = np.where(np.isfinite(y64), err / bound, np.inf)
    mismatch = float(np.mean(np.asarray(y, np.float16) != yhat.astype(np.float16)))
    return dict(ratio=ratio, max_ratio=float(ratio.max()), mismatch=mismatch, yhat=yhat, err=err, bound=bound)


def partial_layer(p, s, a, k):
    """Layer 8: fp32 partial sums p (no bias) against S.  ratio = |p - S| / E_acc; median = median of |p - S| / A."""
    err = np.abs(np.asarray(p, np.float64) - s)
    ratio = err / e_acc(a, k)
    rel = err / np.where(a > 0, a, 1.0)
    return dict(ratio=ratio, max_ratio=float(ratio.max()), median=float(np.median(rel)), err=err, bound=e_acc(a, k))


# ---- tiles the kernels cut each layer into (restated from pilot_api.cu, for the failure messages) ---------------------------------

BLOCK_M = 128


def _choose_box(wo, ho, conv1):
    """pilot_api.cu choose_box (lines 72-88)."""
    best, bx, by, bn = -1.0, 1, 1, 1
    for x in range(1, min(wo, BLOCK_M) + 1):
        for y in range(1, ho + 1):
            if x * y > BLOCK_M:
                break
            if conv1 and ((6 * x + 23) // 4 + 1) * (2 * y + 3) > 128 * 6:
                continue
            nmax = BLOCK_M // (x * y) if (x == wo and not conv1) else 1
            for n in range(1, nmax + 1):
                tiles = ((wo + x - 1) // x) * ((ho + y - 1) // y) / n
                eff = wo * ho / (tiles * BLOCK_M)
                if eff > best + 1e-9 or (eff > best - 1e-9 and x > bx):
                    best, bx, by, bn = eff, x, y, n
    return bx, by, bn


def _choose_row_box(wo, xmax=BLOCK_M, nmax=BLOCK_M):
    """pilot_api.cu choose_row_box (lines 91-100) and the k_pilot_conv1r variant (lines 363-368)."""
    best, bx, bn = -1.0, 1, 1
    for x in range(1, min(wo, xmax) + 1):
        xt, n = (wo + x - 1) // x, min(BLOCK_M // x, nmax)
        eff = wo * n / (xt * BLOCK_M)
        if eff > best + 1e-9 or (eff > best - 1e-9 and x > bx):
            best, bx, bn = eff, x, n
    return bx, bn


def layer_kernels(h, w, rowconv=True, frames_16_aligned=True, full_house=False):
    """layer (1..8) -> (kernel name, (bx, by, bn) box of output columns, rows, frames) as pilot_api.cu build / run_layer pick them."""
    out, hi, wi = {}, h, w
    for i, (k, s, f) in enumerate(ref.CONVS):
        ho, wo = (hi - k) // s + 1, (wi - k) // s + 1
        npad = 32 if f <= 32 else 64 if f <= 64 else 128
        if i == 0:
            if rowconv and w % 16 == 0 and frames_16_aligned:
                bx, bn = _choose_row_box(wo, 40, 4)
                out[1] = ("k_pilot_conv1r", (bx, 7, bn))
            else:
                out[1] = ("k_pilot_conv1", _choose_box(wo, ho, True))
        elif rowconv and i in (1, 2):
            bx, bn = _choose_row_box(wo)
            out[i + 1] = (f"k_pilot_rowconv<{f}>", (bx, 256 // f, bn))
        else:
            out[i + 1] = (f"k_pilot_gemm<{npad},{ {32: 5, 64: 4, 128: 3}[npad]}>", _choose_box(wo, ho, False))
        hi, wi = ho, wo
    out[8] = ("k_pilot_gemm<256,4,f32>" if full_house else "k_pilot_gemm<128,3,f32>", (1, 1, BLOCK_M))
    return out


def worst(report, box, count=6, frame0=0):
    """The `count` largest err / bound elements of an (N, H, W, C) report: (frame, y, x, channel), their position in the layer's box
    (bx, by, bn), err, bound and the exact value.  frame0: the batch index of the report's first frame."""
    r = report["ratio"]
    bx, by, bn = box
    exact = report.get("yhat")
    lines = []
    for f in np.argsort(r, axis=None)[::-1][:count]:
        i = np.unravel_index(f, r.shape)
        n, yy, xx, c = i
        n += frame0
        lines.append(f"(n={n}, y={yy}, x={xx}, c={c}) in box (n%{bn}={n % bn}, y%{by}={yy % by}, x%{bx}={xx % bx}): "
                     f"err/bound={r[i]:.3g} err={report['err'][i]:.4g} bound={report['bound'][i]:.4g}"
                     + (f" exact={exact[i]:.6g}" if exact is not None else ""))
    return "\n  ".join(lines)


# ---- fmaf, bit for bit -------------------------------------------------------------------------------------------------------

def fmaf(a, b, c):
    """Correctly rounded float32 a * b + c, element-wise on numpy arrays.  The fp64 product of two float32 is exact; TwoSum gives the
    fp64 sum s and its exact error e; RN32(s) equals RN32(a*b + c) unless s is a float32 midpoint reached by rounding (e != 0), in which
    case the exact value lies on e's side of the midpoint."""
    a = np.asarray(a, np.float32).astype(np.float64)
    b = np.asarray(b, np.float32).astype(np.float64)
    c = np.asarray(c, np.float32).astype(np.float64)
    p = a * b
    s = p + c
    bp = s - c
    e = (p - bp) + (c - (s - bp))                                 # TwoSum: p + c = s + e exactly
    r = s.astype(np.float32)
    d = s - r.astype(np.float64)                                  # exact: r is within one float32 spacing of s
    toward = np.nextafter(r, np.where(d > 0, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
    tie = (d != 0) & (2.0 * d == toward.astype(np.float64) - r.astype(np.float64))
    fix = tie & (e != 0) & (np.sign(e) == np.sign(d))             # the exact value is past the midpoint, away from r
    return np.where(fix, toward, r).astype(np.float32)


def _dense_chain(w, b, x, relu):
    """dense_warp (pilot_kernels.cuh:1109-1118): acc = b[j]; acc = fmaf(in[k], w[k][j], acc) for k ascending; fmaxf(acc, 0)."""
    acc = np.broadcast_to(np.asarray(b, np.float32), (x.shape[0], len(b))).copy()
    for k in range(x.shape[1]):
        acc = fmaf(x[:, k:k + 1], w[k][None, :], acc)
    return np.maximum(acc, np.float32(0)) if relu else acc


def heads_exact(wts, model_type, partial, ldp, spd_feature=None, loc_feature=None):
    """k_pilot_heads (pilot_kernels.cuh:1123-1168) restated bit for bit: (N, 2) float32 from the GPU's layer-8 partial sums
    (N, ldp) and the features.

    The order of every sum is the kernel's: the first Dense layer is fl32(partial + bias), then fmaf over head 0's feature branch
    (n_prev rows, the full-house steering head only), then over this head's own branch; every other Dense layer starts from its bias
    and runs k ascending.  ReLU is fmaxf.  Head 0 of the full-house model writes output slot 1 (speed), head 1 slot 0 (steering);
    the other models have one head with two outputs.  A change to the summation order in the kernel must change this restatement in the
    same commit."""
    part = np.asarray(partial, np.float32).reshape(-1, ldp)
    n = part.shape[0]
    full = model_type == ref.CNN_2D_FULL_HOUSE
    f32 = lambda v: np.asarray(v, np.float32).reshape(n, 1)
    if full:
        heads = [(("feature1", "feature2", "feature3"), ("dense1", "dense2", "dense3", "output_speed"), f32(loc_feature), 1),
                 (("current_spd_1", "current_spd_2", "current_spd_3"), ("dense4", "dense5", "dense6", "out_steering"), f32(spd_feature), 0)]
    elif model_type == ref.CNN_2D_SPD_FTR:
        heads = [(("feature1", "feature2", "feature3"), ("dense1", "dense2", "dense3", "output_layer"), f32(spd_feature), 0)]
    else:
        heads = [((), ("dense1", "dense2", "dense3", "output_layer"), None, 0)]
    out = np.zeros((n, 2), np.float32)
    keep = np.zeros((n, 0), np.float32)
    flat = None
    for h, (fnames, dnames, feat, slot) in enumerate(heads):
        y = np.zeros((n, 0), np.float32)
        if fnames:
            y = feat
            for nm in fnames:
                y = _dense_chain(wts[f"{nm}/kernel"], wts[f"{nm}/bias"], y, True)
        k1 = np.asarray(wts[f"{dnames[0]}/kernel"], np.float32)
        n_prev = keep.shape[1] if (full and h == 1) else 0
        flat = k1.shape[0] - y.shape[1] - n_prev
        acc = (part[:, 128 * h:128 * h + 100] + np.asarray(wts[f"{dnames[0]}/bias"], np.float32)).astype(np.float32)
        xs = np.concatenate([keep[:, :n_prev], y], 1)
        for k in range(xs.shape[1]):
            acc = fmaf(xs[:, k:k + 1], k1[flat + k][None, :], acc)
        q = np.maximum(acc, np.float32(0))
        q = _dense_chain(wts[f"{dnames[1]}/kernel"], wts[f"{dnames[1]}/bias"], q, True)
        q = _dense_chain(wts[f"{dnames[2]}/kernel"], wts[f"{dnames[2]}/bias"], q, True)
        o = _dense_chain(wts[f"{dnames[3]}/kernel"], wts[f"{dnames[3]}/bias"], q, False)
        out[:, slot:slot + o.shape[1]] = o
        if h == 0:
            keep = y
    return out
