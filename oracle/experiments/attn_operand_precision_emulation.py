"""TEST INFRASTRUCTURE / EVIDENCE -- what fp16 GEMM operands cost the attention (centre-of-mass) CNN.

Runs oracle/attn_oracle_np.attn_forward in float64 twice: as is, and with the operands of the tensor-core GEMMs rounded
where the kernels round them -- the batch-normed activations that feed aconv_2 .. aconv_5 and afc_1, and the filters /
weights of those five layers -- to fp16 (11 significand bits, round to nearest, saturating at +-65504 like
cvt.rn.satfinite).  aconv_1 (the fp32 SIMT stem) and afc_out (the fp32 tail) stay exact, and so does everything
between the GEMMs, so the numbers are the floor an fp16-operand kernel with fp32 accumulation can reach.  Also runs the
bf16 hi + lo split of the default mode (16 significand bits) for comparison.

Reported per tensor: max|a - b| / max|b| (hgru_oracle_np.rel_err) against the exact forward, and the error of the three
outputs (u / height, v / width, d / max depth) in pixels and millimetres at 424 x 512 and a 10 m depth scale, the crop
stage's scaling.  Cases: the golden weights of tests/golden/attn_ref.npz (its own frames), and random-init weights at
the reference widths (64 .. 1024, fc 1024, random batch norm) on Kinect-size frames.

    python oracle/experiments/attn_operand_precision_emulation.py [--out FILE.json]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from monkey_pose_b200 import initialization as init  # noqa: E402
from oracle import attn_oracle_np as anp  # noqa: E402
from oracle import hgru_oracle_np as onp  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", "tests", "golden", "attn_ref.npz")
TENSORS = ("pool1", "pool2", "pool3", "pool4", "pool5", "fc1", "out_put")
BAR = 2.5e-3
SCALE = (424.0, 512.0, 10000.0)       # image_orig_size[0], [1], image_max_depth: tr * SCALE = centre of mass


def fp16(x):
    return np.clip(np.asarray(x, np.float64), -65504.0, 65504.0).astype(np.float16).astype(np.float64)


def bf16_hilo(x):
    import torch
    t = torch.as_tensor(np.asarray(x, np.float64))
    hi = t.to(torch.bfloat16).to(torch.float64)
    return (hi + (t - hi).to(torch.bfloat16).to(torch.float64)).numpy()


class _GemmOperandsRounded(object):
    """Stands in for hgru_oracle_np inside attn_oracle_np: conv_layer / fc_layer round both operands of the layers
    whose weights are in `ids` (aconv_2..5, afc_1); every other function is the original."""

    def __init__(self, rnd, ids):
        self.rnd, self.ids = rnd, ids

    def __getattr__(self, name):
        return getattr(onp, name)

    def conv_layer(self, x, filt, bias):
        if id(filt) in self.ids:
            return onp.conv_layer(self.rnd(x), self.rnd(filt), bias)
        return onp.conv_layer(x, filt, bias)

    def fc_layer(self, x, w, b):
        if id(w) in self.ids:
            return onp.fc_layer(self.rnd(x), self.rnd(w), b)
        return onp.fc_layer(x, w, b)


def forward(frames, P, rnd=None):
    if rnd is None:
        return anp.attn_forward(frames, P, trace=True)[1]
    ids = {id(P["%s/%s_filters" % (n, n)]) for n in anp.CONV_NAMES[1:]} | {id(P["afc_1/afc_1_weights"])}
    saved, anp.onp = anp.onp, _GemmOperandsRounded(rnd, ids)
    try:
        return anp.attn_forward(frames, P, trace=True)[1]
    finally:
        anp.onp = saved


def compare(frames, P):
    ref = forward(frames, P)
    res = {}
    for arm, rnd in (("fp16", fp16), ("bf16x3", bf16_hilo)):
        got = forward(frames, P, rnd)
        r = {k: onp.rel_err(got[k], ref[k])[0] for k in TENSORS}
        d = np.abs(got["out_put"] - ref["out_put"]) * np.array(SCALE)
        r["out_abs_err"] = {"u_px_max": float(d[:, 0].max()), "v_px_max": float(d[:, 1].max()),
                            "d_mm_max": float(d[:, 2].max()), "u_px_mean": float(d[:, 0].mean()),
                            "v_px_mean": float(d[:, 1].mean()), "d_mm_mean": float(d[:, 2].mean())}
        r["worst"] = max(r[k] for k in TENSORS)
        res[arm] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--frames", type=int, default=4, help="frames of the random-init case")
    a = ap.parse_args()
    z = np.load(GOLDEN)
    Pg = {k[4:]: z[k] for k in z.files if k.startswith("var:")}
    rng = np.random.default_rng(3)
    frames = rng.uniform(0.06, 0.4, size=(a.frames, 424, 512, 1)).astype(np.float32)
    frames[rng.uniform(size=frames.shape) < 0.05] = 0.0
    Pr = init.attn_params((64, 128, 256, 512, 1024), 1024, 3, seed=5, random_bn=True)
    golden = "golden (widths %s, fc %d)" % (tuple(int(v) for v in z["widths"]), int(z["fc_hidden"]))
    out = {"bar": BAR,
           golden: compare(z["frames"], Pg),
           "random init (widths (64, 128, 256, 512, 1024), fc 1024, %d frames 424x512)" % a.frames: compare(frames, Pr)}
    ok = True
    for case, arms in out.items():
        if case == "bar":
            continue
        print(case)
        print("  %-7s" % "arm" + "".join("%10s" % k for k in TENSORS) + "   |du| px  |dv| px  |dd| mm (max)")
        for arm, r in arms.items():
            e = r["out_abs_err"]
            print("  %-7s" % arm + "".join("%10.2e" % r[k] for k in TENSORS)
                  + "   %7.4f  %7.4f  %7.4f" % (e["u_px_max"], e["v_px_max"], e["d_mm_max"]))
        ok &= arms["fp16"]["worst"] < BAR
    out["fp16_meets_bar"] = bool(ok)
    print("fp16 %s the %.1e bar on every tensor" % ("meets" if ok else "FAILS", BAR))
    if a.out:
        json.dump(out, open(a.out, "w"), indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
