#!/usr/bin/env python
"""Generates tests/golden/ref_baseline_golden.npz by running the REFERENCE's own layer code (oracle/_ref, built by
oracle/ref_shim/build_ref.py from a checkout of the reference) on a GPU, at the BASELINE.json shapes of ref_cases.py:

    python tests/golden/make_baseline_golden.py OUT.npz          (on a GPU; then copy OUT.npz to tests/golden/)

Correlation d=21 through CorrelationLayer::Forward_gpu, and predict_flow_final of FlowNet2-C / -CSS / FlowNet2 through
oracle.ref.RefNet (the reference's layer classes in GPU mode, synthetic weights as in tests/test_ref_gpu.py).  Only an evenly
spaced sample of each output is stored (ref_cases.baseline_sample); the inputs are regenerated from seeds.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_cases as RC  # noqa: E402
from oracle import ref as R  # noqa: E402
from oracle.net import synth_weights  # noqa: E402
from tests.util import rng, smooth_images  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_baseline_golden.npz")
    import torch
    assert torch.cuda.is_available(), "needs a GPU: the reference's layers run in GPU mode"
    import flownet2_b200 as F
    R.set_mode(True, 0)
    g = {}
    for shape in RC.BASELINE_CORR_SHAPES:
        a, b = RC.baseline_corr_inputs(shape)
        top, = R.run_layer(RC.BASELINE_CORR_TEXT, [a, b])
        g[RC.baseline_corr_key(shape)] = RC.baseline_sample(top, RC.BASELINE_SAMPLES["corr"])
        print(shape, "absmax %.4g" % float(np.abs(top).max()), flush=True)
    for model, w, h in RC.BASELINE_NETS:
        proto = F.fill_template(F.model_template(model), w, h)
        weights, _ = synth_weights(F.fill_template(F.model_template(model), 64, 64), 1701, proto)
        img0, img1 = smooth_images(rng(1701), 1, h, w)
        flow = R.RefNet(proto, weights, batch=1).forward(img0=img0, img1=img1).blob("predict_flow_final")
        g[RC.baseline_net_key(model, w, h)] = RC.baseline_sample(flow, RC.BASELINE_SAMPLES["net"])
        print(model, w, h, "absmax %.4g" % float(np.abs(flow).max()), flush=True)
    g["device"] = np.array(torch.cuda.get_device_name(0))
    np.savez_compressed(out, **g)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
