"""Case list shared by tests/golden/make_ref_golden.py (runs the REFERENCE's own layer code, oracle/_ref, on the GPU box
and writes tests/golden/ref_golden.npz) and by the tests that compare the oracle (CPU) and the CUDA kernels (GPU) with
those vectors.  Inputs are regenerated from the seeds below, only the reference's outputs are stored.

A layer case: name -> dict(text=prototxt of one layer, inputs=fn(rng)->[bottoms], params=fn(rng, bottoms)->[blobs] or None,
ntop, backward=bool (top diffs drawn after the inputs), tol = what the GPU/oracle comparison may differ by, and why).
"""
import numpy as np


def rng_for(name):
    return np.random.default_rng([1701] + [ord(c) for c in name])


def _normal(*shape):
    return lambda r: r.standard_normal(shape).astype(np.float32)


def _corr(name, C, H, W, pad, k, md, s1, s2, typ="MULTIPLY", N=2, backward=False):
    text = ('name: "%s" type: "Correlation" bottom: "a" bottom: "b" top: "t" correlation_param { pad: %d kernel_size: %d '
            'max_displacement: %d stride_1: %d stride_2: %d correlation_type: %s }' % (name, pad, k, md, s1, s2, typ))
    return dict(text=text, inputs=lambda r: [r.standard_normal((N, C, H, W)).astype(np.float32),
                                              r.standard_normal((N, C, H, W)).astype(np.float32)],
                ntop=1, backward=backward, kind="correlation", args=(pad, k, md, s1, s2, 0 if typ == "MULTIPLY" else 1))


def _corr1d(name, C, H, W, pad, k, md, s1, s2, sd=0, typ="MULTIPLY", N=2, backward=True):
    text = ('name: "%s" type: "Correlation1D" bottom: "a" bottom: "b" top: "t" correlation_param { pad: %d kernel_size: %d '
            'max_displacement: %d stride_1: %d stride_2: %d single_direction: %d correlation_type: %s }' % (name, pad, k, md, s1, s2, sd, typ))
    return dict(text=text, inputs=lambda r: [r.standard_normal((N, C, H, W)).astype(np.float32),
                                              r.standard_normal((N, C, H, W)).astype(np.float32)],
                ntop=1, backward=backward, kind="correlation1d", args=(pad, k, md, s1, s2, sd, 0 if typ == "MULTIPLY" else 1))


def _resample(name, shape, oh, ow, typ, antialias=True):
    text = ('name: "%s" type: "Resample" bottom: "x" top: "y" resample_param { width: %d height: %d type: %s antialias: %s }'
            % (name, ow, oh, typ, "true" if antialias else "false"))
    return dict(text=text, inputs=lambda r: [r.standard_normal(shape).astype(np.float32)], ntop=1, kind="resample",
                args=(oh, ow, {"NEAREST": 1, "LINEAR": 2, "CUBIC": 3}[typ], antialias))


def _warp_inputs(shape):
    def f(r):
        N, C, H, W = shape
        img = r.uniform(0, 1, shape).astype(np.float32)
        flow = r.uniform(-6, 6, (N, 2, H, W)).astype(np.float32)
        flow[0, :, 2, 3] = 100.0                       # out of range -> fill value
        flow[-1, 0, 1, 1] = -float(W)
        flow[0, :, 0, 0] = 0.0                         # exact integer coordinate
        flow[0, 0, H - 1, W - 1] = 0.0; flow[0, 1, H - 1, W - 1] = 0.0   # right/bottom clamp
        return [img, flow]
    return f


AUG_COMMON = "augment_during_test: true "


def _aug_params(n_iter, shape_top, mean_val=0.4):
    def f(r, bottoms):
        C, H, W = shape_top
        return [np.full((1, 1, 1, 1), n_iter, np.float32),
                (mean_val + 0.05 * r.standard_normal((1, C, H, W))).astype(np.float32),
                (mean_val + 0.02 * np.arange(C)).astype(np.float32).reshape(1, C, 1, 1)]
    return f


# (N,42) coefficient blob in ARRAY form (fields with default 1 stored as logarithms, augmentation_layer_base.cpp:352-365)
COEFF_DEFAULT = np.array([0, 0, 0, 0, 1, 1, 1, 0, 1, 1, 1, 1] + [1, 1, 1, 0, 0, 0, 1, 1, 1, 1, 1, 1, 0, 0, 0, 1, 1, 1, 1, 0, 1, 0] + [0] * 8,
                         np.float32)
EIGVEC = [0.51, 0.56, 0.65, 0.79, 0.01, -0.62, 0.35, -0.83, 0.44]


def coeff_blob(r, N, spatial=True, chroma=True, eigen=True, effects=True):
    v = np.tile(COEFF_DEFAULT, (N, 1)).astype(np.float64)
    if spatial:
        v[:, 0] = r.integers(0, 2, N)                         # mirror
        v[:, 1:3] = r.uniform(-0.1, 0.1, (N, 2))             # dx dy
        v[:, 3] = r.uniform(-0.3, 0.3, N)                     # angle
        v[:, 4:6] = np.exp(r.uniform(-0.2, 0.2, (N, 2)))      # zoom
    if chroma:
        v[:, 6] = np.exp(r.normal(0, 0.2, N)); v[:, 7] = r.normal(0, 0.05, N); v[:, 8] = np.exp(r.normal(0, 0.2, N))
        v[:, 9:12] = np.exp(r.normal(0, 0.1, (N, 3)))
    if eigen:
        v[:, 12:34] = np.where(COEFF_DEFAULT[12:34] == 1, np.exp(r.uniform(-0.2, 0.2, (N, 22))), r.uniform(-0.05, 0.05, (N, 22)))
    if effects:
        v[:, 38] = r.uniform(-3.1, 3.1, N); v[:, 39] = r.uniform(-5, 5, N); v[:, 40] = r.uniform(0.1, 0.3, N)   # shadow
    v[0] = COEFF_DEFAULT                                       # one all-default sample (clear_defaults path)
    with np.errstate(divide="ignore", invalid="ignore"):
        arr = np.where(np.abs(COEFF_DEFAULT) < 1e-3, v, np.log(v))
    return arr.astype(np.float32).reshape(N, 42, 1, 1)


def _aug_train(name, flags):
    text = ('name: "%s" type: "DataAugmentation" bottom: "x" bottom: "p" top: "y" augmentation_param { augment_during_test: true '
            'crop_width: 24 crop_height: 16 max_multiplier: 1 %s }' % (name, " ".join("chromatic_eigvec: %g" % e for e in EIGVEC)))
    return dict(text=text, inputs=lambda r: [r.uniform(0.02, 0.98, (3, 3, 20, 28)).astype(np.float32), coeff_blob(r, 3, **flags)],
                ntop=1, kind="aug_train", args=(24, 16))


LAYER_CASES = {
    # ---- Correlation (correlation_layer.cu:46-114, 253-293; backward :118-249, :298-427) -------------------------------
    "corr_fn2c": _corr("corr_fn2c", 64, 10, 12, 20, 1, 20, 1, 2),                  # FlowNet2-C's parameters, 441 channels
    "corr_d9": _corr("corr_d9", 32, 12, 14, 8, 1, 8, 1, 2, backward=True),
    "corr_k3": _corr("corr_k3", 8, 16, 16, 4, 3, 4, 2, 1, backward=True),
    "corr_s2_1": _corr("corr_s2_1", 16, 9, 11, 3, 1, 3, 1, 1, backward=True),
    "corr_sub": _corr("corr_sub", 16, 9, 11, 2, 1, 2, 1, 1, typ="SUBTRACT", backward=True),
    "corr_c40": _corr("corr_c40", 40, 7, 9, 4, 1, 4, 1, 2),                        # C not a multiple of 32 (lane-strided sum)
    # ---- Correlation1D (correlation_layer1d.cu): x displacements only; both / left / right; SUBTRACT -------------------------
    "corr1d_both": _corr1d("corr1d_both", 16, 7, 19, 8, 1, 8, 1, 2),
    "corr1d_left": _corr1d("corr1d_left", 16, 7, 19, 8, 1, 8, 1, 2, sd=-1),
    "corr1d_right": _corr1d("corr1d_right", 16, 7, 19, 8, 1, 8, 1, 2, sd=1),
    "corr1d_k3": _corr1d("corr1d_k3", 8, 11, 21, 4, 3, 4, 2, 1),
    "corr1d_sub": _corr1d("corr1d_sub", 8, 6, 15, 3, 1, 3, 1, 1, typ="SUBTRACT"),
    # ---- Resample (resample_layer.cu:40-125,128-206) ----------------------------------------------------------------------
    "rs_lin_up": _resample("rs_lin_up", (2, 3, 13, 17), 26, 34, "LINEAR"),
    "rs_lin_flow_up": _resample("rs_lin_flow_up", (1, 2, 16, 32), 61, 128, "LINEAR"),     # 112x256 -> 436x1024 in small
    "rs_lin_img_up": _resample("rs_lin_img_up", (1, 3, 25, 40), 32, 40, "LINEAR"),        # 436 -> 448 rows, same width
    "rs_lin_down_aa": _resample("rs_lin_down_aa", (2, 3, 13, 17), 5, 7, "LINEAR", True),
    "rs_lin_down_noaa": _resample("rs_lin_down_noaa", (2, 3, 13, 17), 5, 7, "LINEAR", False),
    "rs_cubic_up": _resample("rs_cubic_up", (1, 2, 11, 15), 23, 31, "CUBIC"),
    "rs_cubic_down": _resample("rs_cubic_down", (1, 2, 22, 30), 9, 13, "CUBIC"),
    "rs_nearest_down": _resample("rs_nearest_down", (1, 2, 20, 30), 10, 15, "NEAREST"),
    "rs_nearest_up2": _resample("rs_nearest_up2", (1, 2, 10, 15), 20, 30, "NEAREST"),
    "rs_same": _resample("rs_same", (1, 2, 9, 10), 9, 10, "LINEAR"),
    # ---- DataAugmentation, deploy use (data_augmentation_layer.cu:321-637, .cpp:86-158) -----------------------------------
    "aug_deploy_pc": dict(text='name: "a" type: "DataAugmentation" bottom: "x" top: "y" augmentation_param { ' + AUG_COMMON +
                          'recompute_mean: 1000 mean_per_pixel: false crop_width: 24 crop_height: 20 }',
                          inputs=lambda r: [r.uniform(0, 1, (2, 3, 20, 24)).astype(np.float32)],
                          params=_aug_params(2000, (3, 20, 24)), ntop=1, kind="aug_deploy", args=(24, 20, 1000, False)),
    "aug_deploy_pp": dict(text='name: "a" type: "DataAugmentation" bottom: "x" top: "y" augmentation_param { ' + AUG_COMMON +
                          'recompute_mean: 1000 mean_per_pixel: true crop_width: 24 crop_height: 20 }',
                          inputs=lambda r: [r.uniform(0, 1, (2, 3, 20, 24)).astype(np.float32)],
                          params=_aug_params(2000, (3, 20, 24)), ntop=1, kind="aug_deploy", args=(24, 20, 1000, True)),
    "aug_deploy_update": dict(text='name: "a" type: "DataAugmentation" bottom: "x" top: "y" augmentation_param { ' + AUG_COMMON +
                              'recompute_mean: 1000 mean_per_pixel: false crop_width: 24 crop_height: 20 }',
                              inputs=lambda r: [r.uniform(0, 1, (2, 3, 20, 24)).astype(np.float32)],
                              params=_aug_params(5, (3, 20, 24)), ntop=1, kind="aug_deploy", args=(24, 20, 1000, False),
                              keep_params=True),
    "aug_deploy_crop": dict(text='name: "a" type: "DataAugmentation" bottom: "x" top: "y" augmentation_param { ' + AUG_COMMON +
                            'crop_width: 16 crop_height: 12 mean: 0.4 mean: 0.42 mean: 0.44 mean_per_pixel: false }',
                            inputs=lambda r: [r.uniform(0, 1, (2, 3, 20, 24)).astype(np.float32)],
                            ntop=1, kind="aug_deploy", args=(16, 12, 0, False)),
    # ---- DataAugmentation, training use with a given coefficient blob (:446-587) ------------------------------------------
    "aug_train_spatial": _aug_train("aug_train_spatial", dict(spatial=True, chroma=False, eigen=False, effects=False)),
    "aug_train_chroma": _aug_train("aug_train_chroma", dict(spatial=False, chroma=True, eigen=False, effects=False)),
    "aug_train_eigen": _aug_train("aug_train_eigen", dict(spatial=False, chroma=False, eigen=True, effects=False)),
    "aug_train_effects": _aug_train("aug_train_effects", dict(spatial=False, chroma=False, eigen=False, effects=True)),
    "aug_train_all": _aug_train("aug_train_all", dict(spatial=True, chroma=True, eigen=True, effects=True)),
    # ---- ChannelNorm (channel_norm_layer.cu:17-30), FlowWarp (flow_warp_layer.cu:59-122,170-229) ---------------------------
    "chnorm2": dict(text='name: "n" type: "ChannelNorm" bottom: "x" top: "y"', inputs=lambda r: [r.standard_normal((2, 2, 9, 11)).astype(np.float32)],
                    ntop=1, kind="channel_norm"),
    "chnorm3": dict(text='name: "n" type: "ChannelNorm" bottom: "x" top: "y"', inputs=lambda r: [r.standard_normal((2, 3, 9, 11)).astype(np.float32)],
                    ntop=1, kind="channel_norm"),
    "warp_zero": dict(text='name: "w" type: "FlowWarp" bottom: "i" bottom: "f" top: "o"', inputs=_warp_inputs((2, 3, 13, 17)), ntop=1,
                      backward=True, kind="flow_warp", args=(False,)),
    "warp_nan": dict(text='name: "w" type: "FlowWarp" bottom: "i" bottom: "f" top: "o" flow_warp_param { fill_value: NOT_A_NUMBER }',
                     inputs=_warp_inputs((2, 3, 13, 17)), ntop=1, kind="flow_warp", args=(True,)),
    # ---- conv / deconv through the reference's im2col + cuBLAS path (conv_layer.cu:8-23, deconv_layer.cu:8-23) -------------
    "conv_s2": dict(text='name: "c" type: "Convolution" bottom: "x" top: "y" convolution_param { num_output: 24 kernel_size: 5 stride: 2 pad: 2 }',
                    inputs=_normal(2, 6, 19, 23), params=lambda r, b: [(0.2 * r.standard_normal((24, 6, 5, 5))).astype(np.float32),
                                                                       r.standard_normal(24).astype(np.float32)],
                    ntop=1, kind="conv", args=(2, 2, False)),
    "conv_3x3": dict(text='name: "c" type: "Convolution" bottom: "x" top: "y" convolution_param { num_output: 32 kernel_size: 3 stride: 1 pad: 1 }',
                     inputs=_normal(1, 40, 12, 14), params=lambda r, b: [(0.1 * r.standard_normal((32, 40, 3, 3))).astype(np.float32),
                                                                         r.standard_normal(32).astype(np.float32)],
                     ntop=1, kind="conv", args=(1, 1, False)),
    "deconv_4x4": dict(text='name: "d" type: "Deconvolution" bottom: "x" top: "y" convolution_param { num_output: 16 kernel_size: 4 stride: 2 pad: 1 }',
                       inputs=_normal(2, 20, 7, 9), params=lambda r, b: [(0.1 * r.standard_normal((20, 16, 4, 4))).astype(np.float32),
                                                                         r.standard_normal(16).astype(np.float32)],
                       ntop=1, kind="conv", args=(2, 1, True)),
}

def case_inputs(name):
    """-> (bottoms, params or None, top_diffs or None) for a layer case, deterministic."""
    c = LAYER_CASES[name]
    r = rng_for(name)
    inp = c["inputs"](r)
    bottoms = inp if isinstance(inp, list) else [inp]
    params = c["params"](r, bottoms) if c.get("params") else None
    return bottoms, params, r


# ---- whole nets ------------------------------------------------------------------------------------------------------
# (model, width, height, batch): small enough for the CPU oracle in seconds; the BASELINE shapes below are compared on the
# GPU (tests/test_ref_gpu.py) live against the float64 oracle and against the stored reference outputs.
NET_CASES = {
    "S_128x96": ("FlowNet2-S", 128, 96, 1),
    "C_192x100": ("FlowNet2-C", 192, 100, 1),
    "CSS_128x128": ("FlowNet2-CSS", 128, 128, 1),
    "FN2_128x64": ("FlowNet2", 128, 64, 1),
}


# ---- BASELINE.json shapes ----------------------------------------------------------------------------------------------
# Correlation d=21, k=1 (FlowNet2-C) at the feature maps of configs 2, 3, 4, and the three nets of those configs at batch 1.
# tests/golden/make_baseline_golden.py stores the reference's outputs for them in ref_baseline_golden.npz, as an evenly spaced
# sample of each flattened output (baseline_sample): the whole tensors would be 30-50 MB each.
BASELINE_CORR_SHAPES = [(8, 256, 40, 56), (4, 256, 48, 96), (4, 256, 56, 128)]
BASELINE_CORR_TEXT = ('name: "c" type: "Correlation" bottom: "a" bottom: "b" top: "t" correlation_param { pad: 20 kernel_size: 1 '
                      'max_displacement: 20 stride_1: 1 stride_2: 2 }')
BASELINE_NETS = [("FlowNet2-C", 448, 320), ("FlowNet2-CSS", 768, 384), ("FlowNet2", 1024, 436)]
BASELINE_SAMPLES = {"corr": 4096, "net": 8192}


def baseline_corr_inputs(shape):
    r = np.random.default_rng(shape[0] * 1000 + shape[2])
    return r.standard_normal(shape).astype(np.float32), r.standard_normal(shape).astype(np.float32)


def baseline_corr_key(shape):
    return "corr/%dx%dx%dx%d" % tuple(shape)


def baseline_net_key(model, w, h):
    return "net/%s_%dx%d" % (model, w, h)


def baseline_sample(a, n):
    """n evenly spaced elements of the flattened array (every channel and row is hit)."""
    a = np.asarray(a).reshape(-1)
    return a[(np.arange(n, dtype=np.int64) * a.size) // n]
