"""Evaluates the layer cases of tests/golden/ref_cases.py with (a) the CPU oracle and (b) the CUDA engine, so that both can be
compared with tests/golden/ref_golden.npz -- vectors produced by the REFERENCE's own layer code on a B200
(tests/golden/make_ref_golden.py).

Tolerances (relative to max|reference|, stated per kind in TOL) are what separates the reference's GPU build (nvcc default
-fmad=true, lane-strided / cuBLAS summation orders) from an unfused restatement of the same arithmetic -- measured when the
vectors were generated: correlation / warp / norm / linear resample agree to 1-3 float ulps, bicubic resample to 2e-6 (negative
taps cancel), conv against cuBLAS SGEMM to 6e-7.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import ref_cases as RC  # noqa: E402

from oracle import oracle as O  # noqa: E402

GOLD = os.path.join(HERE, "golden", "ref_golden.npz")
BASELINE_GOLD = os.path.join(HERE, "golden", "ref_baseline_golden.npz")        # tests/golden/make_baseline_golden.py

# kind -> relative tolerance (of max |reference output|) for "same arithmetic, different rounding order"
TOL = {"correlation": 6e-7, "correlation1d": 6e-7, "resample": 1.5e-6, "resample_cubic": 6e-6, "channel_norm": 4e-7, "flow_warp": 5e-7, "conv": 3e-6,
       "aug_deploy": 6e-7, "aug_train": 3e-5, "backward": 1e-6}


def golden():
    return np.load(GOLD)


def tol_for(name, key="top0"):
    c = RC.LAYER_CASES[name]
    if key.startswith("bdiff"):
        return TOL["backward"]
    if c["kind"] == "resample" and c["args"][2] == 3:
        return TOL["resample_cubic"]
    return TOL[c["kind"]]


def rel_err(got, want):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    ng, nw = np.isnan(got), np.isnan(want)
    assert (ng == nw).all(), "NaN pattern differs"
    d = np.abs(np.where(ng, 0, got) - np.where(nw, 0, want))
    scale = max(1e-30, float(np.abs(np.where(nw, 0, want)).max()))
    return float(d.max()) / scale


def coeff_values(params):
    """(N,42,1,1) array-form blob -> coefficient values after array_to_coeff + clear_defaults
    (augmentation_layer_base.cpp:339-379)."""
    p = params.reshape(params.shape[0], 42)
    vals = np.where(np.abs(RC.COEFF_DEFAULT) < 1e-3, p, np.exp(p)).astype(np.float32)
    return np.where(np.abs(RC.COEFF_DEFAULT - vals) < 1e-3, RC.COEFF_DEFAULT, vals)


def oracle_augment(x, params, crop_w, crop_h, eigvec, max_mult, space=None):
    """DataAugmentationLayer::Forward_gpu given the coefficient blob (data_augmentation_layer.cu:446-587), from oracle pieces.
    space: use these chromatic-eigenspace statistics instead of computing them (the reference's own are racy, see
    oracle/ref_shim/ref_capi.cpp ref_layer_debug_eigenspace)."""
    N = x.shape[0]
    vals = coeff_values(params)
    mats = np.stack([O.transmat_from_coeff(crop_w, crop_h, x.shape[3], x.shape[2], mirror=float(vals[n, 0]), angle=float(vals[n, 3]),
                                           dx=float(vals[n, 1]), dy=float(vals[n, 2]), zoom_x=float(vals[n, 4]), zoom_y=float(vals[n, 5]))
                     for n in range(N)])
    out = O.spatial_augmentation(x, mats, crop_h, crop_w)
    eig = vals[:, 12:34]
    if np.any(eig != RC.COEFF_DEFAULT[12:34]):
        out = O.chromatic_eigen_augmentation(out, eig, O.chromatic_eigenspace(x, eigvec) if space is None else space, max_mult)
    chroma = vals[:, 6:12]
    if np.any(chroma != RC.COEFF_DEFAULT[6:12]):
        out = O.color_contrast_augmentation(out, chroma, max_mult)
    eff = np.zeros((N, 9), np.float32)
    eff[:, 0:4] = vals[:, 34:38]
    eff[:, 4], eff[:, 5] = np.cos(vals[:, 38]), np.sin(vals[:, 38])
    eff[:, 6:9] = vals[:, 39:42]
    if np.any((eff[:, 0] != 0) & (eff[:, 1] != 0)) or np.any(eff[:, 3] > 0) or np.any(eff[:, 7] > 0):
        out = O.apply_effects(out, eff, max_mult)
    return out


def oracle_eval(name, gold=None):
    """-> {key: ndarray} with the keys the golden file holds for this case.  gold: the golden archive (only the reference's
    chromatic-eigenspace statistics are taken from it, for the aug_train cases)."""
    c = RC.LAYER_CASES[name]
    bottoms, params, r = RC.case_inputs(name)
    k, out = c["kind"], {}
    if k == "correlation":
        pad, ks, md, s1, s2, typ = c["args"]
        out["top0"] = O.correlation_fwd(bottoms[0], bottoms[1], pad, ks, md, s1, s2, typ, exact_order=True)
        if c.get("backward"):
            td = r.standard_normal(out["top0"].shape).astype(np.float32)
            if typ == 0:
                out["bdiff0"], out["bdiff1"] = O.correlation_bwd(bottoms[0], bottoms[1], td, pad, ks, md, s1, s2)
            else:
                out["bdiff0"], out["bdiff1"] = O.correlation_bwd_ex(bottoms[0], bottoms[1], td, pad, ks, md, s1, s2, 1)
    elif k == "correlation1d":
        pad, ks, md, s1, s2, sd, typ = c["args"]
        out["top0"] = O.correlation1d_fwd(bottoms[0], bottoms[1], pad, ks, md, s1, s2, sd, typ)
        if c.get("backward"):
            td = r.standard_normal(out["top0"].shape).astype(np.float32)
            out["bdiff0"], out["bdiff1"] = O.correlation_bwd_ex(bottoms[0], bottoms[1], td, pad, ks, md, s1, s2, typ, True, sd)
    elif k == "resample":
        oh, ow, t, aa = c["args"]
        out["top0"] = O.resample_fwd(bottoms[0], oh, ow, t, aa)
    elif k == "channel_norm":
        out["top0"] = O.channel_norm(bottoms[0])
    elif k == "flow_warp":
        out["top0"] = O.flow_warp_fwd(bottoms[0], bottoms[1], c["args"][0])
        if c.get("backward"):
            td = r.standard_normal(out["top0"].shape).astype(np.float32)
            out["bdiff0"], out["bdiff1"] = O.flow_warp_bwd(bottoms[0], bottoms[1], td)
    elif k == "conv":
        st, pd, dec = c["args"]
        out["top0"] = (O.deconv_fwd if dec else O.conv_fwd)(bottoms[0], params[0], params[1], st, pd, f64acc=True)
    elif k == "aug_deploy":
        cw, ch, rm, mpp = c["args"]
        x = bottoms[0]
        mats = np.stack([O.transmat_from_coeff(cw, ch, x.shape[3], x.shape[2])] * x.shape[0])
        top = O.spatial_augmentation(x, mats, ch, cw)
        if rm > 0:
            num_iter = float(int(params[0].reshape(-1)[0]) + 1)                      # :353-354
            top, pp, pc = O.mean_subtract(top, 0, num_iter, rm, mpp, params[1].reshape(top.shape[1:]), params[2].reshape(-1))
            if c.get("keep_params"):
                out["param0"] = np.full((1, 1, 1, 1), num_iter, np.float32)
                out["param1"] = pp.reshape(params[1].shape)
                out["param2"] = pc.reshape(params[2].shape)
        else:
            top, _, _ = O.mean_subtract(top, 1, mean_pc=np.array([0.4, 0.42, 0.44], np.float32))
        out["top0"] = top
    elif k == "aug_train":
        cw, ch = c["args"]
        space = gold["L/%s/space" % name] if gold is not None and "L/%s/space" % name in gold.files else None
        out["top0"] = oracle_augment(bottoms[0], bottoms[1], cw, ch, RC.EIGVEC, 1.0, space)
        out["space"] = O.chromatic_eigenspace(bottoms[0], RC.EIGVEC)[:25]
    else:
        raise KeyError(k)
    return out


def check_eigenspace(ref_space, true_space):
    """The reference's statistics vs the exact ones: the mean is an atomicAdd sum (order-dependent in the last ulps); max_abs_eig,
    max_rgb, min_rgb come from the lossy fatomicMax / fatomicMin (data_augmentation_layer.cu:117-143): each is SOME pixel's value,
    bounded by the true extremum.  Returns whether the reference's extrema equal the true ones (they usually do not)."""
    assert np.abs(ref_space[3:6] - true_space[3:6]).max() <= 1e-6                    # mean_rgb
    assert np.all(ref_space[6:9] <= true_space[6:9] + 1e-7) and np.all(ref_space[6:9] > 0)
    assert np.all(ref_space[9:12] <= true_space[9:12] + 1e-7)
    assert np.all(ref_space[12:15] >= true_space[12:15] - 1e-7)
    assert np.array_equal(ref_space[16:25], true_space[16:25])                        # eigvec
    mx = ref_space[6:9].astype(np.float64)                                             # derived values follow THEIR max_abs_eig
    assert abs(float(ref_space[15]) - float(np.sqrt((mx * mx).sum()))) <= 1e-6
    return bool(np.array_equal(ref_space[6:15], true_space[6:15]))


# ---- training-side cases (tests/golden/train_cases.py) ----------------------------------------------------------------------
def _gens_of(layer_text):
    """{generator name: {field: value}} of the augmentation_param of a layer block."""
    from oracle.net import parse_prototxt, get
    ap = get(parse_prototxt(layer_text), "augmentation_param", [])
    gens = {}
    for k, v in ap:
        if isinstance(v, list):
            d = {}
            for kk, vv in v:
                d[kk] = vv if kk == "rand_type" else (vv == "true" if vv in ("true", "false") else float(vv))
            gens[k] = d
    return gens


def train_oracle_eval(name):
    """-> {key: ndarray} with the keys tests/golden/train_golden.npz holds for this case, computed by the oracle."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import train_cases as TC
    c = TC.TRAIN_CASES[name]
    bottoms, params, r = TC.train_inputs(name)
    k, out = c["kind"], {}
    if k == "conv_bwd":
        st, pd, dec = c["args"]
        out["top0"] = (O.deconv_fwd if dec else O.conv_fwd)(bottoms[0], params[0], params[1], st, pd, f64acc=True)
        td = r.standard_normal(out["top0"].shape).astype(np.float32)
        out["bdiff0"], out["pdiff0"], out["pdiff1"] = O.conv_bwd(bottoms[0], params[0], td, st, pd, dec)
    elif k == "l1loss":
        b1 = bottoms[1] if len(bottoms) > 1 else None
        loss, _ = O.l1loss_fwd(bottoms[0], b1, **c["args"])
        out["top0"] = np.array([loss], np.float32)
        g0, g1 = O.l1loss_bwd(bottoms[0], b1, c["top_diff"], **c["args"])
        out["bdiff0"] = g0
        if b1 is not None:
            out["bdiff1"] = g1
    elif k == "downsample":
        out["top0"] = O.downsample_fwd(bottoms[0], *c["args"])
    elif k == "flow_aug":
        cw, ch = c["args"]
        out["top0"] = O.flow_augmentation(bottoms[0], bottoms[1], bottoms[2], cw, ch)
    elif k == "gen_aug":
        mode, image = c["args"]
        gens = _gens_of(c["text"])
        if image:
            arr = O.generate_augmentation_parameters(None, "regenerate", gens, 48, 32, bottoms[0].shape[3], bottoms[0].shape[2], num=bottoms[0].shape[0])
        else:
            arr = O.generate_augmentation_parameters(bottoms[0], mode, gens, 48, 32, 64, 48)
        out["top0"] = arr.reshape(-1, 42, 1, 1)
    else:
        raise KeyError(k)
    return out


TRAIN_TOL = {
    # relative to the largest entry of the tensor
    "conv_bwd": 2e-6,        # fp32 cuBLAS gemm orders against float64 accumulation
    "l1loss": 2e-6,          # cublasSdot order; powf(x, 0.5) against sqrtf
    "downsample": 2e-6,      # FMA contraction of the reference's accumulation
    "flow_aug": 2e-6,        # cos/sin/exp of the host libm, FMA contraction in the kernel (|flow| ~ 10)
    "gen_aug": 2e-6,         # log/exp round trips of the array form
}
