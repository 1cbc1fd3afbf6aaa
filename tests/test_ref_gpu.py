"""GPU parity against the REFERENCE itself.

(1) CUDA kernels (through the C-ABI) vs tests/golden/ref_golden.npz -- vectors the reference's own layer code produced on a
    B200 (tests/golden/make_ref_golden.py; inputs regenerated from seeds, tests/golden/ref_cases.py).
(2) At the BASELINE.json shapes: the engine vs the float64-accumulating CPU oracle (live) with the north_star's STRICT 1e-4
    max-abs on predict_flow_final, and vs tests/golden/ref_baseline_golden.npz -- samples of what the reference's layers
    computed on a B200 for the same seeded inputs (tests/golden/make_baseline_golden.py).
"""
import numpy as np
import pytest

from oracle import oracle as O
from oracle.net import OracleNet, synth_weights, write_caffemodel
from tests import refcheck as RCK
from tests.refcheck import RC
from tests.util import maxabs, rng, smooth_images

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ops(fn2):
    from flownet2_b200 import ops as o
    return o


@pytest.fixture(scope="module")
def gold():
    return RCK.golden()


@pytest.fixture(scope="module")
def baseline_gold():
    return np.load(RCK.BASELINE_GOLD)


def dev(a, channels_last=False):
    t = torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()
    return t.contiguous(memory_format=torch.channels_last) if channels_last and t.dim() == 4 and t.shape[1] > 1 else t


def host(t):
    return t.contiguous().cpu().numpy()


def engine_augment(ops, x, params, crop_w, crop_h, space, max_mult):
    """The same composition as refcheck.oracle_augment with the engine's kernels (fn2_spatial_augmentation, ...)."""
    N = x.shape[0]
    vals = RCK.coeff_values(params)
    mats = np.stack([O.transmat_from_coeff(crop_w, crop_h, x.shape[3], x.shape[2], mirror=float(vals[n, 0]), angle=float(vals[n, 3]),
                                           dx=float(vals[n, 1]), dy=float(vals[n, 2]), zoom_x=float(vals[n, 4]), zoom_y=float(vals[n, 5]))
                     for n in range(N)])
    out = ops.spatial_augmentation(dev(x), dev(mats), crop_h, crop_w)
    eig = vals[:, 12:34]
    if np.any(eig != RC.COEFF_DEFAULT[12:34]):
        sp = torch.zeros(32, device="cuda")
        sp[:25] = dev(space[:25])
        out = ops.chromatic_eigen_augmentation(out, dev(eig), sp, max_mult)
    chroma = vals[:, 6:12]
    if np.any(chroma != RC.COEFF_DEFAULT[6:12]):
        out = ops.color_contrast_augmentation(out, dev(chroma), max_mult)
    eff = np.zeros((N, 9), np.float32)
    eff[:, 0:4] = vals[:, 34:38]
    eff[:, 4], eff[:, 5] = np.cos(vals[:, 38]), np.sin(vals[:, 38])
    eff[:, 6:9] = vals[:, 39:42]
    if np.any(eff[:, 7] > 0):
        out = ops.apply_effects(out, dev(eff), max_mult)
    return host(out)


def engine_eval(fn2, ops, name, gold, channels_last):
    c = RC.LAYER_CASES[name]
    bottoms, params, r = RC.case_inputs(name)
    k, out = c["kind"], {}
    if k == "correlation":
        pad, ks, md, s1, s2, typ = c["args"]
        a, b = dev(bottoms[0], channels_last), dev(bottoms[1], channels_last)
        top = ops.correlation(a, b, pad, ks, md, s1, s2, typ)
        out["top0"] = host(top)
        if c.get("backward"):
            td = dev(r.standard_normal(top.shape).astype(np.float32), channels_last)
            g0, g1 = ops.correlation_backward(a, b, td, pad, ks, md, s1, s2, typ)
            out["bdiff0"], out["bdiff1"] = host(g0), host(g1)
    elif k == "correlation1d":
        pad, ks, md, s1, s2, sd, typ = c["args"]
        a, b = dev(bottoms[0], channels_last), dev(bottoms[1], channels_last)
        top = ops.correlation1d(a, b, pad, ks, md, s1, s2, sd, typ)
        out["top0"] = host(top)
        if c.get("backward"):
            td = dev(r.standard_normal(top.shape).astype(np.float32), channels_last)
            g0, g1 = ops.correlation1d_backward(a, b, td, pad, ks, md, s1, s2, sd, typ)
            out["bdiff0"], out["bdiff1"] = host(g0), host(g1)
    elif k == "resample":
        oh, ow, t, aa = c["args"]
        out["top0"] = host(ops.resample(dev(bottoms[0], channels_last), oh, ow, t, aa))
    elif k == "channel_norm":
        out["top0"] = host(ops.channel_norm(dev(bottoms[0], channels_last)))
    elif k == "flow_warp":
        img, flow = dev(bottoms[0], channels_last), dev(bottoms[1], channels_last)
        top = ops.flow_warp(img, flow, c["args"][0])
        out["top0"] = host(top)
        if c.get("backward"):
            td = dev(r.standard_normal(top.shape).astype(np.float32), channels_last)
            gi, gf = ops.flow_warp_backward(img, flow, td)
            out["bdiff0"], out["bdiff1"] = host(gi), host(gf)
    elif k == "conv":
        st, pd, dec = c["args"]
        out["top0"] = host(ops.conv2d(dev(bottoms[0], channels_last), dev(params[0]), dev(params[1]), st, pd, deconv=dec))
    elif k == "aug_deploy":
        cw, ch, rm, mpp = c["args"]
        x = bottoms[0]
        if c.get("keep_params"):
            # running-mean phase: the layer's CustomCopyBlobs does not take the per-pixel mean when mean_per_pixel is false
            # (data_augmentation_layer.cpp:172-183), the reference case set the blob directly -> kernel level here
            mats = np.stack([O.transmat_from_coeff(cw, ch, x.shape[3], x.shape[2])] * x.shape[0])
            top = ops.spatial_augmentation(dev(x), dev(mats), ch, cw)
            num_iter = float(int(params[0].reshape(-1)[0]) + 1)
            pp, pc = dev(params[1]), dev(params[2].reshape(-1))
            ops.mean_update(top, pp, pc, num_iter)
            ops.mean_subtract(top, pp, pc, mpp)
            out["top0"], out["param1"], out["param2"] = host(top), host(pp), host(pc).reshape(params[2].shape)
            out["param0"] = np.full((1, 1, 1, 1), num_iter, np.float32)
        else:
            proto = ('name: "t" input: "x" input_shape { dim: %d dim: %d dim: %d dim: %d } layer { %s }'
                     % (x.shape + (c["text"],)))
            weights = write_caffemodel([("a", "DataAugmentation", params)]) if params else None
            net = fn2.Net(proto, weights, fn2.TEST)
            out["top0"] = net.forward(x=x)["y"]
    elif k == "aug_train":
        cw, ch = c["args"]
        out["top0"] = engine_augment(ops, bottoms[0], bottoms[1], cw, ch, gold["L/%s/space" % name], 1.0)
    return out


@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("name", sorted(RC.LAYER_CASES))
def test_kernels_match_reference_vectors(fn2, ops, gold, name, channels_last):
    if RC.LAYER_CASES[name]["kind"] in ("aug_deploy", "aug_train") and channels_last:
        pytest.skip("layout is the layer's own choice")
    out = engine_eval(fn2, ops, name, gold, channels_last)
    for key, got in out.items():
        want = gold["L/%s/%s" % (name, key)]
        err = RCK.rel_err(got, want)
        assert err <= RCK.tol_for(name, key), (name, key, err)


def test_integer_index_paths_bit_exact(fn2, ops, gold):
    for name in ("rs_nearest_down", "rs_nearest_up2", "rs_same"):
        got = engine_eval(fn2, ops, name, gold, False)["top0"]
        assert np.array_equal(got, gold["L/%s/top0" % name]), name


def test_true_extrema_where_the_reference_races(fn2, ops, gold):
    """fn2_chromatic_eigenspace computes the exact statistics the reference's lossy atomics only approximate
    (oracle/ref_shim/ref_capi.cpp: ref_layer_debug_eigenspace)."""
    bottoms, _, _ = RC.case_inputs("aug_train_eigen")
    space = host(ops.chromatic_eigenspace(dev(bottoms[0]), RC.EIGVEC))[:25]
    true = O.chromatic_eigenspace(bottoms[0], RC.EIGVEC)[:25]
    assert np.abs(space - true).max() <= 1e-6
    RCK.check_eigenspace(gold["L/aug_train_eigen/space"], space)


@pytest.mark.parametrize("cname", sorted(RC.NET_CASES))
def test_small_nets_match_reference_vectors(fn2, gold, cname):
    model, w, h, batch = RC.NET_CASES[cname]
    proto = fn2.fill_template(fn2.model_template(model), w, h)
    _, blob = synth_weights(fn2.fill_template(fn2.model_template(model), 64, 64), 1701, proto)
    img0, img1 = smooth_images(rng(11), batch, h, w)
    net = fn2.Net(proto, blob, fn2.TEST, batch=batch)
    got = net.forward(img0=img0, img1=img1)["predict_flow_final"]
    assert maxabs(got, gold["N/%s/flow" % cname]) <= 1e-4, maxabs(got, gold["N/%s/flow" % cname])


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json shapes, live
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", RC.BASELINE_CORR_SHAPES)
def test_correlation_baseline_shapes(ops, baseline_gold, shape):
    """Correlation d=21, k=1 (FlowNet2-C) at the three feature-map shapes of BASELINE.json's configs 2, 3, 4."""
    a, b = RC.baseline_corr_inputs(shape)
    got = host(ops.correlation(dev(a, True), dev(b, True), 20, 1, 20, 1, 2))
    want = O.correlation_fwd(a, b, 20, 1, 20, 1, 2, 0, exact_order=False)           # float64 accumulation
    assert maxabs(got, want) <= 1e-6, maxabs(got, want)
    ref = baseline_gold[RC.baseline_corr_key(shape)]
    sample = RC.baseline_sample(got, len(ref))
    assert maxabs(sample, ref) <= 1e-6, maxabs(sample, ref)


@pytest.mark.parametrize("model,w,h", RC.BASELINE_NETS)
def test_nets_at_baseline_sizes_strict_1e4(fn2, baseline_gold, model, w, h):
    """BASELINE configs 2, 3, 4 at batch 1: engine vs the float64 oracle AND vs the reference's layers on a B200 (stored sample),
    both with the north_star's absolute 1e-4 on predict_flow_final (|flow| reaches 10-30 px with the synthetic weights)."""
    proto = fn2.fill_template(fn2.model_template(model), w, h)
    _, blob = synth_weights(fn2.fill_template(fn2.model_template(model), 64, 64), 1701, proto)
    img0, img1 = smooth_images(rng(1701), 1, h, w)
    net = fn2.Net(proto, blob, fn2.TEST, batch=1)
    got = net.forward(img0=img0, img1=img1)["predict_flow_final"].copy()
    again = net.forward(img0=img0, img1=img1)["predict_flow_final"].copy()         # graph replay
    assert np.array_equal(got, again)
    del net
    torch.cuda.empty_cache()
    want = OracleNet(proto, blob, batch=1, f64acc=True).forward(img0=img0, img1=img1)["predict_flow_final"]
    assert np.abs(want).max() > 1.0, "degenerate: flow ~ 0"
    assert maxabs(got, want) <= 1e-4, ("engine vs float64 oracle", maxabs(got, want), float(np.abs(want).max()))
    ref = baseline_gold[RC.baseline_net_key(model, w, h)]
    sample = RC.baseline_sample(got, len(ref))
    assert maxabs(sample, ref) <= 1e-4, ("engine vs reference GPU", maxabs(sample, ref))
