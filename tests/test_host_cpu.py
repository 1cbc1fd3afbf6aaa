"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/fn2.h declares,
and the engine's prototxt / caffemodel parsers agree with the REFERENCE's own protobuf schema (fixtures
produced with python/caffe/proto/caffe_pb2.py by tests/golden/make_golden.py).  No compute calls."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from oracle import net as onet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "fn2.h")).read()
    return sorted(set(re.findall(r"FN2_API\s+[\w\s\*]+?\b(fn2_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol(fn2):
    lib = fn2.lib()
    syms = declared_symbols()
    assert len(syms) >= 50
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert b"sm_100a" in lib.fn2_version()


def test_library_is_sm100a_only():
    import subprocess
    from flownet2_b200 import build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")       # the toolkit that built the library
    out = subprocess.run([cuobjdump, "--list-elf", os.path.join(ROOT, "flownet2_b200", "libfn2.so")],
                         capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def canonical(fn2, text):
    lib = fn2.lib()
    n = C.c_size_t()
    rc = lib.fn2_proto_canonical(text.encode(), None, C.byref(n))
    if rc:
        raise fn2.Fn2Error(lib.fn2_last_error().decode())
    buf = C.create_string_buffer(n.value)
    assert lib.fn2_proto_canonical(text.encode(), buf, C.byref(n)) == 0
    return buf.value.decode()


@pytest.mark.parametrize("model", ["FlowNet2-S", "FlowNet2-C", "FlowNet2-CSS", "FlowNet2-SD", "FlowNet2"])
def test_prototxt_parser_matches_reference_protobuf(fn2, model):
    ref = json.load(open(os.path.join(GOLD, "ref_pb2_prototxt.json")))[model]
    text = fn2.fill_template(fn2.model_template(model), 1024, 436)
    # engine parser -> canonical text -> (independent) oracle parser -> structure
    msg = onet.parse_prototxt(canonical(fn2, text))
    layers = onet.getall(msg, "layer")
    # legacy `input:` fields become one Input layer named "input" placed first (upgrade_proto.cpp:953-992)
    assert onet.get(layers[0], "type") == "Input" and onet.get(layers[0], "name") == "input"
    assert onet.getall(layers[0], "top") == ref["inputs"]
    shapes = [[int(d) for d in onet.getall(s, "dim")] for s in onet.getall(onet.get(layers[0], "input_param"), "shape")]
    assert shapes == ref["input_shape"]
    layers = layers[1:]
    assert len(layers) == len(ref["layers"])
    for got, want in zip(layers, ref["layers"]):
        assert onet.get(got, "name") == want["name"] and onet.get(got, "type") == want["type"]
        assert onet.getall(got, "bottom") == want["bottom"] and onet.getall(got, "top") == want["top"]
        if "conv" in want:
            cp = onet.get(got, "convolution_param")
            assert [int(onet.get(cp, "num_output")), [int(v) for v in onet.getall(cp, "kernel_size")],
                    [int(v) for v in onet.getall(cp, "stride")], [int(v) for v in onet.getall(cp, "pad")],
                    onet.get(cp, "bias_term", "true") == "true"] == want["conv"]
        if "corr" in want:
            cp = onet.get(got, "correlation_param")
            assert [int(onet.get(cp, k)) for k in ("pad", "kernel_size", "max_displacement", "stride_1", "stride_2")] + [0] == want["corr"]
        if "resample" in want and want["resample"][0]:
            rp = onet.get(got, "resample_param")
            assert [int(onet.get(rp, "width")), int(onet.get(rp, "height"))] == want["resample"][:2]
        if "coeff" in want:
            got_c = [float(c) for c in onet.getall(onet.get(got, "eltwise_param"), "coeff")]
            assert np.allclose(got_c, want["coeff"], rtol=1e-6)


def test_prototxt_text_format_quirks(fn2):
    text = '''
    name: 'quirks'  # comment
    layer { name: "a" type: "Input" top: "x" input_param { shape: { dim: [1, 3, 8, 8] } } }
    layer <
      name: "c" type: "Convolution" bottom: "x" top: "y";
      convolution_param { num_output: 4, kernel_h: 3 kernel_w: 1 pad_h: 1 stride: 2
                          weight_filler { type: "gaussian" std: 1e-2 } }
      param { lr_mult: .5 }
    >
    layer { name: "s\\"q" type: "ReLU" bottom: "y" top: "y" relu_param { negative_slope: 1e-1 } }
    '''
    out = canonical(fn2, text)
    msg = onet.parse_prototxt(out)
    ls = onet.getall(msg, "layer")
    assert [onet.get(l, "name") for l in ls] == ["a", "c", 's"q']
    assert onet.getall(onet.get(onet.get(ls[0], "input_param"), "shape"), "dim") == ["1", "3", "8", "8"]
    assert onet.get(onet.get(ls[1], "convolution_param"), "kernel_h") == "3"
    with pytest.raises(fn2.Fn2Error, match="prototxt:"):
        canonical(fn2, 'layer { name: "a" type: "Input" ')
    with pytest.raises(fn2.Fn2Error):
        canonical(fn2, 'layer { name "a" }')


def test_caffemodel_reader_matches_reference_protobuf(fn2):
    raw = open(os.path.join(GOLD, "ref_pb2_caffemodel.bin"), "rb").read()
    want = json.load(open(os.path.join(GOLD, "ref_pb2_caffemodel.json")))
    lib = fn2.lib()
    n = C.c_size_t()
    assert lib.fn2_caffemodel_summary(raw, len(raw), None, C.byref(n)) == 0
    buf = C.create_string_buffer(n.value)
    assert lib.fn2_caffemodel_summary(raw, len(raw), buf, C.byref(n)) == 0
    lines = buf.value.decode().strip().split("\n")
    assert len(lines) == len(want)
    for line, w in zip(lines, want):
        parts = line.split(" ")
        assert parts[0] == w["name"] and parts[1] == w["type"]
        blobs = re.findall(r"\[([\d,]*)\] n=(\d+) sum=(\S+)", line)
        assert len(blobs) == len(w["blobs"])
        for (shape, cnt, s), wb in zip(blobs, w["blobs"]):
            assert [int(v) for v in shape.split(",")] == wb["shape"]
            assert int(cnt) == int(np.prod(wb["shape"])) and abs(float(s) - wb["sum"]) < 1e-5
    # the oracle's independent reader sees the same thing (double_data blobs are engine-only)
    layers = onet.parse_caffemodel(raw)
    assert list(layers["conv1"][0].shape) == [4, 3, 3, 3] and list(layers["legacy_conv"][1].shape) == [1, 1, 1, 2]
    assert abs(float(layers["conv1"][0].astype(np.float64).sum()) - want[0]["blobs"][0]["sum"]) < 1e-5


def test_truncated_caffemodel_is_an_error_not_a_crash(fn2):
    raw = open(os.path.join(GOLD, "ref_pb2_caffemodel.bin"), "rb").read()
    lib = fn2.lib()
    n = C.c_size_t()
    assert lib.fn2_caffemodel_summary(raw[:100], 100, None, C.byref(n)) == -3      # FN2_ERR_PARSE
    assert b"truncated" in lib.fn2_last_error()


def test_template_vars_follow_run_flownet():
    import flownet2_b200 as F
    v = F.template_vars(1024, 436)        # scripts/run-flownet.py:39-48
    assert (v["ADAPTED_WIDTH"], v["ADAPTED_HEIGHT"]) == (1024, 448)
    assert v["SCALE_WIDTH"] == 1.0 and abs(v["SCALE_HEIGHT"] - 436 / 448.0) < 1e-12
    assert F.template_vars(448, 320)["ADAPTED_HEIGHT"] == 320


def test_flo_io_against_reference_file(fn2, tmp_path):
    d = np.load(os.path.join(GOLD, "chairs_crop.npz"))
    # first bytes of data/FlyingChairs_examples/0000000-gt.flo: tag, w, h, then (u,v) pairs
    head = d["flo_bytes_head"].tobytes()
    assert head[:4] == b"PIEH" and np.frombuffer(head[4:12], np.int32).tolist() == d["flo_header"].tolist() == [512, 384]
    flow = np.ascontiguousarray(d["flow"].transpose(2, 0, 1))
    p = str(tmp_path / "crop.flo")
    fn2.write_flo(p, flow)
    raw = open(p, "rb").read()
    assert raw[:4] == b"PIEH" and np.frombuffer(raw[4:12], np.int32).tolist() == [64, 64]
    assert np.array_equal(np.frombuffer(raw[12:], np.float32).reshape(64, 64, 2), d["flow"])
    assert np.array_equal(fn2.read_flo(p), flow)
    open(p, "wb").write(b"JUNK" + raw[4:])
    with pytest.raises(fn2.Fn2Error, match="not a .flo"):
        fn2.read_flo(p)


def test_no_compute_without_gpu_is_loud(fn2):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(fn2.Fn2Error):
        fn2.Net(fn2.fill_template(fn2.model_template("FlowNet2-S"), 64, 64))


def test_tcgen05_engine_plan_for_flownet2_shapes(fn2):
    """Host-side planning of the tensor-core convolution engine (no GPU needed): tile width, small-Ci packing mode, split-K for
    the small-spatial layers and the tail split of the last partial wave, at the BASELINE shapes (4 pairs, 1024x448)."""
    from flownet2_b200 import fn2_conv_desc
    lib = fn2.lib()

    def plan(ci, co, k, s, p, H, W, deconv=0, cis=None, guard=1024, N=4):
        d = fn2_conv_desc(ci, co, k, k, s, s, p, p, deconv, 1, 1, 0.1, 0, guard)
        out = (C.c_int32 * 8)()
        assert lib.fn2_conv_plan(C.byref(d), N, H, W, cis if cis is not None else ci, out) == 0
        ws = C.c_size_t()
        assert lib.fn2_conv_workspace_bytes(C.byref(d), N, H, W, C.byref(ws)) == 0
        return list(out), ws.value

    # conv1 of FlowNetC on the dense 3-channel image (pixel stride 4, guard band): kernel-row packing, 7 steps of one box
    pl, _ = plan(3, 64, 7, 2, 3, 448, 1024, cis=4)
    assert pl[0] == 64 and pl[3] == 2 and pl[2] == 7 and pl[1] == 4 * 224 * 512 // 128
    # the same layer on a tensor without the guard promise: tap groups (8 taps of 4 channels per K block)
    pl, _ = plan(3, 64, 7, 2, 3, 448, 1024, cis=4, guard=0)
    assert pl[3] == 1 and pl[2] == 7
    # ... and as a channel-range view of a wider blob: tap groups as well
    pl, _ = plan(3, 64, 7, 2, 3, 448, 1024, cis=12)
    assert pl[3] == 1
    # conv3_1: 448 tiles on 148 SMs -> the 4 tiles of the last wave are K-split, partials fit the workspace
    pl, ws = plan(473, 256, 3, 1, 1, 56, 128)
    assert pl[0] == 128 and pl[1] == 448 and pl[2] == 9 * 15 and pl[4] == 1
    assert pl[5] == 444 and 2 <= pl[6] <= 8 and ws >= (448 - 444) * pl[6] * 128 * 128 * 4
    # conv6_1: 28 tiles with K = 9*1024 -> uniform split-K over the SMs
    pl, ws = plan(1024, 1024, 3, 1, 1, 7, 16)
    assert pl[1] == 32 and 2 <= pl[4] <= 8 and ws >= pl[4] * 4 * 7 * 16 * 1024 * 4
    # fusion interconv0: 16 output channels at full resolution -> taps-on-N engine (mode 3): one pass of 9 x 16 = 144 accumulator
    # columns, K = 3 blocks of 32 channels, 35 strips of 30 complete columns
    pl, ws = plan(82, 16, 3, 1, 1, 448, 1024, cis=96)
    assert pl[3] == 3 and pl[0] == -144 and pl[2] == 3 and pl[4] == 1 and pl[5] == 35 and ws == 0
    # fusion deconv0 (4x4 stride 2, 16 outputs): two passes of 8 taps = 128 columns, 6 K blocks
    pl, _ = plan(162, 16, 4, 2, 1, 224, 512, deconv=1, cis=192)
    assert pl[3] == 3 and pl[0] == -128 and pl[2] == 6 and pl[4] == 2
    # with the taps-on-N engine switched off the per-tap engine plans 27 steps of NT = 16 (checked in a subprocess: the switch is
    # read once per process)
    import subprocess, sys
    code = ("import ctypes as C, flownet2_b200 as F; from flownet2_b200 import fn2_conv_desc; "
            "d = fn2_conv_desc(82, 16, 3, 3, 1, 1, 1, 1, 0, 1, 1, 0.1, 0, 1024); o = (C.c_int32 * 8)(); "
            "F.lib().fn2_conv_plan(C.byref(d), 4, 448, 1024, 96, o); print(list(o))")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, FN2_TN="0"), cwd=ROOT)
    pl = eval(out.stdout.strip().splitlines()[-1])
    assert pl[0] == 16 and pl[3] == 0 and pl[4] == 1 and pl[2] == 27
    # flow predictor (2 output channels) is not a tensor-core layer
    pl, _ = plan(194, 2, 3, 1, 1, 112, 256)
    assert pl[0] == 0
    # deconv5: 4 parity classes of 2x2 taps
    pl, _ = plan(1024, 512, 4, 2, 1, 7, 16, deconv=1)
    assert pl[0] == 128 and pl[2] == 4 * 32


AUG_LAYER = """
layer {
  name: "aug" type: "DataAugmentation" bottom: "img" top: "aug"
  coeff_schedule_param { half_life: 50000 initial_coeff: 0.5 final_coeff: 1 }
  augmentation_param {
    augment_during_test: true crop_width: 48 crop_height: 32
    mirror { rand_type: "bernoulli" prob: 0.5 }
    translate { rand_type: "uniform_bernoulli" mean: 0 spread: 0.4 prob: 1.0 }
    rotate { rand_type: "uniform_bernoulli" mean: 0 spread: 0.4 prob: 1.0 }
    zoom { rand_type: "uniform_bernoulli" exp: true mean: 0.2 spread: 0.4 prob: 1.0 }
    squeeze { rand_type: "uniform_bernoulli" exp: true mean: 0 spread: 0.3 prob: 1.0 }
    gamma { rand_type: "gaussian_bernoulli" exp: true mean: 0 spread: 0.02 prob: 1.0 apply_schedule: false }
    brightness { rand_type: "gaussian_bernoulli" mean: 0 spread: 0.02 prob: 0.5 apply_schedule: false }
    color { rand_type: "gaussian_bernoulli" exp: true mean: 0 spread: 0.02 prob: 0.0 }
    noise { rand_type: "uniform_bernoulli" mean: 0.03 spread: 0.03 prob: 1.0 apply_schedule: false }
  }
}
"""


def test_augmentation_coefficient_sampling(fn2):
    """Host logic of DataAugmentation's training use without a GPU: distributions of caffe_rng_generate (util/rng.cpp:8-114),
    the discount schedule, and generate_valid_spatial_coeffs' guarantee that the 4 crop corners land inside the source image
    (augmentation_layer_base.cpp:102-169).  The random stream itself is unpinned (boost in the reference)."""
    lib = fn2.lib()
    N, W, H, cw, ch = 4000, 64, 48, 48, 32
    out = np.zeros((N, 42), np.float32)
    assert lib.fn2_aug_sample(AUG_LAYER.encode(), 7, N, W, H, C.c_float(1e9), out.ctypes.data_as(C.POINTER(C.c_float))) == 0
    default = np.array([0, 0, 0, 0, 1, 1, 1, 0, 1, 1, 1, 1] + [1, 1, 1, 0, 0, 0, 1, 1, 1, 1, 1, 1, 0, 0, 0, 1, 1, 1, 1, 0, 1, 0] + [0] * 8, np.float32)
    v = np.where(np.abs(default) < 1e-3, out, np.exp(out))                      # array_to_coeff
    mirror, dx, dy, ang, zx, zy = v[:, 0], v[:, 1], v[:, 2], v[:, 3], v[:, 4], v[:, 5]
    assert set(np.unique(mirror)) <= {0.0, 1.0} and 0.4 < mirror.mean() < 0.6
    assert np.abs(dx).max() <= 0.4 + 1e-6 and np.abs(ang).max() <= 0.4 + 1e-6
    # every accepted sample keeps the 4 crop corners inside the source image (or is the all-default fallback after 50 tries)
    for n in range(0, N, 7):
        fallback = np.allclose(v[n, :6], default[:6])
        for x in (0, cw - 1):
            for y in (0, ch - 1):
                x1 = (-x + .5 * cw) if mirror[n] else (x - .5 * cw)
                y1 = y - .5 * ch
                x2 = np.cos(ang[n]) * x1 - np.sin(ang[n]) * y1 + dx[n] * cw
                y2 = np.sin(ang[n]) * x1 + np.cos(ang[n]) * y1 + dy[n] * ch
                x2 = x2 / zx[n] + .5 * W
                y2 = y2 / zy[n] + .5 * H
                ok = 0 <= np.floor(x2) <= W - 2 and 0 <= np.floor(y2) <= H - 2
                assert ok or fallback, (n, x, y, x2, y2)
    gamma, bright, color, noise = v[:, 6], v[:, 7], v[:, 9:12], v[:, 41]
    assert abs(np.log(gamma).mean()) < 2e-3 and abs(np.log(gamma).std() - 0.02) < 2e-3          # exp(N(0, 0.02))
    on = bright != 0
    assert 0.45 < on.mean() < 0.55 and abs(bright[on].std() - 0.02) < 3e-3                      # Bernoulli(0.5) gate
    assert np.all(color == 1.0)                                                                # prob 0 -> tmp = 0 -> exp -> 1
    assert noise.min() >= 0.0 and noise.max() <= 0.06 + 1e-6 and abs(noise.mean() - 0.03) < 2e-3
    # discount schedule: at iteration 0 the scheduled spreads are halved (initial_coeff 0.5), unscheduled ones are not
    early = np.zeros((N, 42), np.float32)
    assert lib.fn2_aug_sample(AUG_LAYER.encode(), 7, N, W, H, C.c_float(0.0), early.ctypes.data_as(C.POINTER(C.c_float))) == 0
    assert np.abs(early[:, 3]).max() <= 0.2 + 1e-6 and np.abs(early[:, 3]).max() > 0.15
    assert abs(early[:, 6].std() - 0.02) < 2e-3
    # same seed, same stream
    again = np.zeros((N, 42), np.float32)
    assert lib.fn2_aug_sample(AUG_LAYER.encode(), 7, N, W, H, C.c_float(1e9), again.ctypes.data_as(C.POINTER(C.c_float))) == 0
    assert np.array_equal(again, out)


def _norm_tree(msg):
    """Order-insensitive form of a parsed prototxt (protobuf's DebugString orders by field number; here: by name, scalars as
    numbers where they parse as such, enum / string tokens as text)."""
    out = []
    for k, v in msg:
        if isinstance(v, list):
            out.append((k, _norm_tree(v)))
        else:
            try:
                out.append((k, float(v)))
            except ValueError:
                out.append((k, v))
    return sorted(out, key=lambda kv: (kv[0], repr(kv[1])))


def test_v1_prototxt_upgrade_matches_the_reference_tests(fn2):
    """NetParameter::FromText upgrades V1 `layers { type: CONVOLUTION blobs_lr: ... }` nets like UpgradeV1Net
    (util/upgrade_proto.cpp:640-949).  Golden pairs: the reference's own NetUpgradeTest.TestSimple / TestImageNet
    (tests/golden/make_upgrade_golden.py)."""
    import json
    from oracle.net import parse_prototxt
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "upgrade_v1_fixtures.json")) as f:
        cases = json.load(f)["cases"]
    assert len(cases) == 2
    for c in cases:
        got = parse_prototxt(canonical(fn2, c["v1"]))
        want = parse_prototxt(canonical(fn2, c["v2"]))
        assert [k for k, _ in got if k == "layers"] == [] and len([1 for k, _ in got if k == "layer"]) >= 4
        assert _norm_tree(got) == _norm_tree(want)
    with pytest.raises(fn2.Fn2Error):
        canonical(fn2, "layers { name: 'x' type: NO_SUCH_TYPE }")


def test_train_prototxt_parser_matches_reference_protobuf(fn2):
    """The authored FlowNet2-C training prototxt, as the reference's own caffe_pb2 reads it (tests/golden/make_train_proto_golden.py:
    every field exists in the reference's caffe.proto) against the engine's parser: layers, bottoms / tops, loss weights,
    propagate_down, L1Loss parameters, augmentation generators, coefficient schedule."""
    ref = json.load(open(os.path.join(GOLD, "ref_pb2_train_prototxt.json")))
    text = fn2.fill_train_template(fn2.train_template("FlowNet2-C"), 448, 320, 512, 384, 8)
    msg = onet.parse_prototxt(canonical(fn2, text))
    layers = onet.getall(msg, "layer")
    assert len(layers) == len(ref["layers"]) == 67
    for got, want in zip(layers, ref["layers"]):
        assert onet.get(got, "name") == want["name"] and onet.get(got, "type") == want["type"]
        assert onet.getall(got, "bottom") == want["bottom"] and onet.getall(got, "top") == want["top"]
        assert np.allclose([float(x) for x in onet.getall(got, "loss_weight")], want["loss_weight"], rtol=1e-6)
        assert [x == "true" for x in onet.getall(got, "propagate_down")] == want["propagate_down"]
        if "l1" in want:
            lp = onet.get(got, "l1_loss_param", [])
            assert [onet.get(lp, "l2_per_location", "false") == "true", onet.get(lp, "l2_prescale_by_channels", "false") == "true",
                    onet.get(lp, "normalize_by_num_entries", "false") == "true"] == want["l1"][:3]
        if "aug" in want:
            ap = onet.get(got, "augmentation_param")
            assert [int(onet.get(ap, "crop_width", 0)), int(onet.get(ap, "crop_height", 0))] == want["aug"]["crop"]
            assert onet.get(ap, "mode", "add") == want["aug"]["mode"]
            gens = {k: v for k, v in ap if isinstance(v, list)}
            assert sorted(gens) == sorted(want["aug"]["generators"])
            for k, g in gens.items():
                w = want["aug"]["generators"][k]
                assert onet.get(g, "rand_type") == w[0] and (onet.get(g, "exp", "false") == "true") == w[1]
                assert np.allclose([float(onet.get(g, "mean", 0)), float(onet.get(g, "spread", 0)), float(onet.get(g, "prob", 1))], w[2:], rtol=1e-6)
        if "schedule" in want:
            cs = onet.get(got, "coeff_schedule_param")
            assert np.allclose([float(onet.get(cs, k)) for k in ("half_life", "initial_coeff", "final_coeff")], want["schedule"])
        if "shapes" in want:
            assert [[int(d) for d in onet.getall(s, "dim")] for s in onet.getall(onet.get(got, "input_param"), "shape")] == want["shapes"]


def _h5_summary(fn2, data):
    lib = fn2.lib()
    lib.fn2_hdf5_summary.argtypes = [C.c_void_p, C.c_size_t, C.c_char_p, C.POINTER(C.c_size_t)]
    buf = (C.c_char * len(data)).from_buffer_copy(data)
    n = C.c_size_t()
    if lib.fn2_hdf5_summary(buf, len(data), None, C.byref(n)):
        raise fn2.Fn2Error(lib.fn2_last_error().decode())
    out = C.create_string_buffer(n.value)
    assert lib.fn2_hdf5_summary(buf, len(data), out, C.byref(n)) == 0
    return out.value.decode().strip().splitlines()


def test_hdf5_reader_on_files_written_by_the_real_library(fn2):
    """The minimal HDF5 reader (csrc/caffe/hdf5_min.cpp) on the reference's own test data, written with h5py / libhdf5
    (tests/golden/ref_hdf5/): shapes, every value (data = arange), and a loud refusal of the gzip-compressed variant."""
    d = os.path.join(GOLD, "ref_hdf5")
    lines = _h5_summary(fn2, open(os.path.join(d, "sample_data.h5"), "rb").read())
    assert lines == ["/data f32 [10,8,6,5] n=2400 sum=2878800 first=0 last=2399", "/label f32 [10,1] n=10 sum=55 first=1 last=10",
                     "/label2 f32 [10,1] n=10 sum=65 first=2 last=11"]
    lines = _h5_summary(fn2, open(os.path.join(d, "solver_data.h5"), "rb").read())
    assert [l.split(" n=")[0] for l in lines] == ["/data f32 [8,3,10,10]", "/targets f32 [8,1]"]
    with pytest.raises(fn2.Fn2Error, match="gzip"):
        _h5_summary(fn2, open(os.path.join(d, "sample_data_2_gzip.h5"), "rb").read())
    with pytest.raises(fn2.Fn2Error, match="signature"):
        _h5_summary(fn2, b"\x00" * 200)
    trunc = open(os.path.join(d, "sample_data.h5"), "rb").read()[:5000]
    with pytest.raises(fn2.Fn2Error, match="outside the file"):
        _h5_summary(fn2, trunc)


def test_hdf5_reader_nested_caffemodel_layout(fn2):
    """/data/<layer>/<blob index> (Net::ToHDF5's layout, net.cpp:905-960) through a test-side writer of the same on-disk structures."""
    from tests.util_h5 import write_caffemodel_h5
    r = np.random.default_rng(3)
    layers = {"conv1": [r.standard_normal((4, 3, 3, 3)).astype(np.float32), r.standard_normal(4).astype(np.float32)],
              "deconv2": [r.standard_normal((2, 5, 4, 4)).astype(np.float32)],
              "img0s_aug": [np.full((1, 1, 1, 1), 1001, np.float32), np.full((1, 3, 1, 1), 0.4, np.float32), np.full((1, 3, 1, 1), 0.4, np.float32)]}
    for k in range(20):                                   # more than one symbol node per group
        layers["extra%02d" % k] = [np.full((2, 2), float(k), np.float32)]
    lines = _h5_summary(fn2, write_caffemodel_h5(layers))
    want = []
    for name in sorted(layers):
        for i, b in enumerate(layers[name]):
            want.append("/data/%s/%d f32 [%s] n=%d sum=%.9g first=%.9g last=%.9g" % (name, i, ",".join(str(d) for d in b.shape), b.size,
                                                                               float(b.astype(np.float64).sum()), float(b.ravel()[0]), float(b.ravel()[-1])))
    assert lines == want


def test_caffemodel_to_hdf5_round_trip(fn2):
    """fn2_caffemodel_to_hdf5 (the host half of Net::ToHDF5): a binary caffemodel -- here the fixture the reference's caffe_pb2 wrote --
    converted to HDF5 and read back by the reader that is pinned on real libhdf5 files: same layers, shapes and values."""
    lib = fn2.lib()
    lib.fn2_caffemodel_to_hdf5.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_size_t)]
    data = open(os.path.join(GOLD, "ref_pb2_caffemodel.bin"), "rb").read()
    desc = json.load(open(os.path.join(GOLD, "ref_pb2_caffemodel.json")))
    buf = (C.c_char * len(data)).from_buffer_copy(data)
    n = C.c_size_t()
    assert lib.fn2_caffemodel_to_hdf5(buf, len(data), None, C.byref(n)) == 0
    out = (C.c_char * n.value)()
    assert lib.fn2_caffemodel_to_hdf5(buf, len(data), out, C.byref(n)) == 0
    lines = _h5_summary(fn2, bytes(out[:n.value]))
    want = {}
    for l in desc:
        for i, b in enumerate(l["blobs"]):
            want["/data/%s/%d" % (l["name"], i)] = b
    assert len(lines) == len(want) == 8
    for line in lines:
        path, rest = line.split(" ", 1)
        b = want[path]
        assert rest.startswith("f32 [%s] " % ",".join(str(d) for d in b["shape"]))
        got_sum = float(rest.split("sum=")[1].split()[0]); got_first = float(rest.split("first=")[1].split()[0])
        assert abs(got_sum - b["sum"]) <= 1e-5 * max(1.0, abs(b["sum"])) and abs(got_first - b["first"]) <= 1e-6 * max(1.0, abs(b["first"]))
