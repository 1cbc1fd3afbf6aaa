"""ctypes front end of oracle/_ref/libref_caffe.so -- the REFERENCE's own layer classes, compiled from
/root/reference where they lie by oracle/ref_shim/build_ref.py.

TEST INFRASTRUCTURE ONLY: importable from tests/, tools/, __graft_entry__ and bench.py's --impl reference /
cpu_baseline legs.  Nothing under flownet2_b200/ may import this module.

What runs: caffe::Layer<float>::SetUp / Forward / Backward of the reference (include/caffe/layer.hpp:67-81,
:483-535) for Correlation, Correlation1D, Resample, DataAugmentation, ChannelNorm, FlowWarp, Convolution,
Deconvolution, ReLU, Eltwise, Concat, Slice, L1Loss, Downsample, FlowAugmentation,
GenerateAugmentationParameters -- in GPU mode the reference's kernels and cuBLAS calls (GPU box only), in CPU
mode the reference's Forward_cpu where one exists (conv/deconv via im2col + OpenBLAS sgemm, ReLU, Eltwise, Concat,
FlowWarp, ChannelNorm; Correlation / Resample / DataAugmentation have none: correlation_layer.cpp:87-90,
resample_layer.cpp:58-62, data_augmentation_layer.cpp:208-212).

RefNet executes a whole deploy prototxt layer by layer with the reference's graph rules (in-order, in-place
tops, net.cpp:386-448); the reference's net.cpp itself is not compiled (it needs protobuf IO / HDF5).
"""
import ctypes as C
import glob
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libref_caffe.so")
_LIB = None
_MODE = None


class RefError(RuntimeError):
    pass


def available():
    return os.path.exists(LIB_PATH)


def build(required=True):
    """Compile oracle/_ref from the reference checkout named by FN2_REFERENCE (an already built library is kept when the
    checkout is absent).  required=False: return None instead of raising when neither exists."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("build_ref", os.path.join(_HERE, "ref_shim", "build_ref.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.build(required=required)


def _find_openblas():
    import scipy
    sp = glob.glob(os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs", "libscipy_openblas-*.so"))
    if sp:
        return sp[0], 0
    npd = glob.glob(os.path.join(os.path.dirname(os.path.dirname(np.__file__)), "numpy.libs", "libscipy_openblas64_-*.so"))
    if npd:
        return npd[0], 1
    raise RefError("no OpenBLAS found in the scipy / numpy wheels")


def lib():
    global _LIB
    if _LIB is None:
        if not available():
            raise RefError("oracle/_ref/libref_caffe.so is not built (python oracle/ref_shim/build_ref.py)")
        l = C.CDLL(LIB_PATH)
        l.ref_last_error.restype = C.c_char_p
        for f in ("ref_blob_create", "ref_layer_create", "ref_layer_param", "ref_blob_gpu_data"):
            getattr(l, f).restype = C.c_void_p
        l.ref_layer_type.restype = C.c_char_p
        l.ref_blob_count.restype = C.c_longlong
        for f in ("ref_blob_destroy", "ref_blob_reshape", "ref_blob_num_axes", "ref_blob_shape", "ref_blob_count", "ref_blob_set",
                  "ref_blob_get", "ref_blob_gpu_data", "ref_layer_destroy", "ref_layer_setup", "ref_layer_reshape",
                  "ref_layer_forward", "ref_layer_backward", "ref_layer_num_params", "ref_layer_param", "ref_layer_type",
                  "ref_layer_uses_custom_copy", "ref_layer_custom_copy", "ref_layer_time_forward"):
            fn = getattr(l, f)
            fn.argtypes = None
        path, ilp64 = _find_openblas()
        if l.ref_load_blas(path.encode(), ilp64) != 0:
            raise RefError("cannot load OpenBLAS: " + l.ref_last_error().decode())
        _LIB = l
    return _LIB


def _check(rc):
    if rc != 0:
        raise RefError(lib().ref_last_error().decode("utf-8", "replace"))


def set_mode(gpu, device=0):
    """Caffe::set_mode (common.hpp:139).  gpu=False runs the reference's Forward_cpu paths."""
    global _MODE
    _check(lib().ref_set_mode(1 if gpu else 0, int(device)))
    _MODE = bool(gpu)


def set_seed(seed):
    _check(lib().ref_set_seed(C.c_uint(seed)))


def blas_threads(n):
    _check(lib().ref_blas_set_threads(int(n)))


class Blob(object):
    def __init__(self, handle=None, shape=None):
        self._own = handle is None
        self.h = C.c_void_p(lib().ref_blob_create()) if handle is None else C.c_void_p(handle)
        if shape is not None:
            self.reshape(shape)

    def __del__(self):
        try:
            if self._own and self.h:
                lib().ref_blob_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def reshape(self, shape):
        s = (C.c_int * len(shape))(*[int(x) for x in shape])
        _check(lib().ref_blob_reshape(self.h, len(shape), s))

    @property
    def shape(self):
        s = (C.c_int * 32)()
        n = lib().ref_blob_shape(self.h, s)
        return tuple(s[:n])

    def set(self, a, diff=False):
        a = np.ascontiguousarray(a, np.float32)
        if tuple(a.shape) != self.shape:
            self.reshape(a.shape)
        _check(lib().ref_blob_set(self.h, a.ctypes.data_as(C.c_void_p), 1 if diff else 0))

    def get(self, diff=False):
        out = np.empty(self.shape, np.float32)
        _check(lib().ref_blob_get(self.h, out.ctypes.data_as(C.c_void_p), 1 if diff else 0))
        return out


class Layer(object):
    """One reference layer.  `text` is the inside of a prototxt `layer { ... }` block."""

    def __init__(self, text, phase=1):
        if _MODE is None:
            raise RefError("call oracle.ref.set_mode(gpu) first")
        h = lib().ref_layer_create(text.encode(), int(phase))
        if not h:
            raise RefError(lib().ref_last_error().decode("utf-8", "replace"))
        self.h = C.c_void_p(h)
        self.bottoms, self.tops = [], []

    def __del__(self):
        try:
            if self.h:
                lib().ref_layer_destroy(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def type(self):
        return lib().ref_layer_type(self.h).decode()

    def setup(self, bottoms, tops):
        self.bottoms, self.tops = list(bottoms), list(tops)
        b = (C.c_void_p * max(1, len(bottoms)))(*[x.h for x in bottoms])
        t = (C.c_void_p * max(1, len(tops)))(*[x.h for x in tops])
        _check(lib().ref_layer_setup(self.h, len(bottoms), b, len(tops), t))

    @property
    def params(self):
        return [Blob(handle=lib().ref_layer_param(self.h, i)) for i in range(lib().ref_layer_num_params(self.h))]

    def forward(self):
        loss = C.c_float(0)
        _check(lib().ref_layer_forward(self.h, C.byref(loss)))
        return loss.value

    def backward(self, propagate_down=None):
        pd = None
        if propagate_down is not None:
            pd = (C.c_int * len(propagate_down))(*[1 if p else 0 for p in propagate_down])
        _check(lib().ref_layer_backward(self.h, pd))

    def time_forward(self, iters=5):
        ms = C.c_float(0)
        _check(lib().ref_layer_time_forward(self.h, int(iters), C.byref(ms)))
        return ms.value

    def debug_eigenspace(self):
        """tChromaticEigenSpace of a DataAugmentation layer after forward (25 floats) -- see ref_capi.cpp for why."""
        out = np.zeros(25, np.float32)
        _check(lib().ref_layer_debug_eigenspace(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def custom_copy(self, arrays):
        """Net::CopyTrainedLayersFrom for DoesUseCustomCopyBlobs() layers (net.cpp:769-778): DataAugmentation's adjust_blobs."""
        blobs = [Blob(shape=a.shape) for a in arrays]
        for b, a in zip(blobs, arrays):
            b.set(a)
        v = (C.c_void_p * len(blobs))(*[b.h for b in blobs])
        _check(lib().ref_layer_custom_copy(self.h, len(blobs), v))


def run_layer(text, bottoms, ntop=1, params=None, phase=1, top_diffs=None, propagate_down=None):
    """Convenience: build one layer, feed numpy bottoms, return tops (and bottom diffs when top_diffs is given)."""
    bl = [Blob(shape=np.shape(b)) for b in bottoms]
    for b, a in zip(bl, bottoms):
        b.set(a)
    tl = [Blob() for _ in range(ntop)]
    layer = Layer(text, phase)
    layer.setup(bl, tl)
    if params is not None:
        for p, a in zip(layer.params, params):
            p.set(np.asarray(a, np.float32).reshape(p.shape))
    layer.forward()
    tops = [t.get() for t in tl]
    if top_diffs is None:
        return tops
    for t, d in zip(tl, top_diffs):
        t.set(d, diff=True)
    layer.backward(propagate_down)
    return tops, [b.get(diff=True) for b in bl], [p.get(diff=True) for p in layer.params]


# ------------------------------------------------------------------------------------------------
# whole nets
# ------------------------------------------------------------------------------------------------
def split_layers(prototxt_text):
    """-> (header text without layer blocks, [text inside each top-level `layer { }` block])."""
    text = re.sub(r"#[^\n]*", "", prototxt_text)
    layers, header, i, n = [], [], 0, len(text)
    pat = re.compile(r"\blayer\s*\{")
    while True:
        m = pat.search(text, i)
        if not m:
            header.append(text[i:])
            break
        header.append(text[i:m.start()])
        depth, j = 1, m.end()
        in_str = None
        while depth:
            c = text[j]
            if in_str:
                if c == "\\":
                    j += 1
                elif c == in_str:
                    in_str = None
            elif c in "\"'":
                in_str = c
            elif c == "{":
                depth += 1
            elif c == "}":
                depth -= 1
            j += 1
        layers.append(text[m.end():j - 1])
        i = j
    return "".join(header), layers


def _names(text, key):
    # top-level fields of the layer block only (nested messages never use bottom/top/name/type)
    return re.findall(r"\b%s\s*:\s*[\"']([^\"']*)[\"']" % key, text)


def insert_splits(specs):
    """InsertSplits (util/insert_splits.cpp:12-72) on a list of (name, type, block text): every top that is read by more than one
    later layer gets a Split layer, the readers are renamed to its tops.  Names follow SplitBlobName (:120-128)."""
    prod = {}                                   # blob name -> (layer index, top index) of its latest producer
    readers = {}                                # (layer, top) -> [(reader layer, bottom index)]
    for li, (name, typ, blk) in enumerate(specs):
        for bi, b in enumerate(_names(blk, "bottom")):
            if b in prod:
                readers.setdefault(prod[b], []).append((li, bi))
        for ti, t in enumerate(_names(blk, "top")):
            prod[t] = (li, ti)
    rename = {}                                 # (reader layer, bottom index) -> new bottom name
    after = {}                                  # layer index -> [split layer specs to insert after it]
    for (li, ti), rs in readers.items():
        if len(rs) < 2:
            continue
        blob = _names(specs[li][2], "top")[ti]
        lname = specs[li][0]
        tops = ["%s_%s_%d_split_%d" % (blob, lname, ti, k) for k in range(len(rs))]
        for k, r in enumerate(rs):
            rename[r] = tops[k]
        text = 'name: "%s_%s_%d_split" type: "Split" bottom: "%s" %s' % (blob, lname, ti, blob, " ".join('top: "%s"' % t for t in tops))
        after.setdefault(li, []).append(("%s_%s_%d_split" % (blob, lname, ti), "Split", text))
    out = []
    for li, (name, typ, blk) in enumerate(specs):
        cnt = [0]

        def repl(m):
            i = cnt[0]
            cnt[0] += 1
            return 'bottom: "%s"' % rename.get((li, i), m.group(1))
        out.append((name, typ, re.sub(r'\bbottom\s*:\s*["\']([^"\']*)["\']', repl, blk)))
        out.extend(after.get(li, []))
    return out


NO_BACKWARD_TYPES = ("DataAugmentation", "GenerateAugmentationParameters", "FlowAugmentation", "Downsample", "Resample", "Input", "Silence")


class RefNet(object):
    """Runs a deploy prototxt through the reference's layer classes (see module docstring).

    weights: {layer name: [ndarray, ...]} as oracle.net.parse_caffemodel returns; source blobs are copied into the
    layer's params like Net::CopyTrainedLayersFrom (net.cpp:752-802), DataAugmentation through its CustomCopyBlobs."""

    def __init__(self, prototxt_text, weights=None, batch=0, phase=1, splits=False):
        from .net import parse_prototxt, getall, get
        header, blocks = split_layers(prototxt_text)
        root = parse_prototxt(header)
        self.input_names = getall(root, "input")
        self.input_shapes = [[int(d) for d in getall(s, "dim")] for s in getall(root, "input_shape")]
        self.blobs, self.layers = {}, []
        specs = []
        for blk in blocks:
            name, typ = _names(blk, "name")[0], _names(blk, "type")[0]
            if typ == "Input":
                msg = parse_prototxt(blk)
                self.input_names += getall(msg, "top")
                self.input_shapes += [[int(d) for d in getall(s, "dim")] for s in getall(get(msg, "input_param", []), "shape")]
                continue
            specs.append((name, typ, blk))
        if batch:
            for s in self.input_shapes:
                s[0] = batch
        for n, s in zip(self.input_names, self.input_shapes):
            self.blobs[n] = Blob(shape=s)
        if splits:                              # a net that will run Backward: fan-out through Split layers like Net::Init
            specs = [("__in__", "Input", " ".join('top: "%s"' % n for n in self.input_names))] + specs
            specs = insert_splits(specs)[1:]
            if specs and specs[0][0].startswith("__in__"):
                pass
        self.specs = specs
        for name, typ, blk in specs:
            bots = [self.blobs[b] for b in _names(blk, "bottom")]
            tops = []
            for t in _names(blk, "top"):
                if t not in self.blobs:
                    self.blobs[t] = Blob()
                tops.append(self.blobs[t])           # same Blob object when top == bottom (in place, net.cpp:394-400)
            layer = Layer(blk, phase)
            layer.setup(bots, tops)
            if weights and name in weights:
                src = weights[name]
                if lib().ref_layer_uses_custom_copy(layer.h):
                    layer.custom_copy(src)
                else:
                    for p, a in zip(layer.params, src):
                        p.set(np.asarray(a, np.float32).reshape(p.shape))
            self.layers.append((name, typ, layer))

    def forward(self, **inputs):
        for n in self.input_names:
            self.blobs[n].set(inputs[n])
        for _, _, layer in self.layers:
            layer.forward()
        return self

    def blob(self, name):
        return self.blobs[name].get()

    def backward(self):
        """Net::Backward (net.cpp:640-655): loss tops seeded with their loss_weight (layer.hpp:455-478), layers in reverse order;
        a layer runs if it has parameters or a bottom that needs a gradient (net.cpp:120-170), never the augmentation / data side."""
        from .net import parse_prototxt, getall, get
        need_blob, plan = set(), []
        for name, typ, layer in self.layers:
            blk = next(b for n, t, b in self.specs if n == name)
            bots, tops = _names(blk, "bottom"), _names(blk, "top")
            need = typ not in NO_BACKWARD_TYPES and (len(layer.params) > 0 or any(b in need_blob for b in bots))
            if need:
                need_blob.update(tops)
            pd = [b in need_blob and typ not in NO_BACKWARD_TYPES for b in bots]
            if typ == "L1Loss":
                pd = [b in need_blob for b in bots]
            plan.append((need, pd, blk, tops))
        for (name, typ, layer), (need, pd, blk, tops) in zip(self.layers, plan):
            if typ.endswith("Loss"):
                lw = [float(x) for x in getall(parse_prototxt(blk), "loss_weight")] or [1.0]
                t = self.blobs[tops[0]]
                t.set(np.full(t.shape if t.shape else (1,), lw[0], np.float32).reshape(t.shape), diff=True)
        for (name, typ, layer), (need, pd, blk, tops) in reversed(list(zip(self.layers, plan))):
            if need:
                layer.backward(pd)
        return self

    def time_layers(self, iters=1):
        return [(n, t, l.time_forward(iters)) for n, t, l in self.layers]


class _OracleLayer(object):
    """Stand-in for the three layer types whose Forward_cpu does not exist in the reference (NOT_IMPLEMENTED / LOG(FATAL)):
    the oracle restatement of their .cu arithmetic, exchanging data with the reference Blobs on the host."""

    def __init__(self, onet, msg, bottoms, tops):
        self.onet, self.msg, self.bottoms, self.tops = onet, msg, bottoms, tops
        outs = onet.run_layer(msg, [np.zeros(b.shape, np.float32) for b in bottoms])       # shape inference (SetUp)
        for t, o in zip(tops, outs):
            t.reshape(o.shape)

    def forward(self):
        outs = self.onet.run_layer(self.msg, [b.get() for b in self.bottoms])
        for t, o in zip(self.tops, outs):
            t.set(o)

    def time_forward(self, iters=1):
        import time
        t0 = time.perf_counter()
        for _ in range(iters):
            self.forward()
        return (time.perf_counter() - t0) * 1e3 / iters


class RefCpuNet(object):
    """The reference's CPU forward of a deploy prototxt, as far as the reference has one: conv / deconv (im2col + OpenBLAS sgemm,
    base_conv_layer.cpp:257-298), ReLU, Eltwise, Concat, FlowWarp, ChannelNorm run the reference's own Forward_cpu; Correlation,
    Resample and DataAugmentation -- for which the reference only has GPU code -- run the oracle port.  This is what bench.py
    times as `--impl reference` / `cpu_baseline` (kind "reference")."""
    ORACLE_TYPES = ("Correlation", "Resample", "DataAugmentation")

    def __init__(self, prototxt_text, weights=None, batch=0, synth_seed=None):
        from .net import OracleNet, parse_prototxt, getall, get
        set_mode(False)
        self.onet = OracleNet(prototxt_text, None, batch=batch, synth_seed=synth_seed)
        if weights:
            self.onet.weights = {k: [np.asarray(a, np.float32) for a in v] for k, v in weights.items()}
        header, blocks = split_layers(prototxt_text)
        self.input_names, self.input_shapes = list(self.onet.input_names), [list(s) for s in self.onet.input_shapes]
        self.blobs, self.layers = {}, []
        for n, s in zip(self.input_names, self.input_shapes):
            self.blobs[n] = Blob(shape=s)
        r = np.random.default_rng(synth_seed if synth_seed is not None else 0)
        for blk in blocks:
            name, typ = _names(blk, "name")[0], _names(blk, "type")[0]
            if typ == "Input":
                continue
            bots = [self.blobs[b] for b in _names(blk, "bottom")]
            tops = []
            for t in _names(blk, "top"):
                if t not in self.blobs:
                    self.blobs[t] = Blob()
                tops.append(self.blobs[t])
            if typ in self.ORACLE_TYPES:
                layer = _OracleLayer(self.onet, parse_prototxt(blk), bots, tops)
            else:
                layer = Layer(blk, 1)
                layer.setup(bots, tops)
                if weights and name in weights:
                    for p, a in zip(layer.params, weights[name]):
                        p.set(np.asarray(a, np.float32).reshape(p.shape))
                elif synth_seed is not None and typ in ("Convolution", "Deconvolution"):
                    ps = layer.params                      # He-initialised weights, zero bias (timing-only runs)
                    shp = ps[0].shape
                    fan = int(np.prod(shp[1:])) if typ == "Convolution" else shp[0] * shp[2] * shp[3]
                    ps[0].set((r.standard_normal(shp) * np.sqrt(2.0 / fan)).astype(np.float32))
                    if len(ps) > 1:
                        ps[1].set(np.zeros(ps[1].shape, np.float32))
            self.layers.append((name, typ, layer))

    def forward(self, **inputs):
        for n in self.input_names:
            self.blobs[n].set(inputs[n])
        for _, _, layer in self.layers:
            layer.forward()
        return self

    def blob(self, name):
        return self.blobs[name].get()
