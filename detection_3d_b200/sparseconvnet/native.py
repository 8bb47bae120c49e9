"""Python face of the native boundary: the functions `sparseconvnet.SCN` exports in the reference
(SCN/pybind.cpp:200-235), same names, argument order and empty-output-tensor convention, backed
by the C-ABI in libscn_b200.so.  Dimension 3 / float32 only, CUDA tensors only.
"""
import ctypes as C

import torch

from .._lib import check, l3, lib
from . import program as _program


def _tr():
    """the recording in progress, if any (sparseconvnet/program.py)"""
    t = _program.active()
    return t if t is not None and t.failed is None else None


def _ints(t):
    return [int(v) for v in (t.tolist() if hasattr(t, "tolist") else t)]


def copy_device_to_tensor(t, src_ptr):
    check(lib().scn_copy_device(C.c_void_p(t.data_ptr()), C.c_void_p(src_ptr), t.numel() * t.element_size(), _stream()))


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev_f32(t, what):
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise RuntimeError(f"{what}: expected a CUDA tensor (this extension has no CPU path)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{what}: expected float32, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{what}: tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def _opt(t, what):
    return None if t is None or t.numel() == 0 else _dev_f32(t, what)


# ---- 16-bit shadows (math modes 'bf16' and 'fp16' only).  A BatchNorm / add output carries a 16-bit
# copy of itself (bfloat16 in 'bf16' mode, float16 in 'fp16' mode) as a Python attribute of the tensor
# object, written by the same kernel that wrote the fp32 values; the next convolution gathers from that
# copy (half the bytes).  The attribute dies with the tensor object and is ignored once the tensor has
# been modified in place (_version) or when the current mode uses the other 16-bit format (the
# convolution then converts the fp32 rows itself), so switching between 'bf16' and 'fp16' is safe.
_MATH = {"mode": 0}
_WEIGHT_IMAGES_DROPPED = [0]  # (statistics only)
_SHADOW_DTYPE = {2: torch.bfloat16, 5: torch.float16}  # math mode -> format of the 16-bit copies


def _new_shadow(t):
    """16-bit buffer for the fp32 feature matrix `t` (or None when the mode / shape does not use one)."""
    dt = _SHADOW_DTYPE.get(_MATH["mode"])
    if dt is None or t.dim() != 2 or t.size(1) % 32 != 0 or t.size(0) == 0:
        return None
    return torch.empty(t.shape, dtype=dt, device=t.device)


def _attach_shadow(t, sh):
    if sh is not None:
        t._scn_bf16 = (sh, t._version)


_TOKENS = iter(range(1, 1 << 40))


def _weight_tag(w):
    """Identifies the contents of a weight tensor for the native operand-image cache: a token that
    is unique per tensor OBJECT (ids and addresses get reused) combined with the in-place version."""
    tok = getattr(w, "_scn_token", None)
    if tok is None or tok[1] != _EPOCH:
        tok = (next(_TOKENS), _EPOCH)
        try:
            w._scn_token = tok
        except Exception:
            return 0
    return (tok[0] << 24) + (w._version & 0xFFFFFF) + 1


def invalidate_weight_cache(module_or_tensor=None):
    """The packed weight images and bf16 copies are keyed by (per-tensor token, Tensor._version).  Writes through `.data`
    (older optimizers, EMA / checkpoint code: `p.data.copy_(...)`) do NOT bump `_version`; call this after such a write --
    with a module, a tensor, or nothing (= every tensor gets a new token on its next use) -- so the next convolution
    rebuilds its operand image.  `load_state_dict` of FPN_Net calls it."""
    global _EPOCH
    if module_or_tensor is None:
        _EPOCH += 1
        return
    ts = [module_or_tensor] if isinstance(module_or_tensor, torch.Tensor) else list(module_or_tensor.parameters()) + list(module_or_tensor.buffers())
    for t in ts:
        for attr in ("_scn_token", "_scn_bf16"):
            if hasattr(t, attr):
                try:
                    delattr(t, attr)
                except Exception:
                    pass


_EPOCH = 0


def _shadow_ptr(t):
    sh = getattr(t, "_scn_bf16", None)
    if sh is None or sh[0].dtype != _SHADOW_DTYPE.get(_MATH["mode"]) or sh[1] != t._version or sh[0].shape != t.shape:
        return None
    return C.c_void_p(sh[0].data_ptr())


class Metadata_3(object):
    """Handle on a device-resident Metadata (reference: Metadata<3>, SCN/Metadata/Metadata.h:44)."""

    def __init__(self):
        if not torch.cuda.is_available():
            raise RuntimeError("detection_3d_b200: no CUDA device (this extension has no CPU fallback)")
        self._h = C.c_void_p()
        check(lib().scn_metadata_create(C.byref(self._h), _stream()))
        self._keep = []
        self._oplog, self._opseen = [], set()  # rulebook requests of this forward, in order (see prefetch)

    def _log(self, kind, a, b, f, s):
        key = (kind,) + tuple(int(v) for t in (a, b, f, s) for v in t)
        if key not in self._opseen:
            self._opseen.add(key)
            self._oplog.append(key)

    def prefetch(self, ops):
        """Hint: build these rulebooks ahead on a worker thread (scn_metadata_prefetch).  `ops` is the
        `_oplog` of an earlier forward of the same network; results do not depend on it."""
        if not ops:
            return
        flat = (C.c_long * (13 * len(ops)))(*[v for op in ops for v in op])
        check(lib().scn_metadata_prefetch(self._h, len(ops), flat))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().scn_metadata_destroy(h)
            except Exception:
                pass
            self._h = None

    # ---- the methods pybind.cpp:12-32 exposes that the hot path uses
    def getNActive(self, spatial_size):
        n = C.c_long()
        check(lib().scn_get_nactive(self._h, l3(spatial_size), C.byref(n)))
        return n.value

    def getBatchSize(self, spatial_size):
        """number of batch items on the grid of `spatial_size` (known on the host: no device round trip)"""
        b = C.c_int()
        check(lib().scn_get_batch_size(self._h, l3(spatial_size), C.byref(b)))
        return b.value

    def getSpatialLocations(self, spatial_size, device="cpu"):
        """int64 [nActive, 4] (x, y, z, batch) in row order; the reference returns a CPU tensor."""
        n = self.getNActive(spatial_size)
        dev = torch.device(device)
        out = torch.zeros((n, 4), dtype=torch.int64, device=dev)
        if n:
            check(lib().scn_get_spatial_locations(self._h, l3(spatial_size), C.c_void_p(out.data_ptr()), int(dev.type == "cuda")))
        return out

    # ---- parity / inspection helpers (no reference counterpart in pybind; rulebooks are public C++ members)
    def iterationOrder(self, spatial_size):
        n = self.getNActive(spatial_size)
        out = torch.zeros(n, dtype=torch.int32)
        check(lib().scn_iteration_order(self._h, l3(spatial_size), C.c_void_p(out.data_ptr())))
        return out

    def _rulebook(self, kind, a, b, c):
        nl = C.c_int()
        lens = (C.c_long * 512)()  # one entry per list: filter volumes up to 512 (8^3, [1, 1, 512])
        check(lib().scn_rulebook_info(self._h, kind, a, b, c, C.byref(nl), lens))
        out = []
        for i in range(nl.value):
            t = torch.zeros(lens[i], dtype=torch.int32)
            if lens[i]:
                check(lib().scn_rulebook_copy(self._h, kind, a, b, c, i, C.c_void_p(t.data_ptr())))
            out.append(t)
        return out

    def inputLayerRuleBook(self):
        z = l3([0, 0, 0])
        return self._rulebook(0, z, z, z)

    def submanifoldRuleBook(self, spatial_size, filter_size):
        n = C.c_long()
        check(lib().scn_submanifold_prepare(self._h, l3(spatial_size), l3(filter_size), C.byref(n)))
        return [t.view(-1, 2) for t in self._rulebook(1, l3(spatial_size), l3(filter_size), l3([0, 0, 0]))]

    def sparseToDenseRuleBook(self, spatial_size):
        """one [n, 2] (row, spatial offset) list per batch item, hash-iteration order (Metadata.cpp:469-483)"""
        z = l3([0, 0, 0])
        return [t.view(-1, 2) for t in self._rulebook(3, l3(spatial_size), z, z)]

    def ruleBook(self, in_size, out_size, filter_size, filter_stride):
        n, r = C.c_long(), C.c_long()
        check(lib().scn_convolution_prepare(self._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), C.byref(n), C.byref(r)))
        return [t.view(-1, 2) for t in self._rulebook(2, l3(in_size), l3(filter_size), l3(filter_stride))]


# ------------------------------------------------------------------ SparseToDense
def SparseToDense_updateOutput(spatial_size, m, input_features, output_features, nPlanes):
    """pybind.cpp SparseToDense_updateOutput; CPU/SparseToDense.cpp:34-66 -> [batch, nPlanes, X, Y, Z], zero where inactive"""
    sz = _ints(spatial_size)
    b = C.c_int()
    check(lib().scn_get_batch_size(m._h, l3(sz), C.byref(b)))
    output_features.resize_(max(b.value, 1), int(nPlanes), *sz)
    if input_features.dim() == 2:
        check(lib().scn_sparse_to_dense_forward(m._h, l3(sz), _dev_f32(input_features, "in") if input_features.numel() else None,
                                                _dev_f32(output_features, "out"), input_features.size(1)))
    else:
        output_features.zero_()


def SparseToDense_updateGradInput(spatial_size, m, input_features, d_input_features, d_output_features):
    """CPU/SparseToDense.cpp:67-101"""
    d_input_features.resize_as_(input_features)
    if input_features.dim() == 2 and input_features.numel():
        check(lib().scn_sparse_to_dense_backward(m._h, l3(_ints(spatial_size)), _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"),
                                                 input_features.size(1)))
    else:
        d_input_features.zero_()


def n_rulebook_bits():
    return lib().scn_n_rulebook_bits()


# ------------------------------------------------------------------ IO layers
def InputLayer_updateOutput(m, spatial_size, coords, input_features, output_features, batch_size, mode):
    """pybind.cpp:154-158.  coords: LongTensor [N, 3|4], CPU (as the reference requires) or CUDA."""
    if coords.dtype != torch.int64 or coords.dim() != 2:
        raise RuntimeError("InputLayer: coords must be a 2-d LongTensor")
    coords = coords.contiguous()
    m._keep.append(coords)
    n_active, max_active = C.c_long(), C.c_int()
    check(lib().scn_input_layer_build(m._h, l3(spatial_size), C.c_void_p(coords.data_ptr()), int(coords.is_cuda), coords.size(0),
                                      coords.size(1), int(batch_size), int(mode), C.byref(n_active), C.byref(max_active)))
    planes = input_features.size(1)
    output_features.resize_(n_active.value, planes)
    if n_active.value:
        check(lib().scn_input_layer_forward(m._h, _dev_f32(input_features, "InputLayer features"), _dev_f32(output_features, "out"), planes))
    tr = _tr()
    if tr is not None:
        if tr.ops:
            tr.fail("more than one InputLayer in a recording")
        tr.add(0, [tr.new_reg(output_features)] + _ints(spatial_size) + [int(mode), int(batch_size), planes])


def InputLayer_updateGradInput(m, d_input_features, d_output_features):
    """pybind.cpp:159-162"""
    rules = m.inputLayerRuleBook()[0]
    n_in, planes = int(rules[2]), d_output_features.size(1)
    d_input_features.resize_(n_in, planes)
    if n_in:
        check(lib().scn_input_layer_backward(m._h, _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"), planes))


def OutputLayer_updateOutput(m, input_features, output_features):
    """pybind.cpp:163-166"""
    hdr = m.inputLayerRuleBook()[0]
    mode, n_in, n_out, planes = int(hdr[0]), int(hdr[2]), int(hdr[3]), input_features.size(1)
    output_features.resize_(n_out if mode == 0 else n_in, planes)
    if output_features.numel():
        check(lib().scn_output_layer_forward(m._h, _dev_f32(input_features, "in"), _dev_f32(output_features, "out"), planes))


def OutputLayer_updateGradInput(m, d_input_features, d_output_features):
    """pybind.cpp:167-170"""
    hdr = m.inputLayerRuleBook()[0]
    n_out, planes = int(hdr[3]), d_output_features.size(1)
    d_input_features.resize_(n_out, planes)
    if d_input_features.numel():
        check(lib().scn_output_layer_backward(m._h, _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"), planes))


# ------------------------------------------------------------------ convolutions
def _w3(weight):
    # (K, groups=1, Cin, Cout)
    if weight.dim() == 4 and weight.size(1) != 1:
        raise RuntimeError("groups > 1 is not supported by this build")
    return weight.size(0), weight.size(-2), weight.size(-1)


def SubmanifoldConvolution_updateOutput(spatial_size, filter_size, m, input_features, output_features, weight, bias):
    """pybind.cpp:134-138 -> returns the multiply-add count like the reference."""
    _, cin, cout = _w3(weight)
    n = m.getNActive(spatial_size)
    m._log(1, spatial_size, (0, 0, 0), filter_size, (0, 0, 0))
    output_features.resize_(n, cout)
    macs = C.c_double()
    check(lib().scn_submanifold_convolution_forward(m._h, l3(spatial_size), l3(filter_size), _dev_f32(input_features, "in"),
                                                    _dev_f32(output_features, "out"), _dev_f32(weight, "weight"), _opt(bias, "bias"),
                                                    cin, cout, C.byref(macs), _shadow_ptr(input_features), _weight_tag(weight), None, None))
    tr = _tr()
    if tr is not None:
        tr.add(1, [tr.reg(input_features), tr.new_reg(output_features)] + _ints(spatial_size) + _ints(filter_size)
               + [tr.param(weight), tr.param(bias), cin, cout])
    return macs.value


def SubmanifoldConvolution_backward(spatial_size, filter_size, m, input_features, d_input_features, d_output_features, weight, d_weight, d_bias):
    """pybind.cpp:139-143"""
    _, cin, cout = _w3(weight)
    if d_input_features is not None:  # None: the caller does not need the input gradient (native side skips it)
        d_input_features.resize_as_(input_features)
    check(lib().scn_submanifold_convolution_backward(m._h, l3(spatial_size), l3(filter_size), _dev_f32(input_features, "in"),
                                                     None if d_input_features is None else _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"),
                                                     _dev_f32(weight, "weight"), _dev_f32(d_weight, "d_weight"), _opt(d_bias, "d_bias"), cin, cout))


def Convolution_updateOutput(in_size, out_size, filter_size, filter_stride, m, input_features, output_features, weight, bias):
    """pybind.cpp:54-59"""
    _, cin, cout = _w3(weight)
    n, r = C.c_long(), C.c_long()
    m._log(2, in_size, out_size, filter_size, filter_stride)
    check(lib().scn_convolution_prepare(m._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), C.byref(n), C.byref(r)))
    output_features.resize_(n.value, cout)
    macs = C.c_double()
    check(lib().scn_convolution_forward(m._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), _dev_f32(input_features, "in"),
                                        _dev_f32(output_features, "out"), _dev_f32(weight, "weight"), _opt(bias, "bias"), cin, cout, C.byref(macs),
                                        _shadow_ptr(input_features), _weight_tag(weight), None, None))
    tr = _tr()
    if tr is not None:
        tr.add(2, [tr.reg(input_features), tr.new_reg(output_features)] + _ints(in_size) + _ints(out_size) + _ints(filter_size)
               + _ints(filter_stride) + [tr.param(weight), tr.param(bias), cin, cout])
    return macs.value


def Convolution_backward(in_size, out_size, filter_size, filter_stride, m, input_features, d_input_features, d_output_features, weight, d_weight, d_bias):
    """pybind.cpp:60-65"""
    _, cin, cout = _w3(weight)
    d_input_features.resize_as_(input_features)
    check(lib().scn_convolution_backward(m._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), _dev_f32(input_features, "in"),
                                         _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"), _dev_f32(weight, "weight"),
                                         _dev_f32(d_weight, "d_weight"), _opt(d_bias, "d_bias"), cin, cout))


def Deconvolution_updateOutput(in_size, out_size, filter_size, filter_stride, m, input_features, output_features, weight, bias):
    """pybind.cpp:78-83"""
    _, cin, cout = _w3(weight)
    n = m.getNActive(out_size)
    m._log(3, in_size, out_size, filter_size, filter_stride)
    output_features.resize_(n, cout)
    macs = C.c_double()
    check(lib().scn_deconvolution_forward(m._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), _dev_f32(input_features, "in"),
                                          _dev_f32(output_features, "out"), _dev_f32(weight, "weight"), _opt(bias, "bias"), cin, cout, C.byref(macs),
                                          _shadow_ptr(input_features), _weight_tag(weight), None, None))
    tr = _tr()
    if tr is not None:
        tr.add(3, [tr.reg(input_features), tr.new_reg(output_features)] + _ints(in_size) + _ints(out_size) + _ints(filter_size)
               + _ints(filter_stride) + [tr.param(weight), tr.param(bias), cin, cout])
    return macs.value


def Deconvolution_backward(in_size, out_size, filter_size, filter_stride, m, input_features, d_input_features, d_output_features, weight, d_weight, d_bias):
    """pybind.cpp:84-89"""
    _, cin, cout = _w3(weight)
    d_input_features.resize_as_(input_features)
    check(lib().scn_deconvolution_backward(m._h, l3(in_size), l3(out_size), l3(filter_size), l3(filter_stride), _dev_f32(input_features, "in"),
                                           _dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"), _dev_f32(weight, "weight"),
                                           _dev_f32(d_weight, "d_weight"), _opt(d_bias, "d_bias"), cin, cout))


# ------------------------------------------------------------------ batch norm
def BatchNormalization_updateOutput(input_features, output_features, saveMean, saveInvStd, runningMean, runningVar, weight, bias, eps,
                                    momentum, train, leakiness, instance_stats=False):
    """pybind.cpp:219-220.  `instance_stats=True` is the eval / track_running_stats=False branch of
    sparseconvnet/batchNormalization.py:51-56 with the mean / unbiased variance computed by the
    kernel instead of by torch ops; runningMean / runningVar are then ignored."""
    n, c = input_features.size(0), input_features.size(1) if input_features.dim() == 2 else 0
    output_features.resize_as_(input_features)
    saveMean.resize_(c)
    saveInvStd.resize_(c)
    mode = 0 if train else (2 if instance_stats else 1)
    sh = _new_shadow(output_features)
    check(lib().scn_batchnorm_forward(_dev_f32(input_features, "in"), _dev_f32(output_features, "out"), n, c, _dev_f32(saveMean, "saveMean"),
                                      _dev_f32(saveInvStd, "saveInvStd"), _opt(runningMean, "runningMean"), _opt(runningVar, "runningVar"),
                                      _opt(weight, "weight"), _opt(bias, "bias"), float(eps), float(momentum), mode, float(leakiness), _stream(),
                                      None if sh is None else C.c_void_p(sh.data_ptr())))
    _attach_shadow(output_features, sh)
    tr = _tr()
    if tr is not None:
        if train and not tr.training:
            tr.fail("training-mode BatchNorm is not recorded")
        tr.add(4, [tr.reg(input_features), tr.new_reg(output_features), c, tr.param(weight), tr.param(bias), tr.param(runningMean),
                   tr.param(runningVar), mode], [eps, momentum, leakiness])


def BatchNormalization_backward(input_features, d_input_features, output_features, d_output_features, saveMean, saveInvStd, runningMean,
                                runningVar, weight, bias, d_weight, d_bias, leakiness):
    """pybind.cpp:221"""
    n, c = input_features.size(0), input_features.size(1)
    d_input_features.resize_as_(input_features)
    check(lib().scn_batchnorm_backward(_dev_f32(input_features, "in"), _dev_f32(d_input_features, "d_in"), _dev_f32(output_features, "out"),
                                       _dev_f32(d_output_features, "d_out"), n, c, _dev_f32(saveMean, "saveMean"), _dev_f32(saveInvStd, "saveInvStd"),
                                       _opt(weight, "weight"), _opt(d_weight, "d_weight"), _opt(d_bias, "d_bias"), float(leakiness), _stream()))


# ------------------------------------------------------------------ NetworkInNetwork
def NetworkInNetwork_updateOutput(input_features, output_features, weight, bias):
    """pybind.cpp:224-225 -> returns nActive * nIn * nOut like the reference"""
    n, cin, cout = input_features.size(0), weight.size(0), weight.size(1)
    output_features.resize_(n, cout)
    macs = C.c_double()
    check(lib().scn_network_in_network_forward(_dev_f32(input_features, "in") if n else None, _dev_f32(output_features, "out") if n else None,
                                               _dev_f32(weight, "weight"), _opt(bias, "bias"), n, cin, cout, C.byref(macs), _stream(),
                                               _shadow_ptr(input_features), _weight_tag(weight)))
    tr = _tr()
    if tr is not None:
        tr.fail("NetworkInNetwork is not recorded")
    return macs.value


def NetworkInNetwork_updateGradInput(d_input_features, d_output_features, weight):
    """pybind.cpp:226"""
    n, cin, cout = d_output_features.size(0), weight.size(0), weight.size(1)
    d_input_features.resize_(n, cin)
    if n:
        check(lib().scn_network_in_network_backward_input(_dev_f32(d_input_features, "d_in"), _dev_f32(d_output_features, "d_out"),
                                                          _dev_f32(weight, "weight"), n, cin, cout, _stream()))


def NetworkInNetwork_accGradParameters(input_features, d_output_features, d_weight, d_bias):
    """pybind.cpp:227-228"""
    n, cin, cout = input_features.size(0), d_weight.size(0), d_weight.size(1)
    check(lib().scn_network_in_network_backward_params(_dev_f32(input_features, "in") if n else None, _dev_f32(d_output_features, "d_out") if n else None,
                                                       _dev_f32(d_weight, "d_weight"), _opt(d_bias, "d_bias"), n, cin, cout, _stream()))


def add_features(a, b):
    """out = a + b for two feature matrices sharing one Metadata (tables.py:28-41, utils.py:61-66)."""
    out = torch.empty_like(a)
    if a.numel():
        sh = _new_shadow(out)
        check(lib().scn_add_features(_dev_f32(a, "a"), _dev_f32(b, "b"), _dev_f32(out, "out"), a.numel(), _stream(),
                                     None if sh is None else C.c_void_p(sh.data_ptr())))
        _attach_shadow(out, sh)
    tr = _tr()
    if tr is not None:
        if a.numel() == 0:
            tr.fail("empty add")
        tr.add(5, [tr.reg(a), tr.reg(b), tr.new_reg(out)])
    return out


def set_math_mode(mode):
    """'fp32' (CUDA cores, exact), 'tf32' or 'bf16' (tcgen05 tensor cores, fp32 accumulate), 'tf32x3' (tcgen05, every fp32
    operand split into two TF32 values hi + lo, three products per step in one fp32 accumulator: fp32-class accuracy at tensor-core
    speed; weight gradients and the convolutions the tensor-core kernel cannot take run on the exact CUDA-core kernels, as in
    'tf32'), or 'fp16' (as 'bf16', with fp16 operands wherever 'bf16' has bf16 ones: 11 significant bits instead of 8, but a range
    of +-65504 -- a larger value becomes inf, as with .half() -- so training needs loss scaling, e.g. torch.amp.GradScaler).
    math_mode() returns the code: 0, 1, 2, 3 or 5."""
    code = {"fp32": 0, "tf32": 1, "bf16": 2, "tf32x3": 3, "fp16": 5}[mode] if isinstance(mode, str) else int(mode)
    check(lib().scn_set_math_mode(code))
    _MATH["mode"] = lib().scn_get_math_mode()


def math_mode():
    return _MATH["mode"]


def kernel_launch_count():
    return lib().scn_kernel_launch_count()


def empty_cache():
    """Hand the library's idle device memory back to the driver (scn_release_cached_memory): Metadata chunks of finished forwards,
    cached weight operand images, scratch buffers -- memory torch.cuda.empty_cache() cannot see.  Synchronises the device; live
    Metadata objects and recorded programs (FPN_Net.reset_program drops a network's) keep theirs.  -> bytes released."""
    _WEIGHT_IMAGES_DROPPED[0] += 1
    n = lib().scn_release_cached_memory()
    if n < 0:
        raise RuntimeError("scn_release_cached_memory failed")
    return n
