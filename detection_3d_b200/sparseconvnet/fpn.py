"""FPN_Net: the sparse ResNet-FPN backbone of Detection_3D (reference:
SparseConvNet/sparseconvnet/fpn_net.py:13-265, built by
maskrcnn_benchmark/modeling/backbone/backbone.py:39-69).

Module tree and parameter names follow the reference so its checkpoints load unchanged:
layers_in_0, layers_in.{0,1}, layers_out.{0,1}, linear, convs_pro2d.i, m_downs.k..., m_shortcuts.k,
m_ups.k.{0,1}, m_mergeds.k.
"""
import numpy as np
import torch
import torch.nn as nn

import os

from . import layers as L
from . import native, program
from .containers import AddTable, ConcatTable, Identity, Sequential, add_feature_planes
from .tensor import SparseConvNetTensor

_PROGRAMS = os.environ.get("SCN_PROGRAM", "1") != "0"  # developer switch: always run layer by layer
_TRAIN_PROGRAMS = os.environ.get("SCN_TRAIN_PROGRAM", "1") != "0"  # training forwards: replay too (one autograd node per forward)


OutputLayer = L.OutputLayer  # (FPN_Net holds one in `layers_out`; the shipped forward never calls it)


_ELEMENT_CHANNELS = {'xyz': 3, 'color': 3, 'normal': 3}


class FPN_Net(nn.Module):
    def __init__(self, full_scale, dimension, raw_elements, reps, nPlanesF, nPlaneM, residual_blocks,
                 fpn_scales_from_top, roi_scales_from_top, downsample, rpn_map_sizes,
                 rpn_3d_2d_selector, leakiness=0, voxel_scale=None, bn_momentum=0.9, track_running_stats=True):
        """downsample = [kernels, strides], one [kx,ky,kz] per level transition."""
        nn.Module.__init__(self)
        self.bn_momentum = bn_momentum
        self.track_running_stats = track_running_stats
        self.dimension = dimension
        self.down_kernels, self.down_strides = downsample[0], downsample[1]
        self.fpn_scales_from_top = fpn_scales_from_top
        self.roi_scales_from_top = roi_scales_from_top
        n_scales = len(nPlanesF)
        assert len(self.down_kernels) == n_scales - 1 == len(self.down_strides), \
            f"nPlanesF len = {n_scales}, kernels num = {len(self.down_kernels)}"
        assert all(len(k) == 3 for k in self.down_kernels) and all(len(s) == 3 for s in self.down_strides)
        self._merge = 'add'
        in_channels = sum(_ELEMENT_CHANNELS[e] for e in raw_elements)

        def bn(c):
            return L.BatchNormLeakyReLU(c, momentum=bn_momentum, leakiness=leakiness, track_running_stats=track_running_stats)

        self.layers_in_0 = Sequential(L.InputLayer(dimension, full_scale, mode=4))
        self.layers_in = Sequential(L.InputLayer(dimension, full_scale, mode=4),
                                    L.SubmanifoldConvolution(dimension, in_channels, nPlanesF[0], 3, False))
        self.layers_out = Sequential(L.BatchNormReLU(nPlanesF[0], momentum=bn_momentum, track_running_stats=track_running_stats),
                                     OutputLayer(dimension))
        self.linear = nn.Linear(nPlanesF[0], 20)
        self.voxel_scale = voxel_scale
        self.rpn_map_sizes = np.array(rpn_map_sizes)
        self.rpn_3d_2d_selector = rpn_3d_2d_selector

        # z-collapsing convolutions that turn the 3-D rpn maps into 2-D ones (fpn_net.py:55-57)
        self.convs_pro2d = nn.ModuleList()
        for zsize in self.rpn_map_sizes[:, -1]:
            self.convs_pro2d.append(L.Convolution(dimension, nPlaneM, nPlaneM, [1, 1, int(zsize)], [1, 1, 1], False))

        def residual_or_vgg_block(m, a, b):  # fpn_net.py:60-76
            if residual_blocks:
                m.add(ConcatTable()
                      .add(Identity() if a == b else L.NetworkInNetwork(a, b, False))
                      .add(Sequential().add(bn(a)).add(L.SubmanifoldConvolution(dimension, a, b, 3, False))
                           .add(bn(b)).add(L.SubmanifoldConvolution(dimension, b, b, 3, False)))
                      ).add(AddTable())
            else:
                m.add(Sequential().add(bn(a)).add(L.SubmanifoldConvolution(dimension, a, b, 3, False)))
            return {'kernel': [1, 1, 1], 'stride': [1, 1, 1]}

        self.m_downs, self.m_shortcuts = nn.ModuleList(), nn.ModuleList()
        self.operations_down = []
        for k in range(n_scales):
            m = Sequential()
            if k > 0:  # fpn_net.py:77-84
                m.add(Sequential().add(bn(nPlanesF[k - 1])).add(
                    L.Convolution(dimension, nPlanesF[k - 1], nPlanesF[k], self.down_kernels[k - 1], self.down_strides[k - 1], False)))
                self.operations_down.append({'kernel': self.down_kernels[k - 1], 'stride': self.down_strides[k - 1]})
            for _ in range(reps):
                op = residual_or_vgg_block(m, nPlanesF[k], nPlanesF[k])
                if k == 0:
                    self.operations_down.append(op)
            self.m_downs.append(m)
            self.m_shortcuts.append(L.SubmanifoldConvolution(dimension, nPlanesF[k], nPlaneM, 1, False))

        self.m_ups, self.m_mergeds = nn.ModuleList(), nn.ModuleList()
        self.operations_up = []
        for k in range(n_scales - 1, 0, -1):  # fpn_net.py:86-93,119-126
            self.m_ups.append(Sequential().add(bn(nPlaneM)).add(
                L.Deconvolution(dimension, nPlaneM, nPlaneM, self.down_kernels[k - 1], self.down_strides[k - 1], False)))
            self.operations_up.append({'kernel': self.down_kernels[k - 1], 'stride': self.down_strides[k - 1]})
            self.m_mergeds.append(L.SubmanifoldConvolution(dimension, nPlaneM, nPlaneM, 3, False))

    def forward(self, net0):
        """net0 = [coords LongTensor [N,4], features float [N,C]] -> (rpn_maps, roi_maps).

        Inference (eval mode, no autograd graph) runs as a recorded program after the first call: the
        first forward is executed layer by layer while `program.Trace` records the native calls, later
        forwards replay them with one native call (same kernels, same order).  Training, a changed math
        mode, unusual inputs or SCN_PROGRAM=0 use the layer-by-layer path."""
        if _PROGRAMS and not self.training and not torch.is_grad_enabled() and len(net0) == 2:
            coords, feats = net0[0], net0[1]
            dev = self.layers_in[0].device
            if dev is None and isinstance(feats, torch.Tensor) and not feats.is_cuda:
                # (extension of the reference's calling convention: host features are accepted when the network lives on a GPU)
                pdev = next(self.parameters()).device
                dev = pdev if pdev.type == "cuda" else None
            mode = native.math_mode()
            prog = self.__dict__.get("_program")
            if (prog is not None and dev is not None and isinstance(feats, torch.Tensor) and not feats.is_cuda and isinstance(coords, torch.Tensor)
                    and coords.dtype == torch.int64 and coords.dim() == 2 and mode == prog.math_mode and not self._has_prefetched(coords)):
                # host features: start the Metadata build first -- it uploads the coordinates, which the forward needs before
                # anything else -- and only then queue the feature copy, which then overlaps the grid build
                md = L.Metadata(self.dimension)
                prog.prepare(md, coords)
                self.__dict__.setdefault("_prefetched", []).append((coords, coords._version, md))
            if dev is not None and isinstance(feats, torch.Tensor):
                feats = feats.to(dev, non_blocking=True)
                net0 = [coords, feats] + list(net0[2:])  # (the layer-by-layer path below must see the device tensor too)
            if prog is not None and isinstance(coords, torch.Tensor) and prog.usable(coords, feats, mode):
                return self._run_program(prog, coords, feats)
            if prog is None and self.__dict__.get("_program_error") is None and isinstance(feats, torch.Tensor) and feats.is_cuda:
                with program.Trace() as tr:
                    rpn_maps, roi_maps = self.forward_fpn(self.layers_in(net0))
                try:
                    self.__dict__["_program"] = program.Program(tr, [(m.features, m.spatial_size) for m in rpn_maps + roi_maps], mode)
                    self.__dict__["_program_n_rpn"] = len(rpn_maps)
                except Exception as e:  # the layer-by-layer path stays in charge
                    self.__dict__["_program_error"] = str(e)
                return rpn_maps, roi_maps
        if (_PROGRAMS and _TRAIN_PROGRAMS and self.training and torch.is_grad_enabled() and len(net0) == 2 and isinstance(net0[1], torch.Tensor)
                and isinstance(net0[0], torch.Tensor)):
            # Training: the first step runs layer by layer under autograd while the calls are recorded; later steps are ONE autograd node
            # whose forward replays the program in training mode and whose backward is scn_program_backward.
            coords, feats = net0[0], net0[1]
            dev = self.layers_in[0].device
            if dev is not None:
                feats = feats.to(dev, non_blocking=True)
                net0 = [coords, feats]
            mode = native.math_mode()
            prog = self.__dict__.get("_program_train")
            if prog is not None and prog.usable(coords, feats, mode):
                md = self._take_prefetched("_prefetched_train", coords) or L.Metadata(self.dimension)
                import detection_3d_b200.sparseconvnet as pkg
                uniq = program.TrainFunction.apply(prog, md, coords, feats, *prog.params)
                pkg.forward_pass_multiplyAdd_count += prog.last_macs
                by_reg = dict(zip(sorted(set(prog.out_regs)), uniq))
                maps = [SparseConvNetTensor(features=by_reg[r], metadata=md, spatial_size=s.clone()) for r, s in zip(prog.out_regs, prog.out_sizes)]
                n = self.__dict__["_program_train_n_rpn"]
                return maps[:n], maps[n:]
            if prog is None and self.__dict__.get("_program_train_error") is None and feats.is_cuda:
                with program.Trace(training=True) as tr:
                    rpn_maps, roi_maps = self.forward_fpn(self.layers_in(net0))
                try:
                    self.__dict__["_program_train"] = program.Program(tr, [(m.features, m.spatial_size) for m in rpn_maps + roi_maps], mode)
                    self.__dict__["_program_train_n_rpn"] = len(rpn_maps)
                except Exception as e:  # the layer-by-layer path stays in charge
                    self.__dict__["_program_train_error"] = str(e)
                return rpn_maps, roi_maps
        return self.forward_fpn(self.layers_in(net0))

    def _has_prefetched(self, coords):
        return any(pre[0] is coords and pre[1] == coords._version for pre in self.__dict__.get("_prefetched", ()))

    def _take_prefetched(self, queue, coords):
        """The Metadata of the oldest entry of `queue` made for this very coordinate tensor, unmodified since (or None)."""
        q = self.__dict__.get(queue)
        for i, pre in enumerate(q or ()):
            if pre[0] is coords and pre[1] == coords._version:
                del q[i]
                return pre[2]
        return None

    def prefetch(self, coords):
        """Start building the Metadata (active-site grids, rulebooks) of the NEXT input now, on the library's build streams,
        while the GPU still computes the work queued before.  A `forward` whose coordinate tensor is this very object, unmodified
        since, uses that Metadata; any other input ignores it.  Results are identical with or without the call.  Device
        coordinates must be complete (not still being written by another stream).  Returns False (and does nothing) until a
        program has been recorded in the current mode -- the second inference forward, the second training step -- or when the
        math mode has changed since.

        Inference (eval mode): may be called for several inputs (first in, first out); calling it TWO buildings ahead hides the
        whole build behind the computation.

        Training (train mode): prepares the next training step (scn_program_prepare_training): its grids, plans and the rule lists
        its backward pass reads are built while the current step runs.  Call it with the next batch's coordinates before the
        current step's forward or backward; at most two steps stay prepared.  Inference and training entries are kept apart:
        neither is used by the other mode, and switching to eval drops the training entries."""
        key = "_program_train" if self.training else "_program"
        prog = self.__dict__.get(key)
        if prog is None or not isinstance(coords, torch.Tensor) or coords.dtype != torch.int64 or coords.dim() != 2:
            return False
        if native.math_mode() != prog.math_mode:
            return False
        prog.throttle()  # before the Metadata is created: it then recycles the memory of the forward that just finished
        native.lib().scn_set_pool_growth(1)  # built ahead: do not queue behind a running forward for memory
        try:
            md = L.Metadata(self.dimension)
            if self.training:
                prog.prepare_training(md, coords)
            else:
                prog.prepare(md, coords)
        finally:
            native.lib().scn_set_pool_growth(0)
        q = self.__dict__.setdefault("_prefetched_train" if self.training else "_prefetched", [])
        q.append((coords, coords._version, md))
        del q[:-2 if self.training else -4]  # at most a few buildings ahead (training: as many as the program keeps prepared)
        return True

    def train(self, mode=True):
        if not mode:  # evaluation: the training steps prepared ahead are dropped and release their memory
            self.__dict__.pop("_prefetched_train", None)
            if self.__dict__.get("_program_train") is not None:
                self.__dict__["_program_train"].drop_prepared()
        return nn.Module.train(self, mode)

    def reset_program(self):
        """Forget the recorded program (call after changing the module tree)."""
        self.__dict__.pop("_program", None)
        self.__dict__.pop("_program_error", None)
        self.__dict__.pop("_prefetched", None)
        for k in ("_program_train", "_program_train_error", "_program_train_n_rpn", "_prefetched_train"):
            self.__dict__.pop(k, None)

    # The recorded program and the Metadata objects built ahead are handles into the native library (ctypes pointers):
    # a copy / pickle of the network (EMA copies, torch.save(model), as with the reference) drops them and records again.
    _RUNTIME_STATE = ("_program", "_program_error", "_program_n_rpn", "_prefetched", "_program_train", "_program_train_error", "_program_train_n_rpn",
                      "_prefetched_train")

    def __getstate__(self):
        state = self.__dict__.copy()
        for k in self._RUNTIME_STATE:
            state.pop(k, None)
        return state

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k not in self._RUNTIME_STATE:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def load_state_dict(self, *args, **kwargs):
        # loaders write through `.data` / copy_ on detached views, which does not always bump Tensor._version: the packed
        # weight images (keyed by token + version) are dropped explicitly
        out = nn.Module.load_state_dict(self, *args, **kwargs)
        native.invalidate_weight_cache(self)
        return out

    def _run_program(self, prog, coords, feats):
        import detection_3d_b200.sparseconvnet as pkg
        md = self._take_prefetched("_prefetched", coords) or L.Metadata(self.dimension)  # built ahead by prefetch()
        outs, macs = prog.run(md, coords, feats)
        pkg.forward_pass_multiplyAdd_count += macs
        maps = [SparseConvNetTensor(features=f, metadata=md, spatial_size=s.clone()) for f, s in zip(outs, prog.out_sizes)]
        n = self.__dict__["_program_n_rpn"]
        return maps[:n], maps[n:]

    def forward_fpn(self, net):
        n_scales = len(self.m_downs)
        downs = []
        for m in self.m_downs:
            net = m(net)
            downs.append(net)
        net = self.m_shortcuts[-1](net)
        ups = [net]
        for k in range(n_scales - 1):
            j = n_scales - 2 - k
            net = self.m_ups[k](net)
            net = add_feature_planes([net, self.m_shortcuts[j](downs[j])])
            ups.append(self.m_mergeds[k](net))
        rpn_maps_3d = [ups[i] for i in self.fpn_scales_from_top]
        rpn_maps_2d = [self.convs_pro2d[i](rpn_maps_3d[i]) for i in range(len(rpn_maps_3d))]
        rpn_maps = rpn_maps_3d + rpn_maps_2d
        rpn_maps = [rpn_maps[i] for i in self.rpn_3d_2d_selector]
        roi_maps = [ups[i] for i in self.roi_scales_from_top]
        for i in range(len(rpn_maps_3d)):
            assert torch.all(rpn_maps_3d[i].spatial_size == torch.tensor(self.rpn_map_sizes[i]))
        # The sequence of rulebooks a forward requests depends on the network only: remember it so that
        # the next forward's Metadata can build them ahead of the layers (native.Metadata_3.prefetch).
        inp = self.layers_in[0]
        if getattr(inp, "prefetch_ops", None) is None and hasattr(net.metadata, "_oplog"):
            inp.prefetch_ops = list(net.metadata._oplog)
        return rpn_maps, roi_maps


def sw4c_fpn432_config():
    """configs/sw4c/sw4c_fpn432_bs1_lr5.yaml + maskrcnn_benchmark/config/defaults.py:44-53,173-175,225,283-284
    as resolved by tools/train_net_sparse3d.py:231-318 (BASELINE.json configs 1-4)."""
    planes = [32, 64, 64, 128, 128, 128, 256, 256, 256]
    return dict(full_scale=[2048, 2048, 512], dimension=3, raw_elements=['xyz', 'color', 'normal'], reps=1, nPlanesF=planes, nPlaneM=128,
                residual_blocks=True, fpn_scales_from_top=[4, 3, 2], roi_scales_from_top=[4, 3],
                downsample=[[[2, 2, 2]] * 8, [[2, 2, 2]] * 8], rpn_map_sizes=[[128, 128, 32], [64, 64, 16], [32, 32, 8]],
                rpn_3d_2d_selector=[1, 3, 4, 5], bn_momentum=0.9, track_running_stats=False)


def c6_fpn4321_config():
    """configs/6c/6c_Fpn4321_bs1_lr5.yaml (BASELINE.json config 5)."""
    cfg = sw4c_fpn432_config()
    cfg.update(full_scale=[4096, 4096, 512], fpn_scales_from_top=[4, 3, 2, 1],
               rpn_map_sizes=[[256, 256, 32], [128, 128, 16], [64, 64, 8], [32, 32, 4]], rpn_3d_2d_selector=[1, 2, 3, 4, 5, 6])
    return cfg
