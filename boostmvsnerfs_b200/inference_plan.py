"""Call-side preparation of the KEPT cuDNN modules for inference (no change to their math).

north_star keeps the 2-D FPN and the 3-D cost regularisers on cuDNN.  Measured on B200
(tools/conv_experiments.py, profiles/round1_conv_variants.md) the stock eval() modules spend a
third of their time in stand-alone batch-norm kernels and NCHW<->NHWC transposes that cuDNN
inserts around its tensor-core kernels.  Two exact-up-to-rounding rewrites remove both:

  * batch-norm folding: eval-mode BN is an affine map per channel, folded into the preceding
    (transposed) convolution's weight and bias (relative difference ~1e-6 in fp32);
  * channels-last memory format for weights and activations (cuDNN's native tensor-core layout);
    our kernels read and write strided tensors, so no transpose is ever materialised.

The folded copies are derived objects: the registered parameters (and therefore state_dict /
checkpoint names) are untouched, and the copies are rebuilt whenever a parameter changes.
"""
import copy

import torch
import torch.nn as nn

from .modules import _CBR


def _fold_pair(conv, bn, transposed=False):
    scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    shape = [1] * conv.weight.dim()
    shape[1 if transposed else 0] = -1
    w = conv.weight * scale.view(shape)
    b = bn.bias - bn.running_mean * scale
    if conv.bias is not None:
        b = b + conv.bias * scale
    conv.weight = nn.Parameter(w, requires_grad=False)
    conv.bias = nn.Parameter(b, requires_grad=False)


class S2DConv5x5(nn.Module):
    """A 5x5 / stride-2 / pad-2 convolution (+bias, +ReLU) evaluated as space-to-depth(2) followed by a
    3x3 / stride-1 / pad-1 convolution on 4x the channels — the same products, regrouped:
        y[i] = sum_ky W[ky] x[2i+ky-2],  ky = 2a+p  ->  sum_{a in 0..2} sum_{p in 0,1} W6[2a+p] z[i+a-1, p],
    z[i,p] = x[2i+p], W6 = W zero-padded to 6 taps.  Why: cuDNN's heuristics pick an FFT-tiling algorithm
    for the FPN's 16->32 5x5/s2 layer at 272x480 (181 launches, 2.3 ms of the 4.9 ms FPN on B200,
    profiles/round1_fpn_layers.md); the regrouped 64->32 3x3 layer runs on its tensor-core path."""

    def __init__(self, conv, relu=True):
        super().__init__()
        assert conv.kernel_size == (5, 5) and conv.stride == (2, 2) and conv.padding == (2, 2) and conv.groups == 1
        w = conv.weight.detach()
        o, c = w.shape[:2]
        w6 = torch.zeros((o, c, 6, 6), dtype=w.dtype, device=w.device)
        w6[:, :, :5, :5] = w
        # channel order of the space-to-depth tensor: (py, px, c)
        w3 = w6.view(o, c, 3, 2, 3, 2).permute(0, 3, 5, 1, 2, 4).reshape(o, 4 * c, 3, 3)
        self.weight = nn.Parameter(w3.contiguous(), requires_grad=False)
        self.bias = None if conv.bias is None else nn.Parameter(conv.bias.detach().clone(), requires_grad=False)
        self.relu = relu

    def forward(self, x):
        N, C, H, W = x.shape
        if H % 2 or W % 2:
            raise ValueError("space-to-depth needs even H and W")
        z = x.permute(0, 2, 3, 1).reshape(N, H // 2, 2, W // 2, 2, C).permute(0, 1, 3, 2, 4, 5)
        z = z.reshape(N, H // 2, W // 2, 4 * C).permute(0, 3, 1, 2)          # NCHW view, channels-last memory
        return self.forward_s2d(z)

    def forward_s2d(self, z):
        """z: the space-to-depth tensor (N, 4C, H/2, W/2), channel order (py, px, c), channels-last memory."""
        if self.relu and self.bias is not None and z.is_cuda and not torch.is_grad_enabled():
            return torch.cudnn_convolution_relu(z, self.weight, self.bias, (1, 1), (1, 1), (1, 1), 1)
        y = torch.nn.functional.conv2d(z, self.weight, self.bias, stride=1, padding=1)
        return torch.relu_(y) if self.relu else y


def folded_copy(module, memory_format=None):
    """Deep copy of a FeatureNet / (Min)CostRegNet with every conv+BN pair folded."""
    m = copy.deepcopy(module).eval()
    with torch.no_grad():
        for mod in list(m.modules()):
            if isinstance(mod, _CBR) and isinstance(mod.bn, (nn.BatchNorm2d, nn.BatchNorm3d)):
                _fold_pair(mod.conv, mod.bn)
                mod.bn = nn.Identity()
            elif (isinstance(mod, nn.Sequential) and len(mod) == 2 and isinstance(mod[0], nn.ConvTranspose3d)
                  and isinstance(mod[1], nn.BatchNorm3d)):
                _fold_pair(mod[0], mod[1], transposed=True)
                mod[1] = nn.Identity()
        if memory_format == torch.channels_last:
            # FPN: regroup the stride-2 5x5 layers (after folding they are conv+bias followed by ReLU)
            for parent in list(m.modules()):
                for name, child in list(parent.named_children()):
                    if (isinstance(child, _CBR) and isinstance(child.conv, nn.Conv2d) and isinstance(child.bn, nn.Identity)
                            and child.conv.kernel_size == (5, 5) and child.conv.stride == (2, 2)):
                        setattr(parent, name, S2DConv5x5(child.conv, relu=True))
    if memory_format is not None:
        m = m.to(memory_format=memory_format)
    for p in m.parameters():
        p.requires_grad_(False)
    return m


class MergedHeadsCostReg(nn.Module):
    """(Min)CostRegNet forward with the two output heads evaluated as ONE 3x3x3 convolution.
    `feat_conv` (8->8) and `depth_conv` (8->1) read the same full-resolution tensor; stacking their
    weights into an 8->9 convolution reads it once (measured on B200: 0.50+0.50 ms -> one pass for
    cost_reg_1, 0.26+0.26 ms for cost_reg_0; profiles/round1_costreg_layers.md).  Same products and
    sums per output channel, so the result is unchanged."""

    # Full-resolution layers on libbmv's tensor-core kernel (csrc/conv3d_mma.cu) instead of cuDNN.  Its
    # fp16-operand / fp32-accumulate arithmetic is TF32-class, so it is used only where PyTorch itself
    # would run the convolution in TF32 (torch.backends.cudnn.allow_tf32, the default); strict-fp32
    # runs keep cuDNN's fp32 kernels.
    tensor_core_convs = True
    # Layers (by name) whose stride-1 convolution runs on the tcgen05 kernel (csrc/conv3d_umma.cu) when its input is
    # fp16: the merged heads (Cin 8) are ~1.7x faster there; the Cin-16 layers are not (profiles/round1l_tcgen05.md).
    umma_layers = ('heads',)
    # The layers that stay on cuDNN (conv3..conv7, <= 1/4 resolution) with fp16 activations and weights (fp32
    # accumulation) when the 3-level net is used: their input (conv2) and consumer (conv9T) are libbmv kernels that take
    # fp16 anyway.  Measured on B200: 144 -> 96 us for cost_reg_1, no gain for the 2-level cost_reg_0 (32 -> 31 us).
    lowres_half = True

    def __init__(self, net):
        super().__init__()
        self.net = net
        w = torch.cat([net.feat_conv[0].weight.detach(), net.depth_conv[0].weight.detach()], dim=0)
        self.heads = nn.Conv3d(8, 9, 3, padding=1, bias=False)
        self.heads.weight = nn.Parameter(w.contiguous(), requires_grad=False)
        self._packed = None

    def _use_tensor_core_convs(self, x):
        from .mlp_pack import CONV3D_K3_SHAPES
        return (self.tensor_core_convs and x.is_cuda and x.dtype in (torch.float32, torch.float16) and x.stride(1) == 1
                and torch.backends.cudnn.allow_tf32 and x.shape[1] in CONV3D_K3_SHAPES
                and isinstance(self.net.conv0.bn, nn.Identity))

    def _half_lowres(self):
        """fp16 copies of conv3..conv7 (folded), rebuilt with the plan (PlanCache keys on the parameter versions)."""
        if getattr(self, '_low16', None) is None:
            low = nn.Module()
            for name in ('conv3', 'conv4', 'conv5', 'conv6', 'conv7'):
                setattr(low, name, copy.deepcopy(getattr(self.net, name)).half())
            self._low16 = low
        return self._low16

    def _packed_weights(self, device):
        if self._packed is None or self._packed['device'] != device:
            from .mlp_pack import fp16_weight_scale, pack_conv3d_k3, pack_conv3d_k3_umma, pack_convT3d_k3s2
            n = self.net
            bias = lambda m: m.bias.detach().float().contiguous().to(device)
            # conv0 consumes the variance volume, whose magnitude follows the feature magnitude squared: its weights are
            # packed x 2^k (so that none of them falls into the fp16 subnormals) and the kernel divides by it
            ws0 = fp16_weight_scale(n.conv0.conv.weight)
            self._packed = {
                'device': device,
                'conv0': (pack_conv3d_k3(n.conv0.conv.weight, ws0).to(device), bias(n.conv0.conv)),
                'conv0_ws': ws0,
                'conv0_scale': torch.tensor([ws0, 1.0 / ws0], device=device),
                'conv1': (pack_conv3d_k3(n.conv1.conv.weight).to(device), bias(n.conv1.conv)),
                'conv2': (pack_conv3d_k3(n.conv2.conv.weight).to(device), bias(n.conv2.conv)),
                'conv9': (pack_convT3d_k3s2(n.conv9[0].weight).to(device), bias(n.conv9[0])),
                'conv11': (pack_convT3d_k3s2(n.conv11[0].weight).to(device), bias(n.conv11[0])),
                'heads': pack_conv3d_k3(self.heads.weight).to(device),
                'heads_umma': pack_conv3d_k3_umma(self.heads.weight).to(device),
            }
        return self._packed

    def input_weight_scale(self, device):
        """The power of two conv0's fp16 weights are packed with (ops.volume_scale(consumer_scale=...))."""
        return self._packed_weights(device)['conv0_ws']

    def forward(self, x, in_scale=None):
        """in_scale: ops.volume_scale(feats, consumer_scale=self.input_weight_scale(dev))[4:6] when x was stored
        pre-multiplied by a power of two (fp16 cost volume)."""
        n = self.net
        fast = self._use_tensor_core_convs(x)
        if in_scale is not None and not fast:
            raise RuntimeError("a range-scaled volume needs the tensor-core convolution path (conv0 undoes the scale)")
        if fast:
            from . import ops
            pk = self._packed_weights(x.device)
            # activations that only feed other fp16-operand libbmv kernels are stored as fp16 and staged by TMA
            h = torch.float16
            s0 = ops.conv3d_k3(x, *pk['conv0'], 8, relu=True, out_dtype=h,                  # ConvBnReLU3D(C, 8)
                               in_scale=in_scale if in_scale is not None else pk['conv0_scale'])
            s1 = ops.conv3d_k3(s0, *pk['conv1'], 16, relu=True, stride=2, out_dtype=h)   # ConvBnReLU3D(8, 16, stride=2)
            half_low = self.lowres_half and n.depth_levels == 3
            # ConvBnReLU3D(16, 16): fp32 where cuDNN's TF32 layers read it, fp16 when they run in fp16 too
            s1 = ops.conv3d_k3(s1, *pk['conv2'], 16, relu=True, out_dtype=h if half_low else torch.float32)
        else:
            half_low = False
            s0 = n.conv0(x)
            s1 = n.conv2(n.conv1(s0))
        low = self._half_lowres() if half_low else n
        s2 = low.conv4(low.conv3(s1))
        y = s2
        if n.depth_levels == 3:
            y = s2 + low.conv7(low.conv6(low.conv5(s2)))
        if fast and y.stride(1) == 1 and s1.stride(1) == 1:
            y = ops.convT3d_k3s2_add(y, *pk['conv9'], 16, skip=s1, out_dtype=torch.float16)
            # the full-resolution result only feeds the fp16-operand heads convolution: store it as fp16 (TMA-staged there)
            y = ops.convT3d_k3s2_add(y, *pk['conv11'], 8, skip=s0, out_dtype=torch.float16)
        else:
            y = s1 + n.conv9(y)
            y = s0 + n.conv11(y)
        if fast and y.stride(1) == 1:
            # feature volume and depth logits as two dense tensors (32-byte voxels for the trilinear fetch)
            logits = torch.empty((y.shape[0], 1) + tuple(y.shape[2:]), device=y.device)
            if 'heads' in self.umma_layers and y.dtype == torch.float16 and y.stride(4) == y.shape[1]:
                feat = ops.conv3d_k3(y, pk['heads_umma'], None, 9, relu=False, out2=logits, split=8, engine='umma')
            else:
                feat = ops.conv3d_k3(y, pk['heads'], None, 9, relu=False, out2=logits, split=8)
            return feat, logits[:, 0]
        out = self.heads(y)
        feat = out[:, :8]
        if out.stride(1) == 1:       # channels-last: 32-byte voxels (what the one-launch render kernel fetches from)
            feat = feat.contiguous(memory_format=torch.channels_last_3d)
        return feat, out[:, 8]


class FusedTopDownFPN(nn.Module):
    """FeatureNet forward with each `_upsample_add(x, lat(c))` step done by one libbmv launch
    (csrc/fpn.cu).  Wraps a folded, channels-last FeatureNet copy; CUDA only."""

    # With TF32-class convolutions allowed (torch.backends.cudnn.allow_tf32, the default) each top-down
    # step AND its smoothing 3x3 convolution run as one launch (csrc/fpn_fused.cu): the 32-channel
    # full-resolution tensor never reaches HBM.
    fused_smooth = True
    # emit the half-resolution features (read only by the level-1 cost volumes) in fp16 instead of fp32: 8-byte taps in
    # K1 (288 -> 263 us on B200), but this kernel's epilogue then stores 4 bytes per lane (half sectors) and gets 22 us
    # slower (an additional copy next to the fp32 maps: +26 us) — net zero on the frame, so it is off by default.
    emit_half_features = False
    # Run the two top-down + smoothing launches (0.47 ms at C2, bound by the L1 data pipe) on a side stream: they only
    # produce the level-1 / level-2 maps, which the frame needs after the level-0 cost-volume chain / at the render, so
    # they overlap the level-0 chain (K1 + 3-D CNN, tensor- and latency-bound).  `ready` then maps 'level_1' / 'level_2'
    # to the events the consumer must wait for (network.StreamedFeats does); None when nothing was deferred.
    side_topdown = False
    # conv1.x, conv2.x and the top layer on libbmv's tensor-core kernel (csrc/conv2d_mma.cu) instead of cuDNN: four
    # launches instead of seven (the 5x5 / stride-2 layers read their input through space-to-depth in the staging loop,
    # the 1x1 top layer runs in conv2.1's epilogue), fp16 intermediates between them.  TF32-class like the rest.
    tensor_core_mid = True
    # {'level_1': consumer_scale}: the caller wants the fp16 cost volume's range scale of that level (ops.volume_scale)
    # computed right behind the launch that produces the level — on the side stream when the top-down steps run there,
    # i.e. under the level-0 chain instead of in front of the level-1 cost volumes (13 us at C2).  Results in `scales`.
    scale_requests = None

    def __init__(self, fpn):
        super().__init__()
        self.fpn = fpn
        self._packed = None
        self._mid = None
        self._side = None
        self.ready = None
        self.scales = {}

    def _scale_buf(self, level, device):
        """Persistent 6-float result / scratch buffer of ops.volume_scale for one level (zeroed once)."""
        bufs = self.__dict__.setdefault('_scale_bufs', {})
        key = (level, device)
        if key not in bufs:
            bufs[key] = torch.zeros(6, device=device)
        return bufs[key]

    def _mid_weights(self, device):
        if self._mid is None or self._mid['device'] != device:
            from .mlp_pack import pack_conv1x1_after, pack_conv2d_k3
            f = self.fpn
            b = lambda m: m.bias.detach().float().contiguous().to(device)
            self._mid = {
                'device': device,
                'c10': (pack_conv2d_k3(f.conv1[0].weight).to(device), b(f.conv1[0])),
                'c11': (pack_conv2d_k3(f.conv1[1].conv.weight).to(device), b(f.conv1[1].conv)),
                'c20': (pack_conv2d_k3(f.conv2[0].weight).to(device), b(f.conv2[0])),
                'c21': (pack_conv2d_k3(f.conv2[1].conv.weight).to(device), b(f.conv2[1].conv)),
                'top': (pack_conv1x1_after(f.toplayer.weight).to(device), b(f.toplayer)),
            }
        return self._mid

    def _mid_ok(self, x):
        f = self.fpn
        return (self.tensor_core_mid and x.shape[-1] % 4 == 0 and x.shape[-2] % 4 == 0
                and isinstance(f.conv1[0], S2DConv5x5) and isinstance(f.conv2[0], S2DConv5x5)
                and f.conv1[0].relu and f.conv2[0].relu and f.conv1[0].bias is not None and f.conv2[0].bias is not None
                and isinstance(f.conv1[1].bn, nn.Identity) and isinstance(f.conv2[1].bn, nn.Identity)
                and f.conv1[1].conv.bias is not None and f.conv2[1].conv.bias is not None
                and tuple(f.conv1[0].weight.shape) == (16, 32, 3, 3) and tuple(f.conv2[0].weight.shape) == (32, 64, 3, 3)
                and tuple(f.toplayer.weight.shape[:2]) == (32, 32) and f.toplayer.bias is not None)

    def _smooth_weights(self, device):
        if self._packed is None or self._packed[0].device != device:
            from .mlp_pack import pack_conv2d_k3_c32, pack_conv2d_k3_c8
            self._packed = (pack_conv2d_k3_c32(self.fpn.smooth1.weight).to(device),
                            pack_conv2d_k3_c32(self.fpn.smooth0.weight).to(device),
                            pack_conv2d_k3_c8(self.fpn.conv0[1].conv.weight).to(device))
        return self._packed

    def forward(self, x):
        from . import ops
        f = self.fpn
        fused = self.fused_smooth and torch.backends.cudnn.allow_tf32
        self.rgb_nhwc4 = None
        quarter = None
        if fused and isinstance(f.conv0[0].bn, nn.Identity):
            a, b = f.conv0[0].conv, f.conv0[1].conv      # the stem reads x with any strides: no layout copy
            if self._mid_ok(x):
                # every tensor between the stem and the top layer is an MMA operand of its consumers (conv1.0 / conv2.0, the
                # 1x1 laterals of the top-down steps): stored as fp16 = the rounding those consumers apply anyway
                h = torch.float16
                c0, self.rgb_nhwc4 = ops.fpn_stem(x, a.weight, a.bias, self._smooth_weights(x.device)[2], b.bias, want_rgb4=True,
                                                  out_dtype=h)
                mw = self._mid_weights(x.device)
                c1 = ops.conv2d_k3(c0, *mw['c10'], 16, relu=True, s2d=True, out_dtype=h)          # conv1.0: 5x5 / stride 2
                c1 = ops.conv2d_k3(c1, *mw['c11'], 16, relu=True, out_dtype=h)                     # conv1.1 (also read by lat1)
                c2 = ops.conv2d_k3(c1, *mw['c20'], 32, relu=True, s2d=True, out_dtype=h)          # conv2.0: 5x5 / stride 2
                quarter = ops.conv2d_k3(c2, *mw['c21'], 32, relu=True, wfrag1x1=mw['top'][0], bias1x1=mw['top'][1])   # conv2.1 + toplayer
            else:
                want_s2d = isinstance(f.conv1[0], S2DConv5x5) and x.shape[-1] % 2 == 0 and x.shape[-2] % 2 == 0
                if want_s2d:
                    c0, self.rgb_nhwc4, z0 = ops.fpn_stem(x, a.weight, a.bias, self._smooth_weights(x.device)[2], b.bias,
                                                          want_rgb4=True, want_s2d=True)
                    c1 = f.conv1[1](f.conv1[0].forward_s2d(z0))
                else:
                    c0, self.rgb_nhwc4 = ops.fpn_stem(x, a.weight, a.bias, self._smooth_weights(x.device)[2], b.bias, want_rgb4=True)
                    c1 = f.conv1(c0)
        else:
            c0 = f.conv0(x.contiguous(memory_format=torch.channels_last))
            c1 = f.conv1(c0)
        if quarter is None:
            c2 = f.conv2(c1)
            quarter = f.toplayer(c2)
        self.ready = None
        self.scales = {}
        if fused:
            w1, w0, _ = self._smooth_weights(x.device)

            def topdown():
                if self.emit_half_features:
                    half, feat1 = ops.fpn_topdown_smooth(quarter, c1, f.lat1.weight, f.lat1.bias, w1, f.smooth1.bias, 16, True, want_half='only')
                else:
                    half, feat1 = ops.fpn_topdown_smooth(quarter, c1, f.lat1.weight, f.lat1.bias, w1, f.smooth1.bias, 16, True)
                if self.scale_requests and 'level_1' in self.scale_requests:
                    self.scales['level_1'] = ops.volume_scale(feat1, consumer_scale=self.scale_requests['level_1'],
                                                              out=self._scale_buf('level_1', feat1.device))
                ev1 = torch.cuda.current_stream().record_event() if self.side_topdown else None
                _, feat0 = ops.fpn_topdown_smooth(half, c0, f.lat0.weight, f.lat0.bias, w0, f.smooth0.bias, 8, False)
                ev0 = torch.cuda.current_stream().record_event() if self.side_topdown else None
                return feat1, feat0, ev1, ev0
            if not self.side_topdown:
                feat1, feat0, _, _ = topdown()
                return quarter, feat1, feat0
            main = torch.cuda.current_stream()
            if self._side is None or self._side.device != x.device:
                self._side = torch.cuda.Stream(device=x.device)
            self._side.wait_stream(main)                   # fork: quarter, c1, c0 are complete on `main` up to here
            with torch.cuda.stream(self._side):
                feat1, feat0, ev1, ev0 = topdown()
            for t in (quarter, c1, c0):                    # caching allocator: these blocks are still read by the side stream
                t.record_stream(self._side)
            for t in (feat1, feat0) + tuple(self.scales.values()):     # ... and these are consumed on `main`
                if torch.is_tensor(t):
                    t.record_stream(main)
            self.ready = {'level_1': ev1, 'level_2': ev0}
            return quarter, feat1, feat0
        half = ops.fpn_topdown(quarter, c1, f.lat1.weight, f.lat1.bias)
        full = ops.fpn_topdown(half, c0, f.lat0.weight, f.lat0.bias)
        return quarter, f.smooth1(half), f.smooth0(full)


class PlanCache:
    """name -> folded copy, invalidated by parameter/buffer version counters."""

    def __init__(self):
        self._c = {}

    @staticmethod
    def _key(module):
        return tuple((t.data_ptr(), t._version) for t in list(module.parameters()) + list(module.buffers()))

    def get(self, name, module, memory_format):
        key = (self._key(module), memory_format)
        hit = self._c.get(name)
        if hit is None or hit[0] != key:
            plan = folded_copy(module, memory_format)
            from .modules import CostRegNet, FeatureNet
            if isinstance(module, CostRegNet):
                plan = MergedHeadsCostReg(plan)
                if memory_format is not None:
                    plan = plan.to(memory_format=memory_format)
            if isinstance(module, FeatureNet) and memory_format == torch.channels_last and \
                    next(module.parameters()).is_cuda:
                plan = FusedTopDownFPN(plan)
            self._c[name] = (key, plan)
        return self._c[name][1]
