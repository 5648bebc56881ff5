"""
Inference-only execution plan for DeepLabv3+/ResNet-101 (pylc_b200.models.deeplab.DeepLab).

The network stays on stock PyTorch / cuDNN tensor-core kernels (north_star).  What this module
removes is the memory-bound glue around the convolutions that eval-mode inference does not need:

  * every BatchNorm is folded into the preceding convolution's weight and bias
    (w' = w * g / sqrt(var + eps), b' = beta - mean * g / sqrt(var + eps)) -- exact in real
    arithmetic, ~1e-6 relative in fp32;
  * conv + bias + ReLU and conv + bias + residual-add + ReLU run as single cuDNN fused calls
    (torch.cudnn_convolution_relu / torch.cudnn_convolution_add_relu), so the [B,C,H,W]
    activations are written once instead of being re-read and re-written by separate BN, add and
    ReLU kernels (about a third of the unfused network's HBM traffic at 512 x 512 tiles);
  * dropout layers (identity in eval mode) are dropped;
  * the three HBM-bound steps between the convolutions -- the stem's 3x3/2 max-pool, the decoder's
    bilinear up-sample + channel concat, and the final x4 bilinear up-sample (emitted directly as
    planar logits for the stitch kernel) -- run as pylc_b200 kernels (csrc/netglue.cu) on the
    channels-last activations: the stock kernels reach 10-30 % of HBM speed on these layouts
    (2.6 ms of a 21.8 ms image), ours are one streaming pass each.

`FusedDeepLab(net)` snapshots the weights of `net`; call `refresh()` after loading a new
state_dict.  Outputs match `net.eval()(x)` to fp32 rounding of the folded weights, not bit for
bit, so the pipeline uses it only when asked (`TiledSegmenter(fuse_network=True)`); parity tests of
the custom kernels never depend on it.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops


def fold_conv_bn(conv, bn):
    """(weight', bias') of conv followed by eval-mode batch-norm."""
    w = conv.weight.detach().double()
    b = conv.bias.detach().double() if conv.bias is not None else torch.zeros(w.shape[0], dtype=torch.float64, device=w.device)
    if bn is None:
        return w.float(), b.float()
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    w = w * scale[:, None, None, None]
    b = (b - bn.running_mean.detach().double()) * scale + bn.bias.detach().double()
    return w.float(), b.float()


# Library routes of a convolution with a ReLU; the plan picks one from the layer's geometry (`_Conv._route`):
#   0  torch.cudnn_convolution_relu / _add_relu: one fused cuDNN call, engine chosen by cuDNN's heuristic
#   1  F.conv2d (engine chosen by torch.backends.cudnn.benchmark when that is on) + in-place add / ReLU: only the
#      convolutions without a ReLU (`_Conv._plain`)
#   2  tap split (3x3, stride 1, padding == dilation >= 6 only): the convolution as nine cuBLAS GEMMs over the flat
#      pixel ranges that do not fall into the zero padding, summed by pylc_tap_combine_relu_f32 (`_Conv._tap_split`)
# Measured on B200 (tools/exp/dilated_conv.py, 45 tiles): cuDNN has an sm100 kernel for the ASPP branches with
# dilation 6 and 12 (0.54 ms) but none for dilation 18 on a 32 x 32 map -- routes 0 and 1, NHWC or NCHW, padded
# by hand or not, all land on `sm80_xmma_fprop_implicit_gemm_tf32...` (1.73 ms) plus two layout conversions
# (0.2 ms): 10 % of the whole network.  With dilation 18 > 32 / 2 every output pixel sees at most two taps per
# axis, i.e. 39 % of the dense products; route 2 computes 62 % (whole flat runs, so that no window is ever copied),
# on the TF32 tensor cores through cuBLAS.
# The route is fixed by geometry, not timed at run time: where two routes take about as long, timing picks
# differently from process to process, their TF32 sums round differently, and so the same input would give
# different near-tied labels from run to run.


class _Conv(object):
    """One folded convolution with an optional fused ReLU / residual add."""
    __slots__ = ("w", "b", "stride", "padding", "dilation", "relu", "taps")

    def __init__(self, conv, bn, relu, channels_last):
        w, b = fold_conv_bn(conv, bn)
        self.w = w.contiguous(memory_format=torch.channels_last) if channels_last else w.contiguous()
        self.b = b.contiguous()
        self.stride, self.padding, self.dilation, self.relu = conv.stride, conv.padding, conv.dilation, relu
        self.taps = None

    def to(self, dtype):
        self.w = self.w.to(dtype)
        self.b = self.b.to(dtype) if self.b is not None else None
        self.taps = None
        return self

    def _tap_split_applies(self, x, residual):
        d = self.dilation[0]
        return (residual is None and self.relu and self.b is not None and x.dtype == torch.float32 and x.is_cuda
                and tuple(self.w.shape[2:]) == (3, 3) and self.w.shape[0] % 4 == 0
                and tuple(self.stride) == (1, 1) and tuple(self.dilation) == (d, d) and tuple(self.padding) == (d, d) and d >= 6
                and d < min(x.shape[2], x.shape[3]) and x.is_contiguous(memory_format=torch.channels_last))

    def _tap_split(self, x, residual=None):
        """3x3 convolution with padding == dilation == d as GEMMs over the tap windows that miss the zero padding.
        out[y, x] = sum_t W_t . in[y + ty*d, x + tx*d].  In the channels-last activation ([B, H*W, C] as flat
        pixels) tap t reads the pixels of the output shifted by s_t = ty*d*W + tx*d, so its product for the flat
        output range [max(0,-s_t), H*W - max(0,s_t)) is ONE strided-batch cuBLAS GEMM on a view -- no copy, no
        transpose.  Rows whose source wrapped into the neighbouring image row (tx != 0) are computed and then
        masked by pylc_tap_combine_relu_f32, which adds the eight tap products to the centre tap's, applies the
        ReLU and writes the result in one streaming pass.  Dilation 18 on 32 x 32: 62 % of the dense products.
        TF32 products, fp32 accumulation -- the library convolution's numerics, summed in another order."""
        B, C, H, W = x.shape
        d, O = self.dilation[0], self.w.shape[0]
        if self.taps is None:                                            # [3, 3, C, O]: one [C, O] matrix per tap
            self.taps = self.w.permute(2, 3, 1, 0).contiguous()
        wt = self.taps
        HW = H * W
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32      # the convolution's own precision class
        try:
            xf = x.permute(0, 2, 3, 1).reshape(B, HW, C)                 # the channels-last storage itself
            out = torch.addmm(self.b, xf.reshape(B * HW, C), wt[1, 1]).view(B, H, W, O)
            taps = []
            for ky in range(3):
                for kx in range(3):
                    if ky == 1 and kx == 1:
                        continue
                    dy, dx = (ky - 1) * d, (kx - 1) * d
                    s_ = dy * W + dx
                    p0, p1 = max(0, -s_), HW - max(0, s_)
                    if p1 <= p0 or abs(dy) >= H or abs(dx) >= W:
                        continue
                    z = torch.bmm(xf[:, p0 + s_:p1 + s_], wt[ky, kx].expand(B, C, O))
                    taps.append((z, p0, dy, dx))
            ops.tap_combine_relu_(out, taps)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        return out.permute(0, 3, 1, 2)                                   # [B, O, H, W], channels-last strides

    def _fused(self, x, residual):
        if residual is not None:
            return torch.cudnn_convolution_add_relu(x, self.w, residual, 1.0, self.b, self.stride, self.padding,
                                                    self.dilation, 1)
        return torch.cudnn_convolution_relu(x, self.w, self.b, self.stride, self.padding, self.dilation, 1)

    def _plain(self, x, residual):
        y = F.conv2d(x, self.w, self.b, self.stride, self.padding, self.dilation)
        if residual is not None:
            y.add_(residual)
        return y.relu_() if self.relu else y

    def _route(self, x, residual):
        """Route 2 (tap split) where the dilation exceeds half the map, so that at most two taps per axis reach any
        output pixel and cuDNN's dense kernel would do more than twice the products (dilation 18 on the 32 x 32
        ASPP input); route 0 (one fused cuDNN call) everywhere else."""
        if self._tap_split_applies(x, residual) and 2 * self.dilation[0] > min(x.shape[2], x.shape[3]):
            return self._tap_split
        return self._fused

    def __call__(self, x, residual=None):
        if x.is_cuda and self.relu:
            return self._route(x, residual)(x, residual)
        return self._plain(x, residual)


class FusedDeepLab(object):
    def __init__(self, net, channels_last=True, dtype=None, glue=True):
        self.net = net
        self.channels_last = channels_last
        self.dtype = dtype
        # the HBM-bound steps between the convolutions (stem max-pool, decoder up-sample + concat, final
        # up-sample) run as pylc_b200 kernels on channels-last f32 activations; eager ops otherwise
        self.glue = glue and channels_last and dtype is None
        self.refresh()

    def refresh(self):
        net, cl = self.net, self.channels_last
        if any(not isinstance(m, nn.BatchNorm2d) for m in (net.backbone.bn1, net.aspp.bn1, net.decoder.bn1)):
            raise ValueError("FusedDeepLab folds BatchNorm2d only")
        mk = lambda conv, bn, relu: self._cast(_Conv(conv, bn, relu, cl))  # noqa: E731
        bb = net.backbone
        self.stem = mk(bb.conv1, bb.bn1, True)
        self.stem_s2d = self._make_s2d_stem(bb.conv1, self.stem) if self.glue else None
        self.blocks = []
        for layer in (bb.layer1, bb.layer2, bb.layer3, bb.layer4):
            stage = []
            for blk in layer:
                c3 = mk(blk.conv3, blk.bn3, True)
                down = None
                if blk.downsample is not None:
                    # the projection's bias moves into conv3's (the two are summed before the ReLU), so
                    # the projection runs as a bias-free convolution with no separate add kernel
                    down = mk(blk.downsample[0], blk.downsample[1], False)
                    c3.b = (c3.b + down.b).contiguous()
                    down.b = None
                stage.append((mk(blk.conv1, blk.bn1, True), mk(blk.conv2, blk.bn2, True), c3, down))
            self.blocks.append(stage)
        a = net.aspp
        self.aspp = [mk(m.atrous_conv, m.bn, True) for m in (a.aspp1, a.aspp2, a.aspp3, a.aspp4)]
        self.aspp_pool = mk(a.global_avg_pool[1], a.global_avg_pool[2], True)
        self.aspp_out = mk(a.conv1, a.bn1, True)
        self._aspp_fold = None
        d = net.decoder
        self.dec_low = mk(d.conv1, d.bn1, True)
        self.dec1 = mk(d.last_conv[0], d.last_conv[1], True)
        self.dec2 = mk(d.last_conv[4], d.last_conv[5], True)
        self.dec_out = mk(d.last_conv[8], None, False)
        return self

    @staticmethod
    def _make_s2d_stem(conv1, stem):
        """The 7x7 stride-2 pad-3 stem over 3 channels as a 4x4 stride-1 convolution over the 2x2
        space-to-depth image (ops.tile_gather_norm_s2d's layout): zero-extend the (BN-folded) kernel to
        8x8 (one zero row/column in front), then w4[o, (py*2+px)*3+c, U, V] = w8[o, c, 2U+py, 2V+px];
        input channels 12..15 carry zero weights.  Same products and sums as the 7x7 form."""
        if tuple(conv1.kernel_size) != (7, 7) or tuple(conv1.stride) != (2, 2) or tuple(conv1.padding) != (3, 3) \
                or conv1.in_channels != 3:
            return None
        w7 = stem.w.contiguous().float()                                    # [O, 3, 7, 7] folded weights
        O = w7.shape[0]
        w8 = torch.zeros((O, 3, 8, 8), dtype=w7.dtype, device=w7.device)
        w8[:, :, 1:, 1:] = w7
        w4 = torch.zeros((O, 16, 4, 4), dtype=w7.dtype, device=w7.device)
        for py in range(2):
            for px in range(2):
                w4[:, (py * 2 + px) * 3:(py * 2 + px) * 3 + 3] = w8[:, :, py::2, px::2]
        s = _Conv.__new__(_Conv)
        s.w = w4.contiguous(memory_format=torch.channels_last)
        s.b, s.stride, s.padding, s.dilation, s.relu, s.taps = stem.b, (1, 1), (0, 0), (1, 1), True, None
        return s

    def _aspp_out_folded(self, cat4, pooled):
        """ASPP's 1x1 projection (reference aspp.py:88-100: conv1 over the concatenation of the four atrous
        branches and the up-sampled image-pooling branch) without materialising the pooled branch: a bilinear
        up-sample of a 1x1 map (align_corners=True) is that pixel everywhere, so its share of the projection is one
        vector per image, W_p . pooled[b] + bias, added to the projection of the other four branches:
            relu(W_a . cat4[b, :, y, x] + (W_p . pooled[b] + bias))
        One strided-batch TF32 GEMM on the channels-last concatenation (the vector enters as its beta = 1 operand)
        and an in-place ReLU; the up-sample kernel, a fifth of the concat and a fifth of the projection's K go."""
        B, K, H, W = cat4.shape
        conv = self.aspp_out
        O = conv.w.shape[0]
        if self._aspp_fold is None:
            w = conv.w.reshape(O, -1)                                    # [O, 1280] folded 1x1 weights
            self._aspp_fold = (w[:, :K].t().contiguous(), w[:, K:].t().contiguous())
        wa, wp = self._aspp_fold
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32
        try:
            v = torch.addmm(conv.b, pooled.reshape(B, -1), wp)           # [B, O]
            out = torch.baddbmm(v.unsqueeze(1), cat4.permute(0, 2, 3, 1).reshape(B, H * W, K), wa.expand(B, K, O))
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        return out.relu_().view(B, H, W, O).permute(0, 3, 1, 2)

    def _cast(self, conv):
        return conv.to(self.dtype) if self.dtype is not None else conv

    def features(self, x, s2d=False):
        """Decoder output [B, n_classes, H/4, W/4] (before the final x4 bilinear up-sample).
        s2d: `x` is the space-to-depth stem input [B, 16, H/2+3, W/2+3] of ops.tile_gather_norm_s2d."""
        if self.dtype is not None:
            x = x.to(self.dtype)
        if self.channels_last:
            x = x.contiguous(memory_format=torch.channels_last)
        glue = self.glue and x.is_cuda and x.dtype == torch.float32
        x = self.stem_s2d(x) if s2d else self.stem(x)
        x = ops.maxpool3x3s2_nhwc(x) if glue else F.max_pool2d(x, 3, stride=2, padding=1)
        low = None
        for si, stage in enumerate(self.blocks):
            for c1, c2, c3, down in stage:
                skip = x if down is None else down(x)
                x = c3(c2(c1(x)), residual=skip)
            if si == 0:
                low = x
        pooled = self.aspp_pool(F.adaptive_avg_pool2d(x, 1))
        if glue:
            x = self._aspp_out_folded(torch.cat([br(x) for br in self.aspp], dim=1), pooled)
        else:
            pooled = F.interpolate(pooled, size=x.shape[2:], mode='bilinear', align_corners=True)
            x = self.aspp_out(torch.cat([br(x) for br in self.aspp] + [pooled], dim=1))
        low = self.dec_low(low)
        if glue:      # up-sample + concat in one pass (one write of the [B,304,H/4,W/4] tensor, nothing else)
            x = ops.upsample_concat_nhwc(x, low)
        else:
            x = torch.cat((F.interpolate(x, size=low.shape[2:], mode='bilinear', align_corners=True), low), dim=1)
        return self.dec_out(self.dec2(self.dec1(x)))

    @torch.no_grad()
    def decoder_s2d(self, xs):
        """The decoder's output [B, n_classes, T/4, T/4] (channels-last f32) from space-to-depth tiles: the
        network WITHOUT its final x4 bilinear up-sample, which ops.stitch_upsample_argmax_colour evaluates."""
        if self.stem_s2d is None:
            raise ValueError("space-to-depth stem unavailable for this network / plan")
        return self.features(xs, s2d=True).float().contiguous(memory_format=torch.channels_last)

    @torch.no_grad()
    def decoder(self, x):
        return self.features(x).float().contiguous(memory_format=torch.channels_last)

    @torch.no_grad()
    def forward_s2d(self, xs):
        """Logits [B, n_classes, T, T] from space-to-depth tiles (T = 2 * (xs.shape[2] - 3))."""
        if self.stem_s2d is None:
            raise ValueError("space-to-depth stem unavailable for this network / plan")
        y = self.features(xs, s2d=True).float()
        size = (2 * (xs.shape[2] - 3), 2 * (xs.shape[3] - 3))
        return ops.upsample_nhwc_to_nchw(y, size)

    @torch.no_grad()
    def __call__(self, x):
        y = self.features(x).float()
        if self.glue and y.is_cuda and y.is_contiguous(memory_format=torch.channels_last):
            return ops.upsample_nhwc_to_nchw(y, x.shape[2:])      # planar logits straight from the NHWC decoder output
        y = y.contiguous()                                   # small [B,C,H/4,W/4]: make it NCHW here ...
        return F.interpolate(y, size=x.shape[2:], mode='bilinear', align_corners=True)   # ... so the logits are NCHW
