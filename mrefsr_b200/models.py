"""The MRefSR network around the hot path ("next" row of SURVEY.md section 8f: the callers either side).

Mirrors, with identical module / parameter names (so reference checkpoints load):
  * ContrasMultiExtractorSep      basicsr/archs/contras_multi_extractor_arch.py:10-64   (VGG16 -> conv3_1)
  * MRAPARestorationNet           basicsr/archs/ref_mrapa_restoration_arch.py:79-259
    (ContentExtractor, DynamicAggregationRestoration with DynAgg x3 and MRAPAFusion x3)
and `MRefSRPipeline`, the inference flow of MultiRefRestorationModel.test()
(basicsr/models/multi_ref_restoration_model.py:281-294) with the Python loops over references and batch items
replaced by batched calls: one matcher launch for all B*R pairs, the R references of a scale stacked into the batch
dimension of the offset convolutions and of ONE fused DynAgg launch (offsets / masks / pre-offsets assembled in the
DCN gather), one fusion launch per scale.  The plain convolutions stay cuDNN library calls.
"""
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn import init

from .archs import CorrespondenceGenerationArch
from .dynagg import DynAgg
from . import trunk as T
from .fusion import MRAPAFusion
from .matcher import feature_match_index_batched, pre_offsets

_VGG16_TO_CONV3_1 = [('conv1_1', (3, 64)), ('relu1_1', None), ('conv1_2', (64, 64)), ('relu1_2', None), ('pool1', 'M'),
                     ('conv2_1', (64, 128)), ('relu2_1', None), ('conv2_2', (128, 128)), ('relu2_2', None),
                     ('pool2', 'M'), ('conv3_1', (128, 256))]


@torch.no_grad()
def default_init_weights(module_list, scale=1, bias_fill=0, **kwargs):
    """arch_util.py:43-70 (conv / linear branch)."""
    if not isinstance(module_list, list):
        module_list = [module_list]
    for module in module_list:
        for m in module.modules():
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                init.kaiming_normal_(m.weight, **kwargs)
                m.weight.data *= scale
                if m.bias is not None:
                    m.bias.data.fill_(bias_fill)


def srntt_init_weights(net, init_gain=0.02):
    """arch_util.py:18-40 with init_type='normal'."""
    def init_func(m):
        name = m.__class__.__name__
        if hasattr(m, 'weight') and ('Conv' in name or 'Linear' in name):
            init.normal_(m.weight.data, 0.0, init_gain)
            if hasattr(m, 'bias') and m.bias is not None:
                init.constant_(m.bias.data, 0.0)
    net.apply(init_func)


def _lib_supports(t):
    """channel count of a channels-last fp32 / bf16 activation served by the fused training epilogue"""
    from . import _lib
    return bool(_lib.lib().mrefsr_bias_act_train_supported(t.shape[1], 1 if t.dtype == torch.bfloat16 else 0))


def make_layer(basic_block, num_basic_block, **kwarg):
    return nn.Sequential(*[basic_block(**kwarg) for _ in range(num_basic_block)])


class ResidualBlockNoBN(nn.Module):
    """arch_util.py:88-117."""

    def __init__(self, num_feat=64, res_scale=1, pytorch_init=False):
        super().__init__()
        self.res_scale = res_scale
        self.conv1 = nn.Conv2d(num_feat, num_feat, 3, 1, 1, bias=True)
        self.conv2 = nn.Conv2d(num_feat, num_feat, 3, 1, 1, bias=True)
        self.relu = nn.ReLU(inplace=True)
        if not pytorch_init:
            default_init_weights([self.conv1, self.conv2], 0.1)

    def forward(self, x):
        if T.fast_ok(x):    # inference: conv -> [bias + ReLU] -> conv -> [bias, * res_scale, + x], two epilogue passes
            t = T.conv_bias_act(x, self.conv1, T.ACT_LEAKY, 0.0)
            return T.conv_bias_act(t, self.conv2, T.ACT_NONE, residual=x, scale=self.res_scale)
        if T.train_ok(x):   # training: bias / ReLU / residual epilogues and their backward (+ bias gradients) fused
            t = T.conv_bias_act_train(x, self.conv1, T.ACT_LEAKY, 0.0)
            if t is not None:
                out = T.conv_bias_act_train(t, self.conv2, T.ACT_NONE, residual=x, scale=self.res_scale)
                if out is not None:
                    return out
        return x + self.conv2(self.relu(self.conv1(x))) * self.res_scale


class ContrasExtractorLayer(nn.Module):
    """VGG16 features up to conv3_1 (no ReLU after it), parameters under `model.<layer>`."""

    def __init__(self):
        super().__init__()
        layers = OrderedDict()
        for name, spec in _VGG16_TO_CONV3_1:
            if spec is None:
                layers[name] = nn.ReLU(inplace=True)
            elif spec == 'M':
                layers[name] = nn.MaxPool2d(kernel_size=2, stride=2)
            else:
                layers[name] = nn.Conv2d(spec[0], spec[1], 3, padding=1)
        self.model = nn.Sequential(layers)
        self.register_buffer('mean', torch.Tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1))
        self.register_buffer('std', torch.Tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1))

    def forward(self, batch):
        x = (batch - self.mean) / self.std
        if T.fast_ok(x):
            return T.run_sequential(self.model, x)
        return self.model(x)


class ContrasMultiExtractorSep(nn.Module):
    """Same forward contract as the reference (list of {'dense_features1','dense_features2'} dicts) plus
    `forward_batched` which runs all references through the second tower in one call."""

    def __init__(self):
        super().__init__()
        self.feature_extraction_image1 = ContrasExtractorLayer()
        self.feature_extraction_image2 = ContrasExtractorLayer()

    def forward(self, image1, image_list):
        f1 = self.feature_extraction_image1(image1)
        return [{'dense_features1': f1, 'dense_features2': self.feature_extraction_image2(im)} for im in image_list]

    def forward_batched(self, image1, refs):
        """image1 [B,3,H,W], refs [B,R,3,H,W] -> (f1 [B,256,h,w], f2 [B*R,256,h,w])."""
        return self.feature_extraction_image1(image1), self.feature_extraction_image2(refs.flatten(0, 1))


class ContentExtractor(nn.Module):
    def __init__(self, in_nc=3, out_nc=3, nf=64, n_blocks=16):
        super().__init__()
        self.conv_first = nn.Conv2d(in_nc, nf, 3, 1, 1)
        self.body = make_layer(ResidualBlockNoBN, n_blocks, num_feat=nf)
        self.lrelu = nn.LeakyReLU(negative_slope=0.1, inplace=True)
        default_init_weights([self.conv_first], 0.1)

    def forward(self, x):
        if T.fast_ok(x):
            return self.body(T.conv_bias_act(x, self.conv_first, T.ACT_LEAKY, 0.1))
        if T.train_ok(x):
            t = T.conv_bias_act_train(x, self.conv_first, T.ACT_LEAKY, 0.1)
            if t is not None:
                return self.body(t)
        return self.body(self.lrelu(self.conv_first(x)))


class DynamicAggregationRestoration(nn.Module):
    """ref_mrapa_restoration_arch.py:140-259, same attribute names."""

    def __init__(self, ngf=64, n_blocks=16, groups=8):
        super().__init__()
        for name, c in (('small', 256), ('medium', 128), ('large', 64)):
            setattr(self, f'{name}_offset_conv1', nn.Conv2d(ngf + c, c, 3, 1, 1, bias=True))
            setattr(self, f'{name}_offset_conv2', nn.Conv2d(c, c, 3, 1, 1, bias=True))
            setattr(self, f'{name}_dyn_agg', DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=groups,
                                                     extra_offset_mask=True))
            setattr(self, f'head_{name}', MRAPAFusion(nf=ngf, ref_nf=c))
            setattr(self, f'body_{name}', make_layer(ResidualBlockNoBN, n_blocks, num_feat=ngf))
        self.tail_small = nn.Sequential(nn.Conv2d(ngf, ngf * 4, 3, 1, 1), nn.PixelShuffle(2), nn.LeakyReLU(0.1, True))
        self.tail_medium = nn.Sequential(nn.Conv2d(ngf, ngf * 4, 3, 1, 1), nn.PixelShuffle(2), nn.LeakyReLU(0.1, True))
        self.tail_large = nn.Sequential(nn.Conv2d(ngf, ngf // 2, 3, 1, 1), nn.LeakyReLU(0.1, True),
                                        nn.Conv2d(ngf // 2, 3, 3, 1, 1))
        self.lrelu = nn.LeakyReLU(negative_slope=0.1, inplace=True)

    _SCALES = (('small', 'relu3_1'), ('medium', 'relu2_1'), ('large', 'relu1_1'))

    def _split_conv1(self, conv, n_x, channels_last):
        """(weight[:, :n_x], weight[:, n_x:]) of an offset_conv1 as dense tensors, cached until the weight changes."""
        cache = self.__dict__.setdefault('_conv1_split', {})
        key = id(conv)
        ver = (conv.weight._version, conv.weight.data_ptr(), channels_last)
        if key not in cache or cache[key][0] != ver:
            fmt = torch.channels_last if channels_last else torch.contiguous_format
            w = conv.weight.detach()
            cache[key] = (ver, w[:, :n_x].contiguous(memory_format=fmt), w[:, n_x:].contiguous(memory_format=fmt))
        return cache[key][1], cache[key][2]

    batch_refs = True    # forward(): run the R references of a scale as one batch (same arithmetic per sample)

    def _forward_refs_batched(self, x, pre_offset_list, img_ref_feat_list):
        """forward() with the Python loop over references folded into the batch dimension (autograd-capable: this is
        the training path).  Per scale: the references' features / pre-offsets stacked [B, R] -> B*R, conv1 split by
        input channels so that its x half runs once per image instead of once per (image, reference) and no
        repeat / cat of x is materialised, ONE offset-conv / DynAgg / lrelu chain over B*R samples, and the fusion head
        on the stacked tensor (MRAPAFusion.forward would stack the list again)."""
        r = len(img_ref_feat_list)
        keys = [k for _, k in self._SCALES]
        feats = {k: torch.stack([f[k] for f in img_ref_feat_list], 1).flatten(0, 1) for k in keys}   # [B*R, C, H, W]
        pres = {k: torch.stack([p[k] for p in pre_offset_list], 1).flatten(0, 1) for k in keys}     # [B*R, 9, H, W, 2]
        return self._forward_stacked(x, pres, feats, r)

    def _forward_stacked(self, x, pres, feats, r):
        """The same on tensors that are already stacked over the references: pres / feats = {layer: [B*R, ...]}, pairs laid
        out [B, R] (what MRefSRPipeline.correspondences returns: no per-reference lists, no re-stacking).
        pres may instead be the int64 arg-max map [B*R, h-2, w-2] at the 1/4-resolution grid
        (correspondences(..., as_max_idx=True)): each DynAgg then runs forward_fused at its flow scale 1 / 2 / 4, whose
        autograd node builds offsets and masks inside the DCN gather in the forward and in the backward."""
        fused = torch.is_tensor(pres)
        for s, (name, key) in zip((1, 2, 4), self._SCALES):
            conv1, conv2 = getattr(self, f'{name}_offset_conv1'), getattr(self, f'{name}_offset_conv2')
            agg = getattr(self, f'{name}_dyn_agg')
            feat = feats[key]
            feat_c = feat           # the DCN reads planes (NCHW); the convolution takes the trunk's layout
            if x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous():
                feat_c = feat.contiguous(memory_format=torch.channels_last)
            nx = x.shape[1]
            ox = F.conv2d(x, conv1.weight[:, :nx], None, conv1.stride, conv1.padding)         # once per image
            # the bias rides on the per-image half (1 / R of the elements; its gradient = the fused epilogue's one-pass
            # reduction over that half's gradient instead of torch's reduction over all B*R samples)
            fused_bias = conv1.bias is not None and T.train_ok(ox) and _lib_supports(ox)
            if fused_bias:
                ox = T.BiasActFunction.apply(ox, conv1.bias, T.ACT_NONE, 0.0, None, 1.0)
            of = F.conv2d(feat_c, conv1.weight[:, nx:], None if fused_bias else conv1.bias, conv1.stride, conv1.padding)
            o = (of.unflatten(0, (-1, r)) + ox.unsqueeze(1)).flatten(0, 1)
            if T.layout_of(of) == 1:
                o = o.contiguous(memory_format=torch.channels_last)
            o = self.lrelu(o)
            o2 = T.conv_bias_act_train(o, conv2, T.ACT_LEAKY, 0.1)
            o = o2 if o2 is not None else self.lrelu(conv2(o))
            if fused:
                y = agg.forward_fused([feat, o], pres, s, out_slope=0.1, out_like_conv=True)  # [B*R, C, H, W]
            elif agg.fused_autograd and T.layout_of(o) == 1:
                # the leaky ReLU and the hand-off to the fusion head in the trunk's dtype / layout ride on the DynAgg
                # node's one conversion pass (instead of an activation pass, then a cast (autocast) and a layout
                # conversion (cuDNN) per convolution that reads the aligned features)
                y = agg([feat, o], pres[key], out_slope=0.1, out_like_conv=True)              # [B*R, C, H, W]
            else:
                y = self.lrelu(agg([feat, o], pres[key]))
            h = getattr(self, f'head_{name}').forward_stacked(x, y, r)
            h = getattr(self, f'body_{name}')(h) + x
            tail = getattr(self, f'tail_{name}')
            if T.train_ok(h):
                if name == 'large':     # conv -> lrelu -> conv
                    x = T.conv_act(T.conv_act(h, tail[0], T.ACT_LEAKY, 0.1), tail[2])
                else:                   # conv -> pixel shuffle -> lrelu == conv -> lrelu -> pixel shuffle
                    x = F.pixel_shuffle(T.conv_act(h, tail[0], T.ACT_LEAKY, 0.1), 2).contiguous(
                        memory_format=torch.channels_last)
            else:
                x = tail(h)
        return x

    def forward(self, x, pre_offset_list, img_ref_feat_list, n_refs=None):
        """Reference contract: lists over references of pre_offset / VGG feature dicts.  Also accepted: the same tensors
        already stacked over the references ({layer: [B*R, ...]} dicts, pairs laid out [B, R]) with n_refs = R, where the
        pre-offset dict may be replaced by the matcher's int64 arg-max map [B*R, h-2, w-2] (the fused DynAgg path)."""
        if isinstance(img_ref_feat_list, dict):
            if n_refs is None or not (isinstance(pre_offset_list, dict) or torch.is_tensor(pre_offset_list)):
                raise ValueError('stacked references: pass a {layer: [B*R, ...]} feature dict, a pre-offset dict or the '
                                 'arg-max map, and n_refs')
            return self._forward_stacked(x, pre_offset_list, img_ref_feat_list, int(n_refs))
        if (self.batch_refs and len(img_ref_feat_list) > 1 and len(pre_offset_list) == len(img_ref_feat_list) and
                all(f[k].shape == img_ref_feat_list[0][k].shape for f in img_ref_feat_list for _, k in self._SCALES)):
            return self._forward_refs_batched(x, pre_offset_list, img_ref_feat_list)
        for name, key in self._SCALES:
            conv1, conv2 = getattr(self, f'{name}_offset_conv1'), getattr(self, f'{name}_offset_conv2')
            agg = getattr(self, f'{name}_dyn_agg')
            swapped = []
            for pre_offset, feat in zip(pre_offset_list, img_ref_feat_list):
                o = self.lrelu(conv1(torch.cat([x, feat[key]], 1)))
                o = self.lrelu(conv2(o))
                swapped.append(self.lrelu(agg([feat[key], o], pre_offset[key])))
            h = getattr(self, f'head_{name}')(x, swapped)
            h = getattr(self, f'body_{name}')(h) + x
            x = getattr(self, f'tail_{name}')(h)
        return x

    def forward_batched(self, x, max_idx, ref_feats, n_refs):
        """Inference fast path.  max_idx int64 [B*R,h-2,w-2] (pairs laid out [B,R]); ref_feats {layer: [B*R,C,H,W]}.
        The R references are stacked into the batch of the offset convolutions and of ONE fused DynAgg launch."""
        r = n_refs
        for s, (name, key) in zip((1, 2, 4), self._SCALES):
            conv1, conv2 = getattr(self, f'{name}_offset_conv1'), getattr(self, f'{name}_offset_conv2')
            agg = getattr(self, f'{name}_dyn_agg')
            feat = ref_feats[key]                                           # [B*R, C, H, W]
            fast = T.fast_ok(x, feat)
            if fast:
                # conv1 over cat([x repeated per reference, feat]) split by input channels: the x half is computed
                # once per image and enters the feat half's epilogue as a per-image, pre-activation term -- no
                # repeat_interleave, no cat, (R-1)/R of the x-half FLOPs gone
                wx, wf = self._split_conv1(conv1, x.shape[1], T.layout_of(x) == 1)
                ox = F.conv2d(x, wx, None, conv1.stride, conv1.padding)
                o = T.dense(F.conv2d(feat, wf, None, conv1.stride, conv1.padding))
                o = T.bias_act_(o, conv1.bias, T.ACT_LEAKY, 0.1, residual=T.dense(ox), res_div=r, res_pre=True)
                o = T.conv_bias_act(o, conv2, T.ACT_LEAKY, 0.1)
                y = agg.forward_fused([feat, o], max_idx, s, out_slope=0.1)   # lrelu folded into the DCN epilogue
            else:
                xr = x.repeat_interleave(r, dim=0)                          # [B*R, ngf, H, W]
                o = self.lrelu(conv1(torch.cat([xr, feat], 1)))
                o = self.lrelu(conv2(o))
                y = self.lrelu(agg.forward_fused([feat, o], max_idx, s))    # [B*R, C, H, W]
            h = getattr(self, f'head_{name}').forward_stacked(x, y, r)     # y is already [B*R, C, H, W]
            h = getattr(self, f'body_{name}')(h) + x
            tail = getattr(self, f'tail_{name}')
            if fast and T.fast_ok(h):
                if name == 'large':     # conv -> lrelu -> conv
                    x = T.conv_bias_act(T.conv_bias_act(h, tail[0], T.ACT_LEAKY, 0.1), tail[2])
                else:                   # conv -> pixel shuffle -> lrelu == conv -> lrelu -> pixel shuffle
                    x = F.pixel_shuffle(T.conv_bias_act(h, tail[0], T.ACT_LEAKY, 0.1), 2)
                    if T.layout_of(h) == 1:     # pixel_shuffle hands back NCHW: keep the channels-last trunk intact
                        x = T.to_nhwc(x)
            else:
                x = tail(h)
        return x


class MRAPARestorationNet(nn.Module):
    """ref_mrapa_restoration_arch.py:99-137."""

    def __init__(self, ngf=64, n_blocks=16, groups=8):
        super().__init__()
        self.content_extractor = ContentExtractor(in_nc=3, out_nc=3, nf=ngf, n_blocks=n_blocks)
        self.dyn_agg_restore = DynamicAggregationRestoration(ngf, n_blocks, groups)
        srntt_init_weights(self, init_gain=0.02)
        for name in ('small', 'medium', 'large'):
            getattr(self.dyn_agg_restore, f'{name}_dyn_agg').init_offset()

    def forward(self, x, pre_offset_list, img_ref_feat_list, n_refs=None):
        base = F.interpolate(x, None, 4, 'bilinear', False)
        return self.dyn_agg_restore(self.content_extractor(x), pre_offset_list, img_ref_feat_list, n_refs) + base

    def forward_batched(self, x, max_idx, ref_feats, n_refs):
        base = F.interpolate(x, None, 4, 'bilinear', False)
        return self.dyn_agg_restore.forward_batched(self.content_extractor(x), max_idx, ref_feats, n_refs) + base


class MRefSRPipeline(nn.Module):
    """net_extractor -> net_map -> net_g as MultiRefRestorationModel.test() wires them
    (multi_ref_restoration_model.py:281-294), batched over references."""

    def __init__(self, ngf=64, n_blocks=16, groups=8, match_mode='auto'):
        super().__init__()
        self.net_extractor = ContrasMultiExtractorSep()
        self.net_map = CorrespondenceGenerationArch(patch_size=3, stride=1,
                                                    vgg_layer_list=['relu1_1', 'relu2_1', 'relu3_1'], vgg_type='vgg19',
                                                    match_mode=match_mode)
        self.net_g = MRAPARestorationNet(ngf=ngf, n_blocks=n_blocks, groups=groups)
        self.match_mode = match_mode
        self._channels_last = False

    def channels_last_(self):
        """Run the plain-convolution trunk in torch.channels_last (cuDNN's native layout for its tensor-core kernels:
        no NCHW<->NHWC conversion around every convolution).  The alignment kernels take it from there: the DCN
        gathers from the NHWC features as they are and writes NHWC, the glue kernels follow the tensor's layout."""
        self.to(memory_format=torch.channels_last)
        self._channels_last = True
        return self

    @torch.no_grad()
    def forward(self, img_in_lq, img_in_up, img_refs):
        """img_in_lq [B,3,H/4,W/4], img_in_up [B,3,H,W] (the LR input upsampled x4), img_refs [B,R,3,H,W] -> SR [B,3,H,W]."""
        b, r = img_refs.shape[:2]
        if self._channels_last:
            img_in_lq = img_in_lq.contiguous(memory_format=torch.channels_last)
            img_in_up = img_in_up.contiguous(memory_format=torch.channels_last)
            img_refs = img_refs.flatten(0, 1).contiguous(memory_format=torch.channels_last).unflatten(0, (b, r))
        f1, f2 = self.net_extractor.forward_batched(img_in_up, img_refs)
        max_idx, _ = feature_match_index_batched(f1, f2, 3, 1, 1, True, True, normalize_pixels=True, in_div=r,
                                                 mode=self.match_mode)
        ref_feats = self.net_map.vgg(img_refs.flatten(0, 1))
        return self.net_g.forward_batched(img_in_lq, max_idx, ref_feats, r)

    @torch.no_grad()
    def correspondences(self, img_in_up, img_refs, as_max_idx=False):
        """The frozen half of a training step (MultiRefRestorationModel.optimize_parameters evaluates net_extractor and
        net_map per reference under no_grad, multi_ref_restoration_model.py:281-294 has the same loop for testing), batched
        over the references: one extractor pass over B*R reference images, ONE matcher launch for all pairs, one VGG pass.
        img_in_up [B,3,H,W], img_refs [B,R,3,H,W] -> (pre_offsets, ref_feats, R): {layer: [B*R, 9, s*h, s*w, 2]} and
        {layer: [B*R, C, s*h, s*w]} with pairs laid out [B, R] -- the stacked form net_g.forward accepts.
        as_max_idx: return the matcher's int64 arg-max map [B*R, h-2, w-2] in place of the pre-offsets (no pre-offset
        tensors are written; net_g then trains on the fused DynAgg path)."""
        b, r = img_refs.shape[:2]
        if self._channels_last:     # (channels_last_(): the frozen nets run cuDNN's NHWC kernels without layout conversions)
            img_in_up = img_in_up.contiguous(memory_format=torch.channels_last)
            img_refs = img_refs.flatten(0, 1).contiguous(memory_format=torch.channels_last).unflatten(0, (b, r))
        f1, f2 = self.net_extractor.forward_batched(img_in_up, img_refs)
        idx, _ = feature_match_index_batched(f1, f2, 3, 1, 1, True, True, normalize_pixels=True, in_div=r,
                                             mode=self.match_mode)
        pres = idx if as_max_idx else dict(zip(('relu3_1', 'relu2_1', 'relu1_1'), pre_offsets(idx)))
        feats = self.net_map.vgg(img_refs.flatten(0, 1))
        return pres, {k: feats[k] for k in ('relu3_1', 'relu2_1', 'relu1_1')}, r

    def forward_ragged(self, samples, max_batch=16, graphs=False):
        """Images with different reference counts / sizes (LMR-shaped groups, BASELINE config 3): samples[i] =
        (lq [3,h,w], up [3,H,W], refs [R_i,3,H,W]); images sharing (R, H, W) go through one batched `forward`.
        Returns the SR images in input order (parallel.run_ragged; shard a ragged batch over ranks with
        parallel.shard_ragged first).

        graphs=True replays one captured CUDA graph per shape class (batch, R, H, W) instead of launching the ~700
        kernels of a forward eagerly: the groups of a ragged batch are small (1-3 images), so the eager path is bound
        by the host.  Graphs are captured on first use and kept (`clear_graphs()` drops them -- call it after the
        weights were re-allocated or updated through anything but in-place writes)."""
        from .parallel import run_ragged
        if not graphs:
            return run_ragged(self, samples, max_batch)
        cache = self.__dict__.setdefault('_ragged_graphs', {})

        def fwd(lq, up, refs):
            key = (tuple(lq.shape), tuple(up.shape), tuple(refs.shape), str(lq.device))
            g = cache.get(key)
            if g is None:
                g = cache[key] = self.graphed(lq, up, refs)
            return g(lq, up, refs).clone()      # the graph's static output is overwritten by its next replay
        return run_ragged(fwd, samples, max_batch)

    def clear_graphs(self):
        self.__dict__.pop('_ragged_graphs', None)

    def graphed(self, img_in_lq, img_in_up, img_refs, warmup=3):
        """Capture `forward` for these shapes into a CUDA graph and return a GraphedForward runner.  The forward is
        ~700 kernel launches for 25 ms of GPU work, so launched eagerly it is one slow host core away from being
        launch-bound; replaying the graph removes the host from the loop."""
        return GraphedForward(self, img_in_lq, img_in_up, img_refs, warmup)

    @torch.no_grad()
    def forward_reference_order(self, img_in_lq, img_in_up, img_refs):
        """The reference's own operator order (one net_map call per reference, materialised pre-offsets, DynAgg through
        the modulated_deform_conv boundary): slower, used to cross-check `forward`."""
        refs = list(img_refs.unbind(1))
        feats = self.net_extractor(img_in_up, refs)
        pres, rfs = [], []
        for f, ref in zip(feats, refs):
            pre, rf = self.net_map(f, ref)
            pres.append(pre)
            rfs.append(rf)
        # the cross-check keeps the reference's structure: Python loop over references, DynAgg as the two operator Functions
        dar = self.net_g.dyn_agg_restore
        aggs = [getattr(dar, f'{n}_dyn_agg') for n in ('small', 'medium', 'large')]
        saved = (dar.batch_refs, [a.fused_autograd for a in aggs])
        dar.batch_refs = False
        for a in aggs:
            a.fused_autograd = False
        try:
            return self.net_g(img_in_lq, pres, rfs)
        finally:
            dar.batch_refs = saved[0]
            for a, v in zip(aggs, saved[1]):
                a.fused_autograd = v


class GraphedForward:
    """CUDA-graph replay of MRefSRPipeline.forward for fixed shapes.  Inputs are copied into static device buffers
    (from host or device tensors, asynchronously on the current stream), the graph is replayed, and the static
    output tensor is returned (valid until the next call; `out=` copies it into a caller tensor, e.g. pinned host
    memory, on the same stream)."""

    def __init__(self, net, img_in_lq, img_in_up, img_refs, warmup=3):
        dev = next(net.parameters()).device
        self.static_in = [torch.empty(t.shape, dtype=torch.float32, device=dev) for t in (img_in_lq, img_in_up, img_refs)]
        for s_, t in zip(self.static_in, (img_in_lq, img_in_up, img_refs)):
            s_.copy_(t)
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):           # warm-up off the capture: cuDNN plans, workspaces, lazy module init
            for _ in range(max(1, warmup)):
                net(*self.static_in)
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: CUDA calls of other threads (the NCCL watchdog under torchrun) must not invalidate the capture
        with torch.cuda.graph(self.graph, capture_error_mode='thread_local'):
            self.static_out = net(*self.static_in)

    def __call__(self, img_in_lq, img_in_up, img_refs, out=None):
        for s_, t in zip(self.static_in, (img_in_lq, img_in_up, img_refs)):
            s_.copy_(t, non_blocking=True)
        self.graph.replay()
        if out is not None:
            out.copy_(self.static_out, non_blocking=True)
            return out
        return self.static_out
