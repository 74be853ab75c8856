"""3D voxel networks of GenRe / ShapeHD — drop-in for the reference's networks/networks.py.

Same public names, constructor signatures, NCDHW fp32 in/out and — because load_state_dict in the reference is
strict and positional (models/netinterface.py:422-424) — the same ``state_dict`` keys and shapes:

    Unet_3D           enc{1..6}.net.{0,1}.*, full_conv_block.0.*, dec{1..5}.net.{0,1}.*, dec6.net.*   (networks.py:147-190)
    VoxelDecoder      main.{0,1,3,4,8,9,11,12,14,15,17}.*  (two empty Sequentials at 6,7)              (networks.py:25-61)
    VoxelGenerator    main.{0,1,3,4,6,7,9,10,12,13,15}.*                                              (networks.py:64-104)
    VoxelDiscriminator main.{0,2,4,6,8,10}.weight                                                     (networks.py:107-144)

Layers are created in the reference's order, so a model built under the same torch seed has bit-identical
parameters (tests/test_networks.py checks digests recorded from the reference).

Every convolution is a ``Conv3d`` / ``ConvTranspose3d`` below: a torch parameter container whose CUDA forward can be
routed to the hand-written sm_100a implicit-GEMM kernels (genre_shapehd_b200/ops_conv.py) layer by layer; layers
without a custom kernel run on cuDNN exactly like the reference does.
"""
import torch
import torch.nn as nn
from torch import cat

from genre_shapehd_b200 import ops_conv


class Conv3d(nn.Conv3d):
    """nn.Conv3d parameters + dispatch of the CUDA forward to the sm_100a kernel when one covers the layer."""

    def forward(self, x):
        y = ops_conv.conv3d(x, self) if x.is_cuda else None
        if y is None and x.is_cuda and self.padding_mode == "zeros":
            y = ops_conv.exact_fallback(x, self, False)         # <= 8^3 layers in the fp32-accurate modes: 3xTF32 on cuDNN
        return y if y is not None else super().forward(x)


class ConvTranspose3d(nn.ConvTranspose3d):
    def forward(self, x, output_size=None):
        y = ops_conv.conv_transpose3d(x, self) if output_size is None else None
        if y is None and output_size is None and x.is_cuda:
            y = ops_conv.gemm_conv(x, self)
        if y is None and x.is_cuda and self.padding_mode == "zeros":
            y = ops_conv.exact_fallback(x, self, True, output_size)
        return y if y is not None else super().forward(x, output_size)


class FusedSequential(nn.Sequential):
    """nn.Sequential (same state_dict keys) whose CUDA forward hands conv [-> BatchNorm3d] -> ReLU/LeakyReLU/Sigmoid runs to
    ops_conv.fused_block: one kernel with the eval-mode normalisation and the activation in its epilogue.  Anything
    not covered (training-mode BN, autograd, unsupported shapes, CPU) runs module by module like nn.Sequential."""

    def forward(self, x):
        mods = list(self)
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, (Conv3d, ConvTranspose3d)) and x.is_cuda:
                j = i + 1
                bn = mods[j] if j < len(mods) and isinstance(mods[j], nn.BatchNorm3d) else None
                j += bn is not None
                act = mods[j] if j < len(mods) and isinstance(mods[j], (nn.ReLU, nn.LeakyReLU, nn.Sigmoid)) else None
                if act is not None:
                    y = ops_conv.fused_block(x, m, bn, act)
                    if y is not None:
                        x, i = y, j + 1
                        continue
                    if ops_conv.BN_TRAIN and bn is not None and bn.training:
                        z = ops_conv.bn_act_train(m(x), bn, act)          # conv module, then BN+act in one op
                        if z is not None:
                            x, i = z, j + 1
                            continue
            x = m(x)
            i += 1
        return x


# ---- layer helpers (names and arguments of networks.py:225-284) ------------------------------------------------
def relu():
    return nn.ReLU(inplace=True)


def relu_leaky():
    return nn.LeakyReLU(0.2, inplace=True)


def maxpool():
    return nn.MaxPool2d(3, stride=2, padding=0)


def dropout():
    return nn.Dropout(p=0.5, inplace=False)


def conv3d_half(n_ch_in, n_ch_out, bias):
    return Conv3d(n_ch_in, n_ch_out, 4, stride=2, padding=1, dilation=1, groups=1, bias=bias)


def deconv3d_2x(n_ch_in, n_ch_out, bias):
    return ConvTranspose3d(n_ch_in, n_ch_out, 4, stride=2, padding=1, dilation=1, groups=1, bias=bias)


def conv3d_minus3(n_ch_in, n_ch_out, bias):
    return Conv3d(n_ch_in, n_ch_out, 4, stride=1, padding=0, dilation=1, groups=1, bias=bias)


def deconv3d_add3(n_ch_in, n_ch_out, bias):
    return ConvTranspose3d(n_ch_in, n_ch_out, 4, stride=1, padding=0, dilation=1, groups=1, bias=bias)


def batchnorm1d(n_feat):
    return nn.BatchNorm1d(n_feat, eps=1e-5, momentum=0.1, affine=True)


def batchnorm(n_feat):
    return nn.BatchNorm2d(n_feat, eps=1e-5, momentum=0.1, affine=True)


def batchnorm3d(n_feat):
    return nn.BatchNorm3d(n_feat, eps=1e-5, momentum=0.1, affine=True)


def fc(n_in, n_out):
    return nn.Linear(n_in, n_out, bias=True)


class ViewAsLinear(nn.Module):
    @staticmethod
    def forward(x):
        return x.view(x.shape[0], -1)


class ImageEncoder(nn.Module):
    """2.5D sketch -> 200-d code (networks.py:6-22).  A 2D ResNet-18 (torchvision's, randomly initialised): outside the
    hot path."""

    def __init__(self, input_nc, encode_dims=200):
        super().__init__()
        import torchvision
        resnet_m = torchvision.models.resnet18(weights=None)
        resnet_m.conv1 = nn.Conv2d(input_nc, 64, 7, stride=2, padding=3, bias=False)
        resnet_m.avgpool = nn.AdaptiveAvgPool2d(1)
        resnet_m.fc = nn.Linear(512, encode_dims)
        self.main = nn.Sequential(resnet_m)

    def forward(self, x):
        return self.main(x)


def _deconv_stack(n_in, widths, bias, last_sigmoid=False, pad_slots=()):
    """ConvT(k4,s1) to 4^3, then ConvT(k4,s2,p1) doublings with BN+ReLU between, ending in a 1-channel ConvT.
    ``pad_slots``: indices (in the final Sequential) where the reference keeps empty nn.Sequential() placeholders."""
    layers = [deconv3d_add3(n_in, widths[0], bias), batchnorm3d(widths[0]), relu()]
    for cin, cout in zip(widths[:-1], widths[1:]):
        while len(layers) in pad_slots:
            layers.append(nn.Sequential())
        layers.append(deconv3d_2x(cin, cout, bias))
        if cout != 1:
            layers += [batchnorm3d(cout), relu()]
    if last_sigmoid:
        layers.append(nn.Sigmoid())
    return FusedSequential(*layers)


class VoxelDecoder(nn.Module):
    """200-d code -> 128^3 occupancy logits (networks.py:25-61); state_dict keys main.{0,1,3,4,8,9,...,17}."""

    def __init__(self, n_dims=200, nf=512):
        super().__init__()
        self.main = _deconv_stack(n_dims, [nf, nf // 2, nf // 4, nf // 8, nf // 16, 1], True, pad_slots=(6, 7))

    def forward(self, x):
        return self.main(x.view(x.size(0), -1, 1, 1, 1))


class VoxelGenerator(nn.Module):
    """3D-GAN generator (networks.py:64-104)."""

    def __init__(self, nz=200, nf=64, bias=False, res=128):
        super().__init__()
        if res == 64:
            widths = [nf * 8, nf * 4, nf * 2, nf, 1]
        elif res == 128:
            widths = [nf * 8, nf * 4, nf * 2, nf, nf, 1]
        else:
            raise NotImplementedError(res)
        self.main = _deconv_stack(nz, widths, bias, last_sigmoid=True)

    def forward(self, x):
        return self.main(x)


class VoxelDiscriminator(nn.Module):
    """3D-GAN / WGAN-GP critic without normalisation layers (networks.py:107-144)."""

    def __init__(self, nf=64, bias=False, res=128):
        super().__init__()
        if res not in (64, 128):
            raise NotImplementedError(res)
        chans = [1, nf, nf * 2, nf * 4, nf * 8]
        layers = []
        for cin, cout in zip(chans[:-1], chans[1:]):
            layers += [conv3d_half(cin, cout, bias), relu_leaky()]
        layers.append(conv3d_minus3(chans[-1], 1, bias))
        if res == 128:
            # the reference creates the extra nf->nf stage last and splices it in after the first stage
            # (networks.py:128-139); same creation order => same parameters under the same seed
            layers[2:2] = [conv3d_half(nf, nf, bias), relu_leaky()]
        self.main = FusedSequential(*layers)

    def forward(self, x):
        y = self.main(x)
        return y.view(-1, 1).squeeze(1)


class Conv3d_block(nn.Module):
    """Conv3d + BatchNorm3d + LeakyReLU(0.01) (networks.py:193-203)."""

    def __init__(self, ncin, ncout, kernel_size, stride, pad, dropout=False):
        super().__init__()
        self.net = nn.Sequential(Conv3d(ncin, ncout, kernel_size, stride, pad), nn.BatchNorm3d(ncout), nn.LeakyReLU())

    def forward(self, x):
        y = ops_conv.conv3d(x, self.net[0], self.net[1], self.net[2].negative_slope) if x.is_cuda else None
        if y is None and ops_conv.BN_TRAIN and x.is_cuda and self.net[1].training:
            c = self.net[0](x)
            z = ops_conv.bn_act_train(c, self.net[1], self.net[2])
            return z if z is not None else self.net[2](self.net[1](c))
        return y if y is not None else self.net(x)


class Deconv3d_skip(nn.Module):
    """cat(x, skip) -> ConvTranspose3d [+ BatchNorm3d + LeakyReLU] (networks.py:206-222)."""

    def __init__(self, ncin, ncout, kernel_size, stride, pad, extra=0, is_activate=True):
        super(Deconv3d_skip, self).__init__()
        deconv = ConvTranspose3d(ncin, ncout, kernel_size, stride, pad, extra)
        self.net = nn.Sequential(deconv, nn.BatchNorm3d(ncout), nn.LeakyReLU()) if is_activate else deconv

    def forward(self, x, skip_in, keep_blocked=False):
        """keep_blocked: the caller promises the result only feeds another Deconv3d_skip (Unet_3D.forward does for
        dec5 -> dec6), so a custom kernel may leave it in its blocked layout (ops_conv.BlockedActivation)."""
        if not x.is_cuda:
            y = None
        elif isinstance(self.net, nn.Sequential):
            y = ops_conv.deconv_skip(x, skip_in, self.net[0], self.net[1], self.net[2].negative_slope, keep_blocked)
        else:
            y = ops_conv.deconv_skip(x, skip_in, self.net)
        if y is not None:
            return y
        if isinstance(x, ops_conv.BlockedActivation):
            x = x.ncdhw()
        if ops_conv.BN_TRAIN and x.is_cuda and isinstance(self.net, nn.Sequential) and self.net[1].training:
            c = self.net[0](cat((x, skip_in), dim=1))
            z = ops_conv.bn_act_train(c, self.net[1], self.net[2])
            return z if z is not None else self.net[2](self.net[1](c))
        return self.net(cat((x, skip_in), dim=1))


class Unet_3D(nn.Module):
    """GenRe's voxel refiner: [B,2,128^3] -> [B,1,128^3] (networks.py:147-190)."""

    # (in, out, kernel, stride, pad) in units of nf; enc6 / dec1 work at 1^3 <-> 4^3
    _ENC = [(None, 1, 8, 2, 3), (1, 2, 4, 2, 1), (2, 4, 4, 2, 1), (4, 8, 4, 2, 1), (8, 16, 4, 2, 1), (16, 32, 4, 1, 0)]
    _DEC = [(64, 16, 4, 1, 0), (32, 8, 4, 2, 1), (16, 4, 4, 2, 1), (8, 2, 4, 2, 1), (4, 1, 8, 2, 3)]

    def __init__(self, nf=20, in_channel=2, no_linear=False):
        super(Unet_3D, self).__init__()
        self.nf = nf
        for i, (ci, co, k, s, p) in enumerate(self._ENC, 1):
            setattr(self, "enc%d" % i, Conv3d_block(in_channel if ci is None else ci * nf, co * nf, k, s, p))
        self.full_conv_block = nn.Sequential(nn.Linear(32 * nf, 32 * nf), nn.LeakyReLU())
        for i, (ci, co, k, s, p) in enumerate(self._DEC, 1):
            setattr(self, "dec%d" % i, Deconv3d_skip(ci * nf, co * nf, k, s, p, 0))
        self.dec6 = Deconv3d_skip(2 * nf, 1, 4, 2, 1, 0, is_activate=False)
        self.no_linear = no_linear

    def forward(self, x):
        skips = []
        for i in range(1, 7):
            x = getattr(self, "enc%d" % i)(x)
            skips.append(x)
        enc6 = skips[-1]
        if not self.no_linear:
            b = enc6.size(0)
            x = self.full_conv_block(enc6.view(b, self.nf * 32)).view(b, self.nf * 32, 1, 1, 1)
        for i in range(1, 7):
            x = getattr(self, "dec%d" % i)(x, skips[6 - i], keep_blocked=(i == 5))   # dec5's only consumer is dec6
        return x
