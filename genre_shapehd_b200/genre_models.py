"""GenRe and ShapeHD model classes, built on this package's ops and 3D networks.

    GenReNet         RGB + silhouette -> depth (2D U-ResNet-18) -> camera back-projection -> spherical render ->
                     inpainting (2D U-ResNet-18) -> spherical back-projection -> Unet_3D refiner logits
    ShapeHDNet       2.5D sketches -> MarrNet-2 voxels, scored by a frozen 3D-GAN critic
    WganGenerator / WganCritic   the 3D-GAN pair of the WGAN-GP critic step

State dict keys, parameter shapes and the order in which layers are created follow the published GenRe-ShapeHD
models, so a net built under a given torch seed gets the same random initialisation, and published checkpoints load
with ``load_state_dict``.  The two 2D U-ResNet-18s stay on torch (cuDNN): they are outside the hot path.
"""
import torch
import torch.nn as nn
import torchvision

from networks.networks import ImageEncoder, Unet_3D, ViewAsLinear, VoxelDecoder, VoxelDiscriminator, VoxelGenerator
from toolbox.cam_bp.cam_bp.functions import SphericalBackProjection
from toolbox.cam_bp.cam_bp.modules.camera_backprojection_module import Camera_back_projection_layer
from toolbox.spherical_proj import gen_sph_grid, render_spherical, sph_pad

SCALE_25D = 100          # 2.5D maps (depth, normal, silhouette) are stored as [0, 1] * 100


def _deconv(cin, cout, k, stride=1, padding=0, bias=False):
    return nn.ConvTranspose2d(cin, cout, k, stride=stride, padding=padding, bias=bias, output_padding=1 if stride > 1 else 0)


class RevBasicBlock(nn.Module):
    """ResNet basic block mirrored for upsampling: the stride sits on the second (transposed) convolution."""

    def __init__(self, cin, cout, stride=1, upsample=None):
        super().__init__()
        self.deconv1 = _deconv(cin, cout, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(cout)
        self.relu = nn.ReLU(inplace=True)
        self.deconv2 = _deconv(cout, cout, 3, stride, padding=1)
        self.bn2 = nn.BatchNorm2d(cout)
        self.upsample = upsample

    def forward(self, x):
        out = self.bn2(self.deconv2(self.relu(self.bn1(self.deconv1(x)))))
        out += x if self.upsample is None else self.upsample(x)
        return self.relu(out)


def _rev_stage(cin, cout, stride):
    up = nn.Sequential(_deconv(cin, cout, 1, stride), nn.BatchNorm2d(cout)) if stride != 1 or cin != cout else None
    return nn.Sequential(RevBasicBlock(cin, cout, stride, up), RevBasicBlock(cout, cout))


def _rev_unet18_decoder(out_planes):
    """The U-Net decoder of a ResNet-18: four mirrored stages (input channels include the skip connections) and a
    head upsampling x4.  Returns (stages, head layers); the layers are created in the published model's order."""
    head_deconv = nn.ConvTranspose2d(128, 64, 3, stride=2, padding=1, output_padding=1)
    head_out = _deconv(64, out_planes, 7, 2, padding=3)
    head_bn = nn.BatchNorm2d(64)
    stages = [_rev_stage(cin, cout, s) for cin, cout, s in ((512, 256, 2), (512, 128, 2), (256, 64, 2), (128, 64, 1))]
    return stages, [head_deconv, head_bn, nn.ReLU(inplace=True), head_out]


class UResNet18(nn.Module):
    """ResNet-18 encoder and one U-Net decoder per output map (``decoder_<name>``).  ``inpaint=True`` is the variant of
    the spherical-map inpainting net: every decoder ends in one shared 8x8 transposed convolution (``deconv2``)."""

    def __init__(self, out_planes, names, input_planes=3, inpaint=False):
        super().__init__()
        resnet = torchvision.models.resnet18(weights=None)
        in_conv = nn.Conv2d(input_planes, 64, kernel_size=7, stride=2, padding=3, bias=False)
        stem = resnet.conv1 if input_planes == 3 else in_conv
        self.encoder = nn.ModuleList([nn.Sequential(stem, resnet.bn1, resnet.relu, resnet.maxpool),
                                      resnet.layer1, resnet.layer2, resnet.layer3, resnet.layer4])
        self.encoder_out = None
        if inpaint:
            self.deconv2 = nn.ConvTranspose2d(64, 1, kernel_size=8, stride=2, padding=3, bias=False)
        self.names = list(names)
        for planes, name in zip(out_planes, self.names):
            stages, head = _rev_unet18_decoder(planes)
            if inpaint:
                head[-1] = self.deconv2
            setattr(self, "decoder_" + name, nn.ModuleList(stages + [nn.Sequential(*head)]))

    def forward(self, im):
        feats = []
        for f in self.encoder:
            im = f(im)
            feats.append(im)
        self.encoder_out = feats[-1]
        out = {}
        for name in self.names:
            dec = getattr(self, "decoder_" + name)
            x = feats[-1]
            for i, f in enumerate(dec):
                x = f(x)
                if i < len(dec) - 1:
                    x = torch.cat((x, feats[-(i + 2)]), dim=1)
            out[name] = x
        return out


class DepthNet(UResNet18):
    """MarrNet-1 of GenRe: normal, relative depth and silhouette maps of an RGB image, plus the (min, max) of the absolute
    depth regressed from the encoder's 8x8 output (``depth_minmax``)."""

    def __init__(self):
        super().__init__([3, 1, 1], ["normal", "depth", "silhou"])
        self.decoder_minmax = nn.Sequential(
            nn.Conv2d(512, 512, 2, stride=2), nn.Conv2d(512, 512, 4, stride=1), ViewAsLinear(),
            nn.Linear(512, 256), nn.BatchNorm1d(256), nn.ReLU(inplace=True),
            nn.Linear(256, 128), nn.BatchNorm1d(128), nn.ReLU(inplace=True),
            nn.Linear(128, 2))

    def forward(self, input_struct):
        out = super().forward(input_struct.rgb)
        out["depth_minmax"] = self.decoder_minmax(self.encoder_out)
        return out


class DepthInpaintNet(nn.Module):
    """Depth estimation, its back-projection into the voxel grid, the spherical map rendered from it and the
    inpainted full spherical map."""

    def __init__(self, joint_train=False, padding_margin=16):
        super().__init__()
        self.net1 = DepthNet()
        self.net2 = UResNet18([1], ["spherical"], input_planes=1, inpaint=True)
        self.proj_depth = Camera_back_projection_layer()
        self.render_spherical = render_spherical()
        self.joint_train = joint_train
        self.padding_margin = padding_margin

    def forward(self, input_struct):
        with torch.set_grad_enabled(self.joint_train and torch.is_grad_enabled()):
            out = self.net1(input_struct)
        proj = self.proj_depth(self.get_abs_depth(out, input_struct))
        sph_in = sph_pad(self.render_spherical(torch.clamp(proj * 50, 1e-5, 1 - 1e-5)), self.padding_margin)
        out["proj_depth"] = proj * 50
        out["pred_sph_partial"] = sph_in
        out["pred_sph_full"] = self.net2(sph_in)["spherical"]
        return out

    @staticmethod
    def get_abs_depth(pred, input_struct):
        """absolute depth of the silhouette's pixels (0 elsewhere), transposed and flipped into the camera's frame"""
        rel = pred["depth"] / SCALE_25D
        minmax = pred["depth_minmax"].detach()
        dmin, dmax = minmax[:, 0].view(-1, 1, 1, 1), minmax[:, 1].view(-1, 1, 1, 1)
        depth = (1 - rel) * (dmax - dmin + 1e-4) + dmin
        depth[(input_struct.silhou / SCALE_25D).detach() < 0.5] = 0
        return torch.flip(depth.permute(0, 1, 3, 2), [2])


class GenReNet(nn.Module):
    """The full GenRe model.  ``forward(input_struct)`` takes ``.rgb`` [B,3,256,256] and ``.silhou`` [B,1,256,256]
    (x100) and returns a dict whose ``pred_voxel`` [B,1,128,128,128] holds the refiner's occupancy logits.  Unless
    ``joint_train``, the depth and inpainting nets run without gradients."""

    def __init__(self, joint_train=False, padding_margin=16):
        super().__init__()
        self.depth_and_inpaint = DepthInpaintNet(joint_train, padding_margin)
        self.refine_net = Unet_3D()
        self.proj_depth = Camera_back_projection_layer()
        self.joint_train = joint_train
        self.register_buffer("grid", gen_sph_grid())
        self.margin = padding_margin

    def forward(self, input_struct):
        with torch.set_grad_enabled(self.joint_train and torch.is_grad_enabled()):
            out = self.depth_and_inpaint(input_struct)
        pred_proj_sph = self.backproject_spherical(out["pred_sph_full"])
        proj_depth = torch.clamp(out["proj_depth"] / 50, 1e-5, 1 - 1e-5)
        out["pred_proj_depth"] = proj_depth
        out["pred_voxel"] = self.refine_net(torch.cat((pred_proj_sph, proj_depth), dim=1))
        out["pred_proj_sph_full"] = pred_proj_sph
        return out

    def backproject_spherical(self, sph):
        """shifted distance field of the inpainted spherical map (its margin cropped), zero in voxels no ray reached"""
        n, _, h, w = sph.shape
        m = self.margin
        grid = self.grid.expand(n, -1, -1, -1, -1)
        tdf, cnt = SphericalBackProjection.apply(1 - sph[:, :, m:h - m, m:w - m], grid, 128)
        return (-tdf + 1 / 128) * 128 * torch.clamp(cnt.detach(), 0, 1)


class MarrNet2(nn.Module):
    """2.5D sketches (depth + normal, masked by the silhouette) -> 128^3 voxel logits"""

    def __init__(self, in_planes=4, encode_dims=200, silhou_thres=0):
        super().__init__()
        self.encoder = ImageEncoder(in_planes, encode_dims=encode_dims)
        self.decoder = VoxelDecoder(n_dims=encode_dims, nf=512)
        self.silhou_thres = silhou_thres

    def forward(self, input_struct):
        depth, normal = input_struct.depth, input_struct.normal
        bg = input_struct.silhou <= self.silhou_thres
        depth[bg] = 0                                    # in place, as the published model does
        normal[bg.repeat(1, 3, 1, 1)] = 0
        return self.decoder(self.encoder(torch.cat((depth, normal), 1)))


class WganGenerator(VoxelGenerator):
    def __init__(self, nz=200):
        super().__init__(nz=nz, nf=64, bias=False, res=128)
        self.nz = nz

    def forward(self, batch_size):
        x = torch.randn(batch_size, self.nz, 1, 1, 1, device=next(self.parameters()).device)
        return x, super().forward(x)


class WganCritic(VoxelDiscriminator):
    def __init__(self):
        super().__init__(nf=64, bias=False, res=128)

    def forward(self, x):
        return super().forward(x.unsqueeze(1) if x.dim() == 4 else x)


class ShapeHDNet(nn.Module):
    """MarrNet-2 being fine-tuned, a frozen copy of it, and the frozen critic that scores the fine-tuned voxels"""

    def __init__(self):
        super().__init__()
        self.marrnet2 = MarrNet2(4)
        self.marrnet2_noft = MarrNet2(4)
        self.d = WganCritic()
        for p in list(self.d.parameters()) + list(self.marrnet2_noft.parameters()):
            p.requires_grad = False
        self.sigmoid = nn.Sigmoid()

    def forward(self, input_struct):
        pred = {"voxel_noft": self.marrnet2_noft(input_struct), "voxel": self.marrnet2(input_struct)}
        pred["is_real"] = self.d(self.sigmoid(pred["voxel"]))
        return pred
