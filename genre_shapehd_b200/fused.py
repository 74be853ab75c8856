"""Opt-in fused form of GenRe's 3D glue (SURVEY §8f-1).  Inference only.

The reference's model files are frozen callers, so the drop-in ops cannot remove what the callers do between them:
    depth_pred_with_sph_inpaint.py:120-126   proj = cam_bp(depth);  sph_in = render(clamp(proj * 50, 1e-5, 1 - 1e-5));
                                             sph_in = sph_pad(sph_in);  out['proj_depth'] = proj * 50
    genre_full_model.py:120-143              crop, 1 - x, spherical back-projection, mask = clamp(cnt, 0, 1),
                                             (-tdf + 1/128) * 128 * mask;  clamp(proj_depth / 50, 1e-5, 1 - 1e-5);  cat
— about 19 dense passes over 128^3 volumes per batch.  ``GenRe3DGlue`` computes the same tensors with the elementwise
work folded into the kernels (csrc/render_sph.cu pre-transform, csrc/sph_bp.cu fused entry, csrc/layout.cu clamp-copy):

    glue = GenRe3DGlue().to(device)
    proj, sph_in = glue.project_and_render(abs_depth)            # cam_bp + render_spherical + sph_pad
    refine_in = glue.refine_input(proj, pred_sph_full)           # [B,2,128,128,128], ready for Unet_3D

A model that wants it calls these two methods instead of the glue lines; nothing in the frozen callers changes.
Differences to the op-by-op path are rounding only (the (x*50)/50 round trip and the order of the affine in the
spherical back-projection): tests/test_gpu_toolbox.py bounds them at 1e-5.
"""
import torch

from genre_shapehd_b200 import _lib
from toolbox.cam_bp.cam_bp.modules.camera_backprojection_module import Camera_back_projection_layer
from toolbox.spherical_proj import gen_sph_grid, render_forward, render_spherical, sph_pad


class GenRe3DGlue(torch.nn.Module):
    def __init__(self, res=128, sph_res=128, z_res=256, margin=16, scale=50.0, lo=1e-5, hi=1 - 1e-5):
        super().__init__()
        self.res, self.margin, self.scale, self.lo, self.hi = res, margin, float(scale), float(lo), float(hi)
        self.proj_depth = Camera_back_projection_layer(res)
        self.render = render_spherical(sph_res, z_res)
        self.register_buffer("grid", gen_sph_grid(sph_res))          # [1,1,S,S,3], as Net.register_buffer('grid', ...)

    @torch.no_grad()
    def project_and_render(self, abs_depth, fl=418.3, cam_dist=2.2):
        """-> (proj [B,1,R,R,R] = shifted TDF, as Camera_back_projection_layer returns it;
               sph_in [B,1,S+2m,S+2m] = sph_pad(render_spherical(clamp(proj * scale, lo, hi))))"""
        proj = self.proj_depth(abs_depth, fl, cam_dist)
        r = self.render
        n = proj.shape[0]
        sph = proj.new_empty((n, 1, r.sph_res, r.sph_res))
        render_forward(proj, n, self.res, r._dirs_on(proj.device), r.sph_res, r.z_res, r.depth_weight, sph,
                       pre=(self.scale, self.lo, self.hi))
        return proj, sph_pad(sph, self.margin)

    @torch.no_grad()
    def refine_input(self, proj, pred_sph_full):
        """-> cat((backproject_spherical(pred_sph_full), clamp(proj, lo, hi)), dim=1), written once"""
        b, _, h, w = pred_sph_full.shape
        m, r3 = self.margin, self.res ** 3
        _lib.require_cuda(proj, pred_sph_full)
        _lib.require_f32(proj, pred_sph_full)
        out = proj.new_empty((b, 2, self.res, self.res, self.res))
        crop = pred_sph_full[:, :, m:h - m, m:w - m]                 # a view: the kernel walks its strides
        grid = self.grid.expand(b, -1, -1, -1, -1)
        ws, nbytes = _lib.workspace_for(b, crop.shape[2] * crop.shape[3], self.res, proj.device)
        st = _lib.stream_ptr(proj)
        _lib.call("genre_b200_sph_bp_forward_fused", crop.data_ptr(), b, 1, crop.shape[2], crop.shape[3], *crop.stride(),
                  grid.data_ptr(), *grid.stride(), -1.0, 1.0, out.data_ptr(), 2 * r3, self.res, ws.data_ptr(), nbytes, st)
        p = proj.contiguous()
        _lib.call("genre_b200_scale_clamp_strided", p.data_ptr(), b, r3, 1.0, self.lo, self.hi,
                  out.data_ptr() + 4 * r3, 2 * r3, st)
        return out


@torch.no_grad()
def genre_forward_fused(net, input_struct, glue=None):
    """Batched, mesh-free GenRe inference: the same tensors as the frozen ``Net.forward`` (models/genre_full_model.py:116-132;
    same keys, same values up to rounding) with the 3D glue of the callers folded into the kernels (``GenRe3DGlue``).

    It also stands in for the published test path ``Model.forward_with_trimesh`` (genre_full_model.py:202-233), which renders the
    spherical map on the CPU through marching cubes + trimesh ray casting (util_sph.py:36-57), needs batch size 1 and is not
    differentiable: here the spherical map comes from the differentiable renderer, for any batch, on the device (SURVEY 8f-4).

    net: genre_shapehd_b200.genre_models.GenReNet, eval mode.  Returns the dict of its forward."""
    dn = net.depth_and_inpaint
    if glue is None:
        glue = getattr(net, "_gb_glue", None)
        if glue is None or glue.grid.device != net.grid.device:
            glue = GenRe3DGlue(margin=net.margin).to(net.grid.device)
            net.__dict__["_gb_glue"] = glue
    out = dn.net1(input_struct)                                              # depth_pred_with_sph_inpaint.py:115-119
    abs_depth = dn.get_abs_depth(out, input_struct)                         # :133-142
    proj, sph_in = glue.project_and_render(abs_depth)                       # :120-126 cam_bp, clamp(proj * 50), render, sph_pad
    out_2 = dn.net2(sph_in)
    out["proj_depth"] = proj * glue.scale
    out["pred_sph_partial"] = sph_in
    out["pred_sph_full"] = out_2["spherical"]
    refine_input = glue.refine_input(proj, out["pred_sph_full"])            # genre_full_model.py:125-127,134-143
    out["pred_proj_sph_full"] = refine_input[:, 0:1]
    out["pred_proj_depth"] = refine_input[:, 1:2]
    out["pred_voxel"] = net.refine_net(refine_input)
    return out
