"""Dispatch of the 3D convolutions of networks/networks.py to the hand-written sm_100a kernels.

``conv3d(x, module)`` / ``conv_transpose3d(x, module)`` / ``deconv_skip(...)`` return the result computed by this
library's kernels, or ``None`` when no kernel covers the layer (shape / dtype / device / autograd) — the caller then
runs the layer the way the reference does (torch.nn -> cuDNN; in the fp32-accurate mode through ``exact_fallback``).

Kernels and what they cover (routing conditions are the ``*_supported`` predicates below, all of them tested both ways):
  csrc/convt3d.cu          tcgen05 implicit GEMM on halo tiles: ConvTranspose3d k 4 / 8, s 2 (planes 16 or 32 wide), Conv3d
                           k 4 s 2 via parity sub-volumes, Conv3d k 8 s 2 via space-to-depth, the 1-channel ConvTranspose3d
                           with 27 union taps; forward under autograd too, tensor-core input gradients for the k 8 layers
  csrc/convflat.cu         the same GEMM over a flattened, zero-separated volume for coarse sides <= 8^3 (inference)
  csrc/convt_c1_col2im.cu  the 1-channel ConvTranspose3d on 64-wide volumes as a tap GEMM + shared-memory col2im (inference)
  csrc/skinny_gemm.cu      Conv3d whose kernel covers its input / ConvTranspose3d of a 1^3 input: FP32 weight streaming (inference)
  csrc/convt_c1.cu, convt_c1_wgrad.cu, bn_train.cu   FP32-pipe 1-channel stencil and its gradients; training BatchNorm3d + activation
Operand modes: see PRECISION below ("exact" = fp16 hi/lo split, fp32-accurate, the default).

Activations cross the halo kernels in a channel-blocked layout [B*D][C/4][H][W][4] (fp32) or [B*D][parts*C/8][H][W][8] (fp16,
hi | lo' parts); ``to_blocked`` / ``from_blocked`` / ``space_to_depth_*`` convert at the boundary (csrc/layout.cu).
"""
import os

import torch

from . import _lib

ENABLED = os.environ.get("GENRE_B200_CONV", "1") != "0"
# Dispatch policy.  Every kernel is correct on every layer it supports; which layers are ROUTED to it is decided by
# end-to-end measurements on a B200 (kernel + the NCDHW <-> channel-blocked conversions of csrc/layout.cu around it;
# profiles/r01_conv_summary.md), B = 16, against cuDNN with TF32 allowed:
#   convt_k8   ConvTranspose3d k=8 s=2 (Unet_3D.dec5: 7.2 -> 1.35 ms)
#   conv_k8s2  Conv3d k=8 s=2 on few input channels (Unet_3D.enc1: 16.6 -> 0.8 ms)
#   convt_c1   ConvTranspose3d k=4 -> 1 channel on already-blocked inputs (Unet_3D.dec6: 2.1 -> 1.3 ms)
#   convt_k4   ConvTranspose3d k=4 s=2 (dec4 0.30 -> 0.23, VoxelDecoder/Generator stages 1.26 -> 1.01, 1.87 -> 1.46 ms)
#   conv_k4s2  Conv3d k=4 s=2 (discriminator 1.18 -> 0.86 ms per layer, Unet_3D.enc2/enc3)
#   convt_c1_convert   the 1-channel layer when its input must first be converted; FP32-pipe kernel, so only up to
#                      C1_MAX_CIN input channels (VoxelDecoder's 32 -> 1 wins, VoxelGenerator's 64 -> 1 does not)
# GENRE_B200_CONV_POLICY = comma list restricts the set ("all" = everything, the default).
#   convt_c1_tc   the 1-channel layer on the tensor cores (3 union taps, 8 output classes as N columns); tried first
#   gemm          ConvTranspose3d on a 1^3 input (dec1, the decoders' first layer) as one cuBLAS GEMM (0.34 -> 0.085 ms)
#   convt_c1_train   the 1-channel layer under autograd: exact forward + custom input/weight gradients (cuDNN's wgrad: 40 ms)
#   conv_k8s2_wgrad  Unet_3D.enc1's weight gradient (first-order backward only; double backward stays on aten)
#   conv_k4s2_s2d    Conv3d(1 or 2 -> 64, k4 s2) as 3 taps over the 2x space-to-depth input (VoxelDiscriminator main.0:
#                    cuDNN 2.6 ms in eval at B=16 and a 35 ms kernel per call in the WGAN-GP step at B=8)
#   flat          the k4 s2 convolutions of the small volumes (coarse side <= 8^3: Unet_3D.enc4, enc5, dec2, dec3 and the 4^3 / 8^3
#                 stages of the ShapeHD nets) on the flattened-volume kernel (csrc/convflat.cu); fp16 / f16x2 modes, inference
#   skinny        Conv3d whose kernel covers its whole input (Unet_3D.enc6) / ConvTranspose3d on a 1^3 input (dec1, the decoders'
#                 first layer) in eval mode as weight-streaming FP32 products (csrc/skinny_gemm.cu); every precision mode (exact fp32)
#   convt_c1_col2im  the 1-channel layer on 64-wide volumes as a GEMM over the 64 taps + shared-memory col2im (csrc/convt_c1_col2im.cu):
#                    Unet_3D.dec6 1.33 ms (FP32 stencil) / 0.67 ms (MODE 4, fp16) -> see profiles/r02_summary.md; fp16 and f16x2 modes
_all_policy = {"convt_c1_col2im", "skinny", "flat", "conv_k4s2_s2d", "conv_k8s2_wgrad", "convt_c1_train", "convt_k8", "conv_k8s2", "convt_c1", "convt_k4", "conv_k4s2", "convt_c1_convert", "convt_c1_tc", "gemm"}
_default_policy = set(_all_policy)
_env = os.environ.get("GENRE_B200_CONV_POLICY", "")
POLICY = set(_all_policy) if _env in ("", "all") else set(x for x in _env.split(",") if x)
C1_MAX_CIN = 48
K4S2_MIN_CIN = 8
# Operand mode of the tensor-core kernels (GENRE_B200_CONV_PRECISION, or `with ops_conv.precision(mode):`):
#   "exact" (DEFAULT)  fp32-accurate: the reference's fp32 semantics (north_star: occupancies within 1e-4).  Implemented by
#                      EXACT_IMPL: "f16x2" = fp16 hi/lo operand split, 2 MMAs per K step, separate accumulators for the
#                      hi*hi and the cross terms; "fp32x3" = 3xTF32 with the three products along K (3 MMAs per K=8 step)
#   "f16"              single pass, fp16 operands (10-bit mantissa, 5-bit exponent), fp32 accumulation: opt-in, tested at
#                      4e-3 * max|ref| per layer; inputs beyond fp16's range are the caller's responsibility
#   "tf32"             single pass, TF32 operands (what cuDNN does while torch.backends.cudnn.allow_tf32 is on)
# torch.backends.cudnn.allow_tf32 = False upgrades a single-pass mode to "exact" (PyTorch's own switch for fp32 convolutions).
PRECISION = os.environ.get("GENRE_B200_CONV_PRECISION", "exact")
EXACT_IMPL = os.environ.get("GENRE_B200_CONV_EXACT_IMPL", "f16x2")
# k=8 ConvTranspose3d with Cout <= 20 (Unet_3D.dec5): merge the four (y,x) parity classes into one N=80 MMA stream
MERGE_PARITIES = os.environ.get("GENRE_B200_CONV_MERGE", "1") != "0"


# With torch.backends.cudnn.allow_tf32 off the caller asks for fp32 convolutions: the kernels then run the 3xTF32 scheme
# (operands split into TF32 hi + lo parts, A_lo*W_hi + A_hi*W_lo + A_hi*W_hi accumulated in fp32: ~1e-5 relative error, set by the accumulator's truncation,
# 3x the MMAs of the TF32 mode) so that occupancies match the fp32 reference within 1e-4.  "0": fall back to cuDNN fp32.
EXACT_WHEN_TF32_OFF = os.environ.get("GENRE_B200_CONV_EXACT", "1") != "0"


_FORCED_MODE = None   # set by _forced_mode(): gradient convolutions use TF32 operands (fp16 would flush small gradients)
_OVERRIDE = None      # set by precision()
_EXACT = ("exact", "fp32x3", "f16x2")


class _forced_mode:
    """internal: single-pass operand type of the convolutions issued inside (never downgrades an exact mode)"""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        global _FORCED_MODE
        self.old, _FORCED_MODE = _FORCED_MODE, self.mode

    def __exit__(self, *exc):
        global _FORCED_MODE
        _FORCED_MODE = self.old


class precision:
    """public: `with ops_conv.precision("f16"):` selects the operand mode of the custom convolutions issued inside"""

    def __init__(self, mode):
        if mode not in ("exact", "f16", "tf32", "fp32x3", "f16x2"):
            raise ValueError("unknown conv precision %r" % (mode,))
        self.mode = mode

    def __enter__(self):
        global _OVERRIDE
        self.old, _OVERRIDE = _OVERRIDE, self.mode

    def __exit__(self, *exc):
        global _OVERRIDE
        _OVERRIDE = self.old


def _mode():
    """operand mode of the next launch: 'f16' | 'tf32' (single pass) or the fp32-accurate 'f16x2' | 'fp32x3'.
    Inside _forced_mode("tf32") (gradient convolutions) an exact mode means fp32x3: gradients need fp32's exponent range,
    which the fp16 hi/lo split does not have."""
    base = _OVERRIDE or PRECISION
    if base in _EXACT or not torch.backends.cudnn.allow_tf32:
        if _FORCED_MODE == "tf32" or base == "fp32x3":
            return "fp32x3"
        return base if base == "f16x2" else EXACT_IMPL
    return _FORCED_MODE or base


def cudnn_precision():
    """cuDNN flags for GRADIENT convolutions this module hands to cuDNN: the caller's global setting (PyTorch's default allows
    TF32).  The north_star's 1e-4 bound is on the forward outputs; gradients follow PyTorch's switch, as they do upstream:
    `torch.backends.cudnn.allow_tf32 = False` makes them fp32."""
    import contextlib
    return contextlib.nullcontext()


def exact_fallback(x, m, transposed, output_size=None):
    """Forward of a layer NO custom kernel covers (the <= 8^3 layers of the nets) in the fp32-accurate modes, inference only: cuDNN
    fp32 convolutions without tensor cores are 10-20x slower than its TF32 ones (Unet_3D's five small layers: 0.6 -> 11 ms at
    batch 16), and plain TF32 would put a 10-bit mantissa into an otherwise fp32-accurate network.  So the layer is evaluated as
    the 3xTF32 operand split on cuDNN's TF32 kernels:  conv(x_lo, w_hi) + conv(x_hi, [w_hi | w_lo])  with hi = the
    TF32 rounding (exactly representable: cuDNN's own operand conversion is then lossless) and fp32 accumulation.
    Returns None when not applicable (autograd, single-pass modes, TF32 disallowed globally -> plain cuDNN fp32)."""
    if not (x.is_cuda and x.dtype == torch.float32 and _mode() in ("f16x2", "fp32x3") and torch.backends.cudnn.allow_tf32
            and not _needs_grad(x, m.weight, m.bias) and output_size is None):
        return None
    f = torch.nn.functional
    cdim = 1 if transposed else 0            # output-channel axis of the weight tensor

    def split(w):                            # (W_hi | W_lo) stacked along the output channels, and W_hi: cached per weight version
        wh = _tf32_hi(w)
        return torch.cat((wh, w - wh), dim=cdim).contiguous(), wh
    wcat, wh = _cached_pack(m, ("exact_fallback",), split)
    xh = _tf32_hi(x)
    xl = x - xh
    if transposed:
        conv = lambda a, b: f.conv_transpose3d(a, b, None, m.stride, m.padding, m.output_padding, m.groups, m.dilation)
    else:
        conv = lambda a, b: f.conv3d(a, b, None, m.stride, m.padding, m.dilation, m.groups)
    both = conv(xh, wcat)                    # x_hi * (W_hi | W_lo): one launch, 2 * Cout channels
    c = m.out_channels
    y = conv(xl, wh)
    y += both[:, c:]
    y += both[:, :c]
    if m.bias is not None:
        y += m.bias.detach().view(1, -1, 1, 1, 1)
    return y


def describe_mode():
    m = _mode()
    return {"f16": "f16 single pass (10-bit operand mantissa, fp32 accumulate)", "tf32": "tf32 single pass (10-bit operand mantissa)",
            "fp32x3": "exact: 3xTF32 operand split (fp32-accurate, tested <= 1e-4)",
            "f16x2": "exact: fp16 hi/lo operand split, 2 MMAs per K step (fp32-accurate, tested <= 1e-4)"}[m]


def _f16():
    return _mode() == "f16"


def _x3():
    return _mode() == "fp32x3"


def _x2():
    return _mode() == "f16x2"


def _op_flag():
    """`op` argument of the C ABI: 0 = TF32 operands, 1 = fp16, 2 = fp16 hi/lo split"""
    return 2 if _x2() else 1 if _f16() else 0


def _tf32_hi(w):
    """w rounded to TF32 (nearest, ties away - cvt.rna.tf32.f32) but kept in fp32 storage"""
    i = w.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _split3(t):
    """blocked fp32 [BD,CG,H,W,4] -> [BD,3CG,H,W,4] = (lo | hi | hi) blocks (csrc/layout.cu split3_kernel)"""
    bd, cg, h, w, _ = t.shape
    out = torch.empty((bd, 3 * cg, h, w, 4), device=t.device, dtype=torch.float32)
    _lib.call("genre_b200_blocked_split3", t.data_ptr(), cg, bd, h, w, out.data_ptr(), _lib.stream_ptr(t))
    return out


def _split2(t):
    """blocked fp32 [BD,CG4,H,W,4] -> fp16 [BD, 2*CG8, H, W, 8]: CG8 = ceil(CG4/2) groups of hi = fp16(a) followed by CG8
    groups of lo' = fp16((a - hi) * 2^11): the activation operand of the f16x2 mode (csrc/layout.cu split2_f16_kernel)"""
    bd, cg4, h, w, _ = t.shape
    cg8 = (cg4 + 1) // 2
    out = torch.empty((bd, 2 * cg8, h, w, 8), device=t.device, dtype=torch.float16)
    _lib.call("genre_b200_blocked_split2_f16", t.data_ptr(), cg4, bd, h, w, out.data_ptr(), _lib.stream_ptr(t))
    return out


def _finish_operand(xb):
    """fp32 blocked conversion result -> the operand of the current exact mode (no-op for the single-pass modes)"""
    if _x3():
        return _split3(xb)
    if _x2():
        return _split2(xb)
    return xb


def _parts():
    """operand parts stacked along the channel-group axis of an activation tensor (the kernels take per-part group counts)"""
    return 2 if _x2() else 1


def _x3_operands(src0, src1):
    """in fp32x3 mode the (possibly two-source) K range becomes ONE tensor of lo | hi | hi blocks"""
    if not _x3():
        return src0, src1
    t = src0 if src1 is None else torch.cat((src0, src1), dim=1)
    return _split3(t.contiguous()), None


def _pack(module, key, make, chunk_dim, half=None):
    """packed weights of `module` for the current mode (cached per parameter version; repacking is one gather through the
    layer's pack plan).  fp32x3: (W_hi | W_lo | W_hi) along the K-chunk axis, matching the (lo | hi | hi) activation
    blocks: the two small cross terms are accumulated first (the tensor core's fp32 accumulator truncates, so a step's
    error scales with the partial sum it is added to)."""
    if half is None:
        half = _f16()
    x3, x2 = _x3(), _x2()

    def build(w):
        plan = _pack_plan(module, key, make)
        if x2:      # [W_hi | W_lo'] side by side along N: the n-group axis is the third from last of every packed layout
            hi = w.half().float()
            return torch.cat((_apply_plan(plan, hi, True), _apply_plan(plan, (w - hi) * 2048.0, True)), dim=-3).contiguous()
        if not x3:
            return _apply_plan(plan, w, half)
        hi = _tf32_hi(w)
        p_hi, p_lo = _apply_plan(plan, hi, False), _apply_plan(plan, w - hi, False)
        return torch.cat((p_hi, p_lo, p_hi), dim=chunk_dim).contiguous()
    return _cached_pack(module, key + (("x2",) if x2 else ("x3",) if x3 else ("half",) if half else ()), build)


def _group():
    """channels per 16-byte channel group of the kernel operands (weights, K-chunk sizing)"""
    return 8 if (_f16() or _x2()) else 4


def _act_group():
    """channels per group of the NCDHW -> blocked conversions: fp16 groups of 8 in the single-pass fp16 mode; fp32 groups of 4
    otherwise (the exact modes split them afterwards: _finish_operand)"""
    return 8 if _f16() else 4


def _on_device(x, group, dtype):
    """the CUDA layout kernels (csrc/layout.cu) take contiguous fp32 NCDHW and write fp32 groups of 4, fp16 groups of 8, or
    (group 16) the fp16 hi/lo parts of groups of 8 channels"""
    return (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
            and ((group == 4 and dtype in (None, torch.float32)) or (group in (8, 16) and dtype == torch.float16)))


def _x2_direct(x):
    """can the NCDHW -> hi/lo operand conversion run as one pass of the layout kernels?"""
    return _x2() and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()


def _permuted_copy(view, dtype):
    """materialise a permuted view in ONE pass, the cast (if any) riding on the copy"""
    out = torch.empty(view.shape, device=view.device, dtype=dtype or view.dtype)
    out.copy_(view)
    return out


def to_blocked(x, group=4, dtype=None):
    """NCDHW [B,C,D,H,W] (C % group == 0) -> [B*D, C/group, H, W, group] contiguous (optionally cast)."""
    b, c, d, h, w = x.shape
    if group == 16:     # hi | lo' parts of groups of 8 channels (the f16x2 operand), CUDA only
        out = torch.empty((b * d, 2 * (c // 8), h, w, 8), device=x.device, dtype=torch.float16)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 0, 16, 0, out.data_ptr(), _lib.stream_ptr(x))
        return out
    if _on_device(x, group, dtype):
        out = torch.empty((b * d, c // group, h, w, group), device=x.device, dtype=dtype or x.dtype)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 0, group, 0, out.data_ptr(), _lib.stream_ptr(x))
        return out
    v = x.reshape(b, c // group, group, d, h, w).permute(0, 3, 1, 4, 5, 2)
    return _permuted_copy(v, dtype).view(b * d, c // group, h, w, group)


def _to_operand(x):
    if _x2():   # the fp32 blocked twin a previous custom layer left behind saves the NCDHW round trip
        twin = _cached_blocked(x)
        if twin is not None and twin.shape[1] * 4 == x.shape[1] and twin.shape[0] == x.shape[0] * x.shape[2]:
            return _split2(twin)
        if _x2_direct(x) and x.shape[1] % 8 == 0:
            return to_blocked(x, 16, torch.float16)
        return _split2(to_blocked(x, 4))
    return to_blocked(x, 8, torch.float16) if _f16() else to_blocked(x, 4)


def from_blocked(y, batch, channels):
    """[B*D, cg, H, W, 4] -> NCDHW [B, channels, D, H, W] (drops channel padding).  The blocked tensor stays attached to
    the result so that a following custom layer can consume it without converting back."""
    bd, cg, h, w, _ = y.shape
    d = bd // batch
    if y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and 4 * (cg - 1) < channels:
        out = torch.empty((batch, channels, d, h, w), device=y.device, dtype=torch.float32)
        _lib.call("genre_b200_blocked_to_ncdhw", y.data_ptr(), cg, batch, channels, d, h, w, out.data_ptr(), _lib.stream_ptr(y))
    else:
        out = y.view(batch, d, cg, h, w, 4).permute(0, 2, 5, 1, 3, 4).reshape(batch, cg * 4, d, h, w)[:, :channels]
    out._gb_blocked = (y, out._version)   # valid until `out` is modified in place (e.g. an inplace ReLU)
    return out


class BlockedActivation:
    """An activation that exists only in the blocked layout (the output of a custom layer whose sole consumer is the
    next custom layer, e.g. Unet_3D.dec5 -> dec6).  Quacks like the NCDHW tensor for the dispatch checks; ncdhw()
    materialises it if a consumer turns out to need the plain layout."""
    is_cuda, dtype, requires_grad = True, torch.float32, False

    def __init__(self, y, batch, channels):
        bd, cg, h, w, _ = y.shape
        self._gb_blocked, self.batch, self.shape = y, batch, torch.Size((batch, channels, bd // batch, h, w))
        self.device = y.device

    def dim(self):
        return 5

    def size(self, i=None):
        return self.shape if i is None else self.shape[i]

    def ncdhw(self):
        return from_blocked(self._gb_blocked, self.batch, self.shape[1])


def _cached_blocked(x):
    """the blocked twin a custom layer attached to its NCDHW result, unless that result was since modified in place"""
    if isinstance(x, BlockedActivation):
        return x._gb_blocked
    hit = getattr(x, "_gb_blocked", None)
    if hit is None or hit[1] != x._version:
        return None
    return hit[0]


def _blocked_f32(x):
    """fp32 group-of-4 blocked view of an NCDHW tensor: the cached one if x came out of a custom layer"""
    y = _cached_blocked(x)
    if y is not None and y.shape[1] * 4 >= x.shape[1] and y.shape[0] == x.shape[0] * x.shape[2] \
            and (y.shape[1] - 1) * 4 < x.shape[1] + 4 and x.shape[1] % 4 == 0:
        return y
    return to_blocked(x, 4)


def pack_convt_weights(weight, npad, group=4):
    """ConvTranspose3d weight [Cin, Cout, K, K, K] -> the per-stage shared-memory images the kernel bulk-copies:
    [8 parity][T z-tap][Cin/(2g) chunk][T*T (y,x) taps][2 k-core][npad/8 n-group][8 n][g k]  (T = K/2; g = 4 fp32
    or 8 fp16 elements per 16-byte core-matrix row)."""
    cin, cout, k = weight.shape[0], weight.shape[1], weight.shape[2]
    t, pad = k // 2, k // 2 - 1
    g = group
    k0 = [(p + pad) % 2 for p in (0, 1)]
    wp = weight.new_zeros((cin, npad, k, k, k))
    wp[:, :cout] = weight
    out = weight.new_empty((2, 2, 2, t, cin // (2 * g), t, t, 2, npad // 8, 8, g))
    for pz in (0, 1):
        for py in (0, 1):
            for px in (0, 1):
                sub = wp[:, :, k0[pz]::2, k0[py]::2, k0[px]::2]                      # [Cin, npad, tz, ty, tx]
                sub = sub.reshape(cin // (2 * g), 2, g, npad // 8, 8, t, t, t)        # (kc, kk, e, ng, r, tz, ty, tx)
                out[pz, py, px] = sub.permute(5, 0, 6, 7, 1, 3, 4, 2)                 # (tz, kc, ty, tx, kk, ng, r, e)
    out = out.contiguous()
    return _finish_pack(out, g)


def pack_convt_merged_weights(weight, cpad, group=4):
    """ConvTranspose3d weight [Cin, Cout, K, K, K] (stride 2, padding K/2-1) for the merged-parity kernel (MODE 2):
    [2 z-parity][T z-tap][Cin/(2g) chunk][(T+1)^2 union (y,x) taps][2 k-core][N/8][8][g],  N = 4*cpad, column
    n = (py*2+px)*cpad + co.  Union tap u reads input j + T/2 - u; class p uses it as its tap t = u - 1 + p (k = k0_p + 2t)
    when 0 <= t < T, and holds zeros otherwise."""
    cin, cout, k = weight.shape[0], weight.shape[1], weight.shape[2]
    t, pad, g = k // 2, k // 2 - 1, group
    tu, n = t + 1, 4 * cpad
    k0 = [(p + pad) % 2 for p in (0, 1)]
    weq = weight.new_zeros((cin, n, 2, t, tu, tu))                       # (ci, n, pz, tz, uy, ux)
    for py in (0, 1):
        for px in (0, 1):
            c0 = (py * 2 + px) * cpad
            for uy in range(tu):
                ty = uy - 1 + py
                if not 0 <= ty < t:
                    continue
                for ux in range(tu):
                    tx = ux - 1 + px
                    if not 0 <= tx < t:
                        continue
                    for pz in (0, 1):
                        # [Cin, Cout, tz]
                        weq[:, c0:c0 + cout, pz, :, uy, ux] = weight[:, :, k0[pz]::2, k0[py] + 2 * ty, k0[px] + 2 * tx]
    sub = weq.reshape(cin // (2 * g), 2, g, n // 8, 8, 2, t, tu, tu)    # (kc, kk, e, ng, r, pz, tz, uy, ux)
    out = sub.permute(5, 6, 0, 7, 8, 1, 3, 4, 2).contiguous()           # (pz, tz, kc, uy, ux, kk, ng, r, e)
    return _finish_pack(out, g)


def pack_convt_c1_tc_weights(weight, segments, group=4):
    """ConvTranspose3d weight [Cin, 1, 4, 4, 4] (stride 2, padding 1) for kernel MODE 4: [3 z-tap][chunk][9 taps][2][2][8][g].
    N = 16 columns, n = (qz*2+qy)*2+qx < 8 the output classes; union tap u reads input j + 1 - u and serves class q as its
    tap t = u - 1 + q (kernel index k = (q+1)%2 + 2t).  `segments` = [(real channels, padded channels), ...] of the
    concatenated sources: padded rows are zero."""
    g = group
    kmap = {(0, 1): 1, (0, 2): 3, (1, 0): 0, (1, 1): 2}                  # (q, u) -> k
    ktot = sum(pc for _, pc in segments)
    weq = weight.new_zeros((ktot, 16, 3, 3, 3))
    rows, c0, r0 = [], 0, 0
    for real, padded in segments:
        rows.append((r0, c0, real))
        c0, r0 = c0 + real, r0 + padded
    assert c0 == weight.shape[0] and ktot % (2 * g) == 0
    for (qz, uz), kz in kmap.items():
        for (qy, uy), ky in kmap.items():
            for (qx, ux), kx in kmap.items():
                n = (qz * 2 + qy) * 2 + qx
                for r0, c0, real in rows:
                    weq[r0:r0 + real, n, uz, uy, ux] = weight[c0:c0 + real, 0, kz, ky, kx]
    sub = weq.reshape(ktot // (2 * g), 2, g, 2, 8, 3, 3, 3)               # (kc, kk, e, ng, r, tz, ty, tx)
    out = sub.permute(5, 0, 6, 7, 1, 3, 4, 2).contiguous()
    return _finish_pack(out, g)


def pack_convt_c1_col2im_weights(weight, segments, group=8):
    """ConvTranspose3d weight [Cin, 1, 4, 4, 4] for csrc/convt_c1_col2im.cu: [K step][2 kcore][8 n-groups][8 n][8 k], the GEMM's
    N = 64 columns are the taps in phase-major order n = t*8 + r, tap k = 2t + r per dimension (t, r = (z,y,x) bit triples);
    `segments` = [(real channels, padded channels), ...] of the concatenated sources (padded rows zero)."""
    ktot = sum(pc for _, pc in segments)
    assert ktot % 16 == 0
    weq = weight.new_zeros((ktot, 64))
    r0 = c0 = 0
    for real, padded in segments:
        for n in range(64):
            t, r = n >> 3, n & 7
            kz, ky, kx = (2 * ((t >> (2 - i)) & 1) + ((r >> (2 - i)) & 1) for i in range(3))
            weq[r0:r0 + real, n] = weight[c0:c0 + real, 0, kz, ky, kx]
        c0, r0 = c0 + real, r0 + padded
    assert c0 == weight.shape[0]
    sub = weq.reshape(ktot // 16, 2, 8, 8, 8)                                   # (ks, kk, e, ng, r)
    return _finish_pack(sub.permute(0, 1, 3, 4, 2).contiguous(), group)         # (ks, kk, ng, r, e)


_PLAN_MODE = False    # while True the packers run on an index tensor: no dtype conversion at the end


def _finish_pack(out, g):
    return out if _PLAN_MODE or g != 8 else out.half()


def _pack_plan(module, key, make):
    """Every packer is a pure rearrangement (copies, permutes, zero padding) of the weight entries, so it is run ONCE per
    (layer, layout) on a tensor of 1-based element numbers; the result is a gather index + zero mask that repacks the
    real weights with one kernel whenever they change (every optimiser step in training)."""
    global _PLAN_MODE
    plans = module.__dict__.setdefault("_gb_plans", {})
    plan = plans.get(key)
    if plan is None or plan[0].device != module.weight.device:
        w = module.weight
        _PLAN_MODE = True
        try:
            numbered = make(torch.arange(1, w.numel() + 1, dtype=torch.float64).view(w.shape))
        finally:
            _PLAN_MODE = False
        idx = numbered.to(torch.int64)
        plan = ((idx - 1).clamp_(min=0).to(w.device), (idx > 0).to(w.device))
        plans[key] = plan
    return plan


def _apply_plan(plan, w, half):
    out = torch.where(plan[1], w.reshape(-1)[plan[0]], torch.zeros((), device=w.device, dtype=w.dtype))
    return out.half() if half else out


def _cached_pack(module, key, make):
    """Packed weights live ON the module (they die with it; a global cache keyed by id() could hand a recycled id the
    weights of a dead layer) and are rebuilt when the parameter is updated in place (optimizer step, load_state_dict).
    `key` ends with the group size g (8 = fp16 units) or ..., g, "x3"."""
    w = module.weight
    cache = module.__dict__.setdefault("_gb_packed", {})
    ver = (w._version, w.data_ptr(), str(w.device))
    hit = cache.get(key)
    if hit is None or hit[0] != ver:
        hit = (ver, make(w.detach()))
        cache[key] = hit
    return hit[1]


def _convt_supported(shape_bcdhw, module):
    b, c, d, h, w = shape_bcdhw
    k = module.kernel_size[0]
    if ("convt_k8" if k == 8 else "convt_k4") not in POLICY:
        return False
    return (ENABLED and tuple(module.kernel_size) == (k, k, k) and k in (4, 8) and tuple(module.stride) == (2, 2, 2)
            and tuple(module.padding) == (k // 2 - 1,) * 3 and tuple(module.output_padding) == (0, 0, 0)
            and tuple(module.dilation) == (1, 1, 1) and module.groups == 1 and w in (16, 32) and h % 16 == 0
            and c % (2 * _group()) == 0 and module.out_channels <= 64)


def convt3d_s2_blocked(src0, src1, batch, module, bn=None, slope=1.0):
    """Run the kernel on blocked operands (fp32 groups of 4 or fp16 groups of 8, matching PRECISION); returns the
    blocked fp32 output [B*2D, cgo, 2H, 2W, 4], or None when `bn` needs batch statistics."""
    src0, src1 = _x3_operands(src0, src1)
    bd, cg0, h, w, _ = src0.shape
    cg1 = src1.shape[1] if src1 is not None else 0
    cg0, cg1 = cg0 // _parts(), cg1 // _parts()
    cout = module.out_channels
    cgo = (cout + 3) // 4
    dev = src0.device
    g = 8 if src0.dtype == torch.float16 else 4
    merged = MERGE_PARITIES and module.kernel_size[0] == 8 and cout <= 20
    npad = 20 if merged else 32 if cout <= 32 else 64
    aff = _affine(module, bn, npad, dev)
    if aff is None:
        return None
    out = torch.empty((bd * 2, cgo, 2 * h, 2 * w, 4), device=dev, dtype=torch.float32)
    if merged:
        # the four (y,x) parity classes share one MMA stream: N = 4 x 20 columns (csrc/convt3d.cu MODE 2)
        wpack = _pack(module, ("convt_merged", 20, g), lambda wt: pack_convt_merged_weights(wt, 20, g), 2)
        _lib.call("genre_b200_convt3d_s2_merged_forward", src0.data_ptr(), cg0, src1.data_ptr() if src1 is not None else None,
                  cg1, batch, bd // batch, h, w, wpack.data_ptr(), 8, 80, _op_flag() if g == 8 else 0, aff[0].data_ptr(),
                  aff[1].data_ptr(), float(slope), out.data_ptr(), cgo, _lib.stream_ptr(src0))
        return out
    wpack = _pack(module, ("convt", npad, g), lambda wt: pack_convt_weights(wt, npad, g), 4)
    _lib.call("genre_b200_convt3d_s2_forward", src0.data_ptr(), cg0, src1.data_ptr() if src1 is not None else None, cg1,
              batch, bd // batch, h, w, wpack.data_ptr(), module.kernel_size[0], npad, _op_flag() if g == 8 else 0,
              aff[0].data_ptr(), aff[1].data_ptr(), float(slope), out.data_ptr(), cgo, _lib.stream_ptr(src0))
    return out


def _no_autograd(*tensors):
    """The kernels are forward-only: they run when no gradient is needed.  torch.backends.cudnn.allow_tf32 (PyTorch's own
    switch, on by default, for the cuDNN path they replace) selects the operand mode, see _mode()."""
    if not torch.backends.cudnn.allow_tf32 and not EXACT_WHEN_TF32_OFF:
        return False
    return not (torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors))


def space_to_depth_blocked(x, group=4, dtype=None, cpad=0):
    """NCDHW [B,C,D,H,W] (even extents, group | 8) -> blocked [B*D/2, C*8/group, H/2, W/2, group] whose channel
    index is ((c*2 + pz)*2 + py)*2 + px for input position (2z'+pz, 2y'+py, 2x'+px); cpad > 8C appends zero channels."""
    b, c, d, h, w = x.shape
    if group == 16:
        ncg = max(c * 8, cpad) // 8
        out = torch.empty((b * (d // 2), 2 * ncg, h // 2, w // 2, 8), device=x.device, dtype=torch.float16)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 1, 16, cpad if cpad > c * 8 else 0,
                  out.data_ptr(), _lib.stream_ptr(x))
        return out
    assert 8 % group == 0
    if _on_device(x, group, dtype):
        ncg = max(c * 8, cpad) // group
        out = torch.empty((b * (d // 2), ncg, h // 2, w // 2, group), device=x.device, dtype=dtype or x.dtype)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 1, group, cpad if cpad > c * 8 else 0,
                  out.data_ptr(), _lib.stream_ptr(x))
        return out
    if cpad > c * 8:
        y = space_to_depth_blocked(x, group, dtype)
        pad = y.new_zeros((y.shape[0], (cpad - c * 8) // group) + tuple(y.shape[2:]))
        return torch.cat((y, pad), dim=1)
    s = 8 // group                                       # channel groups per input channel
    # pz,py,px bits split as (j, e) with j the top log2(s) bits: view dims b c z' pz y' py x' px
    t = x.reshape(b, c, d // 2, 2, h // 2, 2, w // 2, 2)
    if s == 1:      # e = (pz,py,px)
        v = t.permute(0, 2, 1, 4, 6, 3, 5, 7)            # b z' c y' x' pz py px
    else:           # s == 2: j = pz, e = (py,px)
        v = t.permute(0, 2, 1, 3, 4, 6, 5, 7)            # b z' c pz y' x' py px
    return _permuted_copy(v, dtype).view(b * (d // 2), c * s, h // 2, w // 2, group)


def space_to_depth4_blocked(x, group=4, dtype=None):
    """NCDHW [B,C,D,H,W] (extents % 4 == 0) -> blocked [B*D/4, 64C/group, H/4, W/4, group], channel index
    ((c*4 + rz)*4 + ry)*4 + rx for input position (4z'+rz, 4y'+ry, 4x'+rx)."""
    b, c, d, h, w = x.shape
    if group == 16:
        out = torch.empty((b * (d // 4), 2 * (c * 64 // 8), h // 4, w // 4, 8), device=x.device, dtype=torch.float16)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 3, 16, 0, out.data_ptr(), _lib.stream_ptr(x))
        return out
    out_shape = (b * (d // 4), c * 64 // group, h // 4, w // 4, group)
    if _on_device(x, group, dtype):
        out = torch.empty(out_shape, device=x.device, dtype=dtype or x.dtype)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 3, group, 0, out.data_ptr(), _lib.stream_ptr(x))
        return out
    t = x.reshape(b, c, d // 4, 4, h // 4, 4, w // 4, 4).permute(0, 2, 1, 3, 5, 7, 4, 6)   # b z' c rz ry rx y' x'
    t = t.reshape(b * (d // 4), c * 64 // group, group, h // 4, w // 4).permute(0, 1, 3, 4, 2)
    return _permuted_copy(t, dtype)


def pack_conv_k8s2_s4d_weights(weight, cpad, group=4, split_z=False):
    """Conv3d weight [Cout, Cin, 8, 8, 8] (stride 2, padding 3) -> the 3-tap stride-1 convolution over the 64*Cin
    4x-space-to-depth channels whose N = 8*cpad columns are the 8 output classes q of the 2x finer output grid:
    [3 z-tap][chunk][9 taps][2][N/8][8][g].  Per dimension: output 2j+q reads input 4j + 2q - 3 + k; coarse cell
    j + 1 - t, sub-position r  =>  k = 7 - 4t + r - 2q (zero weight when outside [0, 8))."""
    cout, cin = weight.shape[0], weight.shape[1]
    g, n = group, 8 * cpad
    q = torch.arange(2).view(2, 1, 1)
    t = torch.arange(3).view(1, 3, 1)
    r = torch.arange(4).view(1, 1, 4)
    k = 7 - 4 * t + r - 2 * q                                             # [q, t, r]
    valid = ((k >= 0) & (k < 8)).to(weight.device)
    kc = k.clamp(0, 7).to(weight.device)
    kz, vz = kc.view(2, 3, 4, 1, 1, 1, 1, 1, 1), valid.view(2, 3, 4, 1, 1, 1, 1, 1, 1)
    ky, vy = kc.view(1, 1, 1, 2, 3, 4, 1, 1, 1), valid.view(1, 1, 1, 2, 3, 4, 1, 1, 1)
    kx, vx = kc.view(1, 1, 1, 1, 1, 1, 2, 3, 4), valid.view(1, 1, 1, 1, 1, 1, 2, 3, 4)
    full = weight[:, :, kz, ky, kx] * (vz & vy & vx).to(weight.dtype)      # [co, c, qz,tz,rz, qy,ty,ry, qx,tx,rx]
    weq = full.permute(1, 4, 7, 10, 2, 5, 8, 0, 3, 6, 9)                  # c rz ry rx | qz qy qx co | tz ty tx
    weq = torch.nn.functional.pad(weq, (0, 0, 0, 0, 0, 0, 0, cpad - cout)).reshape(cin * 64, n, 3, 3, 3)
    if split_z:   # [2 qz] x the 4-class (y,x) form: N = 4*cpad columns per z class
        sub = weq.reshape(cin * 64 // (2 * g), 2, g, 2, n // 16, 8, 3, 3, 3)   # (kc, kk, e, qz, ng, r, tz, ty, tx)
        out = sub.permute(3, 6, 0, 7, 8, 1, 4, 5, 2).contiguous()              # (qz, tz, kc, ty, tx, kk, ng, r, e)
        return _finish_pack(out, g)
    sub = weq.reshape(cin * 64 // (2 * g), 2, g, n // 8, 8, 3, 3, 3)      # (kc, kk, e, ng, r, tz, ty, tx)
    out = sub.permute(5, 0, 6, 7, 1, 3, 4, 2).contiguous()                # (tz, kc, ty, tx, kk, ng, r, e)
    return _finish_pack(out, g)


def pack_conv_k4s2_s2d_weights(weight, cpad, npad, group=4):
    """Conv3d weight [Cout, Cin, 4, 4, 4] (stride 2, padding 1), FEW input channels -> the 3-tap stride-1 convolution over the
    8*Cin space-to-depth channels (zero-padded to cpad): [3 z-tap][cpad/(2g)][9 taps][2][npad/8][8][g].  Per dimension:
    output o reads input 2o - 1 + k = 2(o + 1 - t) + r  =>  k = 3 - 2t + r (zero weight outside [0, 4))."""
    cout, cin = weight.shape[0], weight.shape[1]
    g = group
    t = torch.arange(3).view(3, 1)
    r = torch.arange(2).view(1, 2)
    k = 3 - 2 * t + r                                                       # [t, r]
    valid = ((k >= 0) & (k < 4)).to(weight.device)
    kc = k.clamp(0, 3).to(weight.device)
    kz, vz = kc.view(3, 2, 1, 1, 1, 1), valid.view(3, 2, 1, 1, 1, 1)
    ky, vy = kc.view(1, 1, 3, 2, 1, 1), valid.view(1, 1, 3, 2, 1, 1)
    kx, vx = kc.view(1, 1, 1, 1, 3, 2), valid.view(1, 1, 1, 1, 3, 2)
    full = weight[:, :, kz, ky, kx] * (vz & vy & vx).to(weight.dtype)        # [co, c, tz,rz, ty,ry, tx,rx]
    weq = full.permute(1, 3, 5, 7, 0, 2, 4, 6).reshape(cin * 8, cout, 3, 3, 3)   # (c rz ry rx | co | tz ty tx)
    weq = torch.nn.functional.pad(weq, (0, 0, 0, 0, 0, 0, 0, npad - cout, 0, cpad - cin * 8))
    sub = weq.reshape(cpad // (2 * g), 2, g, npad // 8, 8, 3, 3, 3)          # (kc, kk, e, ng, r, tz, ty, tx)
    out = sub.permute(5, 0, 6, 7, 1, 3, 4, 2).contiguous()                   # (tz, kc, ty, tx, kk, ng, r, e)
    return _finish_pack(out, g)


def _conv_k4s2_s2d_supported(x, m):
    """few input channels (the critic's 1 -> 64 first layer): the 8*Cin space-to-depth channels fit one K chunk"""
    return ("conv_k4s2_s2d" in POLICY and ENABLED and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
            and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2) and tuple(m.padding) == (1, 1, 1)
            and tuple(m.dilation) == (1, 1, 1) and m.groups == 1 and m.padding_mode == "zeros" and x.shape[1] <= 2
            and 32 < m.out_channels <= 64 and all(v % 2 == 0 for v in x.shape[2:]) and x.shape[4] // 2 in (16, 32, 64)
            and (x.shape[3] // 2) % 16 == 0)


def _conv_k4s2_s2d(x, m, bn, slope):
    cout, npad, g = m.out_channels, 64, _group()
    aff = _affine(m, bn, npad, x.device)
    if aff is None:
        return None
    cpad = -(-x.shape[1] * 8 // (2 * g)) * 2 * g          # the 8*Cin channels rounded up to whole K chunks
    wpack = _pack(m, ("k4s2_s2d", cpad, npad, g), lambda w: pack_conv_k4s2_s2d_weights(w, cpad, npad, g), 1)
    if _x2_direct(x):
        xb = space_to_depth_blocked(x, 16, torch.float16, cpad)
    else:
        xb = _finish_operand(space_to_depth_blocked(x, _act_group(), torch.float16 if _f16() else None, cpad))
    b = x.shape[0]
    bd, cg, h, w, _ = xb.shape
    cgo = (cout + 3) // 4
    out = torch.empty((bd, cgo, h, w, 4), device=x.device, dtype=torch.float32)
    _lib.call("genre_b200_conv3d_taps_forward", xb.data_ptr(), cg // _parts(), None, 0, b, bd // b, h, w, wpack.data_ptr(), 3, 1, npad,
              _op_flag(), aff[0].data_ptr(), aff[1].data_ptr(), 1.0 if slope is None else float(slope),
              out.data_ptr(), cgo, _lib.stream_ptr(x))
    return from_blocked(out, b, cout)


def pack_conv_k8s2_weights(weight, npad, group=4):
    """Conv3d weight [Cout, Cin, 8, 8, 8] (stride 2, padding 3) -> the equivalent 5-tap stride-1 convolution over the
    8*Cin space-to-depth channels, packed per stage: [5 z-tap][Cin chunk][25 taps][2][npad/8][8][4].
    Input index 2(o+delta)+pi = 2o - 3 + k  =>  k = 2 delta + 3 + pi, delta = 2 - t (kernel: input = j + 2 - t)."""
    cout, cin = weight.shape[0], weight.shape[1]
    t5 = 5
    weq = weight.new_zeros((cin, 2, 2, 2, npad, t5, t5, t5))   # (ci, pz, py, px, n, tz, ty, tx)
    for pz in (0, 1):
        for py in (0, 1):
            for px in (0, 1):
                for tz in range(t5):
                    kz = 2 * (2 - tz) + 3 + pz
                    if not 0 <= kz < 8:
                        continue
                    for ty in range(t5):
                        ky = 2 * (2 - ty) + 3 + py
                        if not 0 <= ky < 8:
                            continue
                        for tx in range(t5):
                            kx = 2 * (2 - tx) + 3 + px
                            if 0 <= kx < 8:
                                weq[:, pz, py, px, :cout, tz, ty, tx] = weight[:, :, kz, ky, kx].t()
    ceq, g = cin * 8, group
    sub = weq.reshape(ceq // (2 * g), 2, g, npad // 8, 8, t5, t5, t5)      # (kc, kk, e, ng, r, tz, ty, tx)
    out = sub.permute(5, 0, 6, 7, 1, 3, 4, 2).contiguous()                # (tz, kc, ty, tx, kk, ng, r, e)
    return _finish_pack(out, g)


def _packed_conv(module, npad):
    g = _group()
    return _pack(module, ("k8s2", npad, g), lambda w: pack_conv_k8s2_weights(w, npad, g), 1)


def _conv_k8s2_supported(x, m):
    return ("conv_k8s2" in POLICY and ENABLED and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and tuple(m.kernel_size) == (8, 8, 8)
            and tuple(m.stride) == (2, 2, 2) and tuple(m.padding) == (3, 3, 3) and tuple(m.dilation) == (1, 1, 1)
            and m.groups == 1 and m.out_channels <= 32 and x.shape[1] % 2 == 0 and x.shape[1] <= 8
            and all(v % 2 == 0 for v in x.shape[2:]) and x.shape[4] // 2 in (16, 32, 64) and (x.shape[3] // 2) % 16 == 0
            and m.padding_mode == "zeros")


def space_to_depth_sources(x, cpad, group, dtype):
    """NCDHW [B,C,D,H,W] (even extents) -> [B*D/2, 8*cpad/group, H/2, W/2, group]: the 8 parity sub-volumes one after the
    other along the channel-group axis (sub-volume s = (pz*2+py)*2+px holds in[2z'+pz, 2y'+py, 2x'+px]), each zero-padded
    from C to cpad channels."""
    b, c, d, h, w = x.shape
    if group == 16:
        out = torch.empty((b * (d // 2), 2 * 8 * (cpad // 8), h // 2, w // 2, 8), device=x.device, dtype=torch.float16)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 2, 16, cpad, out.data_ptr(), _lib.stream_ptr(x))
        return out
    if _on_device(x, group, dtype):
        out = torch.empty((b * (d // 2), 8 * (cpad // group), h // 2, w // 2, group), device=x.device, dtype=dtype or x.dtype)
        _lib.call("genre_b200_ncdhw_to_blocked", x.data_ptr(), b, c, d, h, w, 2, group, cpad, out.data_ptr(), _lib.stream_ptr(x))
        return out
    if cpad != c:
        x = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, 0, 0, cpad - c))
    t = x.reshape(b, cpad // group, group, d // 2, 2, h // 2, 2, w // 2, 2)      # b cg e z' pz y' py x' px
    v = t.permute(0, 3, 4, 6, 8, 1, 5, 7, 2)                                      # b z' pz py px cg y' x' e
    return _permuted_copy(v, dtype).view(b * (d // 2), 8 * (cpad // group), h // 2, w // 2, group)


def pack_conv_k4s2_weights(weight, cpad, npad, group):
    """Conv3d weight [Cout, Cin, 4, 4, 4] (stride 2, padding 1) -> [2 z-tap][8*cpad/(2g) chunk][4 taps][2][npad/8][8][g]:
    sub-volume s = (pz,py,px) and tap t use kernel index k = 3 - 2t - p per dimension."""
    cout, cin = weight.shape[0], weight.shape[1]
    g = group
    weq = weight.new_zeros((8, cpad, npad, 2, 2, 2))                              # (s, ci, n, tz, ty, tx)
    for pz in (0, 1):
        for py in (0, 1):
            for px in (0, 1):
                sidx = (pz * 2 + py) * 2 + px
                for tz in (0, 1):
                    for ty in (0, 1):
                        for tx in (0, 1):
                            weq[sidx, :cin, :cout, tz, ty, tx] = weight[:, :, 3 - 2 * tz - pz, 3 - 2 * ty - py, 3 - 2 * tx - px].t()
    sub = weq.reshape(8 * cpad // (2 * g), 2, g, npad // 8, 8, 2, 2, 2)           # (kc, kk, e, ng, r, tz, ty, tx)
    out = sub.permute(5, 0, 6, 7, 1, 3, 4, 2).contiguous()                        # (tz, kc, ty, tx, kk, ng, r, e)
    return _finish_pack(out, g)


def _conv_k4s2_supported(x, m):
    return ("conv_k4s2" in POLICY and ENABLED and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and tuple(m.kernel_size) == (4, 4, 4)
            and tuple(m.stride) == (2, 2, 2) and tuple(m.padding) == (1, 1, 1) and tuple(m.dilation) == (1, 1, 1)
            and m.groups == 1 and m.out_channels <= 128 and x.shape[1] >= K4S2_MIN_CIN and m.padding_mode == "zeros"
            and all(v % 2 == 0 for v in x.shape[2:]) and x.shape[4] // 2 in (16, 32) and (x.shape[3] // 2) % 16 == 0)


def _versions(*tensors):
    return tuple((t._version, t.data_ptr()) if t is not None else None for t in tensors)


def _affine(m, bn, npad, dev):
    """(scale, shift) [npad] of the epilogue: bias, and eval-mode BatchNorm folded in; None if bn needs batch statistics.
    Cached on the conv module until one of the source tensors is modified in place or replaced."""
    cout = m.out_channels
    if bn is not None and (bn.training or not bn.track_running_stats):
        return None
    ver = (_versions(m.bias, *((bn.running_mean, bn.running_var, bn.weight, bn.bias) if bn is not None else ())),
           bn.eps if bn is not None else None, str(dev))
    cache = m.__dict__.setdefault("_gb_affine", {})
    hit = cache.get(npad)
    if hit is not None and hit[0] == ver:
        return hit[1]
    scale = shift = None
    with torch.no_grad():
        if bn is not None:
            inv = torch.rsqrt(bn.running_var + bn.eps)
            scale = inv * (bn.weight if bn.weight is not None else 1.0)
            bias = m.bias.detach() if m.bias is not None else torch.zeros_like(bn.running_mean)
            shift = (bias - bn.running_mean) * scale + (bn.bias if bn.bias is not None else 0.0)
        sc = torch.ones(npad, device=dev) if scale is None else torch.nn.functional.pad(scale.float(), (0, npad - cout), value=1.0)
        if shift is None:
            shift = m.bias.detach() if m.bias is not None else torch.zeros(cout, device=dev)
        out = (sc.contiguous(), torch.nn.functional.pad(shift.float(), (0, npad - cout)).contiguous())
    cache[npad] = (ver, out)
    return out


def _conv_k4s2(x, m, bn, slope):
    cout = m.out_channels
    npad = 32 * ((cout + 31) // 32)
    aff = _affine(m, bn, npad, x.device)
    if aff is None:
        return None
    g = _group()
    cin = x.shape[1]
    cpad = (cin + 2 * g - 1) // (2 * g) * (2 * g)      # a K chunk (2 channel groups) must not straddle sub-volumes
    wpack = _pack(m, ("k4s2", cpad, npad, g), lambda w: pack_conv_k4s2_weights(w, cpad, npad, g), 1)
    if _x2_direct(x):
        xb = space_to_depth_sources(x, cpad, 16, torch.float16)
    else:
        xb = _finish_operand(space_to_depth_sources(x, cpad, _act_group(), torch.float16 if _f16() else None))
    b = x.shape[0]
    bd, _, h, wd, _ = xb.shape
    cgo = (cout + 3) // 4
    out = torch.empty((bd, cgo, h, wd, 4), device=x.device, dtype=torch.float32)
    _lib.call("genre_b200_conv3d_k4s2_forward", xb.data_ptr(), cpad // g, 3 if _x3() else 1, b, bd // b, h, wd, wpack.data_ptr(), npad,
              _op_flag(), aff[0].data_ptr(), aff[1].data_ptr(), 1.0 if slope is None else float(slope),
              out.data_ptr(), cgo, _lib.stream_ptr(x))
    return from_blocked(out, b, cout)


# ---- small volumes: the flattened, zero-separated implicit GEMM (csrc/convflat.cu) ------------------------------------------
FLAT_MAX = int(os.environ.get("GENRE_B200_CONV_FLAT_MAX", "8"))      # coarse-side extent routed to the flat kernel (larger planes belong to the halo kernels of csrc/convt3d.cu)


def flat_npad(cout):
    """accumulator tile width: the one of {64, 80} that pads Cout least (80 on a tie: fewer N tiles)"""
    return 64 if -(-cout // 64) * 64 < -(-cout // 80) * 80 else 80


def flat_shifts(h, w, transposed):
    """[8 groups][8 taps] position shifts of csrc/convflat.cu (group = output parity class of a transposed conv, or input
    sub-volume of a strided conv; tap t = (tz,ty,tx); bit 2 = z) in a volume whose rows / planes are w+1 / (h+1)(w+1) positions"""
    table = []
    for g in range(8):
        row = []
        for t in range(8):
            d = []
            for k in range(3):
                par, tt = (g >> (2 - k)) & 1, (t >> (2 - k)) & 1
                d.append(((1 - tt) if par else -tt) if transposed else 1 - par - tt)
            row.append(d[0] * (h + 1) * (w + 1) + d[1] * (w + 1) + d[2])
        table.append(row)
    return table


def pack_flat_convt_weights(weight, npad, group=8):
    """ConvTranspose3d weight [Cin, Cout, 4, 4, 4] (stride 2, padding 1) ->
    [8 class][ntile][ceil(Cin/16) K step][8 taps][2 kcore][npad/8][8 n][8 k]: class parity p, tap t reads the input at shift
    d = (1 - t if p else -t), kernel index k = p + 1 - 2 d, per dimension."""
    cin, cout = weight.shape[0], weight.shape[1]
    cpad, nt = -(-cin // 16) * 16, -(-cout // npad)
    weq = weight.new_zeros((8, 8, cpad, nt * npad))                               # (class, tap, ci, n)

    def kidx(par, t):
        return par + 1 - 2 * ((1 - t) if par else -t)
    for cls in range(8):
        for tap in range(8):
            kz, ky, kx = (kidx((cls >> (2 - k)) & 1, (tap >> (2 - k)) & 1) for k in range(3))
            weq[cls, tap, :cin, :cout] = weight[:, :, kz, ky, kx]
    sub = weq.reshape(8, 8, cpad // 16, 2, 8, nt, npad // 8, 8)                   # (class, tap, kc, kk, e, ntile, ng, r)
    return _finish_pack(sub.permute(0, 5, 2, 1, 3, 6, 7, 4).contiguous(), group)  # (class, ntile, kc, tap, kk, ng, r, e)


def pack_flat_conv_weights(weight, npad, group=8):
    """Conv3d weight [Cout, Cin, 4, 4, 4] (stride 2, padding 1, Cin % 16 == 0) -> [1][ntile][8*Cin/16 K step][8 taps][2][npad/8][8][8]:
    K = the 8 parity sub-volumes of the input, sub-volume parity p and tap t use kernel index 3 - 2t - p (shift 1 - p - t)."""
    cout, cin = weight.shape[0], weight.shape[1]
    nt = -(-cout // npad)
    weq = weight.new_zeros((8, 8, cin, nt * npad))                                # (tap, sub-volume, ci, n)
    for sv in range(8):
        for tap in range(8):
            kz, ky, kx = (3 - 2 * ((tap >> (2 - k)) & 1) - ((sv >> (2 - k)) & 1) for k in range(3))
            weq[tap, sv, :, :cout] = weight[:, :, kz, ky, kx].t()
    sub = weq.reshape(8, 8 * cin // 16, 2, 8, nt, npad // 8, 8)                   # (tap, kc, kk, e, ntile, ng, r)
    return _finish_pack(sub.permute(4, 1, 0, 2, 5, 6, 3).contiguous().unsqueeze(0), group)


def _flat_common(m):
    return ("flat" in POLICY and ENABLED and (_f16() or _x2()) and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2)
            and tuple(m.padding) == (1, 1, 1) and tuple(m.dilation) == (1, 1, 1) and m.groups == 1
            and m.out_channels >= 8)     # fewer output channels: the one-channel kernels (an N tile here is 64 columns)


def _flat_source_ok(x):
    return torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.shape[1] % 8 == 0


def _flat_convt_supported(sources, m):
    return (isinstance(m, torch.nn.ConvTranspose3d) and _flat_common(m) and tuple(m.output_padding) == (0, 0, 0)
            and all(_flat_source_ok(x) and x.shape[2:] == sources[0].shape[2:] and x.shape[0] == sources[0].shape[0] for x in sources)
            and max(sources[0].shape[2:]) <= FLAT_MAX and sum(x.shape[1] for x in sources) == m.in_channels
            and _no_autograd(*sources, m.weight, m.bias))


def _flat_conv_supported(x, m):
    return (isinstance(m, torch.nn.Conv3d) and _flat_common(m) and m.padding_mode == "zeros" and _flat_source_ok(x)
            and x.shape[1] % 16 == 0 and x.shape[1] == m.in_channels and all(v % 2 == 0 for v in x.shape[2:])
            and max(x.shape[2:]) <= 2 * FLAT_MAX and _no_autograd(x, m.weight, m.bias))


def _flat_run(sources, m, bn, slope, transposed):
    cout = m.out_channels
    npad = flat_npad(cout)
    dev = sources[0].device
    aff = _affine(m, bn, -(-cout // npad) * npad, dev)
    if aff is None:
        return None
    b = sources[0].shape[0]
    if transposed:
        d, h, w = sources[0].shape[2:]
        groups = sum(x.shape[1] for x in sources) // 8
        wpack = _pack(m, ("flat_convt", npad, 8), lambda wt: pack_flat_convt_weights(wt, npad), 2)
    else:
        d, h, w = (v // 2 for v in sources[0].shape[2:])
        groups = sources[0].shape[1]
        wpack = _pack(m, ("flat_conv", npad, 8), lambda wt: pack_flat_conv_weights(wt, npad), 2)
    cgs = groups + (groups & 1)
    parts = _parts()
    positions = _lib.load().genre_b200_convflat_positions(b, d, h, w, None)
    operand = torch.empty((parts, cgs, positions, 8), device=dev, dtype=torch.float16)
    st = _lib.stream_ptr(sources[0])
    off = 0
    for x in sources:
        x = x.contiguous()
        _lib.call("genre_b200_convflat_pack", x.data_ptr(), x.shape[1], b, d, h, w, 0 if transposed else 1, operand.data_ptr(), off, cgs,
                  parts, 0, st)
        off += x.shape[1] // 8 if transposed else x.shape[1]
    if off < cgs:
        _lib.call("genre_b200_convflat_pack", None, 0, b, d, h, w, 0, operand.data_ptr(), off, cgs, parts, cgs - off, st)
    od, oh, ow = (2 * d, 2 * h, 2 * w) if transposed else (d, h, w)
    out = torch.empty((b, cout, od, oh, ow), device=dev, dtype=torch.float32)
    _lib.call("genre_b200_convflat_forward", operand.data_ptr(), cgs, b, d, h, w, 1 if transposed else 0, wpack.data_ptr(), npad,
              _op_flag(), aff[0].data_ptr(), aff[1].data_ptr(), 1.0 if slope is None else float(slope), out.data_ptr(), cout, st)
    return out


# ---- the 1^3 end of the U-Net: weight-streaming FP32 products (csrc/skinny_gemm.cu) ------------------------------------------
def _skinny_ok(x, m):
    return ("skinny" in POLICY and ENABLED and torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
            and m.groups == 1 and tuple(m.dilation) == (1, 1, 1) and tuple(m.padding) == (0, 0, 0) and m.weight.dtype == torch.float32
            and not (torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (x, m.weight, m.bias))))


def _skinny_conv_supported(x, m):
    """Conv3d whose kernel is its whole input: one output voxel per (sample, channel)"""
    return (isinstance(m, torch.nn.Conv3d) and _skinny_ok(x, m) and m.padding_mode == "zeros" and tuple(x.shape[2:]) == tuple(m.kernel_size)
            and x.shape[1] == m.in_channels and (x.shape[1] * x.shape[2] * x.shape[3] * x.shape[4]) % 4 == 0)


def _skinny_convt_supported(x, m):
    """ConvTranspose3d of a 1^3 input: the output is the kernel weighted by the input channels"""
    return (isinstance(m, torch.nn.ConvTranspose3d) and _skinny_ok(x, m) and tuple(x.shape[2:]) == (1, 1, 1) and x.shape[1] == m.in_channels
            and tuple(m.output_padding) == (0, 0, 0) and (m.out_channels * m.kernel_size[0] * m.kernel_size[1] * m.kernel_size[2]) % 4 == 0)


def _aligned(t):
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _skinny_run(x, m, bn, slope, transposed):
    cout = m.out_channels
    aff = _affine(m, bn, cout, x.device)
    if aff is None:
        return None
    b = x.shape[0]
    x2 = _aligned(x.reshape(b, -1))
    w = _aligned(m.weight.detach())
    k = x2.shape[1]
    if transposed:
        kvol = m.kernel_size[0] * m.kernel_size[1] * m.kernel_size[2]
        n, div, shape = cout * kvol, kvol, (b, cout) + tuple(m.kernel_size)
    else:
        n, div, shape = cout, 1, (b, cout, 1, 1, 1)
    nbytes = _lib.load().genre_b200_skinny_gemm_workspace_bytes(b, n, k, 0 if transposed else 1)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    out = torch.empty(shape, device=x.device, dtype=torch.float32)
    _lib.call("genre_b200_skinny_gemm", x2.data_ptr(), w.data_ptr(), b, n, k, 0 if transposed else 1, div, aff[0].data_ptr(),
              aff[1].data_ptr(), 1.0 if slope is None else float(slope), out.data_ptr(), ws.data_ptr(), nbytes, _lib.stream_ptr(x))
    return out


def _needs_grad(*tensors):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


class _ConvInputGrad(torch.autograd.Function):
    """Input gradient of a Conv3d as a differentiable node of its own, used when the first backward is recorded
    (create_graph=True: WGAN-GP's gradient penalty, wgangp.py:144-164).  Its derivative with respect to the incoming
    gradient is the layer's FORWARD convolution applied to the grad-of-grad, which autograd would otherwise hand to cuDNN
    (for the critic's layers: three 35 ms kernels, 106 of the 142 ms of a critic step at B=8); here it runs on the custom
    forward kernel."""

    @staticmethod
    def forward(ctx, gy, weight, x, m):
        conf = (list(m.stride), list(m.padding), list(m.dilation), False, [0, 0, 0], m.groups)
        with cudnn_precision():
            gx, _, _ = torch.ops.aten.convolution_backward(gy, x, weight, None, *conf, [True, False, False])
        ctx.save_for_backward(gy, weight)
        ctx.m, ctx.conf = m, conf
        return gx

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, ggx):
        gy, weight = ctx.saved_tensors
        m = ctx.m
        ggx = ggx.contiguous()
        g_gy = g_w = None
        if ctx.needs_input_grad[0]:
            # no grad mode here: the custom forward kernel (bias is not part of it).  Grad-of-grads of a penalty are ~1e-4..1e-7:
            # never fp16 operands (subnormal / flushed), TF32 at least (the exact modes stay exact)
            with _forced_mode("tf32"):
                g_gy = conv3d(ggx, m)
            if g_gy is None:
                with cudnn_precision():
                    g_gy = torch.nn.functional.conv3d(ggx, weight, None, m.stride, m.padding, m.dilation, m.groups)
            elif m.bias is not None:
                g_gy = g_gy - m.bias.detach().view(1, -1, 1, 1, 1)
        if ctx.needs_input_grad[1]:
            with cudnn_precision():
                _, g_w, _ = torch.ops.aten.convolution_backward(gy, ggx, weight, None, *ctx.conf, [False, True, False])
        return g_gy, g_w, None, None


# Input gradients of the two k=8 layers of Unet_3D on the tensor cores (first-order backward only).  On by default since
# round 2 (GPU-validated: tests/test_gpu_conv.py::test_tensor_core_input_gradients_of_the_k8_layers); GENRE_B200_CONV_TC_BACKWARD=0
# hands them back to cuDNN.
TC_BACKWARD = os.environ.get("GENRE_B200_CONV_TC_BACKWARD", "1") != "0"


def dgrad_convt_k8s2(gy, m):
    """Input gradient of ConvTranspose3d(Cin -> Cout, k8, s2, p3) (Unet_3D.dec5, networks.py:166): out[2i-3+k] += x[i] W[ci,co,k]
    =>  dx[ci, i] = sum_{co,k} gy[co, 2i - 3 + k] W[ci, co, k] = Conv3d(Cout -> Cin, k8, s2, p3) of gy with the SAME weight
    tensor read as [out = Cin, in = Cout, 8, 8, 8]: the 5-tap form over the 2x space-to-depth of gy (kernel MODE 1, N = 96)."""
    cin_t, cout_t = m.in_channels, m.out_channels
    b, _, d, h, w = gy.shape
    if not (gy.is_cuda and gy.dtype == torch.float32 and cin_t <= 96 and (cout_t * 8) % 8 == 0 and d % 2 == 0 and h % 32 == 0
            and (w // 2) in (16, 32, 64)):
        return None
    with torch.no_grad(), _forced_mode("tf32"):
        g = _group()
        wpack = _pack(m, ("dgrad_k8s2", 96, g), lambda wt: pack_conv_k8s2_weights(wt, 96, g), 1)
        xb = space_to_depth_blocked(gy.contiguous(), g)
        if _x3():
            xb = _split3(xb)
        bd, cg, hh, ww, _ = xb.shape
        cgo = (cin_t + 3) // 4
        one = m.__dict__.get("_gb_dgrad_affine")
        if one is None or one[0].device != gy.device:
            one = m.__dict__["_gb_dgrad_affine"] = (torch.ones(96, device=gy.device), torch.zeros(96, device=gy.device))
        out = torch.empty((bd, cgo, hh, ww, 4), device=gy.device, dtype=torch.float32)
        _lib.call("genre_b200_conv3d_taps_forward", xb.data_ptr(), cg, None, 0, b, bd // b, hh, ww, wpack.data_ptr(), 5, 2, 96,
                  0, one[0].data_ptr(), one[1].data_ptr(), 1.0, out.data_ptr(), cgo, _lib.stream_ptr(gy))
        dx = from_blocked(out, b, cin_t)
        dx.__dict__.pop("_gb_blocked", None)
        return dx


def dgrad_conv_k8s2(gy, m):
    """Input gradient of Conv3d(Cin -> Cout, k8, s2, p3) with Cin <= 20 (Unet_3D.enc1, networks.py:151) = ConvTranspose3d(Cout ->
    Cin, k8, s2, p3) of gy with the SAME weight tensor read as [in = Cout, out = Cin, 8, 8, 8]: the merged-parity kernel
    (MODE 2) over 32-wide x tiles.  Cout is zero-padded to a multiple of 8 (whole K chunks)."""
    cin, cout = m.in_channels, m.out_channels
    b, _, d, h, w = gy.shape
    if not (gy.is_cuda and gy.dtype == torch.float32 and cin <= 20 and h % 16 == 0 and (w == 16 or w % 32 == 0)):
        return None
    pad = (-cout) % 8
    with torch.no_grad(), _forced_mode("tf32"):
        g = _group()
        wpack = _pack(m, ("dgrad_convt_merged", 20, g, pad),
                      lambda wt: pack_convt_merged_weights(torch.nn.functional.pad(wt, (0, 0) * 4 + (0, pad)), 20, g), 2)
        gyp = torch.nn.functional.pad(gy, (0, 0) * 3 + (0, pad)) if pad else gy
        src, _ = _x3_operands(to_blocked(gyp.contiguous(), g), None)
        bd, cg, hh, ww, _ = src.shape
        cgo = (cin + 3) // 4
        one = m.__dict__.get("_gb_dgrad_affine")
        if one is None or one[0].device != gy.device:
            one = m.__dict__["_gb_dgrad_affine"] = (torch.ones(96, device=gy.device), torch.zeros(96, device=gy.device))
        out = torch.empty((bd * 2, cgo, 2 * hh, 2 * ww, 4), device=gy.device, dtype=torch.float32)
        _lib.call("genre_b200_convt3d_s2_merged_forward", src.data_ptr(), cg, None, 0, b, bd // b, hh, ww, wpack.data_ptr(), 8, 80,
                  0, one[0].data_ptr(), one[1].data_ptr(), 1.0, out.data_ptr(), cgo, _lib.stream_ptr(gy))
        dx = from_blocked(out, b, cin)
        dx.__dict__.pop("_gb_blocked", None)
        return dx


class _ConvForward(torch.autograd.Function):
    """Training: the FORWARD of a convolution on the custom kernel (conv + bias only; BatchNorm with batch statistics and
    the activation stay torch modules), the backward on cuDNN through aten::convolution_backward.  The forward is where
    cuDNN is furthest off its pace on these layers (Unet_3D.enc1 16.6 ms, dec5 7.3 ms at B=16)."""

    @staticmethod
    def forward(ctx, x, weight, bias, m):
        transposed = isinstance(m, torch.nn.ConvTranspose3d)
        with torch.no_grad():
            y = (conv_transpose3d if transposed else conv3d)(x.detach(), m)
        if y is None:
            raise RuntimeError("ops_conv: layer not covered (the dispatcher checks support before taking this route)")
        ctx.save_for_backward(x, weight)
        ctx.module = m
        ctx.conf = (transposed, tuple(m.stride), tuple(m.padding), tuple(m.dilation),
                    tuple(m.output_padding) if transposed else (0, 0, 0), m.groups,
                    [m.out_channels] if bias is not None else None)
        y.__dict__.pop("_gb_blocked", None)        # the blocked twin must not ride along into autograd-land
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        transposed, stride, padding, dilation, out_pad, groups, bias_sizes = ctx.conf
        mask = [ctx.needs_input_grad[0], ctx.needs_input_grad[1], bias_sizes is not None and ctx.needs_input_grad[2]]
        gy = gy.contiguous()
        gw_custom = None
        if (mask[1] and not transposed and not torch.is_grad_enabled() and "conv_k8s2_wgrad" in POLICY
                and tuple(weight.shape[2:]) == (8, 8, 8) and stride == (2, 2, 2) and padding == (3, 3, 3)
                and dilation == (1, 1, 1) and groups == 1 and weight.shape[1] <= 2 and weight.shape[0] <= 20
                and x.shape[3] % 16 == 0 and x.shape[4] <= 128 and x.shape[2] % 2 == 0 and x.shape[4] % 2 == 0):
            # Unet_3D.enc1: cuDNN's wgrad for this shape is a 40 ms grouped direct kernel (csrc/convt_c1_wgrad.cu)
            xc = x.contiguous()
            nbytes = _lib.load().genre_b200_conv_k8s2_wgrad_workspace_bytes()
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            gw_custom = torch.empty_like(weight)
            _lib.call("genre_b200_conv_k8s2_wgrad", xc.data_ptr(), gy.data_ptr(), x.shape[0], weight.shape[1], weight.shape[0],
                      x.shape[2], x.shape[3], x.shape[4], gw_custom.data_ptr(), ws.data_ptr(), nbytes, _lib.stream_ptr(x))
            mask[1] = False
        gx = gw = gb = None
        gx_custom = None
        if (TC_BACKWARD and mask[0] and not torch.is_grad_enabled() and ctx.module is not None
                and tuple(weight.shape[2:]) == (8, 8, 8) and stride == (2, 2, 2) and padding == (3, 3, 3) and groups == 1
                and dilation == (1, 1, 1) and out_pad == (0, 0, 0)):
            gx_custom = (dgrad_convt_k8s2 if transposed else dgrad_conv_k8s2)(gy, ctx.module)
            if gx_custom is not None:
                mask[0] = False
        if mask[0] and torch.is_grad_enabled() and not transposed and ctx.module is not None:
            gx_custom = _ConvInputGrad.apply(gy, weight, x, ctx.module)   # double backward stays on the custom forward
            mask[0] = False
        if any(mask):
            with cudnn_precision():
                gx, gw, gb = torch.ops.aten.convolution_backward(gy, x, weight, bias_sizes, list(stride), list(padding),
                                                                  list(dilation), transposed, list(out_pad), groups, mask)
        return (gx_custom if gx_custom is not None else gx), (gw_custom if gw_custom is not None else gw), gb, None


class _ConvTC1Train(torch.autograd.Function):
    """ConvTranspose3d(Cin -> 1, k4, s2, p1) under autograd (Unet_3D.dec6 and the decoders' last layers in training).
    cuDNN's weight gradient for this 1-channel layer is a grouped direct kernel that takes 40.7 of the 60 ms of a Unet_3D
    training step at B=4; here forward = the exact-fp32 FP32-pipe stencil (csrc/convt_c1.cu), input and weight gradients
    = csrc/convt_c1_wgrad.cu (deterministic), bias gradient = a sum."""

    @staticmethod
    def forward(ctx, x, weight, bias, m):
        with torch.no_grad():
            xd = x.detach().contiguous()
            y = convt_c1(to_blocked(xd, 4), None, xd.shape[0], m)
        ctx.save_for_backward(xd, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        b, cin, d, h, w = x.shape
        st = _lib.stream_ptr(x)
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(x)
            _lib.call("genre_b200_convt_c1_dgrad", gy.data_ptr(), weight.detach().contiguous().data_ptr(), b, cin, d, h, w,
                      gx.data_ptr(), st)
        if ctx.needs_input_grad[1]:
            nbytes = _lib.load().genre_b200_convt_c1_wgrad_workspace_bytes(cin)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            gw = torch.empty_like(weight)
            _lib.call("genre_b200_convt_c1_wgrad", x.data_ptr(), gy.data_ptr(), b, cin, d, h, w, gw.data_ptr(),
                      ws.data_ptr(), nbytes, st)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = gy.sum().reshape(1)
        return gx, gw, gb, None


def _convt_c1_train_supported(x, m):
    return (ENABLED and "convt_c1_train" in POLICY and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
            and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2) and tuple(m.padding) == (1, 1, 1)
            and tuple(m.output_padding) == (0, 0, 0) and tuple(m.dilation) == (1, 1, 1) and m.groups == 1
            and m.out_channels == 1 and x.shape[1] % 4 == 0 and x.shape[1] <= 48 and x.shape[3] % 8 == 0
            and x.shape[4] % 4 == 0 and x.shape[4] <= 64)


TRAIN_FORWARD = os.environ.get("GENRE_B200_CONV_TRAIN_FORWARD", "1") != "0"


def _train_forward(x, m, supported):
    """conv-only call under autograd: custom forward + cuDNN backward when the layer is covered, else None"""
    if not (TRAIN_FORWARD and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and supported):
        return None
    return _ConvForward.apply(x, m.weight, m.bias, m)


def conv3d(x, m, bn=None, slope=None):
    """Conv3d on the tcgen05 kernel [+ folded eval BatchNorm3d + LeakyReLU]: k=8,s=2,p=3 on few input channels
    (Unet_3D.enc1) via space-to-depth, or k=4,s=2,p=1 (discriminator, Unet_3D.enc2/enc3) via parity sub-volumes."""
    if not x.is_cuda:
        return None
    if _needs_grad(x, m.weight, m.bias):
        if bn is not None or slope is not None:
            return None     # fused epilogues are inference-only; the caller falls back to module-by-module
        return _train_forward(x, m, _conv_k4s2_supported(x, m) or _conv_k8s2_supported(x, m) or _conv_k4s2_s2d_supported(x, m))
    if not _no_autograd(x, m.weight, m.bias):
        return None
    if _skinny_conv_supported(x, m):
        return _skinny_run(x, m, bn, slope, False)
    if _flat_conv_supported(x, m):
        return _flat_run((x,), m, bn, slope, False)
    if _conv_k4s2_supported(x, m):
        return _conv_k4s2(x, m, bn, slope)
    if _conv_k4s2_s2d_supported(x, m):
        return _conv_k4s2_s2d(x, m, bn, slope)
    if not _conv_k8s2_supported(x, m):
        return None
    if MERGE_PARITIES and m.out_channels <= 20 and all(v % 64 == 0 for v in x.shape[3:]) and x.shape[2] % 4 == 0:
        # 4x space-to-depth: 3 taps over 64*Cin channels, the 8 output classes of the 2x finer grid merged along N
        aff = _affine(m, bn, 20, x.device)
        if aff is None:
            return None
        g, b, cout = _group(), x.shape[0], m.out_channels
        # f16x2 doubles the accumulator columns: 8 classes x 20 x 2 = 320 > 256, so the z class moves to blockIdx.y (N = 80).
        # The other modes keep all 8 classes in N = 160 (the split form measured 0.88 vs 0.80 ms for them).
        split_z = _x2()
        wpack = _pack(m, ("k8s2_s4d", 20, g, split_z), lambda wt: pack_conv_k8s2_s4d_weights(wt, 20, g, split_z),
                      2 if split_z else 1)
        if _x2_direct(x):
            xb = space_to_depth4_blocked(x, 16, torch.float16)
        else:
            xb = _finish_operand(space_to_depth4_blocked(x, _act_group(), torch.float16 if _f16() else None))
        bd, cg, h, w, _ = xb.shape
        cgo = (cout + 3) // 4
        out = torch.empty((bd * 2, cgo, 2 * h, 2 * w, 4), device=x.device, dtype=torch.float32)
        _lib.call("genre_b200_conv3d_k8s2_s4d_forward", xb.data_ptr(), cg // _parts(), b, bd // b, h, w, wpack.data_ptr(), 80 if split_z else 160,
                  _op_flag(), aff[0].data_ptr(), aff[1].data_ptr(), 1.0 if slope is None else float(slope),
                  out.data_ptr(), cgo, _lib.stream_ptr(x))
        return from_blocked(out, b, cout)
    cout, npad = m.out_channels, 32
    aff = _affine(m, bn, npad, x.device)
    if aff is None:
        return None
    sc, sh = aff
    dev = x.device
    if _x2_direct(x):
        xb = space_to_depth_blocked(x, 16, torch.float16)
    else:
        xb = _finish_operand(space_to_depth_blocked(x, 8, torch.float16) if _f16() else space_to_depth_blocked(x))
    b = x.shape[0]
    bd, cg, h, w, _ = xb.shape
    cgo = (cout + 3) // 4
    out = torch.empty((bd, cgo, h, w, 4), device=dev, dtype=torch.float32)
    _lib.call("genre_b200_conv3d_taps_forward", xb.data_ptr(), cg // _parts(), None, 0, b, bd // b, h, w,
              _packed_conv(m, npad).data_ptr(), 5, 2, npad, _op_flag(), sc.data_ptr(), sh.data_ptr(),
              1.0 if slope is None else float(slope), out.data_ptr(), cgo, _lib.stream_ptr(x))
    return from_blocked(out, b, cout)


def _operand_of(x):
    """blocked operand of the tensor-core kernels for activation x (NCDHW tensor or BlockedActivation) in the current
    PRECISION, reusing the fp32 blocked twin a previous custom layer left behind; (operand, padded channels) or None"""
    c = x.shape[1]
    twin = _cached_blocked(x)
    if _x2():       # fp16 hi/lo parts of the (zero-padded) fp32 blocked tensor
        if twin is None:
            if c % 4 != 0 or isinstance(x, BlockedActivation):
                return None
            twin = to_blocked(x, 4)
        return _split2(twin), ((twin.shape[1] + 1) // 2) * 8
    if not _f16():
        if twin is not None:
            return twin, twin.shape[1] * 4
        return (to_blocked(x, 4), c) if c % 4 == 0 and not isinstance(x, BlockedActivation) else None
    if twin is not None:
        bd, cg4, h, w, _ = twin.shape
        out = torch.empty((bd, (cg4 + 1) // 2, h, w, 8), device=twin.device, dtype=torch.float16)
        _lib.call("genre_b200_blocked_f32_to_f16", twin.data_ptr(), cg4, bd, h, w, out.data_ptr(), _lib.stream_ptr(twin))
        return out, out.shape[1] * 8
    return (to_blocked(x, 8, torch.float16), c) if c % 8 == 0 and not isinstance(x, BlockedActivation) else None


def convt_c1_tc(inputs, m, sigmoid=False):
    """ConvTranspose3d(Cin -> 1, k4, s2, p1) over the channel concatenation of `inputs` on the tensor cores (MODE 4);
    NCDHW [B,1,2D,2H,2W] or None if not covered."""
    x0 = inputs[0]
    if _x3() or _x2():
        return None   # fp32 wanted: the FP32-pipe stencil (csrc/convt_c1.cu) is exact and, measured, faster than the split-operand
                      # MMAs once the operand split of its two 336 MB sources is paid (Unet_3D.dec6: 1.33 vs 1.79 ms at B=16)
    if not ("convt_c1_tc" in POLICY and ENABLED and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2)
            and tuple(m.padding) == (1, 1, 1) and tuple(m.output_padding) == (0, 0, 0) and tuple(m.dilation) == (1, 1, 1)
            and m.groups == 1 and m.out_channels == 1 and len(inputs) <= 2
            and all(t.is_cuda and t.dtype == torch.float32 and t.dim() == 5 and t.shape[2:] == x0.shape[2:] for t in inputs)
            and x0.shape[4] in (16, 32, 64) and x0.shape[3] % 16 == 0 and _no_autograd(*inputs, m.weight, m.bias)):
        return None
    ops = [_operand_of(t) for t in inputs]
    if any(o is None for o in ops):
        return None
    g = _group()
    segments = tuple((t.shape[1], o[1]) for t, o in zip(inputs, ops))
    if sum(pc for _, pc in segments) % (2 * g) != 0:
        return None
    wpack = _pack(m, ("c1_tc", segments, g), lambda wt: pack_convt_c1_tc_weights(wt, segments, g), 1)
    b, _, d, h, w = x0.shape
    if m.bias is not None:
        bias = m.bias.detach()
    else:
        bias = m.__dict__.get("_gb_zero_bias")
        if bias is None or bias.device != x0.device:
            bias = m.__dict__["_gb_zero_bias"] = torch.zeros(1, device=x0.device)
    out = torch.empty((b, 1, 2 * d, 2 * h, 2 * w), device=x0.device, dtype=torch.float32)
    s1 = ops[1][0] if len(ops) > 1 else None
    _lib.call("genre_b200_convt_c1_tc_forward", ops[0][0].data_ptr(), ops[0][0].shape[1] // _parts(), s1.data_ptr() if s1 is not None else None,
              s1.shape[1] // _parts() if s1 is not None else 0, b, d, h, w, wpack.data_ptr(), _op_flag() if g == 8 else 0, bias.data_ptr(),
              1 if sigmoid else 0, out.data_ptr(), _lib.stream_ptr(out))
    return out


def convt_c1_col2im(inputs, m):
    """ConvTranspose3d(Cin -> 1, k4, s2, p1) over the channel concatenation of `inputs` on 64-wide volumes: tap GEMM + col2im
    (csrc/convt_c1_col2im.cu); NCDHW [B,1,2D,2H,128] or None if not covered."""
    x0 = inputs[0]
    if not ("convt_c1_col2im" in POLICY and ENABLED and (_f16() or _x2()) and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2)
            and tuple(m.padding) == (1, 1, 1) and tuple(m.output_padding) == (0, 0, 0) and tuple(m.dilation) == (1, 1, 1)
            and m.groups == 1 and m.out_channels == 1 and len(inputs) <= 2
            and all(t.is_cuda and t.dtype == torch.float32 and t.dim() == 5 and t.shape[2:] == x0.shape[2:] for t in inputs)
            and x0.shape[4] == 64 and x0.shape[3] % 8 == 0 and x0.shape[0] <= 65535 and _no_autograd(*inputs, m.weight, m.bias)):
        return None
    ops = [_operand_of(t) for t in inputs]
    if any(o is None for o in ops):
        return None
    segments = tuple((t.shape[1], o[1]) for t, o in zip(inputs, ops))
    if sum(pc for _, pc in segments) % 16 != 0:
        return None
    wpack = _pack(m, ("c1_col2im", segments, 8), lambda wt: pack_convt_c1_col2im_weights(wt, segments), 0)
    b, _, d, h, w = x0.shape
    if m.bias is not None:
        bias = m.bias.detach()
    else:
        bias = m.__dict__.get("_gb_zero_bias")
        if bias is None or bias.device != x0.device:
            bias = m.__dict__["_gb_zero_bias"] = torch.zeros(1, device=x0.device)
    out = torch.empty((b, 1, 2 * d, 2 * h, 2 * w), device=x0.device, dtype=torch.float32)
    s1 = ops[1][0] if len(ops) > 1 else None
    _lib.call("genre_b200_convt_c1_col2im_forward", ops[0][0].data_ptr(), ops[0][0].shape[1] // _parts(), s1.data_ptr() if s1 is not None else None,
              s1.shape[1] // _parts() if s1 is not None else 0, b, d, h, w, wpack.data_ptr(), _op_flag(), bias.data_ptr(), out.data_ptr(),
              _lib.stream_ptr(out))
    return out


def _has_blocked(x):
    return _cached_blocked(x) is not None


def _convt_c1_supported(cin, shape_dhw, m, inputs=()):
    if "convt_c1" not in POLICY:
        return False
    if "convt_c1_convert" not in POLICY and not all(_has_blocked(t) for t in inputs):
        return False
    return (ENABLED and tuple(m.kernel_size) == (4, 4, 4) and tuple(m.stride) == (2, 2, 2) and tuple(m.padding) == (1, 1, 1)
            and tuple(m.output_padding) == (0, 0, 0) and tuple(m.dilation) == (1, 1, 1) and m.groups == 1
            and m.out_channels == 1 and cin % 4 == 0 and cin <= C1_MAX_CIN and shape_dhw[2] % 4 == 0)


def convt_c1(src0, src1, batch, m):
    """ConvTranspose3d(Cin -> 1, k4, s2, p1) on blocked fp32 inputs -> NCDHW [B,1,2D,2H,2W] (csrc/convt_c1.cu)."""
    bd, cg0, h, w, _ = src0.shape
    d = bd // batch
    out = torch.empty((batch, 1, 2 * d, 2 * h, 2 * w), device=src0.device, dtype=torch.float32)
    wt = m.weight.detach().reshape(m.in_channels, 64).contiguous()
    bias = 0.0
    if m.bias is not None:   # the C ABI takes the scalar by value: read it back once per parameter version, not per call
        ver = _versions(m.bias)
        hit = m.__dict__.get("_gb_bias")
        if hit is None or hit[0] != ver:
            hit = m.__dict__["_gb_bias"] = (ver, float(m.bias.detach()))
        bias = hit[1]
    _lib.call("genre_b200_convt_c1_forward", src0.data_ptr(), cg0, src1.data_ptr() if src1 is not None else None,
              src1.shape[1] if src1 is not None else 0, batch, d, h, w, wt.data_ptr(), bias, 0, out.data_ptr(),
              _lib.stream_ptr(src0))
    return out


def conv_transpose3d(x, m, bn=None, slope=None):
    """ConvTranspose3d [-> eval-mode BatchNorm3d folded into the epilogue -> ReLU / LeakyReLU(slope)]; None if not covered
    (the caller then runs the plain modules)."""
    if x.is_cuda and not isinstance(x, BlockedActivation) and _needs_grad(x, m.weight, m.bias):
        if bn is not None or slope is not None or x.dim() != 5:
            return None
        if TRAIN_FORWARD and _convt_c1_train_supported(x, m):
            return _ConvTC1Train.apply(x, m.weight, m.bias, m)
        return _train_forward(x, m, m.out_channels > 1 and _convt_supported(x.shape, m))
    if bn is None and slope is None and m.out_channels == 1:
        y = convt_c1_col2im((x,), m)
        if y is None:
            y = convt_c1_tc((x,), m)
        if y is not None:
            return y
    if not isinstance(x, BlockedActivation) and _skinny_convt_supported(x, m):
        return _skinny_run(x, m, bn, slope, True)
    if not isinstance(x, BlockedActivation) and _flat_convt_supported((x,), m):
        return _flat_run((x,), m, bn, slope, True)
    if (bn is None and slope is None and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
            and _convt_c1_supported(x.shape[1], x.shape[2:], m, (x,)) and _no_autograd(x, m.weight, m.bias)):
        return convt_c1(_blocked_f32(x), None, x.shape[0], m)
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and _convt_supported(x.shape, m)
            and _no_autograd(x, m.weight, m.bias)):
        return None
    y = convt3d_s2_blocked(_to_operand(x), None, x.shape[0], m, bn, 1.0 if slope is None else slope)
    return None if y is None else from_blocked(y, x.shape[0], m.out_channels)


# ---- BatchNorm3d with batch statistics + activation, training mode (csrc/bn_train.cu) --------------------------------
# On by default since round 2 (GPU-validated: tests/test_gpu_conv.py::test_bn_act_train_forward_backward_vs_torch);
# GENRE_B200_BN_TRAIN=0 restores torch's BatchNorm3d kernels.
BN_TRAIN = os.environ.get("GENRE_B200_BN_TRAIN", "1") != "0"


class _BnActTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, bn, slope):
        x = x.contiguous()
        b, c = x.shape[0], x.shape[1]
        sp = x.numel() // (b * c)
        y = torch.empty_like(x)
        mean, invstd = torch.empty(c, device=x.device), torch.empty(c, device=x.device)
        nbytes = _lib.load().genre_b200_bn_workspace_bytes(c)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        track = bn.track_running_stats and bn.running_mean is not None
        _lib.call("genre_b200_bn_act_train_forward", x.data_ptr(), b, c, sp, gamma.data_ptr() if gamma is not None else None,
                  beta.data_ptr() if beta is not None else None, bn.running_mean.data_ptr() if track else None,
                  bn.running_var.data_ptr() if track else None, float(bn.eps), float(bn.momentum), float(slope), y.data_ptr(),
                  mean.data_ptr(), invstd.data_ptr(), ws.data_ptr(), nbytes, _lib.stream_ptr(x))
        if track and bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        ctx.save_for_backward(x, gamma, beta, mean, invstd)
        ctx.slope = float(slope)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        x, gamma, beta, mean, invstd = ctx.saved_tensors
        dy = dy.contiguous()
        b, c = x.shape[0], x.shape[1]
        sp = x.numel() // (b * c)
        dx = torch.empty_like(x)
        dgamma = torch.empty(c, device=x.device) if gamma is not None else None
        dbeta = torch.empty(c, device=x.device) if beta is not None else None
        nbytes = _lib.load().genre_b200_bn_workspace_bytes(c)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        _lib.call("genre_b200_bn_act_train_backward", x.data_ptr(), dy.data_ptr(), b, c, sp,
                  gamma.data_ptr() if gamma is not None else None, beta.data_ptr() if beta is not None else None, mean.data_ptr(),
                  invstd.data_ptr(), ctx.slope, dx.data_ptr(), dgamma.data_ptr() if dgamma is not None else None,
                  dbeta.data_ptr() if dbeta is not None else None, ws.data_ptr(), nbytes, _lib.stream_ptr(x))
        return dx, dgamma, dbeta, None, None


def bn_act_train(x, bn, act=None):
    """act(bn(x)) with batch statistics as 3 streaming kernels forward / 2 backward, or None when not applicable"""
    if not (BN_TRAIN and ENABLED and isinstance(bn, torch.nn.BatchNorm3d) and bn.training and bn.momentum is not None
            and torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
            and (x.numel() // (x.shape[0] * x.shape[1])) % 4 == 0):
        return None
    if act is None:
        slope = 1.0
    elif isinstance(act, torch.nn.ReLU):
        slope = 0.0
    elif isinstance(act, torch.nn.LeakyReLU):
        slope = float(act.negative_slope)
    else:
        return None
    return _BnActTrain.apply(x, bn.weight, bn.bias, bn, slope)


def gemm_conv(x, m):
    """A ConvTranspose3d(k, s=1, p=0) on a 1^3 input IS a plain matrix product,
          out[b, co, :] = sum_ci x[b, ci] * W[ci, co, :]   =   x[B,Cin] @ W[Cin, Cout*k^3],
    bound by reading the weights once (105 MB for Unet_3D.dec1 networks.py:162; VoxelDecoder/VoxelGenerator main.0
    :40,:79): handed to cuBLAS it takes 0.085 ms at B=16 where cuDNN's dgrad engine takes 0.34 ms.  Pure torch ops:
    differentiable, so training takes this route too; fp32 unless torch.backends.cuda.matmul.allow_tf32.
    (The mirror case, Conv3d(k) from k^3 to 1^3 = Unet_3D.enc6, was measured too: the skinny split-K GEMM is slower
    than cuDNN there, 0.134 vs 0.076 ms, so it is not routed.)"""
    if not (ENABLED and "gemm" in POLICY and x.is_cuda and x.dim() == 5 and x.dtype == torch.float32 and m.groups == 1
            and isinstance(m, torch.nn.ConvTranspose3d) and tuple(m.stride) == (1, 1, 1) and tuple(m.padding) == (0, 0, 0)
            and tuple(m.dilation) == (1, 1, 1) and tuple(m.output_padding) == (0, 0, 0) and tuple(x.shape[2:]) == (1, 1, 1)):
        return None
    b = x.shape[0]
    y = (x.reshape(b, m.in_channels) @ m.weight.reshape(m.in_channels, -1)).view(b, m.out_channels, *m.kernel_size)
    if m.bias is not None:
        y = y + m.bias.view(1, -1, 1, 1, 1)
    return y


def fused_block(x, conv, bn, act):
    """conv [-> BatchNorm3d] -> ReLU/LeakyReLU as ONE kernel launch when the conv has a custom kernel: the normalisation
    and activation passes over the activation (0.9 ms of VoxelGenerator's 64^3 stage at B=16) disappear into the epilogue."""
    if isinstance(act, torch.nn.Sigmoid):   # VoxelGenerator's last stage: ConvT(-> 1 channel) -> Sigmoid
        return convt_c1_tc((x,), conv, sigmoid=True) if bn is None and isinstance(conv, torch.nn.ConvTranspose3d) else None
    slope = 0.0 if isinstance(act, torch.nn.ReLU) else float(act.negative_slope)
    if isinstance(conv, torch.nn.ConvTranspose3d):
        return conv_transpose3d(x, conv, bn, slope)
    return conv3d(x, conv, bn, slope)


def deconv_skip(x, skip, conv, bn=None, slope=None, keep_blocked=False):
    """cat(x, skip) -> ConvTranspose3d [-> eval-mode BatchNorm3d folded into the epilogue -> LeakyReLU(slope)] with the
    concatenation walked as two K ranges instead of being materialised.  None if not covered."""
    if bn is None and conv.out_channels == 1:
        y = convt_c1_col2im((x, skip), conv)
        if y is None:
            y = convt_c1_tc((x, skip), conv)
        if y is not None:
            return y
    if (bn is None and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and skip.shape[2:] == x.shape[2:]
            and x.shape[1] % 4 == 0 and skip.shape[1] % 4 == 0
            and _convt_c1_supported(x.shape[1] + skip.shape[1], x.shape[2:], conv, (x, skip))
            and _no_autograd(x, skip, conv.weight, conv.bias)):
        return convt_c1(_blocked_f32(x), _blocked_f32(skip), x.shape[0], conv)
    if isinstance(x, BlockedActivation):
        x = x.ncdhw()
    if (torch.is_tensor(skip) and skip.dim() == 5 and tuple(skip.shape[2:]) == (1, 1, 1) and torch.is_tensor(x) and x.dim() == 5
            and tuple(x.shape[2:]) == (1, 1, 1)):
        xc = torch.cat((x, skip), dim=1)
        return _skinny_run(xc, conv, bn, slope, True) if _skinny_convt_supported(xc, conv) else None
    if _flat_convt_supported((x, skip), conv):
        return _flat_run((x, skip), conv, bn, slope, True)
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and skip.shape[2:] == x.shape[2:]
            and x.shape[1] % _group() == 0 and skip.shape[1] % _group() == 0
            and _convt_supported((x.shape[0], x.shape[1] + skip.shape[1]) + tuple(x.shape[2:]), conv)
            and _no_autograd(x, skip, conv.weight, conv.bias)):
        return None
    if bn is not None and (bn.training or not bn.track_running_stats):
        return None  # batch statistics need the un-normalised output first
    # the concatenation stays two K ranges (a K chunk of 2 channel groups may straddle them: the halo producer picks the
    # source per channel group)
    a, bsrc = _to_operand(x), _to_operand(skip)
    y = convt3d_s2_blocked(a, bsrc, x.shape[0], conv, bn, 1.0 if slope is None else slope)
    if keep_blocked:
        return BlockedActivation(y, x.shape[0], conv.out_channels)
    return from_blocked(y, x.shape[0], conv.out_channels)
