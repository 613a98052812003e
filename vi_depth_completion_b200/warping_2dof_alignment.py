"""Drop-in replacement for the reference's networks/warping_2dof_alignment.py.

Same class name, constructor and method signatures / return tuples as
MARSLab-UMN/vi_depth_completion `Warping2DOFAlignment` (networks/warping_2dof_alignment.py:5-310),
so networks/surface_normal.py (:70, :148, :169) runs unmodified on top of it.  Every method is a thin
host-side wrapper: it checks shapes, allocates the outputs with torch (device memory + streams are
the only things torch is used for) and enqueues the hand-written sm_100a kernels of
libvidc_b200.so on the current CUDA stream through the C ABI in include/vidc_b200.h: the hot entry points through the
operators of the torch C++ extension (_torchops.py) only, the calls no operator takes through ctypes (_cabi.py).

Differences from the reference that are deliberate (see DESIGN.md):
  * the device follows the inputs (the reference pins 'cuda:0', :7);
  * nothing synchronises with the host (the reference reads dozens of device scalars per frame);
  * any canvas size works (the reference hard-codes 240*320 staging buffers, :121-122);
  * gradients: the two reference-shaped methods are differentiable w.r.t. the image (vidc_warp_backward, bilinear /
    nearest; vidc_warp_backward_ordered, bit-reproducible, under torch.use_deterministic_algorithms(True) or with
    deterministic_backward = True) and, as in the reference, w.r.t. I_g and I_a, through both the warped image and the
    returned Cg_H_C (vidc_warp_backward_params, then vidc_frame_params_backward; fixed order, bit-reproducible);
    _build_homography is differentiable w.r.t. I_g and I_a too; the fused entry points, the params= forms, prepare(),
    image_sampler_forward_inverse, warp_normal_image_with_gravity_center_aligned, warp_with_homography and
    interp_mode='bicubic' are forward-only and raise NotImplementedError in backward, for the image and the gravity alike;
  * there is NO CPU / PyTorch fallback: CPU tensors raise RuntimeError.
"""
import ctypes

import numpy as np
import torch

from . import _cabi, _torchops
from ._cabi import VidcCamera, VidcImage, check, lib

__all__ = ["Warping2DOFAlignment"]


def _stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda_f32(t: torch.Tensor, name: str):
    if not isinstance(t, torch.Tensor):
        raise RuntimeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (this module has no CPU fallback), got device {t.device}")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name}: expected scalar type Float but found {t.dtype}")


def _image(t: torch.Tensor) -> VidcImage:
    """(N,C,H,W) tensor -> vidc_image with element strides (no copy for NCHW or channels-last)."""
    n, c, h, w = t.shape
    sn, sc, sh, sw = t.stride()
    return VidcImage(t.data_ptr(), n, c, h, w, sn, sc, sh, sw)


def _gravity(I_g: torch.Tensor, I_a: torch.Tensor, device):
    _require_cuda_f32(I_g, "I_g")
    _require_cuda_f32(I_a, "I_a")
    if I_g.device != device or I_a.device != device:
        raise RuntimeError(f"I_g / I_a must live on {device}, got {I_g.device} / {I_a.device}")
    B, Ba = I_g.shape[0], I_a.shape[0]
    if I_g.numel() != 3 * B or I_a.numel() != 3 * Ba:            # .view(B,3,1) / .view(B,1,3) at :38-39
        raise RuntimeError(f"I_g / I_a: expected 3 components per frame, got shapes {tuple(I_g.shape)} / {tuple(I_a.shape)}")
    # the kernels read 3*B floats from both: a shorter I_a must never reach them.  The reference fails in the same two
    # places: I_a[i] in the loop of :40-41 (IndexError) or the batched product I_a @ I_g at :43 (RuntimeError).
    if Ba < B:
        raise IndexError(f"index {Ba} is out of bounds for dimension 0 with size {Ba} (I_a has {Ba} frames, I_g has {B})")
    if Ba > B:
        raise RuntimeError(f"I_a has {Ba} frames but I_g has {B}: batch dimensions of I_a @ I_g must match (ref :43)")
    return I_g.reshape(B, 3).contiguous(), I_a.reshape(Ba, 3).contiguous()


def _wants_grad(*ts):
    """True when autograd records and one of the tensors requires a gradient."""
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in ts)


def _nd(t):
    """The torch operators carry no autograd kernel: they only ever see detached tensors (torch's not-implemented fallback
    would otherwise hand out a silent None gradient)."""
    return t.detach() if isinstance(t, torch.Tensor) and t.requires_grad else t


def _gravity_backward(w, g, a, gparams, gH=None):
    """dL/dI_g, dL/dI_a from the gradients of the frame parameters (vidc_frame_params_backward)."""
    gg, ga = torch.empty_like(g, memory_format=torch.contiguous_format), torch.empty_like(a, memory_format=torch.contiguous_format)
    with torch.cuda.device(g.device):
        check(lib().vidc_frame_params_backward(ctypes.byref(w._cam), g.data_ptr(), a.data_ptr(), g.shape[0], gparams.data_ptr(),
                                               gH.data_ptr() if gH is not None else None, gg.data_ptr(), ga.data_ptr(),
                                               _stream_ptr(g.device)))
    return gg, ga


class _WarpFn(torch.autograd.Function):
    """Connects the forward-only fused kernels to autograd.  The image gradient is the scatter kernel of vidc_warp_backward;
    under torch.use_deterministic_algorithms(True), or with the warper's deterministic_backward set to True, it is the gather
    kernel of vidc_warp_backward_ordered instead: one fixed summation order, the same bits in every run.  The gradient of
    I_g / I_a (g, a: their (B,3) views) -- the reference's autograd reaches them through the sampling grid -- is
    vidc_warp_backward_params followed by vidc_frame_params_backward, computed only when one of them requires it; x is saved
    for it only then."""

    @staticmethod
    def forward(ctx, x, out, warper, g, a, inverse, mode):
        ctx.warper, ctx.inverse, ctx.mode = warper, inverse, mode
        ctx.in_shape = tuple(x.shape)
        ctx.save_for_backward(g, a, x if (ctx.needs_input_grad[3] or ctx.needs_input_grad[4]) else None)
        return out.view_as(out)

    @staticmethod
    def backward(ctx, grad):
        g, a, x = ctx.saved_tensors
        grad = grad.float()
        gx = _WarpFn._image_grad(ctx, g, a, grad) if ctx.needs_input_grad[0] else None
        gg = ga = None
        if ctx.needs_input_grad[3] or ctx.needs_input_grad[4]:
            w = ctx.warper
            B = g.shape[0]
            gparams = torch.empty((B, _cabi.FRAME_PARAMS_FLOATS), dtype=torch.float32, device=grad.device)
            scratch = torch.empty((max(int(lib().vidc_warp_backward_params_scratch_bytes(ctypes.byref(w._cam), B)), 8) // 8,),
                                  dtype=torch.float64, device=grad.device)
            xi, gi = _image(x), _image(grad)
            with torch.cuda.device(grad.device):
                check(lib().vidc_warp_backward_params(ctypes.byref(w._cam), ctypes.byref(xi), ctypes.byref(gi), g.data_ptr(),
                                                      a.data_ptr(), B, 1 if ctx.inverse else 0, ctx.mode,
                                                      w._params_ws(B, grad.device).data_ptr(), scratch.data_ptr(),
                                                      gparams.data_ptr(), _stream_ptr(grad.device)))
            gg, ga = _gravity_backward(w, g, a, gparams)
        return gx, None, None, gg, ga, None, None

    @staticmethod
    def _image_grad(ctx, g, a, grad):
        w = ctx.warper
        B, C, Hin, Win = ctx.in_shape
        det = w.deterministic_backward
        entry = lib().vidc_warp_backward_ordered if (torch.are_deterministic_algorithms_enabled() if det is None else det) \
            else lib().vidc_warp_backward
        groups = []
        for c0 in range(0, C, 4):                              # feature maps: the scatter kernel takes <= 4 planes per call
            gc = grad[:, c0:c0 + 4]
            gxc = torch.empty((B, gc.shape[1], Hin, Win), dtype=torch.float32, device=grad.device)
            gi = _image(gc)
            with torch.cuda.device(grad.device):
                check(entry(ctypes.byref(w._cam), ctypes.byref(gi), g.data_ptr(), a.data_ptr(), g.shape[0],
                            1 if ctx.inverse else 0, ctx.mode, w._params_ws(g.shape[0], grad.device).data_ptr(),
                            gxc.data_ptr(), Hin, Win, _stream_ptr(grad.device)))
            groups.append(gxc)
        return groups[0] if len(groups) == 1 else torch.cat(groups, 1)


class _HomographyFn(torch.autograd.Function):
    """Cg_H_C (one matrix) or _build_homography's (Cg_H_C, Cg_R_C, Cg_H_C_inv), differentiable w.r.t. I_g / I_a (g, a: their
    (B,3) views) through vidc_frame_params_backward, as the reference's torch ops are."""

    @staticmethod
    def forward(ctx, g, a, warper, *mats):
        ctx.warper, ctx.n = warper, len(mats)
        ctx.save_for_backward(g, a)
        return tuple(m.view_as(m) for m in mats) if len(mats) > 1 else mats[0].view_as(mats[0])

    @staticmethod
    def backward(ctx, *grads):
        g, a = ctx.saved_tensors
        B = g.shape[0]
        gparams = torch.zeros((B, _cabi.FRAME_PARAMS_FLOATS), dtype=torch.float32, device=g.device)
        gH = None
        if ctx.n == 1:
            gH = grads[0].float().reshape(B, 9).contiguous() if grads[0] is not None else None
        else:
            for k, gm in enumerate(grads):                      # fields H, R, Hinv: floats 0, 9, 18
                if gm is not None:
                    gparams[:, 9 * k:9 * k + 9] = gm.float().reshape(B, 9)
        gg, ga = _gravity_backward(ctx.warper, g, a, gparams, gH)
        return (gg, ga, None) + (None,) * ctx.n


class _NoGravityBackward(torch.autograd.Function):
    """Outputs of entry points whose gravity (or Cg_H_C) input requires a gradient they do not compute."""

    @staticmethod
    def forward(ctx, out, *grav):
        return out.view_as(out)

    @staticmethod
    def backward(ctx, *grads):
        raise NotImplementedError(
            "vi_depth_completion_b200: this entry point is not differentiable w.r.t. I_g / I_a (or Cg_H_C); gravity gradients "
            "are computed by warp_with_gravity_center_aligned (bilinear / nearest), "
            "inverse_warp_normal_image_with_gravity_center_aligned and _build_homography")


def _no_gravity_grad(outs, *grav):
    """Wrap the floating-point outputs so that a backward into the gravity raises instead of handing out None."""
    grav = tuple(t for t in grav if isinstance(t, torch.Tensor) and t.requires_grad)
    if not grav or not torch.is_grad_enabled():
        return outs
    return tuple(_NoGravityBackward.apply(o, *grav) if isinstance(o, torch.Tensor) and o.is_floating_point() else o for o in outs)


class _NoBackward(torch.autograd.Function):
    """Outputs of fused entry points that have no backward kernel (renormalising unwarp, rotated forward warp)."""

    @staticmethod
    def forward(ctx, x, out):
        return out.view_as(out)

    @staticmethod
    def backward(ctx, grad):
        raise NotImplementedError(
            "vi_depth_completion_b200: this fused entry point is forward-only; use the reference-shaped methods "
            "(warp_with_gravity_center_aligned / inverse_warp_normal_image_with_gravity_center_aligned) to train through the warp")


def _attach(x, out, warper=None, g=None, a=None, inverse=False, mode=0):
    if torch.is_grad_enabled() and x.requires_grad:
        if warper is not None:
            return _WarpFn.apply(x, out, warper, g, a, inverse, mode)
        return _NoBackward.apply(x, out)
    return out


def _op(fn, *args):
    """Call a torch.ops.vidc operator; the C ABI's batch-mismatch status is the reference's `assert` (:123, :224)."""
    try:
        return fn(*args)
    except RuntimeError as e:
        if "vidc_b200 batch mismatch" in str(e):
            raise AssertionError(str(e).split("vidc_b200 batch mismatch: ", 1)[-1].splitlines()[0]) from None
        raise


_MODES = {"bilinear": _cabi.VIDC_BILINEAR, "nearest": _cabi.VIDC_NEAREST, "bicubic": _cabi.VIDC_BICUBIC}


def _check_interp_mode(interp_mode, allow_bicubic=False):
    """F.grid_sample's own check (the reference forwards interp_mode to it, :150): ValueError for an unknown mode.
    'bicubic' is valid there but never used by the reference's callers (surface_normal.py:148-169 pass 'bilinear' /
    'nearest'): the two reference-shaped forward methods support it (generic kernel, forward only); the fused entry points
    say that they do not instead of silently sampling differently.  Returns the C ABI's mode code."""
    if interp_mode in ("bilinear", "nearest") or (interp_mode == "bicubic" and allow_bicubic):
        return _MODES[interp_mode]
    if interp_mode == "bicubic":
        raise NotImplementedError("depth_mode='bicubic' is not implemented by the fused entry points; use "
                                  "warp_with_gravity_center_aligned(..., interp_mode='bicubic')")
    raise ValueError("nn.functional.grid_sample(): expected mode to be 'bilinear', 'nearest' or 'bicubic', "
                     f"but got: '{interp_mode}'")


class FrameParams:
    """Per-frame parameters of one batch, prepared once (Warping2DOFAlignment.prepare) and shared by warp_rgbd and
    unwarp_normals: the reference rebuilds them in every call (:124, :225) from the same I_g / I_a.  `H` is Cg_H_C (B,3,3)."""
    __slots__ = ("ws", "H", "B", "device", "intr", "grav")

    def __init__(self, ws, H, intr, grav=()):
        self.ws, self.H, self.B, self.device, self.intr = ws, H, H.shape[0], H.device, intr
        self.grav = tuple(t for t in grav if isinstance(t, torch.Tensor) and t.requires_grad)   # forward-only w.r.t. these


class Warping2DOFAlignment:
    # networks/warping_2dof_alignment.py:6
    def __init__(self, fx=577.87061 * 0.5, fy=577.87061 * 0.5, cx=319.87654 * 0.5, cy=239.87603 * 0.5):
        self.fx = fx
        self.fy = fy
        self.cx = cx
        self.cy = cy
        self._cam = VidcCamera()
        check(lib().vidc_camera_init(float(fx), float(fy), float(cx), float(cy), ctypes.byref(self._cam)))
        self.W = np.int64(self._cam.W)
        self.H = np.int64(self._cam.H)
        self.device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        self._const_cache = {}
        self._ws_bytes = {}
        self._intr = (float(fx), float(fy), float(cx), float(cy))      # operator arguments of the torch C++ front end
        # backward of the two reference-shaped methods: None follows torch.are_deterministic_algorithms_enabled(), True always
        # takes the fixed-order gather kernel (bit-reproducible gradients), False always the atomic scatter kernel
        self.deterministic_backward = None

    # ---- constant tensors the reference exposes as attributes (:15-24), built lazily ----------
    def _const(self, name):
        if name not in self._const_cache:
            W, H = int(self.W), int(self.H)
            if name == "K":
                v = torch.tensor(np.array(self._cam.K, dtype=np.float32).reshape(3, 3))
            elif name == "K_inv":
                v = torch.tensor(np.array(self._cam.Kinv, dtype=np.float32).reshape(3, 3))
            elif name == "XX":
                v = torch.arange(W, dtype=torch.float32).view(W, 1).expand(W, H).contiguous()
            elif name == "YY":
                v = torch.arange(H, dtype=torch.float32).view(1, H).expand(W, H).contiguous()
            elif name == "corners_points":
                v = torch.tensor([[0, 0, 1], [W - 1, 0, 1], [0, H - 1, 1], [W - 1, H - 1, 1]], dtype=torch.float32).t()
            elif name == "I3":
                v = torch.eye(3, dtype=torch.float32)
            else:
                raise AttributeError(name)
            self._const_cache[name] = v.to(self.device)
        return self._const_cache[name]

    K = property(lambda self: self._const("K"))
    K_inv = property(lambda self: self._const("K_inv"))
    XX = property(lambda self: self._const("XX"))
    YY = property(lambda self: self._const("YY"))
    corners_points = property(lambda self: self._const("corners_points"))
    I3 = property(lambda self: self._const("I3"))

    def _params_ws(self, B, device):
        """Scratch of vidc_workspace_bytes(cam, B): B vidc_frame_params (192 B each) + the kernels' per-tile tables.  Allocated per call from torch's stream-ordered caching allocator
        (a microsecond), so concurrent use of one instance from several streams never shares scratch."""
        nbytes = self._ws_bytes.get(B)
        if nbytes is None:
            nbytes = self._ws_bytes[B] = max(int(lib().vidc_workspace_bytes(ctypes.byref(self._cam), B)), 4 * _cabi.FRAME_PARAMS_FLOATS)
        return torch.empty((nbytes // 4,), dtype=torch.float32, device=device)

    def _skewsymm(self, x):  # :26-32, kept for API compatibility (pure tensor ops, no host sync)
        x = x.reshape(-1)
        z = torch.zeros((), dtype=x.dtype, device=x.device)
        return torch.stack([torch.stack([z, -x[2], x[1]]), torch.stack([x[2], z, -x[0]]), torch.stack([-x[1], x[0], z])]).float()

    # networks/warping_2dof_alignment.py:35-58
    def _build_homography(self, I_g, I_a):
        _require_cuda_f32(I_g, "I_g")
        _require_cuda_f32(I_a, "I_a")
        out = _op(_torchops.ops().build_homography, _nd(I_g), _nd(I_a), *self._intr)
        if not _wants_grad(I_g, I_a):
            return out
        g, a = _gravity(I_g, I_a, I_g.device)
        return _HomographyFn.apply(g, a, self, *out)

    def frame_params(self, I_g, I_a):
        """Additive: the (B,48) per-frame parameter block (vidc_frame_params) as a tensor."""
        _require_cuda_f32(I_g, "I_g")
        device = I_g.device
        g, a = _gravity(I_g, I_a, device)
        B = g.shape[0]
        out = torch.empty((B, _cabi.FRAME_PARAMS_FLOATS), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            check(lib().vidc_frame_params_compute(ctypes.byref(self._cam), g.data_ptr(), a.data_ptr(), B, out.data_ptr(),
                                                  _stream_ptr(device)))
        return _no_gravity_grad((out,), I_g, I_a)[0]

    def _empty_like_canvas(self, x):
        B, C = x.shape[0], x.shape[1]
        fmt = torch.channels_last if (x.dim() == 4 and C > 1 and x.is_contiguous(memory_format=torch.channels_last)
                                      and not x.is_contiguous()) else torch.contiguous_format
        return torch.empty((B, C, int(self.H), int(self.W)), dtype=torch.float32, device=x.device, memory_format=fmt)

    # networks/warping_2dof_alignment.py:108-156
    def warp_with_gravity_center_aligned(self, x, I_g, I_a, interp_mode='bilinear'):
        _require_cuda_f32(x, "x")
        flag_fix_return = False
        if len(x.shape) == 3:                                   # :110-112
            x = x.view(x.shape[0], 1, x.shape[1], x.shape[2])
            flag_fix_return = True
        if x.dim() != 4:
            raise RuntimeError(f"x: expected a 3-D or 4-D tensor, got {x.dim()}-D")
        mode = _check_interp_mode(interp_mode, allow_bicubic=True)
        _require_cuda_f32(I_g, "I_g")
        _require_cuda_f32(I_a, "I_a")
        needs_graph = torch.is_grad_enabled() and x.requires_grad
        grav_grad = _wants_grad(I_g, I_a)
        # the operators carry no autograd kernel -- the graph is attached below (_attach), so they only ever see detached
        # tensors (torch's not-implemented fallback would otherwise hand out silent zero gradients)
        Cg_H_C, y = _op(_torchops.ops().warp_forward, x.detach() if needs_graph else x, _nd(I_g), _nd(I_a), *self._intr, mode)
        g, a = _gravity(I_g, I_a, x.device) if (needs_graph or grav_grad) else (None, None)
        # the scatter kernel of vidc_warp_backward covers bilinear and nearest; bicubic is forward-only
        if mode == _cabi.VIDC_BICUBIC:
            if needs_graph:
                y = _attach(x, y)
            Cg_H_C, y = _no_gravity_grad((Cg_H_C, y), I_g, I_a)
        else:
            if needs_graph or grav_grad:
                y = _WarpFn.apply(x, y, self, g, a, False, mode)
            if grav_grad:
                Cg_H_C = _HomographyFn.apply(g, a, self, Cg_H_C)
        if flag_fix_return:                                     # :153-154
            return Cg_H_C, y.view(x.shape[0], y.shape[2], y.shape[3])
        return Cg_H_C, y

    # networks/warping_2dof_alignment.py:158-214
    def image_sampler_forward_inverse(self, I_g, I_a):
        _require_cuda_f32(I_g, "I_g")
        device = I_g.device
        g, a = _gravity(I_g, I_a, device)
        B = g.shape[0]
        Rt = torch.empty((B, 3, 3), dtype=torch.float32, device=device)
        grid = torch.empty((B, int(self.H), int(self.W), 2), dtype=torch.float32, device=device)
        inv_grid = torch.empty_like(grid)
        with torch.cuda.device(device):
            check(lib().vidc_sampler_forward_inverse(ctypes.byref(self._cam), g.data_ptr(), a.data_ptr(), B,
                                                     self._params_ws(B, device).data_ptr(), Rt.data_ptr(), grid.data_ptr(),
                                                     inv_grid.data_ptr(), _stream_ptr(device)))
        return _no_gravity_grad((Rt, grid, inv_grid), I_g, I_a)

    # networks/warping_2dof_alignment.py:216-255
    def inverse_warp_normal_image_with_gravity_center_aligned(self, x, I_g, I_a):
        return self._unwarp(x, I_g, I_a, normalize=False, gravity_grad=True)[:2]

    def _unwarp(self, x, I_g, I_a, normalize, want_valid=False, gravity_grad=False):
        """gravity_grad: the reference-shaped method, differentiable w.r.t. I_g / I_a; the fused entry point (unwarp_normals)
        is forward-only w.r.t. them."""
        _require_cuda_f32(x, "x")
        if x.dim() != 4:
            raise RuntimeError(f"x: expected a 4-D tensor, got {x.dim()}-D")
        device = x.device
        grav_grad = _wants_grad(I_g, I_a)
        needs_graph = torch.is_grad_enabled() and x.requires_grad
        if want_valid:                                          # no operator returns the validity plane
            g, a = _gravity(I_g, I_a, device)
            z = self._empty_like_canvas(x)
            Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
            valid = torch.empty((x.shape[0], 1, int(self.H), int(self.W)), dtype=torch.uint8, device=device)
            xi, zi = _image(x), _image(z)
            with torch.cuda.device(device):
                check(lib().vidc_unwarp_normals(ctypes.byref(self._cam), ctypes.byref(xi), g.data_ptr(), a.data_ptr(), g.shape[0],
                                                1 if normalize else 0, self._params_ws(g.shape[0], device).data_ptr(),
                                                Cg_H_C.data_ptr(), ctypes.byref(zi), valid.data_ptr(), _stream_ptr(device)))
        else:
            _require_cuda_f32(I_g, "I_g")
            _require_cuda_f32(I_a, "I_a")
            Cg_H_C, z = _op(_torchops.ops().unwarp_normals, x.detach() if needs_graph else x, _nd(I_g), _nd(I_a), *self._intr,
                            bool(normalize))
            if not (needs_graph or grav_grad):
                return Cg_H_C, z, None
            g, a = _gravity(I_g, I_a, device)
            valid = None
        return self._unwarp_graph(x, z, Cg_H_C, g, a, I_g, I_a, normalize, needs_graph, grav_grad and gravity_grad) + (valid,)

    def _unwarp_graph(self, x, z, Cg_H_C, g, a, I_g, I_a, normalize, needs_graph, grav_diff):
        if grav_diff and not normalize:
            return _HomographyFn.apply(g, a, self, Cg_H_C), _WarpFn.apply(x, z, self, g, a, True, _cabi.VIDC_BILINEAR)
        z = _attach(x, z, self, g, a, True, _cabi.VIDC_BILINEAR) if not normalize else _attach(x, z)
        return _no_gravity_grad((Cg_H_C, z), I_g, I_a)

    # networks/warping_2dof_alignment.py:258-290.  The reference method cannot run (:259 unpacks three
    # return values into two); this implements its evident intent: forward warp, then z = R y.
    def warp_normal_image_with_gravity_center_aligned(self, x, I_g, I_a, interp_mode='bilinear'):
        _require_cuda_f32(x, "x")
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError("x: expected (B,3,H,W)")
        mode = _check_interp_mode(interp_mode, allow_bicubic=True)
        device = x.device
        g, a = _gravity(I_g, I_a, device)
        z = self._empty_like_canvas(x)
        Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
        xi, zi = _image(x), _image(z)
        with torch.cuda.device(device):
            check(lib().vidc_warp_normals_forward(ctypes.byref(self._cam), ctypes.byref(xi), g.data_ptr(), a.data_ptr(),
                                                  g.shape[0], mode,
                                                  self._params_ws(g.shape[0], device).data_ptr(), Cg_H_C.data_ptr(),
                                                  ctypes.byref(zi), _stream_ptr(device)))
        return _no_gravity_grad((Cg_H_C, _attach(x, z)), I_g, I_a)

    # networks/warping_2dof_alignment.py:292-310 (numpy single-image variant, non-uniform kw/kh)
    def warp_with_homography(self, x, Cg_H_C):
        _require_cuda_f32(x, "x")
        if x.dim() != 4:
            raise RuntimeError(f"x: expected a 4-D tensor, got {x.dim()}-D")
        device = x.device
        if isinstance(Cg_H_C, torch.Tensor):                    # stays on its device: no host round trip, no synchronisation
            Hm = Cg_H_C.detach().to(device=device, dtype=torch.float32).reshape(-1, 3, 3)
        else:
            Hm = torch.as_tensor(np.asarray(Cg_H_C, dtype=np.float32)).reshape(-1, 3, 3).to(device)
        if Hm.shape[0] == 1 and x.shape[0] > 1:
            Hm = Hm.expand(x.shape[0], 3, 3)
        Hd = Hm.contiguous()
        y = self._empty_like_canvas(x)
        xi, yi = _image(x), _image(y)
        with torch.cuda.device(device):
            check(lib().vidc_warp_with_homography(ctypes.byref(self._cam), ctypes.byref(xi), Hd.data_ptr(), Hd.shape[0],
                                                  self._params_ws(Hd.shape[0], device).data_ptr(), ctypes.byref(yi),
                                                  _stream_ptr(device)))
        return Cg_H_C, _no_gravity_grad((_attach(x, y),), Cg_H_C)[0]

    # ---- additive fused entry points (SURVEY.md section 8b) ------------------------------------
    def prepare(self, I_g, I_a):
        """Everything the two fused entry points need per frame (homographies, canvas scale, the kernels' per-tile tables),
        computed ONCE for a batch: pass the result as `params=` to warp_rgbd and unwarp_normals, which then launch no
        per-frame kernel of their own.  Valid for this camera and these I_g / I_a values."""
        _require_cuda_f32(I_g, "I_g")
        _require_cuda_f32(I_a, "I_a")
        grav = (I_g, I_a) if _wants_grad(I_g, I_a) else ()
        ws, H = _op(_torchops.ops().frame_params, _nd(I_g), _nd(I_a), *self._intr)
        return FrameParams(ws, _no_gravity_grad((H,), *grav)[0], self._intr, grav)

    def _prepared(self, params, x, name):
        if not isinstance(params, FrameParams):
            raise RuntimeError("params: expected the result of prepare()")
        if params.intr != self._intr:
            raise RuntimeError("params were prepared for a different camera")
        if params.device != x.device:
            raise RuntimeError(f"params live on {params.device}, {name} on {x.device}")
        if params.B != x.shape[0]:
            raise AssertionError(f"{name}.shape[0]={x.shape[0]} != I_g.shape[0]={params.B}")
        return params

    def warp_rgbd(self, x_rgb, x_depth, I_g=None, I_a=None, depth_mode='bilinear', with_mask=True, with_coverage=False, params=None):
        """One pass: warp RGB (B,3,h,w) and sparse depth (B,h,w)/(B,1,h,w) into the gravity-aligned canvas and
        emit the validity mask of surface_normal.py:151.  Returns (Cg_H_C, rgb_w, depth_w, mask_u8[, coverage]).
        params=prepare(I_g, I_a) instead of I_g / I_a: no per-frame kernel in this call."""
        _check_interp_mode(depth_mode)
        _require_cuda_f32(x_rgb, "x_rgb")
        device = x_rgb.device
        mode = _cabi.VIDC_BILINEAR if depth_mode == "bilinear" else _cabi.VIDC_NEAREST
        if params is not None:
            if x_rgb.dim() != 4 or not isinstance(x_depth, torch.Tensor) or not with_mask or with_coverage:
                raise RuntimeError("warp_rgbd(params=...): RGB (B,3,h,w) + depth, mask on, no coverage")
            p = self._prepared(params, x_rgb, "x_rgb")
            _require_cuda_f32(x_depth, "x_depth")
            d4 = x_depth.view(x_depth.shape[0], 1, x_depth.shape[1], x_depth.shape[2]) if x_depth.dim() == 3 else x_depth
            rgb_w, depth_w, mask = _op(_torchops.ops().warp_rgbd_prepared, _nd(x_rgb), _nd(d4), p.ws, *self._intr, mode)
            if x_depth.dim() == 3:
                depth_w = depth_w.view(depth_w.shape[0], depth_w.shape[2], depth_w.shape[3])
            return _no_gravity_grad((p.H, _attach(x_rgb, rgb_w), _attach(x_depth, depth_w), mask), *p.grav)
        if I_g is None or I_a is None:
            raise RuntimeError("warp_rgbd: pass I_g and I_a, or params=prepare(I_g, I_a)")
        if with_mask and not with_coverage and x_depth is not None:
            _require_cuda_f32(x_depth, "x_depth")
            _require_cuda_f32(I_g, "I_g")
            _require_cuda_f32(I_a, "I_a")
            d4 = x_depth.view(x_depth.shape[0], 1, x_depth.shape[1], x_depth.shape[2]) if x_depth.dim() == 3 else x_depth
            Cg_H_C, rgb_w, depth_w, mask = _op(_torchops.ops().warp_rgbd, _nd(x_rgb), _nd(d4), _nd(I_g), _nd(I_a), *self._intr, mode)
            if x_depth.dim() == 3:
                depth_w = depth_w.view(depth_w.shape[0], depth_w.shape[2], depth_w.shape[3])
            return _no_gravity_grad((Cg_H_C, _attach(x_rgb, rgb_w), _attach(x_depth, depth_w), mask), I_g, I_a)   # forward-only
        g, a = _gravity(I_g, I_a, device)                       # coverage, no mask or no depth: no operator takes these
        B = x_rgb.shape[0]
        squeeze = False
        di = dwi = None
        depth_w = None
        if x_depth is not None:
            _require_cuda_f32(x_depth, "x_depth")
            if x_depth.device != device:
                raise RuntimeError(f"x_depth must live on {device}, got {x_depth.device}")
            if x_depth.dim() == 3:
                x_depth = x_depth.view(x_depth.shape[0], 1, x_depth.shape[1], x_depth.shape[2])
                squeeze = True
            depth_w = self._empty_like_canvas(x_depth)
            di, dwi = _image(x_depth), _image(depth_w)
        rgb_w = self._empty_like_canvas(x_rgb)
        mask = torch.empty((B, 1, int(self.H), int(self.W)), dtype=torch.uint8, device=device) if with_mask else None
        cov = torch.empty((B,), dtype=torch.int32, device=device) if with_coverage else None
        Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
        ri, rwi = _image(x_rgb), _image(rgb_w)
        with torch.cuda.device(device):
            check(lib().vidc_warp_rgbd(ctypes.byref(self._cam), ctypes.byref(ri), ctypes.byref(di) if di is not None else None,
                                       g.data_ptr(), a.data_ptr(), g.shape[0], mode, self._params_ws(g.shape[0], device).data_ptr(),
                                       Cg_H_C.data_ptr(), ctypes.byref(rwi), ctypes.byref(dwi) if dwi is not None else None,
                                       mask.data_ptr() if with_mask else None, cov.data_ptr() if with_coverage else None,
                                       _stream_ptr(device)))
        if squeeze:
            depth_w = depth_w.view(B, depth_w.shape[2], depth_w.shape[3])
        out = (Cg_H_C, _attach(x_rgb, rgb_w), depth_w if depth_w is None else _attach(x_depth, depth_w), mask)   # forward-only
        out = _no_gravity_grad(out, I_g, I_a)
        return out + (cov,) if with_coverage else out

    def warp_rgbd_u8(self, rgb_u8, x_depth, I_g=None, I_a=None, depth_mode='bilinear', with_mask=True, with_coverage=False, params=None):
        """warp_rgbd on the frames as the loader decodes them: rgb_u8 is (B,h,w,3) uint8 on the device (dataset.py:468-471,
        before ToTensor).  Same arguments, return tuple and bits as warp_rgbd(to_tensor_u8(rgb_u8), ...); RGB comes out as
        contiguous (B,3,H,W) float32.  The kernel converts each tap itself, so the float copy of the frames is never made."""
        _check_interp_mode(depth_mode)
        if not isinstance(rgb_u8, torch.Tensor) or not rgb_u8.is_cuda or rgb_u8.dtype != torch.uint8 or rgb_u8.dim() != 4:
            raise RuntimeError("rgb_u8: expected a (B,H,W,3) uint8 CUDA tensor")
        if rgb_u8.shape[3] != 3:
            raise RuntimeError(f"rgb_u8: 3 channels, got {rgb_u8.shape[3]}")
        x = rgb_u8.contiguous()
        device = x.device
        mode = _cabi.VIDC_BILINEAR if depth_mode == "bilinear" else _cabi.VIDC_NEAREST
        d4 = None
        if x_depth is not None:
            _require_cuda_f32(x_depth, "x_depth")
            d4 = x_depth.view(x_depth.shape[0], 1, x_depth.shape[1], x_depth.shape[2]) if x_depth.dim() == 3 else x_depth
        cov = None
        if params is not None:
            if d4 is None or not with_mask or with_coverage:
                raise RuntimeError("warp_rgbd_u8(params=...): depth, mask on, no coverage")
            p = self._prepared(params, x, "rgb_u8")
            rgb_w, depth_w, mask = _op(_torchops.ops().warp_rgbd_u8_prepared, x, _nd(d4), p.ws, *self._intr, mode)
            Cg_H_C, grav = p.H, p.grav
        elif I_g is None or I_a is None:
            raise RuntimeError("warp_rgbd_u8: pass I_g and I_a, or params=prepare(I_g, I_a)")
        elif d4 is not None and with_mask and not with_coverage:
            _require_cuda_f32(I_g, "I_g")
            _require_cuda_f32(I_a, "I_a")
            Cg_H_C, rgb_w, depth_w, mask = _op(_torchops.ops().warp_rgbd_u8, x, _nd(d4), _nd(I_g), _nd(I_a), *self._intr, mode)
            grav = (I_g, I_a)
        else:                                                   # coverage, no mask or no depth: no operator takes these
            grav = (I_g, I_a)
            g, a = _gravity(I_g, I_a, device)
            B = x.shape[0]
            di = dwi = depth_w = None
            if d4 is not None:
                if d4.device != device:
                    raise RuntimeError(f"x_depth must live on {device}, got {d4.device}")
                depth_w = self._empty_like_canvas(d4)
                di, dwi = _image(d4), _image(depth_w)
            Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
            rgb_w = torch.empty((B, 3, int(self.H), int(self.W)), dtype=torch.float32, device=device)
            mask = torch.empty((B, 1, int(self.H), int(self.W)), dtype=torch.uint8, device=device) if with_mask else None
            cov = torch.empty((B,), dtype=torch.int32, device=device) if with_coverage else None
            rwi = _image(rgb_w)
            with torch.cuda.device(device):
                check(lib().vidc_warp_rgbd_u8(ctypes.byref(self._cam), x.data_ptr(), B, x.shape[1], x.shape[2],
                                              ctypes.byref(di) if di is not None else None, g.data_ptr(), a.data_ptr(), g.shape[0],
                                              mode, self._params_ws(g.shape[0], device).data_ptr(), Cg_H_C.data_ptr(),
                                              ctypes.byref(rwi), ctypes.byref(dwi) if dwi is not None else None,
                                              mask.data_ptr() if with_mask else None, cov.data_ptr() if with_coverage else None,
                                              _stream_ptr(device)))
        if depth_w is not None:
            if x_depth.dim() == 3:
                depth_w = depth_w.view(depth_w.shape[0], depth_w.shape[2], depth_w.shape[3])
            depth_w = _attach(x_depth, depth_w)                                                  # forward-only
        out = _no_gravity_grad((Cg_H_C, rgb_w, depth_w, mask), *grav)
        return out + (cov,) if with_coverage else out

    def warp_rgb_sparse_depth(self, x_rgb, tracks, counts, fc, cc, I_g, I_a, depth_mode='bilinear', with_mask=True, with_coverage=False):
        """SURVEY row f2: warp RGB (B,3,H,W) and the SPARSE depth given as KLT tracks (B,N,>=4) float64 [id, x, y, z, ...] (valid
        rows per frame in `counts`, loader intrinsics fc, cc: dataset.py:496-510) without building the depth image: the points
        are rasterised on chip and warped analytically.  Same return tuple and the same bits as
        warp_rgbd(x_rgb, rasterize_sparse_depth(tracks, counts, fc, cc, H, W), ...)."""
        _check_interp_mode(depth_mode)
        _require_cuda_f32(x_rgb, "x_rgb")
        if not isinstance(tracks, torch.Tensor) or not tracks.is_cuda or tracks.dtype != torch.float64 or tracks.dim() != 3 or tracks.shape[2] < 4:
            raise RuntimeError("tracks: expected a (B,N,>=4) float64 CUDA tensor")
        device = x_rgb.device
        g, a = _gravity(I_g, I_a, device)
        B = x_rgb.shape[0]
        tr = tracks.contiguous()
        if tr.shape[0] != B:
            raise AssertionError(f"tracks.shape[0]={tr.shape[0]} != x_rgb.shape[0]={B}")
        cnt = None
        if counts is not None:
            cnt = torch.as_tensor(counts, dtype=torch.int32, device=device).contiguous()
            if cnt.shape != (B,):
                raise RuntimeError("counts: expected shape (B,)")
        rgb_w = self._empty_like_canvas(x_rgb)
        depth_w = torch.empty((B, 1, int(self.H), int(self.W)), dtype=torch.float32, device=device)
        mask = torch.empty((B, 1, int(self.H), int(self.W)), dtype=torch.uint8, device=device) if with_mask else None
        cov = torch.empty((B,), dtype=torch.int32, device=device) if with_coverage else None
        Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
        ri, rwi, dwi = _image(x_rgb), _image(rgb_w), _image(depth_w)
        with torch.cuda.device(device):
            check(lib().vidc_warp_rgb_sparse_depth(ctypes.byref(self._cam), ctypes.byref(ri), tr.data_ptr(), cnt.data_ptr() if cnt is not None else None,
                                                   tr.shape[1], tr.shape[2], float(fc[0]), float(fc[1]), float(cc[0]), float(cc[1]),
                                                   g.data_ptr(), a.data_ptr(), g.shape[0],
                                                   _cabi.VIDC_BILINEAR if depth_mode == "bilinear" else _cabi.VIDC_NEAREST,
                                                   self._params_ws(g.shape[0], device).data_ptr(), Cg_H_C.data_ptr(), ctypes.byref(rwi),
                                                   ctypes.byref(dwi), mask.data_ptr() if with_mask else None,
                                                   cov.data_ptr() if with_coverage else None, _stream_ptr(device)))
        out = _no_gravity_grad((Cg_H_C, _attach(x_rgb, rgb_w), depth_w, mask), I_g, I_a)          # forward-only
        return out + (cov,) if with_coverage else out

    def warp_rgbd_packed(self, x_rgbd, I_g, I_a, depth_mode='bilinear', with_mask=True, with_coverage=False):
        """Packed RGBD forward warp: x_rgbd is (B,4,h,w) in channels-last memory format (R,G,B,depth interleaved, 16 B per
        pixel), so each bilinear tap is one 128-bit load.  Returns (Cg_H_C, y_rgbd channels-last, mask_u8[, coverage])."""
        _check_interp_mode(depth_mode)
        _require_cuda_f32(x_rgbd, "x_rgbd")
        if x_rgbd.dim() != 4 or x_rgbd.shape[1] != 4 or not x_rgbd.is_contiguous(memory_format=torch.channels_last):
            raise RuntimeError("x_rgbd: expected a (B,4,H,W) tensor in torch.channels_last memory format")
        device = x_rgbd.device
        g, a = _gravity(I_g, I_a, device)
        B, _, h, w = x_rgbd.shape
        y = torch.empty((B, 4, int(self.H), int(self.W)), dtype=torch.float32, device=device, memory_format=torch.channels_last)
        mask = torch.empty((B, 1, int(self.H), int(self.W)), dtype=torch.uint8, device=device) if with_mask else None
        cov = torch.empty((B,), dtype=torch.int32, device=device) if with_coverage else None
        Cg_H_C = torch.empty((g.shape[0], 3, 3), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            check(lib().vidc_warp_rgbd_packed(ctypes.byref(self._cam), x_rgbd.data_ptr(), B, h, w, g.data_ptr(), a.data_ptr(),
                                              g.shape[0], _cabi.VIDC_BILINEAR if depth_mode == "bilinear" else _cabi.VIDC_NEAREST,
                                              self._params_ws(g.shape[0], device).data_ptr(), Cg_H_C.data_ptr(), y.data_ptr(),
                                              mask.data_ptr() if with_mask else None, cov.data_ptr() if with_coverage else None,
                                              _stream_ptr(device)))
        out = _no_gravity_grad((Cg_H_C, _attach(x_rgbd, y), mask), I_g, I_a)       # forward-only
        return out + (cov,) if with_coverage else out

    def unwarp_normals(self, y, I_g=None, I_a=None, normalize=True, with_valid=False, params=None):
        """One pass: inverse warp + R^T rotation + F.normalize(dim=1) (surface_normal.py:169-170).
        Returns (Cg_H_C, n_hat[, valid_u8]).  params=prepare(I_g, I_a) instead of I_g / I_a: no per-frame kernel here."""
        if params is not None:
            _require_cuda_f32(y, "x")
            if y.dim() != 4 or with_valid:
                raise RuntimeError("unwarp_normals(params=...): a 4-D image, no validity output")
            p = self._prepared(params, y, "x")
            needs_graph = torch.is_grad_enabled() and y.requires_grad
            z = _op(_torchops.ops().unwarp_normals_prepared, y.detach() if needs_graph else y, p.ws, *self._intr, bool(normalize))
            return _no_gravity_grad((p.H, (_attach(y, z) if needs_graph else z)), *p.grav)   # forward-only with a prepared workspace
        if I_g is None or I_a is None:
            raise RuntimeError("unwarp_normals: pass I_g and I_a, or params=prepare(I_g, I_a)")
        H, z, valid = self._unwarp(y, I_g, I_a, normalize=normalize, want_valid=with_valid)
        return (H, z, valid) if with_valid else (H, z)
