"""Drop-in for casapose.pose_estimation.voting_layers_2d.CoordLSVotingWeighted.

Same constructor and call convention as the reference Keras layer
(/root/reference/casapose/pose_estimation/voting_layers_2d.py:5-30):

    layer = CoordLSVotingWeighted(name, num_classes, num_points=9, sigmoid_weights=False,
                                  filter_estimates=False, output_second_largest_component=False)
    coords = layer([seg, direct, w])        # [b, num_classes-1, num_points, 2], (y, x) pixels, float32

The body is one call into the sm_100a library (casa_ls_vote); there is no CPU / PyTorch fallback.
The gradient w.r.t. `direct` and `w` (what TensorFlow's autodiff gives the reference in
train_casapose.py:536-595; `seg` is behind stop_gradient) is casa_ls_vote_backward: `layer.backward(inp,
grad_out)`, or transparently through torch.autograd when `direct` / `w` are torch tensors that require grad.

seg, direct and w may be float32, float16 or bfloat16 (one dtype for all three: they are splits of one network
output).  16-bit inputs are read natively and widened exactly, so outputs equal the call on the .float() tensors.
`layer.backward` returns float32 gradients for every input dtype; through autograd a 16-bit leaf receives its
gradient in its own dtype (the float32 gradient rounded once).

`layer(inp, return_counts=True)` also returns poses_pnp's object availability counts from the same pass over `seg`
(casa_ls_vote_counts): [b, num_classes-1] int32 on the device, the pixels whose softmax(1e6 seg) exceeds 0.1
(/root/reference/casapose/pose_estimation/pose_evaluation.py:183-188)."""
import ctypes as C

import torch

from .. import _lib
from .._carrier import as_cuda_f32, as_cuda_float, current_stream_ptr, ptr


class _LsVoteFn(torch.autograd.Function):
    """torch.autograd carrier of casa_ls_vote / casa_ls_vote_backward (PyTorch only routes the gradient)."""

    @staticmethod
    def forward(ctx, layer, seg, direct, w, return_counts=False, check_finite=True):
        ctx.layer = layer
        ctx.save_for_backward(seg, direct, w)
        res = layer._forward(seg, direct, w, False, check_finite, return_counts)
        if return_counts:
            ctx.mark_non_differentiable(res[1])
        return res

    @staticmethod
    def backward(ctx, grad_out, *grad_counts):
        seg, direct, w = ctx.saved_tensors
        gd, gw = ctx.layer.backward([seg, direct, w], grad_out)
        return None, None, gd.reshape(direct.shape).to(direct.dtype), gw.to(w.dtype), None, None


class CoordLSVotingWeighted:
    def __init__(self, name, num_classes, num_points=9, sigmoid_weights=False, filter_estimates=False,
                 output_second_largest_component=False):
        self.name = name
        self.num_classes = num_classes
        self.num_points = num_points
        self.sigmoid_weights = sigmoid_weights
        self.filter_estimates = filter_estimates
        self.sigmoid_scale = 1.0
        self.output_second_largest_component = output_second_largest_component
        self.height = None
        self.width = None

    def build(self, input_shape):  # voting_layers_2d.py:23-25
        self.width = input_shape[0][2]
        self.height = input_shape[0][1]

    def __call__(self, inp, **kwargs):
        return self.call(inp, **kwargs)

    def call(self, inp, return_debug=False, check_finite=True, *, return_counts=False, **kwargs):
        """coords [b, oc, vn, 2]; with return_counts (coords, counts [b, oc] int32); with return_debug the debug dict
        comes last.  On the autograd path the counts are a non-differentiable output."""
        seg, direct, w = inp
        if not return_debug and torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (direct, w)):
            return _LsVoteFn.apply(self, seg.detach() if isinstance(seg, torch.Tensor) else seg, direct, w, return_counts)
        return self._forward(seg, direct, w, return_debug, check_finite, return_counts)

    def _prepare(self, seg, direct, w):
        seg, dt = as_cuda_float(seg, "seg")
        direct, dt_direct = as_cuda_float(direct, "direct")
        w, dt_w = as_cuda_float(w, "w")
        if not dt == dt_direct == dt_w:
            raise TypeError("seg, direct and w must share one dtype, got %s, %s, %s" % (seg.dtype, direct.dtype, w.dtype))
        if seg.dim() != 4:
            raise ValueError("seg must be [b,h,w,num_classes], got %s" % (tuple(seg.shape),))
        b, h, wd, nc = seg.shape
        if self.height is None:
            self.build([seg.shape, direct.shape, w.shape])
        if nc != self.num_classes:
            raise ValueError("seg has %d channels, layer was built for num_classes=%d" % (nc, self.num_classes))
        vn = self.num_points
        if direct.dim() == 5:
            direct = direct.reshape(b, h, wd, 2 * vn)
        if tuple(direct.shape) != (b, h, wd, 2 * vn) or tuple(w.shape) != (b, h, wd, vn):
            raise ValueError("direct must be [b,h,w,%d] and w [b,h,w,%d]" % (2 * vn, vn))
        return seg, direct, w, (b, h, wd, nc, vn), dt

    def _params(self, b, h, wd, nc, vn, check_finite):
        return _lib.LsParams(b=b, h=h, w=wd, num_classes=nc, vn=vn, sigmoid_weights=int(bool(self.sigmoid_weights)),
                             filter_estimates=int(bool(self.filter_estimates)),
                             second_largest=int(bool(self.output_second_largest_component)), min_component=0,
                             check_finite=int(bool(check_finite)))

    def backward(self, inp, grad_out):
        """(dL/d direct [b,h,w,2*vn], dL/d w [b,h,w,vn]) for dL/d output = grad_out [b,oc,vn,2] — casa_ls_vote_backward.
        Both are float32 whatever the inputs' dtype."""
        seg, direct, w, (b, h, wd, nc, vn), dt = self._prepare(*[t.detach() if isinstance(t, torch.Tensor) else t for t in inp])
        grad_out = as_cuda_f32(grad_out.contiguous() if isinstance(grad_out, torch.Tensor) else grad_out, "grad_out")
        if tuple(grad_out.shape) != (b, nc - 1, vn, 2):
            raise ValueError("grad_out must be [b,%d,%d,2]" % (nc - 1, vn))
        dev = seg.device
        gd = torch.empty((b, h, wd, 2 * vn), dtype=torch.float32, device=dev)
        gw = torch.empty((b, h, wd, vn), dtype=torch.float32, device=dev)
        p = self._params(b, h, wd, nc, vn, False)
        hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
        with torch.cuda.device(dev):
            rc = _lib.lib().casa_ls_vote_backward_typed(hdl, C.byref(p), dt, ptr(seg), ptr(direct), ptr(w), ptr(grad_out), None,
                                                        ptr(gd), ptr(gw), current_stream_ptr(dev))
        _lib.check(rc)
        return gd, gw

    def _forward(self, seg, direct, w, return_debug, check_finite, return_counts=False):
        seg, direct, w, (b, h, wd, nc, vn), dt = self._prepare(seg, direct, w)
        dev = seg.device
        out = torch.empty((b, nc - 1, vn, 2), dtype=torch.float32, device=dev)
        counts = torch.empty((b, nc - 1), dtype=torch.int32, device=dev) if return_counts else None
        p = self._params(b, h, wd, nc, vn, check_finite)
        dbg = None
        dbg_struct = None
        if return_debug:
            dbg = {
                "sums": torch.zeros((b, nc - 1, vn, 5), dtype=torch.float64, device=dev),
                "labels": torch.zeros((b, h, wd), dtype=torch.uint8, device=dev),
                "selected": torch.zeros((b, nc - 1), dtype=torch.int32, device=dev),
                "parent": torch.zeros((b, h, wd), dtype=torch.int32, device=dev),
                "tn": torch.zeros((b, nc - 1), dtype=torch.int32, device=dev),
            }
            dbg_struct = _lib.LsDebug(**{k: ptr(v) for k, v in dbg.items()})
        hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
        dbg_arg = C.byref(dbg_struct) if dbg_struct is not None else None
        with torch.cuda.device(dev):
            if return_counts:
                rc = _lib.lib().casa_ls_vote_counts(hdl, C.byref(p), dt, ptr(seg), ptr(direct), ptr(w), ptr(out), ptr(counts),
                                                    dbg_arg, current_stream_ptr(dev))
            else:
                rc = _lib.lib().casa_ls_vote_typed(hdl, C.byref(p), dt, ptr(seg), ptr(direct), ptr(w), ptr(out), dbg_arg,
                                                   current_stream_ptr(dev))
        _lib.check(rc)
        res = (out,) + ((counts,) if return_counts else ()) + ((dbg,) if return_debug else ())
        return res if len(res) > 1 else out
