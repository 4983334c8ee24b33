"""d3d_b200.box -- pairwise IoU and NMS on (rotated) 2-D boxes.  Mirrors reference d3d/box/__init__.py
(box2d_iou :180-224, box2d_nms :226-276, enums d3d/box/common.h:5-10) on top of the C ABI."""
import enum

import numpy as np
import torch

from .. import _cabi as _c
from . import _frames


class IouType(enum.IntEnum):   # d3d/box/common.h:5-9
    NA = 0
    BOX = 1
    RBOX = 2
    GBOX = 3
    GRBOX = 4
    DBOX = 5
    DRBOX = 6


class SupressionType(enum.IntEnum):   # d3d/box/common.h:10 (reference spelling)
    HARD = 0
    LINEAR = 1
    GAUSSIAN = 2


cuda_available = True


def iou2d_forward_cuda(boxes1, boxes2):
    """AABB IoU of rotated boxes; CUDA tensors [N,5],[M,5] -> [N,M] (reference d3d/box/iou.h:7-9)."""
    return _pairwise(boxes1, boxes2, _c.iou2d)


def iou2dr_forward_cuda(boxes1, boxes2):
    """Rotated IoU; CUDA tensors [N,5],[M,5] -> [N,M] (reference d3d/box/iou.h:14-16; the backward-only
    nx/xflags outputs are not produced)."""
    return _pairwise(boxes1, boxes2, _c.iou2dr)


def giou2dr_forward_cuda(boxes1, boxes2):
    """Rotated GIoU; CUDA tensors [N,5],[M,5] -> [N,M] (reference d3d/box/iou.h:24-26)"""
    return _pairwise_ex(boxes1, boxes2, _c.giou2dr)


def diou2dr_forward_cuda(boxes1, boxes2):
    """Rotated DIoU; CUDA tensors [N,5],[M,5] -> [N,M] (reference d3d/box/iou.h:34-36)"""
    return _pairwise_ex(boxes1, boxes2, _c.diou2dr)


def iou2d_backward_cuda(boxes1, boxes2, grad):
    """(grad_boxes1, grad_boxes2) of the AABB IoU (reference d3d/box/iou.h:10-12)"""
    return _pairwise_backward("iou2d", boxes1, boxes2, grad)


def iou2dr_backward_cuda(boxes1, boxes2, grad, nx=None, xflags=None):
    """(grad_boxes1, grad_boxes2) of the rotated IoU (reference d3d/box/iou.h:17-20); nx / xflags are accepted and ignored"""
    return _pairwise_backward("iou2dr", boxes1, boxes2, grad)


def giou2dr_backward_cuda(boxes1, boxes2, grad, nxm=None, flags=None):
    """(grad_boxes1, grad_boxes2) of the rotated GIoU (reference d3d/box/iou.h:27-30)"""
    return _pairwise_backward("giou2dr", boxes1, boxes2, grad)


def diou2dr_backward_cuda(boxes1, boxes2, grad, nxd=None, flags=None):
    """(grad_boxes1, grad_boxes2) of the rotated DIoU (reference d3d/box/iou.h:37-40)"""
    return _pairwise_backward("diou2dr", boxes1, boxes2, grad)


def _pairwise(b1, b2, table, out=None):
    code = _c.dtype_code(b1.dtype)
    if b2.dtype != b1.dtype:
        raise RuntimeError("boxes1 and boxes2 must have the same dtype")
    n, m = b1.shape[0], b2.shape[0]
    if out is None:
        out = torch.empty((n, m), dtype=b1.dtype, device=b1.device)
    if n == 0 or m == 0:
        return out
    ws = _c.workspace(_c.iou_workspace_bytes(n, m, code), b1.device)
    with torch.cuda.device(b1.device):
        st = table[code](_c.ptr(b1), n, _c.ptr(b2), m, _c.ptr(out), out.stride(0), _c.ptr(ws), ws.numel(), _c.stream_ptr())
    _c.check(st, "box2d_iou")
    return out


def _pairwise_ex(b1, b2, table):
    """GIoU / DIoU forward: no workspace"""
    code = _c.dtype_code(b1.dtype)
    if b2.dtype != b1.dtype:
        raise RuntimeError("boxes1 and boxes2 must have the same dtype")
    n, m = b1.shape[0], b2.shape[0]
    out = torch.empty((n, m), dtype=b1.dtype, device=b1.device)
    if n and m:
        with torch.cuda.device(b1.device):
            st = table[code](_c.ptr(b1), n, _c.ptr(b2), m, _c.ptr(out), out.stride(0), _c.stream_ptr())
        _c.check(st, "box2d_iou")
    return out


def _pairwise_backward(name, b1, b2, grad):
    code = _c.dtype_code(b1.dtype)
    n, m = b1.shape[0], b2.shape[0]
    grad = grad.contiguous()
    g1, g2 = torch.empty_like(b1), torch.empty_like(b2)
    with torch.cuda.device(b1.device):
        st = _c.iou_backward[name][code](_c.ptr(b1), n, _c.ptr(b2), m, _c.ptr(grad), max(m, 1), _c.ptr(g1), _c.ptr(g2), _c.stream_ptr())
    _c.check(st, "box2d_iou backward")
    return g1, g2


def _make_iou_function(name, doc, forward_impl):
    class _F(torch.autograd.Function):
        @staticmethod
        def forward(ctx, boxes1, boxes2):
            boxes1, boxes2 = boxes1.contiguous(), boxes2.contiguous()
            ctx.save_for_backward(boxes1, boxes2)   # the reference also saves nx / xflags (9 B per pair); the backward here recomputes
            return forward_impl(boxes1, boxes2)

        @staticmethod
        def backward(ctx, grad):
            boxes1, boxes2 = ctx.saved_tensors
            return _pairwise_backward(name, boxes1, boxes2, grad)
    _F.__doc__ = doc
    return _F


Iou2D = _make_iou_function("iou2d", "Differentiable IoU function for 2D axis-aligned boxes (reference d3d/box/__init__.py:38-61)",
                           lambda a, b: _pairwise(a, b, _c.iou2d))
Iou2D.__name__ = Iou2D.__qualname__ = "Iou2D"
Iou2DR = _make_iou_function("iou2dr", "Differentiable rotated IoU function for 2D boxes (reference d3d/box/__init__.py:63-84)",
                            lambda a, b: _pairwise(a, b, _c.iou2dr))
Iou2DR.__name__ = Iou2DR.__qualname__ = "Iou2DR"
GIou2DR = _make_iou_function("giou2dr", "Differentiable rotated GIoU function for 2D boxes (reference d3d/box/__init__.py:86-107)",
                             lambda a, b: _pairwise_ex(a, b, _c.giou2dr))
GIou2DR.__name__ = GIou2DR.__qualname__ = "GIou2DR"
DIou2DR = _make_iou_function("diou2dr", "Differentiable rotated DIoU function for 2D boxes (reference d3d/box/__init__.py:109-130)",
                             lambda a, b: _pairwise_ex(a, b, _c.diou2dr))
DIou2DR.__name__ = DIou2DR.__qualname__ = "DIou2DR"


def _check_iou2d(boxes1, boxes2):   # box2d_iou's checks
    if len(boxes1.shape) != 2 or len(boxes2.shape) != 2:
        raise ValueError("Input of rbox_2d_iou should be Nx2 tensors!")
    if boxes1.shape[1] != 5 or boxes2.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")


def box2d_iou(boxes1, boxes2, method="box", precise=True):
    '''
    Differentiable IoU on axis-aligned or rotated 2D boxes (reference d3d/box/__init__.py:180-224)

    :param boxes1: Input boxes, shape is N x 5 (x,y,w,h,r)
    :param boxes2: Input boxes, shape is M x 5 (x,y,w,h,r)
    :param method: 'box' - axis-aligned box, 'rbox' - rotated box,
        'grbox' - giou for rotated box, 'drbox' - diou for rotated box
    :param precise: force using double precision to calculate iou
    '''
    convert_numpy = False
    if isinstance(boxes1, np.ndarray):
        assert isinstance(boxes2, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
        boxes1 = torch.from_numpy(boxes1)
        boxes2 = torch.from_numpy(boxes2)
        convert_numpy = True

    otype = boxes1.dtype
    odev = boxes1.device
    _check_iou2d(boxes1, boxes2)

    iou_type = getattr(IouType, method.upper())
    if iou_type == IouType.BOX:
        impl = Iou2D
    elif iou_type == IouType.RBOX:
        impl = Iou2DR
    elif iou_type == IouType.GRBOX:
        impl = GIou2DR
    elif iou_type == IouType.DRBOX:
        impl = DIou2DR
    else:
        raise ValueError("Unrecognized iou type!")

    b1, b2 = _c.to_device(boxes1), _c.to_device(boxes2)
    if precise:
        b1, b2 = b1.to(torch.float64), b2.to(torch.float64)
    result = impl.apply(b1, b2)
    if precise:
        result = result.to(otype)
    if not odev.type == "cuda":
        result = result.cpu()
    if convert_numpy:
        return result.detach().numpy()
    return result


# rows x columns of the "rbox" tile (IouTile in csrc/iou.cu; keep both in step): a frame of more than 65535 tiles on an axis would make the
# batch call return D3D_ERR_UNSUPPORTED, so it runs the single-frame kernel instead
_IOU_TILE = {torch.float32: (64, 128), torch.float64: (64, 64)}


class _IouBatch(torch.autograd.Function):
    """packed IoU blocks of all frames: the forward is one launch sequence, the backward two launches, whatever the number of frames"""
    @staticmethod
    def forward(ctx, boxes1, boxes2, offsets, nframes, bounds, iou_type, total, big):
        code = _c.dtype_code(boxes1.dtype)
        out = torch.empty(total, dtype=boxes1.dtype, device=boxes1.device)
        od1, od2, odo = offsets
        fwd_max1, fwd_max2, max1, max2 = bounds
        if fwd_max1 and fwd_max2:   # "rbox": the bounds of the frames that fit the tile grid, so the batch kernels skip the others
            ws = None   # "grbox" / "drbox" need no workspace
            if iou_type in (IouType.BOX, IouType.RBOX):
                ws = _c.workspace(_c.iou_batch_workspace_bytes(len(boxes1), len(boxes2), nframes, code), boxes1.device)
            with torch.cuda.device(boxes1.device):
                st = _c.iou_batch[code](_c.ptr(boxes1), len(boxes1), _c.ptr(od1), _c.ptr(boxes2), len(boxes2), _c.ptr(od2), nframes, fwd_max1, fwd_max2,
                                        int(iou_type), _c.ptr(odo), _c.ptr(out), _c.ptr(ws), ws.numel() if ws is not None else 0, _c.stream_ptr())
            _c.check(st, "box2d_iou_batch")
        for _, r, c, k in big:   # "rbox" frames past the batch kernel's tile grid: the single-frame kernel, into their block
            _pairwise(boxes1[r], boxes2[c], _c.iou2dr, out=out[k].view(r.stop - r.start, c.stop - c.start))
        ctx.save_for_backward(boxes1, boxes2, *offsets)
        ctx.args = (nframes, max1, max2, iou_type)
        return out

    @staticmethod
    def backward(ctx, grad):
        boxes1, boxes2, od1, od2, odo = ctx.saved_tensors
        nframes, max1, max2, iou_type = ctx.args
        code = _c.dtype_code(boxes1.dtype)
        grad = grad.contiguous()
        g1, g2 = torch.empty_like(boxes1), torch.empty_like(boxes2)
        with torch.cuda.device(boxes1.device):
            st = _c.iou_batch_backward[code](_c.ptr(boxes1), len(boxes1), _c.ptr(od1), _c.ptr(boxes2), len(boxes2), _c.ptr(od2), nframes, max1, max2,
                                             int(iou_type), _c.ptr(odo), _c.ptr(grad), _c.ptr(g1), _c.ptr(g2), _c.stream_ptr())
        _c.check(st, "box2d_iou_batch backward")
        return g1, g2, None, None, None, None, None, None


def _iou_pair(b1, b2, precise):
    """both packed box sets on the device, in float64 with `precise`; their dtypes are checked before any device work"""
    if not precise:
        _c.dtype_code(b1.dtype)
        if b2.dtype != b1.dtype:
            raise RuntimeError("boxes1 and boxes2 must have the same dtype")
    b1, b2 = _c.to_device(b1), _c.to_device(b2)
    return (b1.to(torch.float64), b2.to(torch.float64)) if precise else (b1, b2)


def box2d_iou_batch(boxes1, boxes2, offsets1=None, offsets2=None, method="box", precise=True):
    '''
    :func:`box2d_iou` on a batch of frames (target assignment and IoU losses of a training batch); differentiable in both box sets.  Per
    frame the values equal :func:`box2d_iou` on that frame bit for bit, and so do the gradients.  Two call forms, like
    :func:`box3d_iou_distance_batch`: lists of per-frame ``boxes1`` [n_f, 5] / ``boxes2`` [m_f, 5] (returns the list of [n_f, m_f]
    matrices, views into one packed buffer), or the frames packed back to back with ``offsets1`` / ``offsets2`` (int64 [nframes + 1], CPU)
    (returns ``(iou_flat, iou_offsets)``: frame f's matrix is ``iou_flat[iou_offsets[f]:iou_offsets[f + 1]].view(n_f, m_f)``).  ``method``
    and ``precise`` as in :func:`box2d_iou`.  numpy in -> numpy out, host tensors in -> host tensors out.  "rbox" frames of more than
    65535 tiles (64 rows, or 128 fp32 / 64 fp64 columns) run the single-frame kernel, into their block; the batch kernels skip them,
    though the workspace still has room for their records.
    '''
    if _frames.empty(boxes1, boxes2):
        return []
    B1, B2, fr = _frames.inputs(boxes1, boxes2, offsets1, offsets2, _check_iou2d, ("boxes1", "boxes2"))
    iou_type = getattr(IouType, method.upper())
    if iou_type not in (IouType.BOX, IouType.RBOX, IouType.GRBOX, IouType.DRBOX):
        raise ValueError("Unrecognized iou type!")
    b1, b2 = _iou_pair(B1, B2, precise)
    n_f, m_f = fr.lengths()
    big = torch.zeros(fr.nframes, dtype=torch.bool)
    if iou_type == IouType.RBOX:
        tr, tc = _IOU_TILE[b1.dtype]
        big = (n_f > 65535 * tr) | (m_f > 65535 * tc)
    bounds = fr.bounds((n_f * m_f > 0) & ~big) + fr.bounds()
    offsets = _frames.to_device(b1.device, fr.rows, fr.cols, fr.blocks)
    flat = _IouBatch.apply(b1.contiguous(), b2.contiguous(), offsets, fr.nframes, bounds, iou_type, int(fr.blocks[-1]), list(fr.each(big)))
    return fr.matrices(flat.to(B1.dtype) if precise else flat)


def _iou_max(B1, B2, fr, method, precise):
    """(max1, idx1, max2, idx2) of the frames `fr` of the packed box sets, frame-local indices, on the caller's side"""
    iou_type = getattr(IouType, method.upper())
    if iou_type not in (IouType.BOX, IouType.RBOX):
        raise ValueError("Unsupported iou type!")
    otype = B1.dtype
    ocode = _c.dtype_code(otype)
    b1, b2 = _iou_pair(B1.detach(), B2.detach(), precise)
    code = _c.dtype_code(b1.dtype)
    dev, total1, total2 = b1.device, len(b1), len(b2)
    max1, max2 = torch.empty(total1, dtype=otype, device=dev), torch.empty(total2, dtype=otype, device=dev)
    idx1, idx2 = torch.empty(total1, dtype=torch.int64, device=dev), torch.empty(total2, dtype=torch.int64, device=dev)
    if fr.nframes and total1 + total2:
        b1, b2 = b1.contiguous(), b2.contiguous()
        od1, od2 = _frames.to_device(dev, fr.rows, fr.cols)
        ws = _c.workspace(_c.iou_max_batch_workspace_bytes(total1, total2, fr.nframes, code), dev)
        with torch.cuda.device(dev):
            st = _c.iou_max_batch[code](_c.ptr(b1), total1, _c.ptr(od1), _c.ptr(b2), total2, _c.ptr(od2), fr.nframes, *fr.bounds(), int(iou_type),
                                        ocode, _c.ptr(max1), _c.ptr(idx1), _c.ptr(max2), _c.ptr(idx2), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box2d_iou_max_batch")
    return fr.outputs(rows=(max1, idx1), cols=(max2, idx2))


def box2d_iou_max(boxes1, boxes2, method="box", precise=True):
    '''
    Best overlap of every box with the other set, without the IoU matrix (target assignment: each anchor's best ground truth and each
    ground truth's best anchor).  Returns ``(max1, idx1, max2, idx2)``: ``max1`` / ``idx1`` [N] are the values and int64 indices that
    ``torch.max(box2d_iou(boxes1, boxes2, method, precise), dim=1)`` returns, ``max2`` / ``idx2`` [M] those of ``dim=0``, bit for bit:
    the comparison is made on the values in the output dtype (with ``precise``, computed in float64 and rounded to the input dtype), ties
    go to the lower index, and NaN is the maximum, at the first NaN's index.  Where torch would raise because the other set is empty,
    the value is 0 and the index -1.  The outputs do not require grad: they are assignment targets, not a differentiable IoU.
    numpy in -> numpy out, host tensors in -> host tensors out.

    :param boxes1: Input boxes, shape is N x 5 (x,y,w,h,r)
    :param boxes2: Input boxes, shape is M x 5 (x,y,w,h,r)
    :param method: 'box' - axis-aligned box, 'rbox' - rotated box
    :param precise: force using double precision to calculate iou
    '''
    numpy_in = isinstance(boxes1, np.ndarray)
    if numpy_in:
        assert isinstance(boxes2, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
        boxes1, boxes2 = torch.from_numpy(boxes1), torch.from_numpy(boxes2)
    _check_iou2d(boxes1, boxes2)
    return _iou_max(boxes1, boxes2, _frames.Frames([0, len(boxes1)], [0, len(boxes2)], False, numpy_in, boxes1.device), method, precise)


def box2d_iou_max_batch(boxes1, boxes2, offsets1=None, offsets2=None, method="box", precise=True):
    '''
    :func:`box2d_iou_max` on a batch of frames in one launch sequence; per frame the outputs equal :func:`box2d_iou_max` on that frame
    bit for bit.  Two call forms, like :func:`box2d_iou_batch`: lists of per-frame ``boxes1`` [n_f, 5] / ``boxes2`` [m_f, 5] (returns the
    list of per-frame ``(max1, idx1, max2, idx2)`` tuples), or the frames packed back to back with ``offsets1`` / ``offsets2`` (int64
    [nframes + 1], CPU) (returns the packed ``(max1 [total1], idx1 [total1], max2 [total2], idx2 [total2])`` with FRAME-LOCAL indices, as
    :func:`match_greedy_batch` gives them).  A box whose frame's other side is empty gets value 0 and index -1.  ``method`` ('box' or
    'rbox') and ``precise`` as in :func:`box2d_iou_max`.  The outputs do not require grad.  numpy in -> numpy out, host tensors in -> host
    tensors out.
    '''
    if _frames.empty(boxes1, boxes2):
        return []
    return _iou_max(*_frames.inputs(boxes1, boxes2, offsets1, offsets2, _check_iou2d, ("boxes1", "boxes2")), method, precise)


def box2d_nms_batch(boxes, scores, offsets=None, iou_method="box", iou_threshold=0, score_threshold=0, precise=True, offsets_dev=None,
                    supression_method="hard", supression_param=0):
    '''
    NMS on a batch of frames in one launch sequence (the reference has no batch form; per frame the result equals
    :func:`box2d_nms` with the same arguments, bit for bit).  Two call forms: lists of per-frame ``boxes`` / ``scores`` (returns a list
    of keep masks), or the frames packed back to back as ``boxes`` [total, 5] / ``scores`` [total] with ``offsets`` (int64
    [nframes + 1], CPU tensor) (returns one keep mask bool[total]).  Frames of more than 8192 boxes fall back to one :func:`box2d_nms`
    call per frame.

    :param iou_method: 'box' - axis-aligned box, 'rbox' - rotated box
    :param offsets_dev: the same offsets already on the device (saves the copy)
    :param supression_method: 'hard', or 'linear' / 'gaussian' (soft-NMS: one CTA walks each frame, the frames run side by side)
    :param supression_param: parameter of the soft decay, as in :func:`box2d_nms`
    '''
    if isinstance(boxes, (list, tuple)):
        if len(boxes) != len(scores):
            raise ValueError("Numbers of boxes and scores are inconsistent!")
        if len(boxes) == 0:
            return []
        blist, slist = [_frames.host(b) for b in boxes], [_frames.host(s_) for s_ in scores]
        fr = _frames.Frames(_frames.offsets_of(len(b) for b in blist), None, True, isinstance(boxes[0], np.ndarray), blist[0].device)
        counts = sum(b.numel() // 5 for b in blist), sum(s_.numel() for s_ in slist)   # boxes: the rows of 5 that the copies below hold
    else:
        numpy_in = isinstance(boxes, np.ndarray)
        if numpy_in:
            boxes, scores = torch.from_numpy(boxes), torch.from_numpy(scores)
        if offsets is None:
            raise ValueError("packed boxes need the frame offsets")
        fr = _frames.Frames(offsets, None, False, numpy_in, boxes.device)
        counts = len(boxes), len(scores)
    fr.expect(*counts, "boxes, scores")
    iou_type = getattr(IouType, iou_method.upper())
    if iou_type not in (IouType.BOX, IouType.RBOX):
        raise ValueError("Unsupported iou type!")
    sup_type = getattr(SupressionType, supression_method.upper())
    if fr.as_list:   # frame by frame to the device (asynchronous copies from pinned host memory), concatenated there
        boxes = torch.cat([_c.to_device(b).reshape(-1, 5) for b in blist], 0)
        scores = torch.cat([_c.to_device(s_).reshape(-1) for s_ in slist], 0)
    b, s_ = _c.to_device(boxes), _c.to_device(scores)
    if precise:
        b, s_ = b.to(torch.float64), s_.to(torch.float64)
    elif s_.dtype != b.dtype:
        s_ = s_.to(b.dtype)
    b, s_ = b.contiguous(), s_.contiguous()
    total, nframes = int(b.shape[0]), fr.nframes
    max_frame = fr.bounds()[0]
    suppressed = torch.zeros(total, dtype=torch.uint8, device=b.device)
    if total > 0 and max_frame > 8192:
        for _, r, _, _ in fr.each(fr.lengths()[0] > 0):
            suppressed[r] = nms2d_cuda(b[r], s_[r], iou_type, sup_type, iou_threshold, score_threshold, supression_param).view(torch.uint8)
    elif total > 0:
        code = _c.dtype_code(b.dtype)
        od = _frames.to_device(b.device, fr.rows)[0] if offsets_dev is None else offsets_dev
        if sup_type == SupressionType.HARD:
            ws = _c.workspace(_c.nms_batch_workspace_bytes(total, nframes, max_frame, code), b.device)
            with torch.cuda.device(b.device):
                st = _c.nms2d_batch[code](_c.ptr(b), _c.ptr(s_), total, _c.ptr(od), nframes, max_frame, int(iou_type), int(SupressionType.HARD),
                                          float(iou_threshold), float(score_threshold), _c.ptr(suppressed), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        else:
            ws = _c.workspace(_c.nms_batch_soft_workspace_bytes(total, nframes, max_frame, code), b.device)
            with torch.cuda.device(b.device):
                st = _c.nms2d_batch_soft[code](_c.ptr(b), _c.ptr(s_), total, _c.ptr(od), nframes, max_frame, int(iou_type), int(sup_type),
                                               float(iou_threshold), float(score_threshold), float(supression_param), _c.ptr(suppressed),
                                               _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box2d_nms_batch")
    keep = fr.outputs(rows=(~suppressed.view(torch.bool),))
    return [k for k, in keep] if fr.as_list else keep[0]


_PLANE = {0: ([1, 2], [1, 2, 4, 5, 6]), 1: ([0, 2], [0, 2, 3, 5, 6]), 2: ([0, 1], [0, 1, 3, 4, 6])}   # box3dp_crop / box3dr_pdist's columns


def _check_axis(project_axis):
    if project_axis not in (0, 1, 2):
        raise ValueError("The projection axis can only be 0-x, 1-y and 2-z!")


def _check_crop2d(points, boxes):   # box2dr_crop's checks
    if len(points.shape) != 2 or points.shape[1] != 2:
        raise ValueError("Input points should be Nx2 tensors!")
    if len(boxes.shape) != 2 or boxes.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")


def _check_pdist2d(points, boxes):   # box2dr_pdist's checks
    if len(boxes.shape) != 2:
        raise ValueError("Input boxes should be Nx2 tensors!")
    if boxes.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")
    if len(points.shape) != 2 or points.shape[1] != 2:
        raise ValueError("Input points should be Nx2 tensors!")


def _check_3d(points, boxes):
    if len(points.shape) != 2 or points.shape[1] != 3:
        raise ValueError("Input points should be Nx3 tensors!")
    if len(boxes.shape) != 2 or boxes.shape[1] != 7:
        raise ValueError("Input boxes should have 7 fields: x, y, z, lx, ly, lz, r")


def _crop_axis_mask(points, boxes, project_axis):
    """box3dp_crop's test along the projected axis, [M, N]"""
    points_p = points[:, [project_axis]].t()
    boxes_p = boxes[:, [project_axis]]
    boxes_pd = boxes[:, [3 + project_axis]] / 2
    return (points_p - boxes_pd < boxes_p) & (boxes_p < points_p + boxes_pd)


def _point_box_pair(points, boxes):
    """points and boxes on the device; their dtypes are checked first"""
    _c.dtype_code(points.dtype)
    if boxes.dtype != points.dtype:
        raise RuntimeError("points and boxes must have the same dtype")
    return _c.to_device(points), _c.to_device(boxes)


def crop_2dr_cuda(points, boxes, out=None):
    """bool[M, N] mask of the points [N,2] inside the rotated boxes [M,5] (reference crop_2dr, d3d/box/utils.h:45; CUDA tensors);
    `out`: a contiguous bool [M, N] to write it into"""
    code = _c.dtype_code(points.dtype)
    if boxes.dtype != points.dtype:
        raise RuntimeError("points and boxes must have the same dtype")
    n, m = points.shape[0], boxes.shape[0]
    mask = torch.empty((m, n), dtype=torch.bool, device=points.device) if out is None else out
    if n and m:
        ws = _c.workspace(_c.crop_workspace_bytes(n, m, code), points.device)
        with torch.cuda.device(points.device):
            st = _c.crop2dr[code](_c.ptr(points), n, _c.ptr(boxes), m, _c.ptr(mask), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box2dr_crop")
    return mask


def box2dr_crop(points, boxes):
    '''
    Crop point points points out given rotated boxes (reference d3d/box/__init__.py:278-287).
    The result is the M x N indicator mask of the points lying in each box (what the reference's crop_2dr returns).

    :param points: The input point points, shape: N x 2
    :param boxes: Input boxes array, shape: M x 5
    '''
    _check_crop2d(points, boxes)
    odev = points.device
    r = crop_2dr_cuda(_c.to_device(points).contiguous(), _c.to_device(boxes).contiguous())
    return r if odev.type == "cuda" else r.cpu()


def box3dp_crop(points, boxes, project_axis=2):
    '''
    Crop point points points out given rotated boxes with boxes projected to given axis (reference d3d/box/__init__.py:289-314)

    :param points: The input point points, shape: N x 3
    :param boxes: Input boxes array, shape: M x 7
    :param project_axis: Axis for the box to be projected to. {0: x, 1: y, 2: z}
    '''
    _check_axis(project_axis)
    pc, bc = _PLANE[project_axis]
    mask_2d = box2dr_crop(points[:, pc], boxes[:, bc])
    return mask_2d & _crop_axis_mask(points, boxes, project_axis).to(mask_2d.device)


class PDist2DR(torch.autograd.Function):
    """Differentiable signed distance from points to rotated boxes (reference d3d/box/__init__.py:149-166 over pdist2dr_forward /
    pdist2dr_backward[_cuda], d3d/box/dist.h:7-23).  Returns T[M boxes, N points]: the signed Euclidean distance to the boundary of the
    closed rectangle with half extents |w|/2, |h|/2 turned by r, positive inside -- the layout of the native function (and of
    box2dr_crop).  The reference's wrapper hands (boxes, points) to a native function declared (points, boxes) and cannot run."""
    @staticmethod
    def forward(ctx, points, boxes):
        code = _c.dtype_code(points.dtype)
        if boxes.dtype != points.dtype:
            raise RuntimeError("points and boxes must have the same dtype")
        n, m = points.shape[0], boxes.shape[0]
        dist = torch.empty((m, n), dtype=points.dtype, device=points.device)
        if n and m:
            with torch.cuda.device(points.device):
                st = _c.pdist2dr[code](_c.ptr(points), n, _c.ptr(boxes), m, _c.ptr(dist), None, _c.stream_ptr())
            _c.check(st, "box2dr_pdist")
        ctx.save_for_backward(points, boxes)
        return dist

    @staticmethod
    def backward(ctx, grad):
        points, boxes = ctx.saved_tensors
        code = _c.dtype_code(points.dtype)
        n, m = points.shape[0], boxes.shape[0]
        grad = grad.contiguous()
        grad_boxes, grad_points = torch.zeros_like(boxes), torch.zeros_like(points)
        if n and m:
            with torch.cuda.device(points.device):
                st = _c.pdist2dr_backward[code](_c.ptr(points), n, _c.ptr(boxes), m, _c.ptr(grad), _c.ptr(grad_boxes), _c.ptr(grad_points), _c.stream_ptr())
            _c.check(st, "box2dr_pdist backward")
        return grad_points, grad_boxes


def seg1d_pdist(points, segs):
    """Signed distance from points [N] to 1-D segments [M, 2] (centre, width), positive inside: [M, N]
    (reference d3d/box/__init__.py:316-328, in the [segments, points] layout of box2dr_pdist)."""
    assert torch.all(segs[:, 1] > 0)
    dsegs = (segs[:, 1] / 2)[:, None]
    ctr = segs[:, 0][:, None]
    return torch.where(points[None, :] > ctr, (ctr + dsegs) - points[None, :], points[None, :] - (ctr - dsegs))


def box2dr_pdist(points, boxes, method="rbox"):
    '''
    Calculate signed distance from points to 2d boxes (surfaces), positive inside (reference d3d/box/__init__.py:330-346).
    Differentiable in points and boxes.

    :param points: target points, shape: N x 2
    :param boxes: target boxes, shape: M x 5
    :param method: 'rbox' - rotated box
    :return: M x N
    '''
    _check_pdist2d(points, boxes)
    if method != "rbox":
        raise ValueError("Only supported rotated boxes by now!")
    odev = points.device
    r = PDist2DR.apply(_c.to_device(points).contiguous(), _c.to_device(boxes).contiguous())
    return r if odev.type == "cuda" else r.cpu()


def box3dr_pdist(points, boxes, project_axis=2):
    '''
    Calculate signed distance from points to 3d boxes (surfaces) (reference d3d/box/__init__.py:348-381)

    :param points: target points, shape: N x 3
    :param boxes: target boxes, shape: M x 7
    :param project_axis: Axis for the box to be projected to. {0: x, 1: y, 2: z}
    :return: M x N
    '''
    _check_axis(project_axis)
    pc, bc = _PLANE[project_axis]
    dist_2d = box2dr_pdist(points[:, pc], boxes[:, bc])
    dist_p = seg1d_pdist(points[:, project_axis], boxes[:, [project_axis, 3 + project_axis]]).to(dist_2d.device)
    # on an edge of the prism (both terms 0) the square root has no derivative: take it of 1 there, so that its backward, which runs
    # for every pair whichever branch is selected, multiplies by a finite number instead of 0 * inf = NaN
    sq = dist_2d.square() + dist_p.square()
    corner = torch.where(sq > 0, -torch.sqrt(torch.where(sq > 0, sq, torch.ones_like(sq))), torch.zeros_like(sq))
    return torch.where(dist_p > 0,
                       torch.where(dist_2d > 0, torch.min(dist_p, dist_2d), dist_2d),
                       torch.where(dist_2d > 0, dist_p, corner))


# ------------------------------------------------------------------ frame-batched point <-> box operators
def _crop_batch(points, boxes, point_offsets, box_offsets, project_axis):
    if _frames.empty(points):   # whatever `boxes` holds
        return []
    P, B, fr = _frames.inputs(points, boxes, point_offsets, box_offsets, _check_crop2d if project_axis < 0 else _check_3d, ("points", "boxes"))
    P, B = _point_box_pair(P, B)
    fr = fr.T   # the masks are [boxes, points] blocks
    code = _c.dtype_code(P.dtype)
    n_b, n_p = fr.lengths()
    mask = torch.empty(int(fr.blocks[-1]), dtype=torch.bool, device=P.device)
    big = n_b * n_p >= int(_c.crop_grid_min_pairs())   # the single-frame grid path is faster on these
    small = (n_b * n_p > 0) & ~big
    if bool(small.any()):
        od_b, od_p, od_m = _frames.to_device(P.device, fr.rows, fr.cols, fr.blocks)
        max_b, max_p = fr.bounds(small)
        ws = _c.workspace(_c.crop_batch_workspace_bytes(len(B), code), P.device)
        with torch.cuda.device(P.device):
            st = _c.crop2dr_batch[code](_c.ptr(P), len(P), _c.ptr(od_p), _c.ptr(B), len(B), _c.ptr(od_b), fr.nframes, max_p, max_b, project_axis,
                                        _c.ptr(od_m), _c.ptr(mask), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box2dr_crop_batch" if project_axis < 0 else "box3dp_crop_batch")
    for _, rb, cp, k in fr.each(big):
        p, b = P[cp], B[rb]
        block = mask[k].view(len(b), len(p))
        if project_axis < 0:
            crop_2dr_cuda(p, b, out=block)
        else:
            pc, bc = _PLANE[project_axis]
            crop_2dr_cuda(p[:, pc].contiguous(), b[:, bc].contiguous(), out=block)
            block &= _crop_axis_mask(p, b, project_axis)
    return fr.matrices(mask)


def box2dr_crop_batch(points, boxes, point_offsets=None, box_offsets=None):
    '''
    :func:`box2dr_crop` on a batch of frames (ground-truth point labels or segmentation targets of a training batch); per frame the mask
    equals :func:`box2dr_crop` on that frame, bit for bit.  Two call forms, like :func:`box3d_iou_distance_batch`: lists of per-frame
    ``points`` [N_f, 2] / ``boxes`` [M_f, 5] (returns the list of bool [M_f, N_f] masks, views into one packed buffer), or the frames
    packed back to back with ``point_offsets`` / ``box_offsets`` (int64 [nframes + 1], CPU) (returns ``(mask_flat, mask_offsets)``: frame
    f's mask is ``mask_flat[mask_offsets[f]:mask_offsets[f + 1]].view(M_f, N_f)``, ``mask_offsets`` the running sum of M_f * N_f).
    numpy in -> numpy out, host tensors in -> host tensors out.
    '''
    return _crop_batch(points, boxes, point_offsets, box_offsets, -1)


def box3dp_crop_batch(points, boxes, point_offsets=None, box_offsets=None, project_axis=2):
    '''
    :func:`box3dp_crop` on a batch of frames: points [N_f, 3], boxes [M_f, 7]; call forms and outputs as :func:`box2dr_crop_batch`, and
    per frame the mask equals :func:`box3dp_crop` on that frame, bit for bit (the test along ``project_axis`` runs in the kernel).
    '''
    _check_axis(project_axis)
    return _crop_batch(points, boxes, point_offsets, box_offsets, project_axis)


def _crop_assign_frame(p, b, project_axis, point_box, box_npoints):
    """one frame's reductions on the device, written into the given int64 slices (the single-frame entry: grid path on large frames)"""
    code = _c.dtype_code(p.dtype)
    n, m = len(p), len(b)
    if n or m:
        ws = _c.workspace(_c.crop_assign_workspace_bytes(n, m, code) if n and m else 0, p.device)
        with torch.cuda.device(p.device):
            st = _c.crop2dr_assign[code](_c.ptr(p), n, _c.ptr(b), m, project_axis, _c.ptr(point_box), _c.ptr(box_npoints), _c.ptr(ws), ws.numel(),
                                         _c.stream_ptr())
        _c.check(st, "box2dr_crop_assign" if project_axis < 0 else "box3dp_crop_assign")


def _crop_assign(points, boxes, project_axis):
    numpy_in = isinstance(points, np.ndarray)
    if numpy_in:
        assert isinstance(boxes, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
        points, boxes = torch.from_numpy(points), torch.from_numpy(boxes)
    (_check_crop2d if project_axis < 0 else _check_3d)(points, boxes)
    P, B = _point_box_pair(points.detach(), boxes.detach())
    point_box = torch.empty(len(P), dtype=torch.int64, device=P.device)
    box_npoints = torch.empty(len(B), dtype=torch.int64, device=P.device)
    _crop_assign_frame(P, B, project_axis, point_box, box_npoints)
    fr = _frames.Frames([0, len(P)], [0, len(B)], False, numpy_in, points.device)   # one frame
    return fr.outputs(rows=(point_box,), cols=(box_npoints,))


def box2dr_crop_assign(points, boxes):
    '''
    The two reductions of :func:`box2dr_crop`'s mask that point labels and box filters use, without the mask.  Returns
    ``(point_box, box_npoints)``: ``point_box`` int64 [N] is the lowest index of a box containing each point, or -1 if there is none
    (``torch.where(mask.any(0), mask.to(torch.uint8).argmax(0), -1)``), and ``box_npoints`` int64 [M] the number of points inside each box
    (``mask.sum(1)``), both exactly equal to those of the mask.  The outputs carry no grad.  numpy in -> numpy out, host tensors in -> host
    tensors out.

    :param points: The input points, shape: N x 2
    :param boxes: Input boxes array, shape: M x 5
    '''
    return _crop_assign(points, boxes, -1)


def box3dp_crop_assign(points, boxes, project_axis=2):
    '''
    :func:`box2dr_crop_assign` for :func:`box3dp_crop`'s mask: points [N, 3], boxes [M, 7] projected to ``project_axis``.

    :param points: The input points, shape: N x 3
    :param boxes: Input boxes array, shape: M x 7
    :param project_axis: Axis for the box to be projected to. {0: x, 1: y, 2: z}
    '''
    _check_axis(project_axis)
    return _crop_assign(points, boxes, project_axis)


def _crop_assign_batch(points, boxes, point_offsets, box_offsets, project_axis):
    if _frames.empty(points):   # whatever `boxes` holds
        return []
    P, B, fr = _frames.inputs(points, boxes, point_offsets, box_offsets, _check_crop2d if project_axis < 0 else _check_3d, ("points", "boxes"))
    P, B = _point_box_pair(P.detach(), B.detach())
    P, B = P.contiguous(), B.contiguous()
    code = _c.dtype_code(P.dtype)
    n_p, n_b = fr.lengths()
    point_box = torch.empty(len(P), dtype=torch.int64, device=P.device)
    box_npoints = torch.empty(len(B), dtype=torch.int64, device=P.device)
    big = n_p * n_b >= int(_c.crop_grid_min_pairs())   # the single-frame entry (grid path) computes these
    if fr.nframes and len(P) + len(B):
        od_p, od_b = _frames.to_device(P.device, fr.rows, fr.cols)
        ws = _c.workspace(_c.crop_assign_batch_workspace_bytes(len(B), code), P.device)
        max_p, max_b = fr.bounds((n_p * n_b > 0) & ~big)
        with torch.cuda.device(P.device):   # bounds of 1 when no frame is left to it: the call still initialises every output slice
            st = _c.crop2dr_assign_batch[code](_c.ptr(P), len(P), _c.ptr(od_p), _c.ptr(B), len(B), _c.ptr(od_b), fr.nframes, max_p or 1, max_b or 1,
                                               project_axis, _c.ptr(point_box), _c.ptr(box_npoints), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box2dr_crop_assign_batch" if project_axis < 0 else "box3dp_crop_assign_batch")
    for _, r, c, _ in fr.each(big):   # after the batch call, which initialises every slice
        _crop_assign_frame(P[r], B[c], project_axis, point_box[r], box_npoints[c])
    return fr.outputs(rows=(point_box,), cols=(box_npoints,))


def box2dr_crop_assign_batch(points, boxes, point_offsets=None, box_offsets=None):
    '''
    :func:`box2dr_crop_assign` on a batch of frames in one launch sequence; per frame the outputs equal :func:`box2dr_crop_assign` on that
    frame exactly.  Two call forms, like :func:`box2dr_crop_batch`: lists of per-frame ``points`` [N_f, 2] / ``boxes`` [M_f, 5] (returns the
    list of per-frame ``(point_box, box_npoints)`` tuples), or the frames packed back to back with ``point_offsets`` / ``box_offsets``
    (int64 [nframes + 1], CPU) (returns the packed ``(point_box [total_points], box_npoints [total_boxes])``, with FRAME-LOCAL box indices
    as :func:`box2d_iou_max_batch` gives them).  The outputs carry no grad.  numpy in -> numpy out, host tensors in -> host tensors out.
    '''
    return _crop_assign_batch(points, boxes, point_offsets, box_offsets, -1)


def box3dp_crop_assign_batch(points, boxes, point_offsets=None, box_offsets=None, project_axis=2):
    '''
    :func:`box3dp_crop_assign` on a batch of frames: points [N_f, 3], boxes [M_f, 7]; call forms and outputs as
    :func:`box2dr_crop_assign_batch`, and per frame the outputs equal :func:`box3dp_crop_assign` on that frame exactly.
    '''
    _check_axis(project_axis)
    return _crop_assign_batch(points, boxes, point_offsets, box_offsets, project_axis)


class _PDistBatch(torch.autograd.Function):
    """packed distances of all frames: forward and backward are one launch each"""
    @staticmethod
    def forward(ctx, points, boxes, offsets, nframes, max_points, max_boxes, project_axis, total):
        code = _c.dtype_code(points.dtype)
        dist = torch.empty(total, dtype=points.dtype, device=points.device)
        if total:
            od_p, od_b, od_d = offsets
            with torch.cuda.device(points.device):
                st = _c.pdist2dr_batch[code](_c.ptr(points), len(points), _c.ptr(od_p), _c.ptr(boxes), len(boxes), _c.ptr(od_b), nframes, max_points,
                                             max_boxes, project_axis, _c.ptr(od_d), _c.ptr(dist), _c.stream_ptr())
            _c.check(st, "box2dr_pdist_batch" if project_axis < 0 else "box3dr_pdist_batch")
        ctx.save_for_backward(points, boxes, *offsets)
        ctx.args = (nframes, max_points, max_boxes, project_axis, total)
        return dist

    @staticmethod
    def backward(ctx, grad):
        points, boxes, od_p, od_b, od_d = ctx.saved_tensors
        nframes, max_points, max_boxes, project_axis, total = ctx.args
        code = _c.dtype_code(points.dtype)
        grad = grad.contiguous()
        grad_points, grad_boxes = torch.zeros_like(points), torch.zeros_like(boxes)
        if total:
            with torch.cuda.device(points.device):
                st = _c.pdist2dr_batch_backward[code](_c.ptr(points), len(points), _c.ptr(od_p), _c.ptr(boxes), len(boxes), _c.ptr(od_b), nframes,
                                                      max_points, max_boxes, project_axis, _c.ptr(od_d), _c.ptr(grad), _c.ptr(grad_boxes),
                                                      _c.ptr(grad_points), _c.stream_ptr())
            _c.check(st, "box2dr_pdist_batch backward" if project_axis < 0 else "box3dr_pdist_batch backward")
        return grad_points, grad_boxes, None, None, None, None, None, None


def _pdist_batch(points, boxes, point_offsets, box_offsets, project_axis):
    if _frames.empty(points):   # whatever `boxes` holds
        return []
    P, B, fr = _frames.inputs(points, boxes, point_offsets, box_offsets, _check_pdist2d if project_axis < 0 else _check_3d, ("points", "boxes"))
    P, B = _point_box_pair(P, B)
    if project_axis >= 0:
        assert torch.all(B[:, 3 + project_axis] > 0)   # seg1d_pdist's condition, once for the batch
    fr = fr.T   # the distances are [boxes, points] blocks
    max_b, max_p = fr.bounds()
    od_b, od_p, od_d = _frames.to_device(P.device, fr.rows, fr.cols, fr.blocks)
    dist = _PDistBatch.apply(P.contiguous(), B.contiguous(), (od_p, od_b, od_d), fr.nframes, max_p, max_b, project_axis, int(fr.blocks[-1]))
    return fr.matrices(dist)


def box2dr_pdist_batch(points, boxes, point_offsets=None, box_offsets=None):
    '''
    :func:`box2dr_pdist` on a batch of frames (centerness and distance targets of a training batch); differentiable in points and boxes.
    Call forms and outputs as :func:`box2dr_crop_batch`, with T [M_f, N_f] distances; per frame the values equal :func:`box2dr_pdist`
    on that frame bit for bit, and the gradients agree to rounding (both sum with atomics).
    '''
    return _pdist_batch(points, boxes, point_offsets, box_offsets, -1)


def box3dr_pdist_batch(points, boxes, point_offsets=None, box_offsets=None, project_axis=2):
    '''
    :func:`box3dr_pdist` on a batch of frames: points [N_f, 3], boxes [M_f, 7]; call forms and outputs as :func:`box2dr_pdist_batch`.
    The combination with the distance along ``project_axis`` runs in the kernel, forward and backward; per frame the values equal
    :func:`box3dr_pdist` bit for bit.  Non-positive extents along the axis raise AssertionError, as in :func:`seg1d_pdist`.
    '''
    _check_axis(project_axis)
    return _pdist_batch(points, boxes, point_offsets, box_offsets, project_axis)


def _dist3d_input(boxes):
    """float32 copy on the device with the sizes clamped to +-1e3: "prevent really weird boxes with unusual size" (matcher.pyx:50-52)"""
    b = _c.to_device(boxes).to(torch.float32).contiguous().clone()
    b[:, 3:6].clamp_(-1e3, 1e3)
    return b


def _check_boxes3d(src_boxes, dst_boxes):
    if len(src_boxes.shape) != 2 or len(dst_boxes.shape) != 2 or src_boxes.shape[1] != 7 or dst_boxes.shape[1] != 7:
        raise ValueError("Input boxes should be Nx7 tensors: x, y, z, lx, ly, lz, rz")


def box3d_iou_distance(src_boxes, dst_boxes, metric="riou"):
    '''
    Distance matrix of the detection evaluator / tracking matcher: ``1 - iou2d * ziou`` in float32, the array
    ``ScoreMatcher.prepare_boxes`` caches (reference d3d/tracking/matcher.pyx:24-82 over box3dr_iou / box3d_iou,
    d3d/dgal_wrap.h:45-91).

    :param src_boxes: boxes to match, shape N x 7: x, y, z, lx, ly, lz, rz (the columns 2..8 of ``Target3DArray.to_numpy()``)
    :param dst_boxes: fixed boxes (such as ground truth boxes), shape M x 7
    :param metric: 'riou' - rotated BEV IoU times the z overlap ratio (DistanceTypes.RIoU), 'iou' - IoU of the BEV
        axis-aligned bounding boxes times the z overlap ratio (DistanceTypes.IoU)
    :return: float32 N x M; numpy in -> numpy out, host tensors in -> host tensor out
    '''
    convert_numpy = False
    if isinstance(src_boxes, np.ndarray):
        assert isinstance(dst_boxes, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
        src_boxes, dst_boxes = torch.from_numpy(src_boxes), torch.from_numpy(dst_boxes)
        convert_numpy = True
    _check_boxes3d(src_boxes, dst_boxes)
    if metric.lower() not in ("riou", "iou"):
        raise ValueError("Unrecognized distance metric!")
    odev = src_boxes.device
    b1, b2 = _dist3d_input(src_boxes), _dist3d_input(dst_boxes)
    n, m = b1.shape[0], b2.shape[0]
    out = torch.empty((n, m), dtype=torch.float32, device=b1.device)
    if n and m:
        ws = _c.workspace(_c.iou3d_distance_workspace_bytes(n, m), b1.device)
        with torch.cuda.device(b1.device):
            st = _c.iou3d_distance(_c.ptr(b1), n, _c.ptr(b2), m, 1 if metric.lower() == "riou" else 0, _c.ptr(out), out.stride(0),
                                   _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box3d_iou_distance")
    if odev.type != "cuda":
        out = out.cpu()
    return out.numpy() if convert_numpy else out


def nms2d_cuda(boxes, scores, iou_type, supression_type, iou_threshold, score_threshold, supression_param):
    """Suppressed mask bool[N] in original order (reference d3d/box/nms.h:6-10, nms_cuda.cu:217-244)."""
    code = _c.dtype_code(boxes.dtype)
    if scores.dtype != boxes.dtype:
        raise RuntimeError("boxes and scores must have the same dtype")
    n = boxes.shape[0]
    suppressed = torch.empty(n, dtype=torch.uint8, device=boxes.device)
    ws = _c.workspace(_c.nms_workspace_bytes(n, code), boxes.device)
    with torch.cuda.device(boxes.device):
        st = _c.nms2d[code](_c.ptr(boxes), _c.ptr(scores), n, int(iou_type), int(supression_type), float(iou_threshold),
                            float(score_threshold), float(supression_param), _c.ptr(suppressed), _c.ptr(ws), ws.numel(),
                            _c.stream_ptr())
    if st == _c.ERR_INVALID and int(iou_type) not in (IouType.BOX, IouType.RBOX):
        raise ValueError("Unsupported iou type!")
    _c.check(st, "box2d_nms")
    return suppressed.view(torch.bool)


def box2d_nms(boxes, scores, iou_method="box", supression_method="hard",
    iou_threshold=0, score_threshold=0, supression_param=0, precise=True):
    '''
    NMS on axis-aligned or rotated 2D boxes (reference d3d/box/__init__.py:226-276).  Returns the
    KEEP mask bool[N] in the original box order.

    :param iou_method: 'box' - axis-aligned box, 'rbox' - rotated box
    :param precise: force using double precision to calculate iou
    :param iou_threshold: IoU threshold for two boxes to be considered as overlapped
    :param score_threshold: Minimum score for a box to be considered as valid
    '''
    convert_numpy = False
    if isinstance(boxes, np.ndarray):
        assert isinstance(scores, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
        boxes = torch.from_numpy(boxes)
        scores = torch.from_numpy(scores)
        convert_numpy = True
    odev = boxes.device

    if len(boxes) != len(scores):
        raise ValueError("Numbers of boxes and scores are inconsistent!")
    if boxes.numel() == 0:
        mask = torch.tensor([], dtype=torch.bool)
        return mask.numpy() if convert_numpy else mask

    iou_type = getattr(IouType, iou_method.upper())
    supression_type = getattr(SupressionType, supression_method.upper())

    b, s = _c.to_device(boxes), _c.to_device(scores)
    if precise:
        b, s = b.to(torch.float64), s.to(torch.float64)
    elif s.dtype != b.dtype:
        s = s.to(b.dtype)
    if len(s.shape) == 2:
        s = s.max(axis=1).values.contiguous()

    suppressed = nms2d_cuda(b, s, iou_type, supression_type, iou_threshold, score_threshold, supression_param)
    mask = ~suppressed
    if odev.type != "cuda":
        mask = mask.cpu()
    if convert_numpy:
        return mask.numpy()
    return mask


def _as_tensor(x, dt):
    return (torch.from_numpy(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else torch.as_tensor(x)).to(dt)


def match_greedy(distance, src_scores, src_tags, dst_tags, thresholds):
    '''
    Greedy score-ordered matching on a distance matrix: ``ScoreMatcher.match`` of the reference (d3d/tracking/matcher.pyx:138-162 over
    match_by_order :93-122) for one or many threshold sets at once -- the detection evaluator's loop over score thresholds
    (d3d/benchmarks.pyx:220-238) is one launch.  Source boxes are visited from the best score down (ties: the later box first, like
    ``np.flip(np.argsort(scores))``); each takes the closest free destination box of its category whose distance is <= the threshold.

    :param distance: float32 N x M, e.g. the result of :func:`box3d_iou_distance`
    :param src_scores: N scores of the source boxes
    :param src_tags, dst_tags: integer category per source / destination box, values in [0, C)
    :param thresholds: T x C (or C for a single set): maximum distance per category
    :return: (src_assignment int32 T x N, dst_assignment int32 T x M) with -1 for unmatched boxes; the leading dimension is dropped
        for a single threshold set.  numpy in -> numpy out.
    '''
    convert_numpy = isinstance(distance, np.ndarray)
    distance = _as_tensor(distance, torch.float32)
    odev = distance.device
    d = _c.to_device(distance).contiguous()
    dev = d.device
    if d.dim() != 2:
        raise ValueError("distance should be an NxM matrix")
    n, m = d.shape
    thr = _as_tensor(thresholds, torch.float32)
    single = thr.dim() == 1
    thr = thr.reshape(1, -1) if single else thr
    scores = _as_tensor(src_scores, torch.float64)
    st, dt_ = _as_tensor(src_tags, torch.int32).to(dev).contiguous(), _as_tensor(dst_tags, torch.int32).to(dev).contiguous()
    if len(scores) != n or len(st) != n or len(dt_) != m:
        raise ValueError("scores / tags do not match the distance matrix")
    order = torch.flip(torch.argsort(scores.cpu(), stable=True), dims=[0]).to(torch.int32).to(dev).contiguous()   # np.flip(np.argsort(scores))
    thr = thr.to(dev).contiguous()
    T, ncat = thr.shape
    sa = torch.empty((T, n), dtype=torch.int32, device=dev)
    da = torch.empty((T, m), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        stt = _c.match_greedy(_c.ptr(d), n, m, d.stride(0) if n else max(m, 1), _c.ptr(order), _c.ptr(st), _c.ptr(dt_), _c.ptr(thr), T, ncat, _c.ptr(sa), _c.ptr(da),
                              _c.stream_ptr())
    _c.check(stt, "match_greedy")
    if single:
        sa, da = sa[0], da[0]
    if odev.type != "cuda" or convert_numpy:
        sa, da = sa.cpu(), da.cpu()
    return (sa.numpy(), da.numpy()) if convert_numpy else (sa, da)


def box3d_iou_distance_batch(src_boxes, dst_boxes, src_offsets=None, dst_offsets=None, metric="riou"):
    '''
    :func:`box3d_iou_distance` on a batch of frames in one launch sequence (the detection evaluator computes one matrix per frame of a
    validation set); per frame the matrix equals :func:`box3d_iou_distance` on that frame, bit for bit.  Two call forms, like
    :func:`box2d_nms_batch`: lists of per-frame ``src_boxes`` [n_f, 7] / ``dst_boxes`` [m_f, 7] (returns the list of [n_f, m_f] float32
    matrices, views into one packed buffer), or the frames packed back to back as ``src_boxes`` [total_src, 7] / ``dst_boxes``
    [total_dst, 7] with ``src_offsets`` / ``dst_offsets`` (int64 [nframes + 1], CPU) (returns ``(dist_flat, dist_offsets)``: frame f's
    matrix is ``dist_flat[dist_offsets[f]:dist_offsets[f + 1]].view(n_f, m_f)``).  numpy in -> numpy out, host tensors in -> host tensors out.

    :param metric: 'riou' or 'iou', as in :func:`box3d_iou_distance`
    '''
    if _frames.empty(src_boxes, dst_boxes):
        return []
    A, B, fr = _frames.inputs(src_boxes, dst_boxes, src_offsets, dst_offsets, _check_boxes3d, ("src_boxes", "dst_boxes"), dtype=torch.float32)
    if metric.lower() not in ("riou", "iou"):
        raise ValueError("Unrecognized distance metric!")
    b1, b2 = _dist3d_input(A), _dist3d_input(B)   # one copy to the device per box set
    dist = torch.empty(int(fr.blocks[-1]), dtype=torch.float32, device=b1.device)
    if dist.numel():
        od1, od2, odd = _frames.to_device(b1.device, fr.rows, fr.cols, fr.blocks)
        ws = _c.workspace(_c.iou3d_distance_batch_workspace_bytes(len(b1), len(b2), fr.nframes), b1.device)
        with torch.cuda.device(b1.device):
            st = _c.iou3d_distance_batch(_c.ptr(b1), len(b1), _c.ptr(od1), _c.ptr(b2), len(b2), _c.ptr(od2), fr.nframes, *fr.bounds(),
                                         1 if metric.lower() == "riou" else 0, _c.ptr(odd), _c.ptr(dist), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box3d_iou_distance_batch")
    return fr.matrices(dist)


def _frame_score_order(scores, src_off_dev, nframes):
    """per frame np.flip(np.argsort(scores, kind="stable")) (descending, ties to the higher index, NaN first) in frame-local indices,
    from device sorts and gathers without a host synchronise"""
    dev, total = scores.device, scores.numel()
    s = torch.where(torch.isnan(scores), float("nan"), scores + 0.0)   # one NaN and one zero, so the device sort orders like the host sort
    fid = torch.repeat_interleave(torch.arange(nframes, device=dev), src_off_dev[1:] - src_off_dev[:-1], output_size=total)
    o = torch.argsort(s, stable=True)                  # ascending over the whole batch
    o = o[torch.argsort(fid[o], stable=True)]          # grouped by frame, ascending inside each frame
    start = src_off_dev[:-1][fid]
    rev = start + src_off_dev[1:][fid] - 1 - torch.arange(total, device=dev)   # reverse each frame's segment
    return (o[rev] - start).to(torch.int32).contiguous()


def match_greedy_batch(distance, src_scores, src_tags, dst_tags, thresholds, src_offsets=None, dst_offsets=None):
    '''
    :func:`match_greedy` on a batch of frames in one launch: per frame and threshold set the assignment equals :func:`match_greedy` on
    that frame.  Two call forms, like :func:`box3d_iou_distance_batch`: lists of per-frame ``distance`` [n_f, m_f], ``src_scores``,
    ``src_tags`` and ``dst_tags`` (returns a list of per-frame ``(src_assignment, dst_assignment)`` pairs shaped as :func:`match_greedy`
    shapes them), or ``distance = (dist_flat, dist_offsets)`` as the packed :func:`box3d_iou_distance_batch` returns it, packed scores and
    tags, and ``src_offsets`` / ``dst_offsets`` (int64 [nframes + 1], CPU) (returns ``(src_assignment [T, total_src], dst_assignment
    [T, total_dst])`` with frame-local indices).  The thresholds (T x C, or C for a single set, which drops the leading dimension) are
    shared by all frames.  Frames of more than 4096 destination boxes fall back to one :func:`match_greedy` call per frame.
    numpy in -> numpy out, host tensors in -> host tensors out.
    '''
    if src_offsets is None and dst_offsets is None:
        frames = list(distance)
        if not len(frames) == len(src_scores) == len(src_tags) == len(dst_tags):
            raise ValueError("distance, scores and tags should hold the same number of frames")
        if not frames:
            return []
        dl = [_as_tensor(d, torch.float32) for d in frames]
        if any(d.dim() != 2 for d in dl):
            raise ValueError("distance should be an NxM matrix")
        fr = _frames.Frames(_frames.offsets_of(d.shape[0] for d in dl), _frames.offsets_of(d.shape[1] for d in dl), True,
                            isinstance(frames[0], np.ndarray), dl[0].device)
        d = torch.cat([x.reshape(-1) for x in dl])
        cat = lambda xs, dt: torch.cat([_as_tensor(x, dt).reshape(-1) for x in xs])  # noqa: E731
        scores, st, dt_ = cat(src_scores, torch.float64), cat(src_tags, torch.int32), cat(dst_tags, torch.int32)
    else:
        if src_offsets is None or dst_offsets is None:
            raise ValueError("packed distances need the frame offsets")
        d, given = distance
        numpy_in = isinstance(d, np.ndarray)
        d = _as_tensor(d, torch.float32)
        fr = _frames.Frames(src_offsets, dst_offsets, False, numpy_in, d.device)
        d = d.reshape(-1)
        if not torch.equal(_frames.offsets(given), fr.blocks) or int(fr.blocks[-1]) != d.numel():
            raise ValueError("distance blocks do not match the frame offsets")
        scores, st, dt_ = _as_tensor(src_scores, torch.float64).reshape(-1), _as_tensor(src_tags, torch.int32), _as_tensor(dst_tags, torch.int32)
    total_src, total_dst = int(fr.rows[-1]), int(fr.cols[-1])
    if len(scores) != total_src or len(st) != total_src or len(dt_) != total_dst:
        raise ValueError("scores / tags do not match the distance matrix")
    thr = _as_tensor(thresholds, torch.float32)
    single = thr.dim() == 1
    thr = thr.reshape(1, -1) if single else thr
    T, ncat = thr.shape
    d = _c.to_device(d)
    dev = d.device
    thr, scores, st, dt_ = thr.to(dev).contiguous(), scores.to(dev).contiguous(), st.to(dev).contiguous(), dt_.to(dev).contiguous()
    max_dst = fr.bounds()[1]
    sa = torch.full((T, total_src), -1, dtype=torch.int32, device=dev)
    da = torch.full((T, total_dst), -1, dtype=torch.int32, device=dev)
    if max_dst > 4096:   # the kernel's taken bitmask holds 4096 destinations
        for _, r, c, k in fr.each():
            sa[:, r], da[:, c] = match_greedy(d[k].view(r.stop - r.start, c.stop - c.start), scores[r], st[r], dt_[c], thr)
    elif T and d.numel():
        os_, od_, odd = _frames.to_device(dev, fr.rows, fr.cols, fr.blocks)
        order = _frame_score_order(scores, os_, fr.nframes)
        with torch.cuda.device(dev):
            stt = _c.match_greedy_batch(_c.ptr(d), _c.ptr(odd), _c.ptr(os_), _c.ptr(od_), fr.nframes, max_dst, _c.ptr(order), _c.ptr(st), _c.ptr(dt_),
                                        _c.ptr(thr), T, ncat, _c.ptr(sa), _c.ptr(da), _c.stream_ptr())
        _c.check(stt, "match_greedy_batch")
    if single:
        sa, da = sa[0], da[0]
    return fr.outputs(rows=(sa,), cols=(da,))
