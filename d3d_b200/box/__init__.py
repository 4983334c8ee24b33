"""d3d_b200.box -- pairwise IoU and NMS on (rotated) 2-D boxes.  Mirrors reference d3d/box/__init__.py
(box2d_iou :180-224, box2d_nms :226-276, enums d3d/box/common.h:5-10) on top of the C ABI."""
import enum

import numpy as np
import torch

from .. import _cabi as _c


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
    if len(boxes1.shape) != 2 or len(boxes2.shape) != 2:
        raise ValueError("Input of rbox_2d_iou should be Nx2 tensors!")
    if boxes1.shape[1] != 5 or boxes2.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")

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
    as_list = isinstance(boxes, (list, tuple))
    if as_list:
        if len(boxes) != len(scores):
            raise ValueError("Numbers of boxes and scores are inconsistent!")
        if len(boxes) == 0:
            return []
        tt = lambda x: torch.from_numpy(x) if isinstance(x, np.ndarray) else x
        numpy_in = isinstance(boxes[0], np.ndarray)
        blist, slist = [tt(b) for b in boxes], [tt(s_) for s_ in scores]
        odev = blist[0].device
        lens = [int(b.shape[0]) for b in blist]
        offsets = torch.zeros(len(lens) + 1, dtype=torch.int64)
        offsets[1:] = torch.tensor(lens).cumsum(0)
        boxes = torch.cat([_c.to_device(b).reshape(-1, 5) for b in blist], 0)
        scores = torch.cat([_c.to_device(s_).reshape(-1) for s_ in slist], 0)
    else:
        numpy_in = isinstance(boxes, np.ndarray)
        if numpy_in:
            boxes, scores = torch.from_numpy(boxes), torch.from_numpy(scores)
        odev = boxes.device
        if offsets is None:
            raise ValueError("packed boxes need the frame offsets")
        offsets = torch.as_tensor(offsets).to(torch.int64).cpu()
    if len(boxes) != len(scores) or int(offsets[-1]) != len(boxes):
        raise ValueError("Numbers of boxes and scores are inconsistent!")
    iou_type = getattr(IouType, iou_method.upper())
    if iou_type not in (IouType.BOX, IouType.RBOX):
        raise ValueError("Unsupported iou type!")
    sup_type = getattr(SupressionType, supression_method.upper())
    b, s_ = _c.to_device(boxes), _c.to_device(scores)
    if precise:
        b, s_ = b.to(torch.float64), s_.to(torch.float64)
    elif s_.dtype != b.dtype:
        s_ = s_.to(b.dtype)
    b, s_ = b.contiguous(), s_.contiguous()
    total, nframes = int(b.shape[0]), int(offsets.numel()) - 1
    max_frame = int((offsets[1:] - offsets[:-1]).max()) if nframes > 0 else 0
    suppressed = torch.zeros(total, dtype=torch.uint8, device=b.device)
    if total > 0 and max_frame > 8192:
        for f in range(nframes):
            lo, hi = int(offsets[f]), int(offsets[f + 1])
            if hi > lo:
                suppressed[lo:hi] = nms2d_cuda(b[lo:hi], s_[lo:hi], iou_type, sup_type, iou_threshold, score_threshold, supression_param).view(torch.uint8)
    elif total > 0:
        code = _c.dtype_code(b.dtype)
        od = offsets.to(b.device, non_blocking=True) if offsets_dev is None else offsets_dev
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
    keep = ~suppressed.view(torch.bool)
    if odev.type != "cuda":
        keep = keep.cpu()
    if as_list:
        out = [keep[int(offsets[f]):int(offsets[f + 1])] for f in range(nframes)]
        return [k.cpu().numpy() for k in out] if numpy_in else out
    return keep.cpu().numpy() if numpy_in else keep


def crop_2dr_cuda(points, boxes):
    """bool[M, N] mask of the points [N,2] inside the rotated boxes [M,5] (reference crop_2dr, d3d/box/utils.h:45; CUDA tensors)"""
    code = _c.dtype_code(points.dtype)
    if boxes.dtype != points.dtype:
        raise RuntimeError("points and boxes must have the same dtype")
    n, m = points.shape[0], boxes.shape[0]
    mask = torch.empty((m, n), dtype=torch.bool, device=points.device)
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
    if len(points.shape) != 2 or points.shape[1] != 2:
        raise ValueError("Input points should be Nx2 tensors!")
    if len(boxes.shape) != 2 or boxes.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")
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
    if project_axis == 0:
        points_2d, boxes_2d = points[:, [1, 2]], boxes[:, [1, 2, 4, 5, 6]]
    elif project_axis == 1:
        points_2d, boxes_2d = points[:, [0, 2]], boxes[:, [0, 2, 3, 5, 6]]
    elif project_axis == 2:
        points_2d, boxes_2d = points[:, [0, 1]], boxes[:, [0, 1, 3, 4, 6]]
    else:
        raise ValueError("The projection axis can only be 0-x, 1-y and 2-z!")
    mask_2d = box2dr_crop(points_2d, boxes_2d)
    points_p = points[:, [project_axis]].t()
    boxes_p = boxes[:, [project_axis]]
    boxes_pd = boxes[:, [3 + project_axis]] / 2
    mask_p = (points_p - boxes_pd < boxes_p) & (boxes_p < points_p + boxes_pd)
    return mask_2d & mask_p.to(mask_2d.device)


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
    if len(boxes.shape) != 2:
        raise ValueError("Input boxes should be Nx2 tensors!")
    if boxes.shape[1] != 5:
        raise ValueError("Input boxes should have 5 fields: x, y, w, h, r")
    if len(points.shape) != 2 or points.shape[1] != 2:
        raise ValueError("Input points should be Nx2 tensors!")
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
    if project_axis == 0:
        points_2d, boxes_2d = points[:, [1, 2]], boxes[:, [1, 2, 4, 5, 6]]
    elif project_axis == 1:
        points_2d, boxes_2d = points[:, [0, 2]], boxes[:, [0, 2, 3, 5, 6]]
    elif project_axis == 2:
        points_2d, boxes_2d = points[:, [0, 1]], boxes[:, [0, 1, 3, 4, 6]]
    else:
        raise ValueError("The projection axis can only be 0-x, 1-y and 2-z!")
    dist_2d = box2dr_pdist(points_2d, boxes_2d)
    dist_p = seg1d_pdist(points[:, project_axis], boxes[:, [project_axis, 3 + project_axis]]).to(dist_2d.device)
    # on an edge of the prism (both terms 0) the square root has no derivative: take it of 1 there, so that its backward, which runs
    # for every pair whichever branch is selected, multiplies by a finite number instead of 0 * inf = NaN
    sq = dist_2d.square() + dist_p.square()
    corner = torch.where(sq > 0, -torch.sqrt(torch.where(sq > 0, sq, torch.ones_like(sq))), torch.zeros_like(sq))
    return torch.where(dist_p > 0,
                       torch.where(dist_2d > 0, torch.min(dist_p, dist_2d), dist_2d),
                       torch.where(dist_2d > 0, dist_p, corner))


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


def _frame_offsets(offsets=None, lens=None):
    """CPU int64 [nframes + 1] from given offsets or from frame lengths"""
    if lens is not None:
        off = torch.zeros(len(lens) + 1, dtype=torch.int64)
        off[1:] = torch.tensor(lens, dtype=torch.int64).cumsum(0)
        return off
    off = torch.as_tensor(offsets).to(torch.int64).cpu().reshape(-1)
    if off.numel() < 1 or int(off[0]) != 0 or bool((off[1:] < off[:-1]).any()):
        raise ValueError("frame offsets must start at 0 and be ascending")
    return off


def _block_offsets(src_off, dst_off):
    """start of every frame's [n_f, m_f] block in the packed distance buffer: the running sum of n_f * m_f"""
    off = torch.zeros_like(src_off)
    off[1:] = ((src_off[1:] - src_off[:-1]) * (dst_off[1:] - dst_off[:-1])).cumsum(0)
    return off


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
    as_list = isinstance(src_boxes, (list, tuple))
    if as_list:
        if not isinstance(dst_boxes, (list, tuple)) or len(src_boxes) != len(dst_boxes):
            raise ValueError("src_boxes and dst_boxes should hold the same number of frames")
        if len(src_boxes) == 0:
            return []
        numpy_in = isinstance(src_boxes[0], np.ndarray)
        tt = lambda x: torch.from_numpy(x) if isinstance(x, np.ndarray) else x  # noqa: E731
        slist, dlist = [tt(b) for b in src_boxes], [tt(b) for b in dst_boxes]
        for a, b in zip(slist, dlist):
            _check_boxes3d(a, b)
        odev = slist[0].device
        src_off, dst_off = _frame_offsets(lens=[len(b) for b in slist]), _frame_offsets(lens=[len(b) for b in dlist])
        b1 = _dist3d_input(torch.cat([b.to(torch.float32) for b in slist]))   # one copy to the device per box set
        b2 = _dist3d_input(torch.cat([b.to(torch.float32) for b in dlist]))
    else:
        numpy_in = isinstance(src_boxes, np.ndarray)
        if numpy_in:
            assert isinstance(dst_boxes, np.ndarray), "Input should be both numpy tensor or pytorch tensor!"
            src_boxes, dst_boxes = torch.from_numpy(src_boxes), torch.from_numpy(dst_boxes)
        if src_offsets is None or dst_offsets is None:
            raise ValueError("packed boxes need the frame offsets")
        _check_boxes3d(src_boxes, dst_boxes)
        odev = src_boxes.device
        src_off, dst_off = _frame_offsets(src_offsets), _frame_offsets(dst_offsets)
        b1, b2 = _dist3d_input(src_boxes), _dist3d_input(dst_boxes)
    if src_off.numel() != dst_off.numel() or int(src_off[-1]) != len(b1) or int(dst_off[-1]) != len(b2):
        raise ValueError("Numbers of boxes and frame offsets are inconsistent!")
    if metric.lower() not in ("riou", "iou"):
        raise ValueError("Unrecognized distance metric!")
    nframes = src_off.numel() - 1
    dist_off = _block_offsets(src_off, dst_off)
    dist = torch.empty(int(dist_off[-1]), dtype=torch.float32, device=b1.device)
    if dist.numel():
        n_f, m_f = src_off[1:] - src_off[:-1], dst_off[1:] - dst_off[:-1]
        offs = torch.cat([src_off, dst_off, dist_off]).to(b1.device, non_blocking=True)   # one copy of the three offset arrays
        od1, od2, odd = offs[:nframes + 1], offs[nframes + 1:2 * nframes + 2], offs[2 * nframes + 2:]
        ws = _c.workspace(_c.iou3d_distance_batch_workspace_bytes(len(b1), len(b2), nframes), b1.device)
        with torch.cuda.device(b1.device):
            st = _c.iou3d_distance_batch(_c.ptr(b1), len(b1), _c.ptr(od1), _c.ptr(b2), len(b2), _c.ptr(od2), nframes, int(n_f.max()), int(m_f.max()),
                                         1 if metric.lower() == "riou" else 0, _c.ptr(odd), _c.ptr(dist), _c.ptr(ws), ws.numel(), _c.stream_ptr())
        _c.check(st, "box3d_iou_distance_batch")
    if odev.type != "cuda" or numpy_in:
        dist = dist.cpu()
    if numpy_in:
        dist, dist_off = dist.numpy(), dist_off.numpy()
    if not as_list:
        return dist, dist_off
    return [dist[int(dist_off[f]):int(dist_off[f + 1])].reshape(int(src_off[f + 1] - src_off[f]), int(dst_off[f + 1] - dst_off[f])) for f in range(nframes)]


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
    as_list = src_offsets is None and dst_offsets is None
    if as_list:
        frames = list(distance)
        if not len(frames) == len(src_scores) == len(src_tags) == len(dst_tags):
            raise ValueError("distance, scores and tags should hold the same number of frames")
        if not frames:
            return []
        numpy_in = isinstance(frames[0], np.ndarray)
        dl = [_as_tensor(d, torch.float32) for d in frames]
        if any(d.dim() != 2 for d in dl):
            raise ValueError("distance should be an NxM matrix")
        odev = dl[0].device
        src_off, dst_off = _frame_offsets(lens=[d.shape[0] for d in dl]), _frame_offsets(lens=[d.shape[1] for d in dl])
        dist_off = _block_offsets(src_off, dst_off)
        d = _c.to_device(torch.cat([x.reshape(-1) for x in dl]))
        cat = lambda xs, dt: torch.cat([_as_tensor(x, dt).reshape(-1) for x in xs])  # noqa: E731
        scores, st, dt_ = cat(src_scores, torch.float64), cat(src_tags, torch.int32), cat(dst_tags, torch.int32)
    else:
        if src_offsets is None or dst_offsets is None:
            raise ValueError("packed distances need the frame offsets")
        d, given = distance
        numpy_in = isinstance(d, np.ndarray)
        d = _as_tensor(d, torch.float32)
        odev = d.device
        d = _c.to_device(d).reshape(-1)
        src_off, dst_off = _frame_offsets(src_offsets), _frame_offsets(dst_offsets)
        if src_off.numel() != dst_off.numel():
            raise ValueError("Numbers of frames in the offsets are inconsistent!")
        dist_off = _block_offsets(src_off, dst_off)
        if not torch.equal(_frame_offsets(given), dist_off) or int(dist_off[-1]) != d.numel():
            raise ValueError("distance blocks do not match the frame offsets")
        scores, st, dt_ = _as_tensor(src_scores, torch.float64).reshape(-1), _as_tensor(src_tags, torch.int32), _as_tensor(dst_tags, torch.int32)
    dev = d.device
    nframes, total_src, total_dst = src_off.numel() - 1, int(src_off[-1]), int(dst_off[-1])
    if len(scores) != total_src or len(st) != total_src or len(dt_) != total_dst:
        raise ValueError("scores / tags do not match the distance matrix")
    thr = _as_tensor(thresholds, torch.float32)
    single = thr.dim() == 1
    thr = (thr.reshape(1, -1) if single else thr).to(dev).contiguous()
    T, ncat = thr.shape
    scores, st, dt_ = scores.to(dev).contiguous(), st.to(dev).contiguous(), dt_.to(dev).contiguous()
    n_f, m_f = src_off[1:] - src_off[:-1], dst_off[1:] - dst_off[:-1]
    max_dst = int(m_f.max()) if nframes else 0
    sa = torch.full((T, total_src), -1, dtype=torch.int32, device=dev)
    da = torch.full((T, total_dst), -1, dtype=torch.int32, device=dev)
    if max_dst > 4096:   # the kernel's taken bitmask holds 4096 destinations
        for f in range(nframes):
            s0, s1, d0, d1 = int(src_off[f]), int(src_off[f + 1]), int(dst_off[f]), int(dst_off[f + 1])
            sa[:, s0:s1], da[:, d0:d1] = match_greedy(d[int(dist_off[f]):int(dist_off[f + 1])].view(s1 - s0, d1 - d0), scores[s0:s1], st[s0:s1],
                                                      dt_[d0:d1], thr)
    elif T and d.numel():
        offs = torch.cat([src_off, dst_off, dist_off]).to(dev, non_blocking=True)   # one copy of the three offset arrays
        os_, od_, odd = offs[:nframes + 1], offs[nframes + 1:2 * nframes + 2], offs[2 * nframes + 2:]
        order = _frame_score_order(scores, os_, nframes)
        with torch.cuda.device(dev):
            stt = _c.match_greedy_batch(_c.ptr(d), _c.ptr(odd), _c.ptr(os_), _c.ptr(od_), nframes, max_dst, _c.ptr(order), _c.ptr(st), _c.ptr(dt_),
                                        _c.ptr(thr), T, ncat, _c.ptr(sa), _c.ptr(da), _c.stream_ptr())
        _c.check(stt, "match_greedy_batch")
    if odev.type != "cuda" or numpy_in:
        sa, da = sa.cpu(), da.cpu()
    if numpy_in:
        sa, da = sa.numpy(), da.numpy()
    if not as_list:
        return (sa[0], da[0]) if single else (sa, da)
    out = []
    for f in range(nframes):
        a, b = sa[:, int(src_off[f]):int(src_off[f + 1])], da[:, int(dst_off[f]):int(dst_off[f + 1])]
        out.append((a[0], b[0]) if single else (a, b))
    return out
