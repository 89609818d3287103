"""The step right after the seeker (SURVEY.md section 8 f1): reading the per-frame proposal files
back and de-duplicating them with a rotated-BEV NMS, on the device.

Reference: pcdet/datasets/augmentor/pseudo_loader.py
  :29-55   bev_nms_cpu -- greedy class-agnostic NMS in descending score order over the N x N matrix
           of boxes_bev_iou_cpu; returns the kept indices in score order;
  :561-679 PseudoLoader.load_pseudos -- torch.load of `<folder>/<frame_id with . -> _>.pth`
           (a list of length 1 holding pred_boxes / pred_scores / pred_labels, or the bare dict)
           -> (K, 8) [x, y, z, dx, dy, dz, heading, label] + (K,) scores;
  :755     the NMS is applied with PSEUDO_NMS_THRESH (0.1 in the self-training config).

Only the file format and the NMS are mirrored here; the score-EMA filtering of load_pseudos is
state of the self-training loop and stays out of scope (SURVEY.md section 2).
"""
import os

import numpy as np
import torch

from .pcdet_ops import iou3d_nms_utils


def bev_nms(boxes, scores, thresh=0.5):
    """Same contract as the reference's bev_nms_cpu(boxes (N,7), scores (N), thresh): indices of
    the kept boxes in descending score order.  Accepts CPU or CUDA tensors (or numpy arrays) and
    answers in kind; the work is one bitmask kernel + one greedy scan kernel on the GPU.
    Ties in the scores: earlier index first (the reference's argsort leaves them undefined)."""
    is_numpy = isinstance(boxes, np.ndarray)
    b = torch.as_tensor(boxes, dtype=torch.float32)
    s = torch.as_tensor(scores, dtype=torch.float32)
    if b.shape[0] == 0:
        out = torch.zeros(0, dtype=torch.long)
        return out.numpy() if is_numpy else out.to(b.device)
    if not torch.cuda.is_available():
        raise RuntimeError("findnpropagate_b200.pseudo_loader.bev_nms needs a CUDA device (no CPU fallback)")
    dev = b.device if b.is_cuda else torch.device("cuda", torch.cuda.current_device())
    keep, _ = iou3d_nms_utils.nms_gpu(b[:, :7].to(dev).contiguous(), s.to(dev), float(thresh))
    keep = keep.to(b.device)
    return keep.numpy() if is_numpy else keep


def seg_nms_keep(boxes_list, scores_list, thresh, device=None):
    """Per frame, the indices of the rows ``load_pseudos(nms_thresh=thresh)`` keeps, in its order (descending score,
    ties by row), for many frames in one fnp_seg_nms_rotated launch.  boxes_list[f]: (K_f, >= 7), scores_list[f]:
    (K_f,).  ValueError for a frame of more than SEG_NMS_MAX boxes."""
    from . import _lib
    ks = np.array([len(s) for s in scores_list], np.int64)
    if ks.max(initial=0) > _lib.SEG_NMS_MAX:
        raise ValueError("frame %d has %d boxes, the NMS takes at most %d per frame"
                         % (int(np.argmax(ks)), int(ks.max()), _lib.SEG_NMS_MAX))
    n = len(ks)
    start = np.concatenate([[0], np.cumsum(ks)]).astype(np.int32)
    if start[-1] == 0:
        return [np.zeros(0, np.int64) for _ in range(n)]
    boxes = np.ascontiguousarray(np.concatenate([np.asarray(b, np.float32)[:, :7] for b in boxes_list]))
    scores = np.concatenate([np.asarray(s, np.float32) for s in scores_list])
    order = np.lexsort((-scores, np.repeat(np.arange(n), ks))).astype(np.int32)    # stable: ties by row
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    d_boxes, d_order, d_start = (torch.from_numpy(a).to(dev) for a in (boxes, order, start))
    keep = torch.empty(boxes.shape[0], dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib.fnp_seg_nms_rotated(d_boxes.data_ptr(), None, d_order.data_ptr(), None, d_start.data_ptr(),
                                                n, int(ks.max()), float(thresh), keep.data_ptr(),
                                                _lib.current_stream(dev)), "fnp_seg_nms_rotated")
    keep = keep.cpu().numpy().astype(bool)
    return [order[start[f]:start[f + 1]][keep[order[start[f]:start[f + 1]]]] - start[f] for f in range(n)]


def pseudo_path(folder, frame_id):
    return os.path.join(str(folder), "%s.pth" % str(frame_id).replace('.', '_'))


def read_pseudos(path):
    """(boxes (K,7) f32, scores (K,) f32, labels (K,)) of one proposal file -- a list of length 1 holding the dict, or
    the bare dict; pred_boxes may have more than 7 columns -- or None when the file does not exist."""
    if not os.path.exists(path):
        return None
    preds = torch.load(path, map_location='cpu', weights_only=False)
    if isinstance(preds, dict):
        pred = preds
    else:
        assert len(preds) == 1, "preds list should have len == 1, got %d" % len(preds)
        pred = preds[0]
    boxes = pred['pred_boxes'].numpy().astype(np.float32)[:, :7]
    scores = pred['pred_scores'].numpy().astype(np.float32)
    return boxes, scores, pred['pred_labels'].numpy()


def load_pseudos(folder, frame_id, labels=None, nms_thresh=None):
    """(K, 8) float32 [box7, label] and (K,) float32 scores of one frame, as load_pseudos returns
    them with filter_by_score=False; a missing file gives empty arrays (the reference prints and
    does the same).  labels: keep only these class labels (the reference's unknowns_only);
    nms_thresh: apply bev_nms at that threshold (reference: PSEUDO_NMS_THRESH)."""
    got = read_pseudos(pseudo_path(folder, frame_id))
    if got is None:
        return np.zeros((0, 8), np.float32), np.zeros((0,), np.float32)
    boxes, scores, lab = got
    if labels is not None:
        m = np.isin(lab, np.asarray(list(labels)))
        boxes, scores, lab = boxes[m], scores[m], lab[m]
    if nms_thresh is not None and boxes.shape[0] > 1:
        keep = bev_nms(boxes, scores, nms_thresh)
        boxes, scores, lab = boxes[keep], scores[keep], lab[keep]
    out = np.zeros((boxes.shape[0], 8), np.float32)
    out[:, :7] = boxes
    out[:, 7] = lab
    return out, scores
