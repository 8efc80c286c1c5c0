"""The periodic test pass of the reference trainer (``train_air_pr.py:314-334``): run the TEST model (z_pres rounded,
``air_number_bbox_location.py:634-635``) on a labelled batch and score the inferred boxes with the detection metrics
(``air/evaluation_detection.py``), everything on the device."""
from __future__ import annotations

import torch

from .. import detection


def _per_image(model, batch, noise, any_reduce, metrics):
    out = model(torch.clamp(batch["images"], 0.0, 1.0), noise=noise, any_reduce=any_reduce, train=False)
    cs = model.cfg.canvas_size
    # the loop may have stopped early: only the executed steps exist (inf_num never exceeds them)
    return out, metrics(batch["pos"], batch["size"], batch["num"], out["rec_shifts"], out["rec_scales"], out["rec_num_digits"], cs)


@torch.no_grad()
def evaluate_detection(model, batch, noise=None):
    """``batch``: a dict from ``DeviceMultiObjectDataset.batch`` (``images``, ``pos``, ``size``, ``num``).  Returns the five
    batch means the reference logs -- precision[11], recall[11], gt IoU, detection IoU, global IoU (:326-334) -- as
    float64 tensors, plus the count accuracy (:1073-1077)."""
    out, (p, r, g, d, m) = _per_image(model, batch, noise, None, detection.detection_metrics)
    accuracy = (out["rec_num_digits"] == batch["num"]).double().mean()
    return dict(precision=p.mean(0), recall=r.mean(0), gt_max_iou=g.mean(), detected_max_iou=d.mean(), global_iou=m.mean(),
                accuracy=accuracy, steps=out["steps"])


SUM_FIELDS = ("precision", "recall", "gt_max_iou", "detected_max_iou", "global_iou", "correct", "images")


@torch.no_grad()
def evaluate_detection_sums(model, batch, noise=None, any_reduce=None, metrics=None):
    """The sum form of ``evaluate_detection`` for a test set sharded over ranks: one float64 vector ``[27]`` of per-image
    SUMS -- precision[11], recall[11], gt IoU, detection IoU, global IoU, correct counts, image count (``SUM_FIELDS``).  Summed
    over the shards (one all-reduce), ``sums_to_means`` turns it into the means ``evaluate_detection`` reports for the whole
    set.  ``any_reduce``: the model's loop condition across ranks (every rank then issues the same collectives);
    ``metrics``: ``detection.detection_metrics`` or a stand-in with its signature and per-image results."""
    out, (p, r, g, d, m) = _per_image(model, batch, noise, any_reduce, metrics or detection.detection_metrics)
    correct = (out["rec_num_digits"] == batch["num"].to(out["rec_num_digits"].device)).double().sum()
    dev = p.device
    return torch.cat([p.sum(0), r.sum(0), torch.stack([g.sum(), d.sum(), m.sum(), correct.to(dev),
                                                         torch.tensor(float(p.shape[0]), dtype=torch.float64, device=dev)])])


def sums_to_means(sums):
    """``evaluate_detection_sums`` vector (summed over shards) -> dict of the means and the count accuracy"""
    n = sums[-1]
    return dict(precision=sums[0:11] / n, recall=sums[11:22] / n, gt_max_iou=sums[22] / n, detected_max_iou=sums[23] / n,
                global_iou=sums[24] / n, accuracy=sums[25] / n, images=n)
