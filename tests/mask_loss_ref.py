"""CPU restatement of the mask term of the generator loss on GT masks (sg2im's ``compute_generator_loss``; the
reference's own source is not in this tree): ``weight * F.binary_cross_entropy(masks_pred, masks_gt)``, the mean over
every element, in whatever dtype ``masks_pred`` has.  torch's arithmetic is the contract of
``canonicalsg2im_b200.model.mask_pred_loss``: per element -(t max(log p, -100) + (1 - t) max(log(1 - p), -100)),
d/dp = weight (p - t) / max((1 - p) p, 1e-12) / n."""
import torch.nn.functional as F


def mask_pred_loss(masks_pred, masks_gt, weight=1.0):
    return weight * F.binary_cross_entropy(masks_pred, masks_gt.to(masks_pred.dtype))
