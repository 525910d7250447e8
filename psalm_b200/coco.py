"""COCO outputs of eval_seg's results, encoded on the device.

The reference's evaluators copy the dense fp32 `instances.pred_masks` [K, H, W] to the host and run
`pycocotools.mask.encode` on every mask: detectron2's `instances_to_coco_json` behind `COCOEvaluator.process`
(psalm/eval/instance_segmentation.py:128,150) and the region script (psalm/eval/region_segmentation.py:282-283).  Here the
run-length encoding runs on the GPU (csrc/rle.cu) and only the compressed counts strings cross to the host: a few
kilobytes per mask instead of 4 * H * W bytes.

Results of the CUDA-graph path (`use_cuda_graph=True`) hold views of the lane's static graph buffers: encode them before
the next submission on that lane (INTEGRATION.md section 2).  Both functions run on the current CUDA stream."""
import torch

from . import _lib, kernels


def encode(masks):
    """`pycocotools.mask.encode` on the device.  masks: CUDA tensor [K, H, W] (or [H, W]), contiguous, fp32 / fp16 / bf16 /
    uint8 / bool holding 0 / 1 (non-zero = foreground).  Returns a list of K dicts {"size": [H, W], "counts": bytes}, each
    identical to what pycocotools returns for the same mask (one dict for a 2-D input, as pycocotools does; [] for
    K == 0, without a launch)."""
    if not isinstance(masks, torch.Tensor):
        raise TypeError("coco.encode: expected a torch.Tensor, got %s" % type(masks).__name__)
    if masks.dim() == 2:
        return encode(masks.unsqueeze(0))[0]
    if masks.dim() != 3:
        raise _lib.PsalmKernelError("coco.encode: expected masks [K, H, W] or [H, W], got %s" % (tuple(masks.shape),))
    kernels._chk(masks, "coco.encode.masks")
    K, H, W = masks.shape
    if K == 0:
        return []
    _, _, strings, offsets = kernels.mask_rle(masks)
    payload = strings.cpu().numpy().tobytes()
    o = offsets.tolist()
    return [{"size": [H, W], "counts": payload[o[k]:o[k + 1]]} for k in range(K)]


def instances_to_coco_json(instances, img_id):
    """detectron2.evaluation.coco_evaluation.instances_to_coco_json for eval_seg's `instances` (instance task): one record
    per prediction with image_id, category_id (`pred_classes`), bbox (`pred_boxes` XYXY -> XYWH), score and segmentation
    (RLE, counts as str).  The masks are encoded on the device; only the RLE strings and the K scores, classes and boxes
    cross to the host."""
    n = len(instances)
    if n == 0:
        return []
    boxes = instances.pred_boxes.tensor.detach().to("cpu", torch.float32).clone()
    boxes[:, 2:] -= boxes[:, :2]                       # BoxMode.XYXY_ABS -> BoxMode.XYWH_ABS
    boxes = boxes.tolist()
    scores = instances.scores.tolist()
    classes = instances.pred_classes.tolist()
    rles = encode(instances.pred_masks)
    for rle in rles:
        rle["counts"] = rle["counts"].decode("utf-8")
    return [{"image_id": img_id, "category_id": classes[k], "bbox": boxes[k], "score": scores[k], "segmentation": rles[k]}
            for k in range(n)]
