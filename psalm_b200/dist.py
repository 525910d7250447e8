"""Multi-GPU plumbing of the hot path: images are independent units (SURVEY.md §8e), so ranks hold full
weight replicas and take disjoint images; there is no collective on the data path.  What crosses NVLink is what
the evaluators consume (what the reference *would* do with detectron2.comm.all_gather,
psalm/eval/segmentation_evaluation/referring_evaluation.py:162-164, but never enables):
  * per step, ONE all_gather of the fixed-size predictions of every image — class_id[Q], score[Q] and the int32
    panoptic id map [H,W] (`pack_predictions` / `gather_predictions`);
  * an all_reduce(SUM) of metric accumulators (confusion matrix, PQ tp/fp/fn/iou) (`reduce_sum`);
  * a MAX reduction of the device-timed step time (`max_over_ranks`).
Backend: NCCL over NVLink on GPUs, gloo in the CPU tests."""
import torch
import torch.distributed as dist


def shard_indices(n_items, rank, world):
    """Round-robin image sharding: rank r takes items i == r (mod world)."""
    return list(range(rank, n_items, world))


def max_over_ranks(values, device):
    """values: list of floats (e.g. elapsed ms) -> element-wise max over ranks."""
    t = torch.tensor(values, dtype=torch.float64, device=device)
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


def compact_record(result, num_queries=100):
    """Fixed-size per-image record [num_queries, 3] fp32: (score, class, mask area) of the instance
    predictions, zero padded — the payload of the final gather."""
    inst = result["instances"]
    rec = torch.zeros(num_queries, 3, dtype=torch.float32, device=inst.scores.device)
    n = min(num_queries, inst.scores.shape[0])
    rec[:n, 0] = inst.scores[:n]
    if inst.has("pred_classes"):
        rec[:n, 1] = inst.pred_classes[:n].float()
    rec[:n, 2] = inst.pred_masks[:n].flatten(1).sum(1)
    return rec


def gather_records(local):
    """local [n_local, Q, 3] -> [world * n_local, Q, 3] in rank order (every rank holds the result)."""
    if not (dist.is_initialized() and dist.get_world_size() > 1):
        return local
    out = [torch.empty_like(local) for _ in range(dist.get_world_size())]
    dist.all_gather(out, local.contiguous())
    return torch.cat(out, 0)


def pack_predictions(results, num_queries=100):
    """Per-image fixed-size payload of the prediction gather (SURVEY.md §8e): meta [n, Q, 2] fp32 = (score, class id)
    of the instance predictions (zero padded, class -1 = empty slot) and the panoptic id map [n, H, W] int32
    (None when the task has no panoptic output)."""
    metas, maps = [], []
    for r in results:
        inst = r.get("instances")
        dev = (inst.scores if inst is not None else r["panoptic_seg"][0]).device
        meta = torch.zeros(num_queries, 2, dtype=torch.float32, device=dev)
        meta[:, 1] = -1.0
        if inst is not None:
            n = min(num_queries, inst.scores.shape[0])
            meta[:n, 0] = inst.scores[:n]
            meta[:n, 1] = inst.pred_classes[:n].float() if inst.has("pred_classes") else 0.0
        metas.append(meta)
        if "panoptic_seg" in r:
            maps.append(r["panoptic_seg"][0])
    return torch.stack(metas), (torch.stack(maps) if maps else None)


def pack_mask_bits(masks):
    """Instance masks [n, H, W] (float 0/1 or bool, as `Instances.pred_masks`) -> bit-packed uint8 [n, H, ceil(W/8)]
    (MSB = leftmost pixel, numpy.packbits order): 1/32 of the bytes of the dense float masks of the reference API, the
    form in which they cross NVLink / PCIe between ranks.  COCO evaluators take the RLE encoded on the device instead
    (`psalm_b200.coco.encode` / `instances_to_coco_json`, a few kilobytes per mask).  Torch ops only: runs on the device
    that holds the masks."""
    n, H, W = masks.shape
    b = masks > 0 if masks.dtype != torch.bool else masks
    pad = (-W) % 8
    if pad:
        b = torch.nn.functional.pad(b, (0, pad))
    w = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], dtype=torch.uint8, device=masks.device)
    return (b.view(n, H, -1, 8).to(torch.uint8) * w).sum(-1, dtype=torch.uint8)


def unpack_mask_bits(bits, W):
    """Inverse of `pack_mask_bits`: uint8 [n, H, ceil(W/8)] -> bool [n, H, W]."""
    w = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], dtype=torch.uint8, device=bits.device)
    return ((bits.unsqueeze(-1) & w) != 0).flatten(-2)[..., :W]


def pack_instance_masks(results, num_queries=100):
    """Bit-packed instance masks of a step for the prediction gather: uint8 [n_images, Q, H, ceil(W/8)] (zero padded to Q
    slots; all images of a step share one output size)."""
    out = []
    for r in results:
        m = r["instances"].pred_masks
        bits = pack_mask_bits(m[:num_queries])
        if bits.shape[0] < num_queries:
            bits = torch.cat([bits, bits.new_zeros((num_queries - bits.shape[0],) + tuple(bits.shape[1:]))], 0)
        out.append(bits)
    return torch.stack(out)


def gather_tensor(t):
    """all_gather of one tensor along dim 0 (rank order); identity without a process group."""
    if t is None or not (dist.is_initialized() and dist.get_world_size() > 1):
        return t
    t = t.contiguous()
    g = torch.empty((dist.get_world_size() * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(g, t)
    return g


def gather_predictions(meta, maps):
    """all_gather of the per-step predictions: ([world*n, Q, 2], [world*n, H, W] or None), rank order."""
    if not (dist.is_initialized() and dist.get_world_size() > 1):
        return meta, maps
    world = dist.get_world_size()
    out = []
    for t in (meta, maps):
        if t is None:
            out.append(None)
            continue
        t = t.contiguous()
        g = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(g, t)
        out.append(g)
    return out[0], out[1]


def reduce_sum(tensors, device):
    """all_reduce(SUM) of metric accumulators (list of tensors, returned on `device`)."""
    outs = []
    for t in tensors:
        t = t.to(device)
        if dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        outs.append(t)
    return outs
