"""Device COCO RLE (coco.encode / csrc/rle.cu) against the dense `pred_masks.cpu()` copy it replaces.

For K = 100 masks at 1024 x 1024 and at 480 x 640 (H x W), fp32 as eval_seg returns them, and three mask kinds: the real
pred_masks of the random-weight instance model (PsalmConfig(), bf16, synthetic weights and image), smooth synthetic blobs
and the checkerboard (H * W runs per mask, the worst case).  Per case, CUDA events, L2 overwritten before every timed pass:
  sizes_us    the first phase alone (psalm_mask_rle_sizes: the one read of the masks), with its bytes/s against 7.7 TB/s
  encode_us   kernels.mask_rle: all three phases and the two host synchronisations that size the outputs
  payload     the RLE strings' bytes and the time of their device-to-host copy
  coco_us     coco.encode end to end (= encode + payload copy + splitting into dicts)
  dense_us    pred_masks.cpu() of the same masks: a lower bound on the host path (it leaves out pycocotools' work)
Card name and power limit are read in the same run.
usage: python tools/bench_rle.py [--iters 50] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from psalm_b200 import _lib, coco, kernels, synth  # noqa: E402
from psalm_b200.layout import PsalmConfig  # noqa: E402

HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def model_masks(geoms):
    """pred_masks [100, H, W] fp32 of the instance task of the full-size random-weight model (C4 configuration)."""
    from psalm_b200.psalm import PSALM
    cfg = PsalmConfig()
    sd = synth.synth_state_dict(cfg, seed=0, device="cuda")
    m = PSALM(sd, cfg, torch.bfloat16, "cuda", "instance")
    del sd
    out = {}
    for H, W in geoms:
        inp = synth.synth_inputs(batch=1, height=H, width=W, task="instance", n_classes=81, seed=3)
        kw = {k: inp[k] for k in ("class_name_ids", "cls_indices", "class_name_embedding_indices", "is_thing_list")
              if k in inp}
        res = m.eval_seg(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"], images=inp["images"],
                         seg_info=inp["seg_info"], **kw)
        out[(H, W)] = res[0]["instances"].pred_masks.clone()
    del m
    torch.cuda.empty_cache()
    return out


def blobs(K, H, W, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    y = torch.arange(H, device="cuda", dtype=torch.float32).view(1, H, 1)
    x = torch.arange(W, device="cuda", dtype=torch.float32).view(1, 1, W)
    f = torch.zeros(K, H, W, device="cuda")
    for _ in range(3):
        cy = torch.rand(K, 1, 1, device="cuda", generator=g) * H
        cx = torch.rand(K, 1, 1, device="cuda", generator=g) * W
        s = (0.03 + 0.2 * torch.rand(K, 1, 1, device="cuda", generator=g)) * max(H, W)
        f += torch.exp(-((y - cy) ** 2 + (x - cx) ** 2) / (2 * s * s))
    return (f > 0.5).float().contiguous()


def checkerboard(K, H, W):
    y = torch.arange(H, device="cuda").view(H, 1)
    x = torch.arange(W, device="cuda").view(1, W)
    return ((y + x) % 2).float().expand(K, H, W).contiguous()


def events_us(fn, iters, flush):
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return {"median": round(ts[len(ts) // 2], 1), "min": round(ts[0], 1), "n": len(ts)}


def measure(masks, iters, flush):
    K, H, W = masks.shape
    L = _lib.lib()
    ws = torch.empty(L.psalm_mask_rle_workspace_bytes(K, H, W), dtype=torch.uint8, device="cuda")
    run_off = torch.empty(K + 1, dtype=torch.int64, device="cuda")

    def sizes():
        _lib.check(L.psalm_mask_rle_sizes(_lib.ptr(masks), _lib.ptr(ws), ws.numel(), _lib.ptr(run_off), K, H, W, _lib.F32,
                                          _lib.stream_ptr()), "psalm_mask_rle_sizes")

    for _ in range(3):   # warm-up of every shape
        sizes()
        kernels.mask_rle(masks)
        coco.encode(masks)
        masks.cpu()
    torch.cuda.synchronize()
    _, _, strings, _ = kernels.mask_rle(masks)
    runs = int(run_off[K])
    mask_bytes = masks.numel() * masks.element_size()
    r = {"K": K, "H": H, "W": W, "mask_bytes": mask_bytes, "runs": runs, "payload_bytes": strings.numel()}
    r["sizes_us"] = events_us(sizes, iters, flush)
    r["sizes_bytes_per_s"] = round(mask_bytes / (r["sizes_us"]["median"] * 1e-6) / 1e9, 1)   # GB/s
    r["sizes_share_of_hbm_bound"] = round(mask_bytes / HBM_BYTES_PER_S / (r["sizes_us"]["median"] * 1e-6), 3)
    r["encode_us"] = events_us(lambda: kernels.mask_rle(masks), iters, flush)
    r["payload_copy_us"] = events_us(lambda: strings.cpu(), iters, flush)
    r["coco_encode_us"] = events_us(lambda: coco.encode(masks), iters, flush)
    r["dense_copy_us"] = events_us(lambda: masks.cpu(), max(5, iters // 5), flush)
    r["encode_plus_payload_us"] = round(r["encode_us"]["median"] + r["payload_copy_us"]["median"], 1)
    r["dense_over_encode_plus_payload"] = round(r["dense_copy_us"]["median"] / r["encode_plus_payload_us"], 1)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rle needs a GPU"
    geoms = [(1024, 1024), (480, 640)]
    t0 = time.time()
    real = model_masks(geoms)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > the 126 MB L2
    res = {"gpu": gpu_info(), "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S, "cases": []}
    for H, W in geoms:
        for kind, masks in (("model_pred_masks", real[(H, W)]), ("blobs", blobs(100, H, W)),
                            ("checkerboard", checkerboard(100, H, W))):
            r = measure(masks, a.iters, flush)
            r["kind"] = kind
            res["cases"].append(r)
            print(json.dumps(r), flush=True)
            del masks
    res["wall_s"] = round(time.time() - t0, 1)
    print(json.dumps(res["gpu"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
