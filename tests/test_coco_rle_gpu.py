"""COCO RLE on the device (csrc/rle.cu through kernels.mask_rle / coco.encode) against the numpy restatement of
pycocotools' maskApi.c (oracle/coco_rle.py), byte for byte: structured and random masks, edge shapes, every accepted dtype,
the real pred_masks of eval_seg's instance and region results, and the error paths."""
import numpy as np
import pytest
import torch

from oracle import coco_rle as R
from psalm_b200 import _lib, coco, kernels, synth
from psalm_b200.layout import PhiConfig, PsalmConfig

pytestmark = pytest.mark.gpu
SMALL = PsalmConfig(phi=PhiConfig(hidden=256, layers=2, heads=4, inter=1024))
SHAPES = [(1, 37), (41, 1), (31, 33), (480, 640), (1333, 800), (1024, 1024)]


def _structured(H, W):
    """empty, full, a single pixel at each corner, vertical / horizontal stripes, checkerboard."""
    y, x = np.mgrid[:H, :W]
    out = [np.zeros((H, W)), np.ones((H, W))]
    for cy, cx in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)):
        m = np.zeros((H, W))
        m[cy, cx] = 1
        out.append(m)
    first = np.zeros((H, W))
    first.flat[0] = 1
    first[min(1, H - 1):, :] = 1                        # first pixel set, then a long run
    out += [first, (x // 3) % 2, (y // 3) % 2, (y + x) % 2]
    return np.stack(out).astype(np.uint8)


def _blobs(K, H, W, seed):
    """smooth masks: thresholded sums of a few Gaussians (long runs: multi-character counts, negative deltas)."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[:H, :W].astype(np.float32)
    out = np.zeros((K, H, W), np.uint8)
    for k in range(K):
        f = np.zeros((H, W), np.float32)
        for _ in range(rng.integers(1, 5)):
            cy, cx = rng.uniform(0, H), rng.uniform(0, W)
            s = rng.uniform(0.03, 0.25) * max(H, W)
            f += np.exp(-((y - cy) ** 2 + (x - cx) ** 2) / (2 * s * s))
        out[k] = f > rng.uniform(0.3, 0.9)
    return out


def _check(masks_u8, dtype=torch.float32):
    """coco.encode of the masks in `dtype` == the oracle's dicts, byte for byte; the counts too."""
    t = torch.from_numpy(masks_u8).to("cuda", dtype)
    got = coco.encode(t)
    assert len(got) == masks_u8.shape[0]
    counts, run_off, _, _ = kernels.mask_rle(t)
    counts, run_off = counts.cpu().numpy(), run_off.cpu().numpy()
    for k, m in enumerate(masks_u8):
        c = R.rle_encode(m)
        assert np.array_equal(counts[run_off[k]:run_off[k + 1]], c), "counts of mask %d" % k
        ref = {"size": list(m.shape), "counts": R.rle_to_string(c)}
        assert got[k] == ref, "mask %d: %r... != %r..." % (k, got[k]["counts"][:40], ref["counts"][:40])


@pytest.mark.parametrize("H,W", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_structured_masks(H, W):
    _check(_structured(H, W))


@pytest.mark.parametrize("density", [0.5, 0.02])
@pytest.mark.parametrize("H,W", SHAPES, ids=["%dx%d" % s for s in SHAPES])
def test_random_masks(H, W, density):
    rng = np.random.default_rng(H * 7 + W)
    _check((rng.random((2, H, W)) < density).astype(np.uint8))


def test_long_runs_and_negative_deltas():
    m = _blobs(6, 1024, 1024, seed=3)
    cs = [R.rle_encode(x).astype(np.int64) for x in m]
    assert max(int(c.max()) for c in cs) >= 1 << 15                       # several 5-bit groups
    assert any((c[3:] - c[1:-2] < 0).any() for c in cs if c.size > 3)     # negative deltas
    _check(m)


@pytest.mark.parametrize("H,W", [(480, 640), (1024, 1024)])
def test_k100(H, W):
    rng = np.random.default_rng(5)
    m = _blobs(100, H, W, seed=H)
    m[::10] = (rng.random((10, H, W)) < 0.02)                              # every tenth mask sparse noise
    _check(m)


def test_k1():
    _check(_blobs(1, 1333, 800, seed=1))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.uint8, torch.bool],
                         ids=["f32", "f16", "bf16", "u8", "bool"])
def test_every_accepted_dtype(dtype):
    rng = np.random.default_rng(11)
    _check(np.concatenate([(rng.random((2, 31, 33)) < 0.4), _structured(31, 33)]).astype(np.uint8), dtype)
    _check(_blobs(3, 200, 300, seed=2), dtype)


def test_two_dimensional_input_and_empty_batch():
    m = _blobs(1, 61, 47, seed=4)[0]
    assert coco.encode(torch.from_numpy(m).cuda().float()) == R.encode(m)
    n = kernels.launches()
    assert coco.encode(torch.zeros(0, 8, 8, device="cuda")) == []
    assert kernels.launches() == n


def test_non_default_stream():
    m = _blobs(4, 256, 192, seed=6)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.from_numpy(m).to("cuda", torch.float32, non_blocking=True)
        t = t * 1.0                                                       # produced on the side stream
        got = coco.encode(t)
    assert got == [R.encode(x) for x in m]


def test_errors():
    with pytest.raises(_lib.PsalmKernelError, match="CUDA"):
        coco.encode(torch.zeros(2, 4, 4))
    with pytest.raises(_lib.PsalmKernelError, match="contiguous"):
        coco.encode(torch.zeros(2, 4, 6, device="cuda")[:, :, ::2])
    with pytest.raises(_lib.PsalmKernelError, match="K, H, W"):
        coco.encode(torch.zeros(1, 2, 4, 4, device="cuda"))
    with pytest.raises(_lib.PsalmKernelError, match="dtype"):
        coco.encode(torch.zeros(2, 4, 4, dtype=torch.int32, device="cuda"))
    with pytest.raises(_lib.PsalmKernelError, match="K >= 1"):
        kernels.mask_rle(torch.zeros(0, 4, 4, device="cuda"))
    L = _lib.lib()
    assert L.psalm_mask_rle_sizes(None, None, 0, None, 1, 4, 4, _lib.F32, None) == -1
    assert b"null pointer" in L.psalm_last_error()


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "eager"])
def test_instance_eval_seg_results(graph):
    from psalm_b200.psalm import PSALM
    sd = synth.synth_state_dict(SMALL, seed=31)
    inp = synth.synth_inputs(batch=1, height=192, width=160, task="instance", n_classes=9, seed=32)
    m = PSALM(sd, SMALL, torch.bfloat16, "cuda", "instance", use_cuda_graph=graph)
    kw = {k: inp[k] for k in ("class_name_ids", "cls_indices", "class_name_embedding_indices", "is_thing_list") if k in inp}
    res = m.eval_seg(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"], images=inp["images"],
                     seg_info=inp["seg_info"], **kw)
    inst = res[0]["instances"]
    dense = inst.pred_masks.cpu().numpy()
    assert dense.shape[0] > 0
    recs = coco.instances_to_coco_json(inst, 7)          # before the next submission on the lane
    assert len(recs) == dense.shape[0]
    for r, mk, s, c in zip(recs, dense, inst.scores.tolist(), inst.pred_classes.tolist()):
        ref = R.encode(mk)
        assert r["segmentation"] == {"size": ref["size"], "counts": ref["counts"].decode()}
        assert r["image_id"] == 7 and r["score"] == s and r["category_id"] == c and r["bbox"] == [0.0] * 4


def test_region_eval_seg_results():
    from psalm_b200.psalm import PSALM
    sd = synth.synth_state_dict(SMALL, seed=9)
    inp = synth.synth_inputs(batch=1, height=160, width=160, task="region", seed=10)
    m = PSALM(sd, SMALL, torch.float32, "cuda", "region")
    res = m.eval_seg(input_ids=inp["input_ids"], attention_mask=inp["attention_mask"], images=inp["images"],
                     seg_info=inp["seg_info"])
    pm = res[0]["instances"].pred_masks
    assert coco.encode(pm) == [R.encode(x) for x in pm.cpu().numpy()]
