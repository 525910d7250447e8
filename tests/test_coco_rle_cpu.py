"""COCO RLE without a GPU: the numpy oracle (oracle/coco_rle.py, maskApi.c restated) against hand-derived vectors,
its round trip, pycocotools itself when installed, and the record layout of coco.instances_to_coco_json."""
import numpy as np
import pytest
import torch

from oracle import coco_rle as R

# (mask rows, counts, string): derived by hand from maskApi.c's rleEncode / rleToString
VECTORS = [
    ([[0, 1], [1, 1]], [1, 3], b"13"),
    (np.ones((3, 3)), [0, 9], b"09"),
    (np.zeros((4, 4)), [16], b"`0"),                    # 16 has bit 4 set: a second group carries the sign
    ([[1]], [0, 1], b"01"),
    ([[1, 0, 1], [0, 1, 0]], [0, 1, 2, 2, 1], b"0121O"),  # last delta is -1
    (np.add.outer(np.arange(4), np.arange(4)) % 2, [1, 1, 1, 2, 1, 1, 2, 1, 1, 2, 1, 1, 1], b"11110O10O10O0"),
]


@pytest.mark.parametrize("mask,counts,string", VECTORS, ids=["2x2", "3x3_ones", "4x4_zeros", "1x1_one", "2x3", "4x4_checker"])
def test_oracle_matches_hand_derived_vectors(mask, counts, string):
    m = np.asarray(mask, dtype=np.uint8)
    c = R.rle_encode(m)
    assert c.dtype == np.uint32 and c.tolist() == counts
    assert R.rle_to_string(c) == string
    assert R.rle_fr_string(string).tolist() == counts
    assert np.array_equal(R.rle_decode(c, *m.shape), m)
    assert R.encode(m) == {"size": list(m.shape), "counts": string}


def test_oracle_string_of_counts_with_a_negative_delta():
    assert R.rle_to_string([1, 5, 1, 2]) == b"151M"       # 2 - 5 = -3
    assert R.rle_fr_string(b"151M").tolist() == [1, 5, 1, 2]


def test_oracle_multi_group_values_round_trip():
    counts = [0, 15, 16, 31, 32, 1023, 1024, 1, 70000, 3, 2 ** 31 - 1, 5, 2 ** 32 - 1]
    s = R.rle_to_string(counts)
    assert R.rle_fr_string(s).tolist() == counts


@pytest.mark.parametrize("seed", range(6))
def test_oracle_round_trip_random_masks(seed):
    rng = np.random.default_rng(seed)
    H, W = rng.integers(1, 60, size=2)
    m = (rng.random((H, W)) < rng.choice([0.02, 0.5, 0.95])).astype(np.uint8)
    c = R.rle_encode(m)
    assert int(c.astype(np.int64).sum()) == H * W
    assert np.all(c[1:] > 0)                               # only the first run may be empty
    assert np.array_equal(R.decode(R.encode(m)), m)


def test_oracle_matches_pycocotools():
    mask_util = pytest.importorskip("pycocotools.mask")
    rng = np.random.default_rng(7)
    for _ in range(20):
        H, W = rng.integers(1, 80, size=2)
        m = (rng.random((H, W)) < rng.uniform(0.01, 0.99)).astype(np.uint8)
        ref = mask_util.encode(np.asfortranarray(m))
        assert R.encode(m) == {"size": [int(v) for v in ref["size"]], "counts": ref["counts"]}


def test_instances_to_coco_json_record_layout(monkeypatch):
    """detectron2's record layout, with the device encoder replaced by the oracle."""
    from psalm_b200 import coco
    from psalm_b200.structures import Boxes, Instances
    monkeypatch.setattr(coco, "encode", lambda masks: [R.encode(m) for m in masks.numpy()])
    masks = torch.zeros(3, 4, 5)
    masks[0, 1:3, 2:4] = 1
    masks[2] = 1
    inst = Instances((4, 5))
    inst.pred_masks = masks
    inst.pred_boxes = Boxes(torch.tensor([[0.0, 0.0, 0.0, 0.0], [1.0, 2.0, 4.0, 6.0], [0.5, 0.5, 1.5, 3.5]]))
    inst.scores = torch.tensor([0.9, 0.25, 0.5])
    inst.pred_classes = torch.tensor([3, 0, 79])
    recs = coco.instances_to_coco_json(inst, 42)
    assert len(recs) == 3
    for k, r in enumerate(recs):
        assert list(r) == ["image_id", "category_id", "bbox", "score", "segmentation"]
        assert r["image_id"] == 42 and isinstance(r["category_id"], int) and isinstance(r["score"], float)
        assert r["segmentation"]["size"] == [4, 5] and isinstance(r["segmentation"]["counts"], str)
        assert np.array_equal(R.decode(r["segmentation"]), masks[k].numpy().astype(np.uint8))
    assert [r["category_id"] for r in recs] == [3, 0, 79]
    assert recs[1]["bbox"] == [1.0, 2.0, 3.0, 4.0] and recs[2]["bbox"] == [0.5, 0.5, 1.0, 3.0]
    assert recs[0]["score"] == pytest.approx(0.9) and recs[2]["segmentation"]["counts"] == "0d0"
    empty = Instances((4, 5))
    empty.pred_masks = torch.zeros(0, 4, 5)
    assert coco.instances_to_coco_json(empty, 1) == []


def test_encode_rejects_cpu_and_bad_rank():
    from psalm_b200 import _lib, coco
    with pytest.raises(_lib.PsalmKernelError, match="CUDA"):
        coco.encode(torch.zeros(2, 4, 4))
    with pytest.raises(_lib.PsalmKernelError, match="K, H, W"):
        coco.encode(torch.zeros(1, 2, 4, 4))
