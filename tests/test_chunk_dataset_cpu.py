"""SURVEY 8(f) row 2 / 8(a) row b2 on the CPU box: the native bag assignment + chunk dataset against (i) the running CPython's set
semantics (the order the reference's greedy loop depends on) and (ii) what the reference's own MatchingMultiviewData class produced
on synthetic COLMAP models (stored under tests/golden by tests/golden/make_golden.py)."""
import ctypes
import os
import random

import numpy as np
import pytest
import torch

from detectorfreesfm_b200 import _lib
from tests import util

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "chunk_dataset_small.pt")
CASES_GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "chunk_dataset_cases.pt")


def _pyset(lib, op, a, b):
    a, b = np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64)
    out = np.zeros(len(a) + len(b) + 1, dtype=np.int64)
    n = ctypes.c_int64(0)
    p = lambda x: x.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    _lib.check(lib.dfsfm_debug_pyset(op, p(a), len(a), p(b), len(b), p(out), ctypes.byref(n)))
    return out[:n.value].tolist()


def test_pyset_workalike_matches_running_cpython(lib):
    """list(set(a)), a - b, a & b, |=, -=, set(set(a)) in CPython's iteration order, over table sizes 8 .. 2048 with collisions"""
    rnd = random.Random(0)
    for _ in range(4000):
        hi = rnd.choice([6, 20, 60, 300, 3000, 100000])
        a = [rnd.randrange(hi) for _ in range(rnd.choice([0, 1, 2, 3, 5, 8, 13, 21, 40, 90, 200]))]
        b = [rnd.choice(a) if a and rnd.random() < 0.5 else rnd.randrange(hi) for _ in range(rnd.choice([0, 1, 2, 3, 5, 8, 13, 30, 100]))]
        sa, sb = set(a), set(b)
        s3 = set(a); s3 |= set(b)
        s4 = set(a); s4 -= set(b)
        want = [list(sa), list(sa - sb), list(sa & sb), list(s3), list(s4), list(set(sa))]
        for op in range(6):
            assert _pyset(lib, op, a, b) == want[op], (op, a, b)


def _as_lists(bags):
    return [{"bag_image_ids": [int(x) for x in b["bag_image_ids"]], "track_ids": [int(x) for x in b["track_ids"]],
             "track_corresponding_imgs": [[int(r), [int(x) for x in q]] for r, q in b["track_corresponding_imgs"]]} for b in bags]


def _compare_items(a, b):
    assert set(a.keys()) == set(b.keys())
    for k in a:
        if k == "images":
            assert len(a[k]) == len(b[k]) and all(torch.equal(x, y) for x, y in zip(a[k], b[k]))
        elif k in ("scales_relative", "view_point_vector"):
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape
            assert torch.allclose(a[k], b[k], rtol=1e-9, atol=1e-9), k      # vectorised float64 geometry: same values up to summation order
        else:
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k


CASES = [dict(n_images=6, n_points=60, max_obs=5, seed=1), dict(n_images=12, n_points=400, max_obs=9, seed=2),
         dict(n_images=30, n_points=900, max_obs=25, seed=3, dup_frac=0.1), dict(n_images=40, n_points=1500, max_obs=12, seed=4, first_image_id=900)]


def _case_args(case):
    """-> (dataset, cfg, worker_split_idxs) of CASES[case]"""
    ds = util.SynthColmapDataset(**CASES[case])
    cfg = {"max_track_length": 16, "chunk": 50 if case != 1 else 2000}
    split = None if case != 3 else list(range(0, len(ds.colmap_3ds), 2))[::-1]      # a worker's share, in its own order
    return ds, cfg, split


def _flat_bags(bags):
    """the bags as one int64 sequence: per bag its image ids, track ids and (reference image, query images) per track, each list
    preceded by its length"""
    flat = []
    for b in _as_lists(bags):
        flat += [len(b["bag_image_ids"])] + b["bag_image_ids"] + [len(b["track_ids"])] + b["track_ids"]
        for ref_img, q in b["track_corresponding_imgs"]:
            flat += [ref_img, len(q)] + q
    return torch.tensor(flat, dtype=torch.int64)


@pytest.mark.parametrize("case", range(len(CASES)))
def test_bags_and_chunks_match_reference_class(case):
    """bags and every chunk dict vs the reference class's, stored as checksums (tests/golden/chunk_dataset_cases.pt): equal shapes,
    dtypes and values up to float64 summation order, the float64 geometry within rtol = atol = 1e-9"""
    from detectorfreesfm_b200.chunk_dataset import B200MatchingMultiviewData
    from tests.golden.make_golden import checksum_close
    g = torch.load(CASES_GOLDEN, weights_only=False)["cases"][case]
    assert g["case"] == CASES[case]
    ds, cfg, split = _case_args(case)
    ours = B200MatchingMultiviewData(ds, cfg, worker_split_idxs=split)
    assert checksum_close(_flat_bags(ours.image_bags), g["bags"])
    assert len(ours) == len(g["items"]) and (len(ours) > 1 or case == 1)
    for i, want in enumerate(g["items"]):
        item = ours[i]
        assert set(item.keys()) == set(want.keys())
        assert len(item.pop("images")) == want["images"]
        for k, v in item.items():
            assert checksum_close(v, want[k], 1e-9 if k in ("scales_relative", "view_point_vector") else 1e-12), (i, k)
    # every query node of every assigned track lands in exactly one chunk
    total = sum(int(ours[i]["track_valid_mask"].sum()) for i in range(len(ours)))
    want = sum(len(set(ds.colmap_3ds[t].image_ids.tolist()) - {int(ours.point3d_assignment[t][0])}) for t in ours.point3d_assignment)
    assert total == want


def test_chunk_dataset_vs_golden():
    """the reference class's own output (generated in the build container by tests/golden/make_golden.py) for one synthetic model"""
    from detectorfreesfm_b200.chunk_dataset import B200MatchingMultiviewData
    g = torch.load(GOLDEN)
    ds = util.SynthColmapDataset(**g["case"])
    ours = B200MatchingMultiviewData(ds, g["cfg"])
    assert _as_lists(ours.image_bags) == g["bags"]
    for i, item in enumerate(g["items"]):
        got = ours[i]
        assert len(got.pop("images")) == len(g["bags"][i]["bag_image_ids"])
        _compare_items(got, item)


def _writeback_case(seed):
    import copy
    import types
    rng = np.random.default_rng(seed)
    ims = {}
    for cid in (3, 7, 11):
        n = 40
        ims[cid] = types.SimpleNamespace(point3D_ids=rng.integers(-1, 12, n).astype(np.int64), xys=rng.normal(0, 100, (n, 2)))
    results = [np.stack([np.r_[rng.normal(0, 50, 2), cid, rng.integers(0, 40)] for cid in rng.choice([3, 7, 11], 30)]) for _ in range(4)]
    return ims, copy.deepcopy(ims), results


def test_colmap_writeback_matches_the_reference_loop():
    """refine_stage.update_refined_kpts_to_colmap_multiview (vectorised, grouped by image) vs the reference's row-by-row loop
    (coarse_sfm_refinement_dataset.py:333-341, restated here): duplicates of a 3-D point in an image all move, later rows win."""
    from detectorfreesfm_b200 import refine_stage as rs
    for seed in range(3):
        a, b, results = _writeback_case(seed)
        for bag in results:                                    # the reference loop
            for row in bag:
                loc, image_id, idx = row[:2], int(row[2]), int(row[3])
                pid = a[image_id].point3D_ids[idx]
                dup = np.concatenate(np.where(a[image_id].point3D_ids == pid), axis=0)
                a[image_id].xys[dup, :] = loc + 0.5
        rs.update_refined_kpts_to_colmap_multiview(b, results)
        assert all(np.array_equal(a[c].xys, b[c].xys) for c in a)


def test_colmap_writeback_matches_the_reference_method():
    """vs the key points CoarseColmapDataset.update_refined_kpts_to_colmap_multiview wrote (tests/golden/chunk_dataset_cases.pt)"""
    from detectorfreesfm_b200 import refine_stage as rs
    want = torch.load(CASES_GOLDEN, weights_only=False)["writeback"]
    _, b, results = _writeback_case(5)
    rs.update_refined_kpts_to_colmap_multiview(b, results)
    assert set(want) == set(b) and all(np.array_equal(want[c], b[c].xys) for c in b)
