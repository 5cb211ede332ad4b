"""Generate the committed golden fixtures by running the UNMODIFIED reference modules (imported from the reference tree via
oracle/ref_shims.py) on seeded inputs.  Needs the reference tree (oracle/ref_shims.py: DFSFM_REFERENCE).
Usage:  python tests/golden/make_golden.py [chunk_dataset | reference_outputs | chunk_dataset_cases ...]   (no argument: all)

Fixtures (small, fp32, torch.save):
  roialign_readme.pt   the reference's own known-answer vector (third_party/RoIAlign.pytorch/README.md:42-96)
  loftr_small.pt       LoFTR coarse_only on a 64x80 pair: conf-matrix digest, match ids, mkpts, mconf, feature digests
  multiview_small.pt   MultiviewMatcher on a 24-track chunk: refined points + std
  postprocess_small.pt Match2Kpts + keypoint_worker + update_matches + transform_keypoints on synthetic matches of 5 images
  refine_worker_small.pt  matchWorker (the reference's refinement host loop) on three small chunks with a stand-in matcher
  image_small.pt       read_grayscale (cv2 decode of a PNG written here, PIL-LANCZOS resize, /255) on three synthetic images
  reference_outputs.pt what tests/test_oracle_vs_reference.py compares the oracle with: LoFTR coarse + fine and MultiviewMatcher
                       whole, RoIAlign C++ as a seeded sample + sums, post-processing and read_grayscale images as checksums
  chunk_dataset_cases.pt  MatchingMultiviewData on the four cases of tests/test_chunk_dataset_cpu.py (bags and every chunk dict
                       as checksums) + CoarseColmapDataset.update_refined_kpts_to_colmap_multiview on one write-back case
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_shims  # noqa: E402
from tests import weights  # noqa: E402
from tests import util  # noqa: E402


def digest(t):
    """order-sensitive summary of a big tensor: strided samples + moments"""
    f = t.flatten().double()
    idx = torch.linspace(0, f.numel() - 1, 257).long()
    return {"shape": list(t.shape), "sum": f.sum().item(), "abs_sum": f.abs().sum().item(), "samples": f[idx].float()}


def main():
    assert ref_shims.available(), "needs /root/reference"
    torch.manual_seed(0)
    # ---- RoIAlign README vector, produced by the reference's own C++ op and python wrapper
    ext = ref_shims.build_ref_roialign()
    image = torch.arange(0., 49).view(1, 1, 7, 7).repeat(2, 1, 1, 1)
    image[0] += 10
    boxes = torch.tensor([[1, 0, 5, 4], [0.5, 3.5, 4, 7]])
    x1, y1, x2, y2 = boxes.split(1, 1)
    sw, sh = (x2 - x1) / 4.0, (y2 - y1) / 4.0
    nb = torch.cat(((y1 + sh / 2 - 0.5) / 6.0, (x1 + sw / 2 - 0.5) / 6.0, (y1 + sh / 2 - 0.5) / 6.0 + sh * 3 / 6.0,
                    (x1 + sw / 2 - 0.5) / 6.0 + sw * 3 / 6.0), 1).contiguous()
    crops = torch.zeros(1)
    ext.forward(image, nb, torch.tensor([0, 1], dtype=torch.int32), 0.0, 4, 4, crops)
    readme = torch.tensor([[[[11.0, 12.0, 13.0, 14.0], [18.0, 19.0, 20.0, 21.0], [25.0, 26.0, 27.0, 28.0], [32.0, 33.0, 34.0, 35.0]]],
                           [[[24.5, 25.375, 26.25, 27.125], [30.625, 31.5, 32.375, 33.25], [36.75, 37.625, 38.5, 39.375], [0.0, 0.0, 0.0, 0.0]]]])
    assert torch.allclose(crops, readme, atol=5e-5, rtol=0), "reference op does not reproduce its README vector (4 printed decimals)"
    torch.save({"image": image, "boxes_norm": nb, "box_index": torch.tensor([0, 1], dtype=torch.int32), "crops": crops},
               os.path.join(HERE, "roialign_readme.pt"))
    # ---- LoFTR
    LoFTR, _ = ref_shims.import_loftr()
    sd = weights.loftr_state_dict(0)
    gold = {}
    for name, (thr, temp) in {"default": (0.2, 0.1), "sharp": (0.2, 0.01)}.items():
        m = LoFTR(ref_shims.loftr_config(thr=thr, temperature=temp)).eval()
        m.load_state_dict(sd, strict=True)
        im0, im1 = util.synth_pair(64, 80, seed=1)
        data = {"image0": im0, "image1": im1, "scale0": torch.tensor([[1.5, 1.25]]), "scale1": torch.tensor([[1.0, 2.0]])}
        with torch.no_grad():
            m(data)
        gold[name] = {"thr": thr, "temperature": temp, "conf": digest(data["conf_matrix"]), "conf_max": data["conf_matrix"].max().item(),
                      "i_ids": data["i_ids"], "j_ids": data["j_ids"], "mconf": data["mconf"], "mkpts0_f": data["mkpts0_f"],
                      "mkpts1_f": data["mkpts1_f"]}
    torch.save(gold, os.path.join(HERE, "loftr_small.pt"))
    # ---- MultiviewMatcher
    MM = ref_shims.import_multiview()
    sdm = weights.multiview_state_dict(0)
    gm = {}
    for name, (W, LW) in {"iter0": (15, 7), "iter1": (11, 3)}.items():
        m = MM(config=ref_shims.multiview_config(W, LW), test=True).eval()
        m.load_state_dict(sdm, strict=True)
        data = util.synth_chunk(M=24, n_img=4, max_views=3, seed=4)
        with torch.no_grad():
            m(data)
        gm[name] = {"W": W, "LW": LW, "query_points_refined": data["query_points_refined"],
                    "reference_points_refined": data["reference_points_refined"][-1], "std": data["std"][-1]}
    torch.save(gm, os.path.join(HERE, "multiview_small.pt"))
    # ---- match -> keypoint -> index post-processing (coarse_match.py:203-237), reference functions themselves
    torch.save(postprocess_golden(), os.path.join(HERE, "postprocess_small.pt"))
    torch.save(image_golden(), os.path.join(HERE, "image_small.pt"))
    torch.save({"results": reference_refine_worker()}, os.path.join(HERE, "refine_worker_small.pt"))
    print("golden fixtures written to", HERE)


def reference_refine_worker():
    """the reference's matchWorker itself (multiview_match_worker.py:111-150): chunk dataset replaced by a list, dict_to_cuda by
    the identity, the matcher by tests.util.StandInRefiner -> list of [K,4] arrays"""
    class ListDataset(torch.utils.data.Dataset):
        colmap_images = {i: None for i in range(4)}

        def __init__(self, colmap_dataset, cfgs, worker_split_idxs=None):
            self.chunks = util.worker_chunks()

        def __len__(self):
            return len(self.chunks)

        def __getitem__(self, i):
            return self.chunks[i]

    mod = ref_shims.import_refine_worker(ListDataset)
    mod.DataLoader = lambda ds, num_workers=0, pin_memory=False: torch.utils.data.DataLoader(ds, num_workers=0)
    return mod.matchWorker(None, util.StandInRefiner(), verbose=False)


def reference_read_grayscale(image_u8, resize, df, tmpdir):
    """the reference's read_grayscale on a losslessly written PNG of image_u8 -> (tensor, scales, original_hw)"""
    import cv2
    utils = ref_shims.import_image_utils()
    path = os.path.join(tmpdir, "img.png")
    assert cv2.imwrite(path, image_u8)
    return utils.read_grayscale(path, resize, df=df, ret_scales=True)


def image_golden():
    import tempfile
    from oracle import image_oracle as io
    out = []
    with tempfile.TemporaryDirectory() as d:
        for seed, (h, w, resize, df) in enumerate([(150, 200, (96,), 8), (97, 61, (128,), 8), (64, 80, None, None)]):
            img = util.synth_photo(h, w, seed)
            t, scales, hw = reference_read_grayscale(img, resize, df, d)
            out.append({"image": torch.from_numpy(img), "resize": resize, "df": df, "tensor": t, "scales": scales, "original_hw": hw})
    return out


def reference_postprocess(matches, names, split=" "):
    """the block of src/coarse_match/coarse_match.py:203-237 with the reference's own functions"""
    M2K, keypoint_worker, update_matches, transform_keypoints = ref_shims.import_postprocess()
    all_kpts = M2K(matches, names, name_split=split)
    keypoints = keypoint_worker(all_kpts[0:len(names)], verbose=False)
    updated = update_matches(matches, keypoints, merge=False, verbose=False, pair_name_split=split)
    keypoints = {k: v for k, v in keypoints.items() if isinstance(v, dict)}
    final_kpts, final_scores = transform_keypoints(keypoints, verbose=False)
    return final_kpts, final_scores, updated


def postprocess_golden():
    import itertools
    from oracle import postprocess_oracle as po
    pairs = [p for p in itertools.combinations(range(5), 2) if 4 not in p]  # image 4 never matched
    matches, names = util.synth_matches(5, pairs, [0, 40, 150], seed=7)
    fk, fs, upd = reference_postprocess(matches, names)
    return {"names": names, "matches": matches, "final_keypoints": fk, "final_scores": fs, "updated_matches": upd}


LOFTR_CASE = {"hw": (64, 96), "seed": 3, "scale0": [[1.5, 1.25]], "scale1": [[1.0, 2.0]], "thr": 0.0, "temperature": 0.01}
MULTIVIEW_CASE = {"M": 20, "n_img": 4, "max_views": 3, "seed": 9}
POSTPROCESS_CASES = [(4, 50), (6, 300), (5, [0, 10, 200]), (3, 1)]
IMAGE_CASES = [(150, 200, (96,), 8), (97, 61, (128,), 8), (64, 80, None, None), (300, 200, (64, 48), None)]


def loftr_case_input():
    im0, im1 = util.synth_pair(*LOFTR_CASE["hw"], seed=LOFTR_CASE["seed"])
    return {"image0": im0, "image1": im1, "scale0": torch.tensor(LOFTR_CASE["scale0"]), "scale1": torch.tensor(LOFTR_CASE["scale1"])}


def roialign_case_input():
    """image [2,3,40,56], 64 boxes (normalised, partly outside the image), box indices"""
    g = torch.Generator().manual_seed(0)
    image = torch.rand(2, 3, 40, 56, generator=g)
    nb = torch.rand(64, 4, generator=g) * 1.4 - 0.2
    nb[:, 2:] = nb[:, :2] + torch.rand(64, 2, generator=g) * 0.6
    bi = torch.randint(0, 2, (64,), generator=g, dtype=torch.int32)
    return image, nb.contiguous(), bi


def postprocess_case_input(seed):
    import itertools
    n, m = POSTPROCESS_CASES[seed]
    pairs = list(itertools.combinations(range(n), 2))
    if seed == 2:
        pairs = [p for p in pairs if 4 not in p]    # image 4 never matched
    return util.synth_matches(n, pairs, m, seed=seed)


def sample_of(t, n=4096):
    """a fixed, seeded sample of a tensor too large to store whole: flat indices, their values, float64 sum and abs-sum"""
    f = t.flatten()
    idx = torch.randperm(f.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
    return {"shape": list(t.shape), "idx": idx, "values": f[idx].clone(), "sum": f.double().sum().item(), "abs_sum": f.double().abs().sum().item()}


def reference_outputs():
    """the reference's own outputs on the inputs tests/test_oracle_vs_reference.py gives the oracle"""
    out = {"loftr": {}}
    LoFTR, _ = ref_shims.import_loftr()
    sd = weights.loftr_state_dict(0)
    for fine in (False, True):
        m = LoFTR(ref_shims.loftr_config(thr=LOFTR_CASE["thr"], fine=fine, temperature=LOFTR_CASE["temperature"])).eval()
        m.load_state_dict(sd, strict=True)
        d = loftr_case_input()
        with torch.no_grad():
            m(d)
        out["loftr"][fine] = {k: d[k] for k in ("conf_matrix", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f")}
    MM = ref_shims.import_multiview()
    m = MM(config=ref_shims.multiview_config(15, 7), test=True).eval()
    m.load_state_dict(weights.multiview_state_dict(0), strict=True)
    d = util.synth_chunk(**MULTIVIEW_CASE)
    with torch.no_grad():
        m(d)
    out["multiview"] = {"query_points_refined": d["query_points_refined"], "reference_points_refined": d["reference_points_refined"][-1],
                        "std": d["std"][-1]}
    ext = ref_shims.build_ref_roialign()
    image, boxes, box_index = roialign_case_input()
    crops = torch.zeros(1)
    ext.forward(image, boxes, box_index, 0.0, 35, 35, crops)
    out["roialign"] = sample_of(crops)
    out["postprocess"] = [tuple({k: checksum(a) for k, a in part.items()} for part in reference_postprocess(*postprocess_case_input(seed)))
                          for seed in range(len(POSTPROCESS_CASES))]
    import tempfile
    out["image"] = []
    with tempfile.TemporaryDirectory() as tmp:
        for seed, (h, w, resize, df) in enumerate(IMAGE_CASES):
            t, scales, hw = reference_read_grayscale(util.synth_photo(h, w, seed), resize, df, tmp)
            out["image"].append((checksum(t), scales, hw))
    return out


def checksum(t):
    """order-sensitive checksum of a tensor or numpy array: shape, dtype, float64 sum and position-weighted sum"""
    f = torch.as_tensor(t).flatten().double()
    return {"shape": list(t.shape), "dtype": str(t.dtype), "sum": f.sum().item(),
            "wsum": (f * torch.arange(1, f.numel() + 1, dtype=torch.float64)).sum().item()}


def checksum_close(t, want, rel=1e-12):
    """``t`` against a stored checksum(): same shape and dtype, both sums equal to within rel * (|t_i| + 1) per element -- with the
    default, equal up to float64 summation order"""
    got = checksum(t)
    f = torch.as_tensor(t).flatten().double().abs()
    pos = torch.arange(1, f.numel() + 1, dtype=torch.float64)
    return (got["shape"] == want["shape"] and got["dtype"] == want["dtype"]
            and abs(got["sum"] - want["sum"]) <= rel * (f.sum().item() + f.numel())
            and abs(got["wsum"] - want["wsum"]) <= rel * ((f * pos).sum().item() + pos.sum().item()))


def chunk_dataset_cases():
    """the reference's MatchingMultiviewData on every case of tests/test_chunk_dataset_cpu.py (the bags and every chunk dict as
    checksums: the whole items would be several MB) and its update_refined_kpts_to_colmap_multiview on write-back case 5"""
    import types
    from tests.test_chunk_dataset_cpu import CASES, _case_args, _writeback_case, _flat_bags
    Ref = ref_shims.import_chunk_dataset()
    cases = []
    for case in range(len(CASES)):
        ds, cfg, split = _case_args(case)
        ref = Ref(ds, cfg, worker_split_idxs=split)
        cases.append({"case": CASES[case], "bags": checksum(_flat_bags(ref.image_bags)),
                      "items": [{k: (len(v) if k == "images" else checksum(v)) for k, v in ref[i].items()} for i in range(len(ref))]})
    a, _, results = _writeback_case(5)
    ref_cls = ref_shims.import_colmap_dataset_class()
    ref_cls.update_refined_kpts_to_colmap_multiview(types.SimpleNamespace(colmap_images=a), results)
    return {"cases": cases, "writeback": {c: a[c].xys for c in a}}


def chunk_dataset_golden():
    """the reference's own MatchingMultiviewData (bags + every chunk dict) on one synthetic COLMAP model"""
    Ref = ref_shims.import_chunk_dataset()
    case = dict(n_images=20, n_points=160, max_obs=18, seed=5, dup_frac=0.1)
    cfg = {"max_track_length": 16, "chunk": 40}
    ref = Ref(util.SynthColmapDataset(**case), cfg)
    bags = [{"bag_image_ids": [int(x) for x in b["bag_image_ids"]], "track_ids": [int(x) for x in b["track_ids"]],
             "track_corresponding_imgs": [[int(r), [int(x) for x in q]] for r, q in b["track_corresponding_imgs"]]} for b in ref.image_bags]
    return {"case": case, "cfg": cfg, "bags": bags, "items": [{k: v for k, v in ref[i].items() if k != "images"} for i in range(len(ref))]}   # images: pass-through of ds[...]


PARTS = {"chunk_dataset": (chunk_dataset_golden, "chunk_dataset_small.pt"), "reference_outputs": (reference_outputs, "reference_outputs.pt"),
         "chunk_dataset_cases": (chunk_dataset_cases, "chunk_dataset_cases.pt")}

if __name__ == "__main__":
    if len(sys.argv) == 1:
        main()
    for part in sys.argv[1:] or list(PARTS):
        fn, name = PARTS[part]
        torch.save(fn(), os.path.join(HERE, name))
