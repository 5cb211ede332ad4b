"""Pin the oracle restatement against the UNMODIFIED reference: its outputs on the inputs below are stored in
tests/golden/reference_outputs.pt by tests/golden/make_golden.py.  The plugin test imports the reference's own hook modules and
runs only where the reference tree is present (oracle/ref_shims.py: DFSFM_REFERENCE)."""
import os

import pytest
import torch

from tests import util  # noqa: E402
from tests.golden import make_golden as mg

from oracle import ref_shims

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.pt")


@pytest.fixture(scope="module")
def ref():
    return torch.load(GOLDEN, weights_only=False)


def test_loftr_coarse_and_fine_match_reference(ref):
    from oracle import loftr_oracle as lo
    from tests import weights
    sd = weights.loftr_state_dict(0)
    for fine in (False, True):
        d = ref["loftr"][fine]
        out = lo.loftr_forward(mg.loftr_case_input(), sd,
                               {"thr": mg.LOFTR_CASE["thr"], "temperature": mg.LOFTR_CASE["temperature"], "fine_enable": fine}, keep=True)
        assert (d["conf_matrix"] - out["conf_matrix"]).abs().max().item() < 1e-6
        assert torch.equal(d["i_ids"], out["i_ids"]) and torch.equal(d["j_ids"], out["j_ids"])
        assert (d["mconf"] - out["mconf"]).abs().max().item() < 1e-6
        assert (d["mkpts0_f"] - out["mkpts0_f"]).abs().max().item() < 1e-3
        assert (d["mkpts1_f"] - out["mkpts1_f"]).abs().max().item() < 1e-3


def test_multiview_matches_reference(ref):
    from oracle import multiview_oracle as mo
    from tests import weights
    sd = weights.multiview_state_dict(0)
    data = util.synth_chunk(**mg.MULTIVIEW_CASE)
    d2 = ref["multiview"]
    out = mo.multiview_forward(data, sd, 15, 7)
    mask = data["track_valid_mask"]
    assert (d2["query_points_refined"] - out["query_points_refined"]).abs().max().item() < 1e-4
    assert (d2["reference_points_refined"] - out["reference_points_refined"])[mask].abs().max().item() < 1e-3
    assert (d2["std"] - out["std"])[mask].abs().max().item() < 1e-4


def test_c_roialign_matches_reference_cpp(ref):
    """the C restatement vs the reference's crop_and_resize.cpp on 64 boxes of 35x35: a seeded sample of 4096 crop values
    bit for bit, and the sums over all of them"""
    from oracle import build_native
    image, nb, bi = mg.roialign_case_input()
    crops = build_native.roialign_forward(image, nb, bi, 35, 35)
    want, got = ref["roialign"], mg.sample_of(crops)
    assert got["shape"] == want["shape"] and torch.equal(got["idx"], want["idx"]) and torch.equal(got["values"], want["values"])
    assert abs(got["sum"] - want["sum"]) <= 1e-12 * want["abs_sum"] and abs(got["abs_sum"] - want["abs_sum"]) <= 1e-12 * want["abs_sum"]


def test_postprocess_oracle_matches_reference(ref):
    """Match2Kpts / keypoint_worker / update_matches / transform_keypoints themselves (stored as checksums) vs
    oracle/postprocess_oracle.py: equal dtypes, shapes and values, including pairs without matches and an image that never appears."""
    from oracle import postprocess_oracle as po
    for seed, want in enumerate(ref["postprocess"]):
        matches, names = mg.postprocess_case_input(seed)
        ora = po.merge_keypoints(matches, names, " ")
        assert set(want[0]) == set(want[1]) == set(names) and set(want[2]) == set(matches)
        for w, o in zip(want, ora):
            for k in w:
                assert mg.checksum_close(o[k], w[k]), (seed, k)


def test_image_oracle_matches_reference_read_grayscale(ref):
    """the reference's read_grayscale (cv2 decode of a PNG, PIL LANCZOS, /255) vs oracle/image_oracle.py: equal tensors, scales."""
    from oracle import image_oracle as io
    for seed, ((h, w, resize, df), (t, scales, hw)) in enumerate(zip(mg.IMAGE_CASES, ref["image"])):
        img = util.synth_photo(h, w, seed)
        to, so, ho = io.read_grayscale_from_array(img, resize, df=df)
        assert mg.checksum_close(to, t) and torch.equal(scales, so) and torch.equal(hw, ho)


def test_refine_worker_loop_matches_reference_match_worker():
    """Row b1: the reference's matchWorker (its real code, with the chunk dataset replaced by a list and dict_to_cuda by the
    identity; output stored in tests/golden/refine_worker_small.pt) and detectorfreesfm_b200.refine_stage.match_worker give
    identical [K,4] arrays for the same chunks and the same (deterministic stand-in) matcher -- including the fact that
    UpdatedQueryPts never freezes anything in the reference."""
    import numpy as np
    from detectorfreesfm_b200 import refine_stage as rs
    ref = torch.load(os.path.join(os.path.dirname(GOLDEN), "refine_worker_small.pt"), weights_only=False)["results"]
    got = rs.match_worker(torch.utils.data.DataLoader(util.worker_chunks(), num_workers=0), util.StandInRefiner(), range(4),
                          device=torch.device("cpu"))
    assert len(ref) == len(got) == 3
    for a, b in zip(ref, got):
        assert a.shape == b.shape and a.shape[1] == 4 and np.array_equal(a, b)


@pytest.mark.skipif(not ref_shims.available(), reason="needs the reference tree: the test patches its own hook modules")
def test_plugin_install_rebinds_both_hooks_and_builds_b200_models(tmp_path, monkeypatch):
    """plugin.install() behind the reference's own hook modules (imported where they lie, third-party deps stubbed):
    * the HP-1 name 'loftr_b200' builds (DetectorWrapper, B200LoFTR) from the reference's yacs config + a checkpoint file, with
      thr / temp_bug_fix overwritten like coarse_match_worker.py:31-35, and other matcher names still reach the original;
    * the HP-2 builder is rebound in BOTH modules that hold the name (multiview_match.py star-imports it, :7) and applies the
      per-iteration window rescale of multiview_match_worker.py:20-34."""
    import os
    from detectorfreesfm_b200 import B200LoFTR, B200MultiviewMatcher
    from detectorfreesfm_b200 import plugin
    from tests import weights
    cm, cmw, mm, mmw = ref_shims.import_hook_modules()
    orig_coarse, orig_refine = cmw.build_model, mmw.build_model
    assert mm.build_model is orig_refine                      # the star import the advisor pointed at
    plugin.install()
    assert cmw.build_model is not orig_coarse and cm.build_model is cmw.build_model
    assert mmw.build_model is not orig_refine and mm.build_model is mmw.build_model
    assert "loftr_b200" in cm.cfgs["matcher"]["model"]
    # ---- HP-1
    ckpt = tmp_path / "outdoor_ds.ckpt"
    torch.save({"state_dict": {"matcher." + k: v for k, v in weights.loftr_state_dict(0).items()}}, ckpt)
    monkeypatch.chdir(ref_shims.REF)                          # the yacs .py configs use cwd-relative paths, like eval_dataset.py
    args = dict(cm.cfgs["matcher"]["model"])
    args.update({"matcher": "loftr_b200", "type": "coarse_only", "match_thr": 0.35})
    args["loftr_b200"] = {**args["loftr_b200"], "weight_path": str(ckpt)}
    detector, matcher = cmw.build_model(args)
    assert isinstance(detector, cmw.DetectorWrapper) and isinstance(matcher, B200LoFTR)
    assert matcher.thr == 0.35 and matcher.fine is False and matcher.temperature == 0.1 and matcher._packed is not None
    args["type"] = "coarse_fine"
    _, matcher_f = cmw.build_model(args)
    assert matcher_f.fine is True
    with pytest.raises(NotImplementedError):                  # unknown names still fall through to the reference's if/elif chain
        cmw.build_model({**args, "matcher": "no_such_matcher", "seed": 0})
    # ---- HP-2
    ckpt2 = tmp_path / "multiview_matcher.ckpt"
    sdm = {"matcher." + k.replace("fine_transformer", "loftr_fine"): v for k, v in weights.multiview_state_dict(0).items()}
    sdm["matcher.loftr_coarse.layers.0.q_proj.weight"] = torch.zeros(4, 4)   # dropped by the reference (:47-49) and by the packer
    sdm["loss.whatever"] = torch.zeros(1)
    torch.save({"state_dict": sdm}, ckpt2)
    yaml_path = os.path.join(ref_shims.REF, "hydra_training_configs", "experiment", "multiview_refinement_matching.yaml")
    margs = {"cfg_path": [yaml_path], "weight_path": [str(ckpt2)], "seed": 666}
    for factor, (w, lw) in {None: (15, 7), 1: (13, 5), 2: (11, 3), 5: (7, 3)}.items():
        m = mm.build_model(margs, rewindow_size_factor=factor, model_idx=0)
        assert isinstance(m, B200MultiviewMatcher) and (m.W, m.LW) == (w, lw) and m._packed is not None
