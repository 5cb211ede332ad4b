"""Two-image backbone pass (dfsfm_coarse_features_pair): the tokens of both images of a pair from one launch per layer are bitwise the
tokens of two one-image calls, and the matcher takes that path only when it applies (coarse-only, same size, neither image cached)."""
import pytest
import torch

from tests import util
from tests import weights

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sd():
    return weights.loftr_state_dict(0, calibrated=True)


def make_matcher(sd):
    from detectorfreesfm_b200 import B200LoFTR
    m = B200LoFTR(util.loftr_config(thr=0.2, temperature=0.1)).cuda().eval()
    m.load_state_dict(sd)
    return m


def spy_pair_calls(m, monkeypatch):
    calls = []
    orig = m.extract_features_pair

    def spy(*a, **k):
        calls.append(a[2:])
        return orig(*a, **k)
    monkeypatch.setattr(m, "extract_features_pair", spy)
    return calls


# 832x832: the benchmark size; 480x640; 352x480: 45 x 61 = 2745 flat rows at 1/8, not a multiple of the 256-row tile, so tiles straddle
# the boundary between the two images at every layer
@pytest.mark.parametrize("hw", [(832, 832), (480, 640), (352, 480)])
def test_pair_tokens_equal_single_image_tokens(sd, hw):
    m = make_matcher(sd)
    im0, im1 = util.synth_image(*hw, seed=21).cuda(), util.synth_image(*hw, seed=22).cuda()
    with torch.no_grad():
        p0, p1 = m.extract_features_pair(im0, im1)
        s0, s1 = m.extract_features(im0), m.extract_features(im1)
        q0, q1 = m.extract_features_pair(im0, im1)   # the pair workspace is reused after single-image calls
    torch.cuda.synchronize()
    assert p0.shape == ((hw[0] // 8) * (hw[1] // 8), 256)
    assert s0.abs().max().item() > 0 and not torch.equal(s0, s1)
    assert torch.equal(p0, s0) and torch.equal(p1, s1)
    assert torch.equal(q0, s0) and torch.equal(q1, s1)


def test_pair_path_fills_the_cache_and_one_cached_image_falls_back(sd, monkeypatch):
    m = make_matcher(sd)
    calls = spy_pair_calls(m, monkeypatch)
    ims = [util.synth_pair(96, 128, seed=s)[i].cuda() for s, i in ((1, 0), (1, 1), (2, 0))]
    ones = torch.ones(1, 2, device="cuda")

    def run(i, j, matcher, keyed=True):
        data = {"image0": ims[i], "image1": ims[j], "scale0": ones, "scale1": ones}
        if keyed:
            data["pair_key"] = ((f"im{i}",), (f"im{j}",))
        matcher(data)
        return data

    d01 = run(0, 1, m)
    assert len(calls) == 1 and ("im0", 96, 128) in m._cache and ("im1", 96, 128) in m._cache
    assert torch.equal(m._cache[("im0", 96, 128)], m.extract_features(ims[0]))
    assert torch.equal(m._cache[("im1", 96, 128)], m.extract_features(ims[1]))
    d02 = run(0, 2, m)                    # image 0 is cached: image 2 alone through the one-image path
    assert len(calls) == 1 and ("im2", 96, 128) in m._cache
    d00 = run(0, 0, m)                    # both cached
    assert len(calls) == 1
    ref = make_matcher(sd)
    for (i, j), d in (((0, 1), d01), ((0, 2), d02), ((0, 0), d00)):
        r = run(i, j, ref, keyed=False)   # no cache: every pair takes the two-image path
        for k in ("i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f"):
            assert torch.equal(d[k], r[k]), (i, j, k)
    assert len(d01["mconf"]) > 0


def test_pair_of_different_sizes_falls_back(sd, monkeypatch):
    m = make_matcher(sd)
    calls = spy_pair_calls(m, monkeypatch)
    im0, im1 = util.synth_image(96, 136, seed=11).cuda(), util.synth_image(120, 88, seed=12).cuda()
    data = {"image0": im0, "image1": im1, "pair_key": (("a",), ("b",))}
    m(data)
    assert len(calls) == 0
    assert tuple(data["hw0_c"]) == (12, 17) and tuple(data["hw1_c"]) == (15, 11)
    assert ("a", 96, 136) in m._cache and ("b", 120, 88) in m._cache
