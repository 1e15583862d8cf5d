"""CPU: host-side logic of the package - prior generation, gt packing, sharding, the drop-in modules'
behaviour without a GPU (loud failure, no fallback)."""
import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import priors as PR, synth
from oracle import ssd_oracle as O


def test_priors_equal_the_oracle_tables():
    assert torch.equal(PR.make_priors(), O.make_priors())
    assert torch.equal(PR.make_priors(PR.SSD512_SPEC), O.make_priors(**O.SSD512))
    assert PR.SSD300_SPEC.num_priors == 8732 and PR.SSD512_SPEC.num_priors == 24564
    p = PR.make_priors()
    assert torch.equal(PR.cxcywh_to_xyxy_host(p), O.cxcywh_to_xyxy(p))
    assert float(p.min()) >= 0.0 and float(p.max()) <= 1.0                        # clamped in cxcywh form...
    assert float(PR.cxcywh_to_xyxy_host(p).min()) < 0.0                           # ...so corners leave the unit square


def test_pack_gt_and_synth_are_deterministic():
    gb, gc = synth.make_gt(5, 6)
    gb2, gc2 = synth.make_gt(5, 6)
    assert synth.digest(*gb, *gc) == synth.digest(*gb2, *gc2)
    boxes, cls, off = synth.pack_gt(gb, gc)
    assert off[0] == 0 and off[-1] == boxes.shape[0] == cls.shape[0]
    assert all(1 <= off[i + 1] - off[i] <= 10 for i in range(6))
    assert boxes.dtype == np.float32 and off.dtype == np.int32
    assert (boxes[:, 2:] >= boxes[:, :2]).all() and boxes.min() >= 0 and boxes.max() <= 1
    b0, c0, o0 = synth.pack_gt([], [])
    assert b0.shape == (0, 4) and o0.tolist() == [0]


def test_shard_ranges_cover_the_batch():
    from objectdetection_ssd_b200.dist import shard_range, shard_lists
    for batch in (0, 1, 7, 8, 256, 257):
        for world in (1, 2, 3, 8):
            spans = [shard_range(r, world, batch) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == batch
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    a, b = shard_lists(1, 2, list(range(5)), torch.arange(5))
    assert a == [3, 4] and b.tolist() == [3, 4]
    with pytest.raises(ValueError):
        shard_range(2, 2, 4)


def test_empty_image_raises_index_error_like_the_reference():
    from objectdetection_ssd_b200.head import PackedGT
    with pytest.raises(IndexError):
        PackedGT([torch.zeros(2, 4), torch.zeros(0, 4)], [torch.zeros(2), torch.zeros(0)], torch.device("cpu"))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour of a process WITHOUT a GPU")
def test_no_cpu_fallback_fails_loudly():
    from objectdetection_ssd_b200 import Losses, Util
    assert Losses.ancs_xywh.shape == (8732, 4) and not Losses.ancs_xywh.is_cuda     # import needs no GPU, no dataset
    pri = Losses.ancs_xywh
    with pytest.raises(RuntimeError, match="no CPU fallback|no CUDA"):
        Util.get_jaccard_tensor1(torch.rand(2, 4), Losses.ancs_xyxy)
    with pytest.raises(RuntimeError, match="no CPU fallback|no CUDA"):
        Losses.ssd((torch.zeros(1, 8732, 4), torch.zeros(1, 8732, 21)), [torch.zeros(1)], [torch.rand(1, 4)])
    with pytest.raises(RuntimeError, match="no CPU fallback|no CUDA"):
        Util.gcxgcy_to_cxcy(torch.zeros(8732, 4), pri)
    # the DataLoader-worker helper stays on the CPU by contract (Util.py:303-316)
    a = torch.tensor([[0.1, 0.1, 0.5, 0.5]])
    assert torch.equal(Util.get_jaccard_tensor11(a, Losses.ancs_xyxy), O.iou_matrix(a, Losses.ancs_xyxy))
    with pytest.raises(AttributeError):
        Util.transform            # outside the head path: only forwarded when the reference's Util is available


def test_missing_library_is_a_loud_error(monkeypatch, tmp_path):
    from objectdetection_ssd_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libssdhead.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_subsampling_matches_strided_indexing():
    from objectdetection_ssd_b200.Util import subsampling
    x = torch.arange(4 * 6 * 5).view(4, 6, 5)
    assert torch.equal(subsampling(x, [2, None, 3]), x[::2, :, ::3])


def test_head_levels_are_views_of_the_reference_layout():
    """Model.py:212-235 restated (permute(0,2,3,1).contiguous().view per conv map, cat over the six levels): the
    per-level tensors `head_levels` hands to the kernels are exactly the pieces of that concatenation, in the same
    prior order, and for channels_last conv outputs they are views (no copy)."""
    from objectdetection_ssd_b200.Losses import head_levels
    g = torch.Generator().manual_seed(3)
    bs = 2
    grids = ((38, 4), (19, 6), (10, 6), (5, 6), (3, 4), (1, 4))
    loc_maps = [torch.randn(bs, a * 4, hw, hw, generator=g) for hw, a in grids]
    conf_maps = [torch.randn(bs, a * 21, hw, hw, generator=g) for hw, a in grids]
    ref_loc = torch.cat([m.permute(0, 2, 3, 1).contiguous().view(bs, -1, 4) for m in loc_maps], dim=1)
    ref_conf = torch.cat([m.permute(0, 2, 3, 1).contiguous().view(bs, -1, 21) for m in conf_maps], dim=1)
    assert ref_loc.shape == (bs, 8732, 4) and ref_conf.shape == (bs, 8732, 21)
    locs, confs = head_levels(loc_maps, conf_maps)
    assert [int(t.shape[1]) for t in confs] == [5776, 2166, 600, 150, 36, 4]
    assert torch.equal(torch.cat(locs, 1), ref_loc) and torch.equal(torch.cat(confs, 1), ref_conf)
    cl = [m.contiguous(memory_format=torch.channels_last) for m in conf_maps]
    _, confs_cl = head_levels(loc_maps, cl)
    assert torch.equal(torch.cat(confs_cl, 1), ref_conf)
    # 1x1 maps have ambiguous strides; every other NHWC conv output is consumed in place
    assert all(v.data_ptr() == m.data_ptr() and v.is_contiguous() for v, m in zip(confs_cl[:5], cl[:5]))


def test_kernel_attributes_are_set_once_per_device_not_per_call():
    """The per-call launch path never sets a function attribute: a call that lowered a kernel's shared-memory limit
    could break another thread's launch of a larger shape between that thread's set and its launch.  The only
    cudaFuncSetAttribute of the library is the once-per-kernel-and-device raise in common.cuh."""
    import glob
    import os
    import re
    csrc = os.path.join(os.path.dirname(PR.__file__), "csrc")
    hits = {}
    for path in glob.glob(os.path.join(csrc, "*.cu*")):
        with open(path) as f:
            text = re.sub(r"//[^\n]*", "", f.read())
        n = len(re.findall(r"\bcudaFuncSetAttribute\s*\(", text))
        if n:
            hits[os.path.basename(path)] = n
    assert hits == {"common.cuh": 1}, hits
    with open(os.path.join(csrc, "common.cuh")) as f:
        text = f.read()
    body = text[text.index("inline cudaError_t smem_limit_once(const void* kernel)"):]
    body = body[:body.index("\n}\n")]
    assert "cudaFuncSetAttribute" in body and "std::lock_guard" in body
