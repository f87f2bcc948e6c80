"""CPU-side checks of the score-ranked evaluation hand-off: argument checks of frr_pack_detections_ranked that return
before any CUDA call, its workspace query, and the Python option checks."""
import pytest
import torch

from faster_rcnn_pytorch_b200 import _lib, ops


@pytest.fixture(scope="module")
def lib():
    from faster_rcnn_pytorch_b200 import build
    build.build()
    return _lib.load()


def test_workspace_bytes_follow_the_ranked_rows(lib):
    # valid mask [B,cap] u8 + order [B,min(max_det,cap)] i32 + count [B] i32, each 256-byte aligned
    assert lib.frr_pack_detections_ranked_workspace_bytes(8, 24000, 100) == 8 * 24000 + 3328 + 256
    assert lib.frr_pack_detections_ranked_workspace_bytes(2, 10, 100) == 256 * 3
    assert lib.frr_pack_detections_ranked_workspace_bytes(1, 0, 100) == 256
    assert lib.frr_pack_detections_ranked_workspace_bytes(1, 10, 0) == 0


@pytest.mark.parametrize("B,cap,max_det,pcm,what", [
    (-1, 10, 100, 0, b"bad sizes"), (1, -1, 100, 0, b"bad sizes"), (1, 10, 0, 0, b"bad sizes"),
    (1, 10, 100, -1, b"bad sizes"), (1, 20000, 16385, 0, b"16384"), (1, 10, 100, 0, b"null pointer")])
def test_ranked_entry_point_rejects_bad_arguments(lib, B, cap, max_det, pcm, what):
    rc = lib.frr_pack_detections_ranked(None, None, None, None, B, cap, max_det, pcm, None, 0, None, None, None, 0, None)
    assert rc == -1 and what in lib.frr_last_error()


def test_ranked_entry_point_accepts_an_empty_batch(lib):
    assert lib.frr_pack_detections_ranked(None, None, None, None, 0, 10, 100, 0, None, 0, None, None, None, 0, None) == 0


@pytest.mark.parametrize("rank,pcm", [("area", 0), ("class", 100), ("score", -1)])
def test_pack_detections_rejects_unknown_selections(rank, pcm):
    z = torch.zeros((1, 4), dtype=torch.int32)
    with pytest.raises(ValueError, match="pack_detections"):
        ops.pack_detections(torch.zeros((1, 4, 4)), z, torch.zeros((1, 4)), z[:, 0], 100, rank=rank, per_class_max=pcm)
