"""CPU: the data-parallel trainer's batch split and device-list validation (riser_b200/parallel.py)."""
import pytest
import torch

from riser_b200.parallel import MAX_DEVICES, _expandable_segments, check_devices, split


def test_split_is_contiguous_in_device_order_and_balanced():
    for G in range(1, MAX_DEVICES + 1):
        for B in range(20):
            s = split(B, G)
            assert len(s) == G
            assert s[0][0] == 0 and s[-1][1] == B
            assert all(s[d][1] == s[d + 1][0] for d in range(G - 1))
            sizes = [hi - lo for lo, hi in s]
            assert min(sizes) >= 0 and max(sizes) - min(sizes) <= 1
            assert s == [(d * B // G, (d + 1) * B // G) for d in range(G)]
    assert split(1, 2) == [(0, 0), (0, 1)]           # the first device is the empty one
    assert split(3, 2) == [(0, 1), (1, 3)]


def test_device_list_validation():
    assert check_devices([0, 1]) == [0, 1]
    assert check_devices(["cuda:3", torch.device("cuda", 1), 2]) == [3, 1, 2]
    assert check_devices(range(8)) == list(range(8))
    for bad in ([], [0, 0], [1, "cuda:1"], list(range(9)), [-1], ["cpu"], ["cuda"], [torch.device("cpu")]):
        with pytest.raises(ValueError):
            check_devices(bad)
    with pytest.raises(TypeError):
        check_devices([0.5])


def test_expandable_segments_setting_is_recognised(monkeypatch):
    for var in ("PYTORCH_CUDA_ALLOC_CONF", "PYTORCH_ALLOC_CONF"):
        monkeypatch.delenv(var, raising=False)
    assert not _expandable_segments()
    monkeypatch.setenv("PYTORCH_CUDA_ALLOC_CONF", "max_split_size_mb:128, expandable_segments:True")
    assert _expandable_segments()
    monkeypatch.setenv("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:False")
    assert not _expandable_segments()
    monkeypatch.setenv("PYTORCH_ALLOC_CONF", "expandable_segments:true")
    assert _expandable_segments()
