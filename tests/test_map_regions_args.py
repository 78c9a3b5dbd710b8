"""CPU test of the arguments DivQuant.map_regions / map_regions_device refuse with a ValueError before the library is
called (dq_map_regions_* would abort on some of them).  No device work: the library is a stub that fails if called."""
import numpy as np
import pytest


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"{name} called although the arguments are refused")


class _ManyPalettes:
    """More palettes than the 2^24 regions the call takes, without building them."""

    def __len__(self):
        return (1 << 24) + 1

    def __iter__(self):
        raise AssertionError("the palettes were read although there are too many")


@pytest.fixture
def dq(pkg):
    d = pkg.DivQuant.__new__(pkg.DivQuant)
    d.lib = _NoLibrary()
    return d


def test_host_form_refuses_bad_arguments(dq):
    px = np.arange(12, dtype=np.uint32)
    pal = np.array([0x102030, 0x405060], np.uint32)
    with pytest.raises(ValueError, match="one tag per pixel"):
        dq.map_regions(px, np.zeros(11, np.uint32), [pal])
    with pytest.raises(ValueError, match="2\\^24"):
        dq.map_regions(px, np.zeros(12, np.uint32), _ManyPalettes())
    with pytest.raises(ValueError, match="1-D array"):
        dq.map_regions(px, np.zeros(12, np.uint32), pal)  # one flat array instead of one palette per region
    with pytest.raises(ValueError, match="24000"):
        dq.map_regions(px, np.zeros(12, np.uint32), [pal, np.zeros(24001, np.uint32)], labels=True)


def test_device_form_refuses_bad_arguments(dq):
    torch = pytest.importorskip("torch")
    px = torch.arange(12, dtype=torch.int32)
    with pytest.raises(ValueError, match="CUDA tensors"):
        dq.map_regions_device(px, torch.zeros(12, dtype=torch.int32), [np.array([1], np.uint32)])
