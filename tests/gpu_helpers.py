"""Helpers shared by the GPU-tier modules (test_gpu_*.py): the `lmz` fixture, bit views, device sizes and a
free-memory precondition.  The CPU tier imports every GPU module at collection time on machines without the library
or a device, so nothing here loads either before a test runs."""
import gc

import numpy as np
import pytest
import torch

# float32 bit patterns of the reference's four rewards (-0.0, -1.0, -0.01, 100.0), indexed by the 2-bit reward code
# the packed state and the rollout's reward codes hold
REWARD_BITS = np.array([0x80000000, 0xBF800000, 0xBC23D70A, 0x42C80000], dtype=np.uint32)
REWARD_F32 = REWARD_BITS.view(np.float32)

CHUNK_BYTES = 1 << 30                  # bytes per chunk of same_bytes


@pytest.fixture(scope="module")
def lmz():
    import gym_lmaze_b200 as g
    from gym_lmaze_b200 import _abi
    _abi.load()                      # must be the in-tree CUDA library; raises if missing
    assert torch.cuda.is_available()
    return g


def u32(x):
    """uint32 view of a tensor (copied to the host) or an array; non-contiguous inputs are copied first."""
    if torch.is_tensor(x):
        x = x.detach().cpu().numpy()
    return np.ascontiguousarray(x).view(np.uint32)


def same_bytes(a, b):
    """Two contiguous tensors of one shape hold the same bytes.  Compared chunk by chunk on the device, so that a
    buffer of many GB needs no whole-buffer temporary."""
    if a.shape != b.shape:
        return False
    a, b = a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8)
    return a.numel() == b.numel() and \
        all(torch.equal(a[lo:lo + CHUNK_BYTES], b[lo:lo + CHUNK_BYTES]) for lo in range(0, a.numel(), CHUNK_BYTES))


def need_free(nbytes):
    """Fail (a B200 has the memory) unless nbytes of device memory are free once torch's cache is released."""
    gc.collect()
    torch.cuda.empty_cache()             # earlier tests' tensors sit in torch's caching allocator
    free_b = torch.cuda.mem_get_info()[0]
    if free_b < nbytes:
        pytest.fail("B200 expected: %d GiB free, need %d GiB" % (free_b >> 30, nbytes >> 30))


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def resident_threads():
    """The most threads the device holds resident: 2,048 per SM."""
    return sms() * 2048
