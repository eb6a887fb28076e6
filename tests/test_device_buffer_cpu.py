"""A failed cc_device_alloc raises and leaves nothing for the buffer's finaliser to release (no GPU needed: device -1 is
refused on any machine)."""

import gc
import sys

import pytest

torch = pytest.importorskip("torch")


def test_failed_allocation_raises_and_finalises_cleanly():
    from collectivecrossing_b200 import _native
    from collectivecrossing_b200.batched import _DeviceBuffer

    seen = []
    hook, sys.unraisablehook = sys.unraisablehook, seen.append
    try:
        with pytest.raises(Exception):
            _DeviceBuffer(_native.library(), -1, (16,), torch.float32)
        gc.collect()
    finally:
        sys.unraisablehook = hook
    assert not seen, [str(u.exc_value) for u in seen]
