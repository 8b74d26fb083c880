"""A destroyed context gives back all of its device memory, including the per-layer wait-cycle counters it allocates
when NHANS_DEBUG_STATS=1."""
import pytest

from nhans_b200.engine import Engine

pytestmark = pytest.mark.gpu

CONTEXTS = 600                      # 600 x 8 KiB of counters: well above the tolerance, however the driver packs them
TOLERANCE = 2 << 20


def test_destroyed_contexts_free_their_device_memory(monkeypatch):
    import torch
    monkeypatch.setenv("NHANS_DEBUG_STATS", "1")        # read by nhans_create
    Engine(0, 0, win_capacity=1, row_capacity=1).close()       # loads the library and the CUDA context
    free0, _ = torch.cuda.mem_get_info(0)
    for _ in range(CONTEXTS):
        Engine(0, 0, win_capacity=1, row_capacity=1).close()
    free1, _ = torch.cuda.mem_get_info(0)
    assert free0 - free1 <= TOLERANCE, "%d contexts kept %.1f MiB of device memory" % (CONTEXTS, (free0 - free1) / 2 ** 20)
