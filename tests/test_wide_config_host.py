"""The launch-plan rule of the solve kernel (layout.cuh choose_solve_config) through cave_plan_choice, on hand-made plan words:
the wide configuration (4: 256 threads, one CTA per SM) is chosen only when the pack's shape enqueued it (word 5 = its dynamic
shared memory, 0 = not enqueued) and the largest hot set fits it but not 256 x 2; every other choice stays as it was."""
import ctypes

import pytest

CAPS = [27520, 56320, 75776, 112640]      # dynamic shared memory of configurations 0..3
WIDE_SMEM = 232448 - 528                  # what a B200 gives one CTA of the solve kernel (the plan kernel writes it)
D = 4950


@pytest.fixture(scope="module")
def lib():
    from cave_b200 import _lib, build
    build.build()
    return _lib.load()


def _choice(lib, hot, avg=None, wide=WIDE_SMEM, n=16, fp32=False, io64=False):
    """Plan words of n instances whose largest hot set is `hot` bytes and average working set `avg` bytes."""
    from cave_b200 import _lib
    avg = hot if avg is None else avg
    words = [n, avg * n, avg * n, hot, hot, wide, 0, 0]
    if fp32:
        words[3] = 10 ** 9                # the fp64 words must not be read
    else:
        words[4] = 10 ** 9
    arr = (ctypes.c_uint64 * 8)(*words)
    t, c, sm = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    idx = lib.cave_plan_choice(arr, D, _lib.F64 if io64 else _lib.F32, _lib.F32 if fp32 else _lib.F64,
                               ctypes.byref(t), ctypes.byref(c), ctypes.byref(sm))
    return idx, (t.value, c.value, sm.value)


@pytest.mark.parametrize("fp32", [False, True])
@pytest.mark.parametrize("wide", [0, WIDE_SMEM])
def test_configurations_0_to_3_are_unchanged(lib, wide, fp32):
    """Hot sets just below and above the capacity of configurations 0..2, with and without the wide configuration."""
    for i, cap in enumerate(CAPS[:3]):
        avg = cap // 2
        assert _choice(lib, cap - 1024, avg, wide, fp32=fp32)[0] == i
        assert _choice(lib, cap - 1023, avg, wide, fp32=fp32)[0] == i + 1
    assert _choice(lib, CAPS[3] - 1024, wide=wide, fp32=fp32)[0] == 3
    assert _choice(lib, 100, wide=wide, fp32=fp32, n=0)[0] == 3             # empty batch
    # an average working set beyond 95 % of 256 x 2 with a largest hot set that fits it: 256 x 2, as before
    assert _choice(lib, CAPS[3] - 1024, avg=CAPS[3], wide=wide, fp32=fp32)[0] == 3


@pytest.mark.parametrize("fp32", [False, True])
def test_wide_configuration_only_between_the_two_capacities(lib, fp32):
    above3 = CAPS[3] - 1023
    assert _choice(lib, above3, wide=0, fp32=fp32)[0] == 3                  # not enqueued: never chosen
    idx, cfg = _choice(lib, above3, fp32=fp32)
    assert idx == 4 and cfg == (256, 1, WIDE_SMEM)
    assert _choice(lib, WIDE_SMEM - 1024, fp32=fp32)[0] == 4                # fits exactly
    assert _choice(lib, WIDE_SMEM - 1023, fp32=fp32)[0] == 3                # fits nowhere: generic placement in 256 x 2
    assert _choice(lib, above3, fp32=fp32, n=0)[0] == 3
    # another wide capacity in the word (another device): the rule and the reported shared memory follow it
    assert _choice(lib, 150000, wide=150000 + 1024, fp32=fp32) == (4, (256, 1, 151024))
    assert _choice(lib, 150001, wide=150000 + 1024, fp32=fp32)[0] == 3


def test_float64_io_counts_the_cost_vector(lib):
    """c in float64 adds 4 bytes per coordinate to every hot set (io_extra)."""
    extra = D * 4
    assert _choice(lib, CAPS[3] - 1024 - extra, io64=True)[0] == 3
    assert _choice(lib, CAPS[3] - 1023 - extra, io64=True)[0] == 4
    assert _choice(lib, WIDE_SMEM - 1024 - extra, io64=True)[0] == 4
    assert _choice(lib, WIDE_SMEM - 1023 - extra, io64=True)[0] == 3
