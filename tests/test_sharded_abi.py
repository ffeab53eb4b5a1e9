"""cpbus_create_sharded / cpbus_shard_range: host logic, no GPU needed.  Argument validation returns the same status codes
with or without a device, and the id partition is the one `sharding` uses."""
import ctypes as C

import pytest

from containerpilot_b200 import _native as nat
from containerpilot_b200 import sharding


def _create_sharded(devices, n_shards=None, stream=None, **kw):
    lib = nat.load()
    cfg = nat.Config(); cfg.n_max_subs = 8; cfg.device = -1
    for k, v in kw.items():
        setattr(cfg, k, v)
    cfg.stream = stream
    n = len(devices) if n_shards is None else n_shards
    devs = (C.c_int32 * max(1, len(devices)))(*devices) if devices is not None else None
    h = C.c_void_p()
    rc = lib.cpbus_create_sharded(C.byref(cfg), devs, n, C.byref(h))
    if rc == 0:
        lib.cpbus_destroy(h)
    else:
        assert not h.value
    return rc


def test_create_sharded_rejects_bad_arguments_before_touching_a_device():
    assert _create_sharded([0, 0], n_max_subs=0) == nat.EINVAL
    assert _create_sharded([0, 0], ring_cap=1000) == nat.EINVAL
    assert _create_sharded([0, 0], ring_cap=1024, batch_cap=100) == nat.EINVAL
    assert _create_sharded([0, 0], timers_per_sub=3) == nat.EINVAL
    assert _create_sharded([0, 0], store_path=9) == nat.EINVAL
    assert _create_sharded(None, n_shards=2) == nat.EINVAL                  # devices == NULL
    assert _create_sharded([0], n_shards=0) == nat.EINVAL
    assert _create_sharded([0] * 65, n_max_subs=1000) == nat.EINVAL         # above the stream's 64 consumers
    assert _create_sharded([0, 0, 0], n_max_subs=2) == nat.EINVAL           # fewer subscribers than shards
    assert _create_sharded([0, 0], stream=1) == nat.EINVAL                  # each shard owns its stream
    lib = nat.load()
    h = C.c_void_p()
    assert lib.cpbus_create_sharded(None, (C.c_int32 * 1)(0), 1, C.byref(h)) == nat.EINVAL


def test_create_sharded_without_a_device_is_enodev():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is visible")
    assert _create_sharded([0, 0, 0, 0], n_max_subs=64) == nat.ENODEV
    assert _create_sharded([0], n_max_subs=64) == nat.ENODEV               # n_shards == 1 is cpbus_create on devices[0]


def _py_range(n, g, k):
    base, extra = divmod(n, g)
    return k * base + min(k, extra), base + (1 if k < extra else 0)


def test_shard_range_tiles_and_inverts():
    lib = nat.load()
    first, count = C.c_uint32(), C.c_uint32()
    for g in range(1, 10):
        for n in range(g, 301):
            nxt = 0
            sizes = []
            for k in range(g):
                assert lib.cpbus_shard_range(n, g, k, C.byref(first), C.byref(count)) == nat.OK
                assert (first.value, count.value) == _py_range(n, g, k) == sharding.shard_range(n, g, k)
                assert first.value == nxt                                   # the pieces tile [0, n) in order
                nxt += count.value
                sizes.append(count.value)
                for i in range(first.value, first.value + count.value):
                    assert sharding.owner_of(i, n, g) == k
            assert nxt == n and max(sizes) - min(sizes) <= 1


def test_shard_range_rejects_bad_arguments():
    lib = nat.load()
    first, count = C.c_uint32(), C.c_uint32()
    assert lib.cpbus_shard_range(10, 0, 0, C.byref(first), C.byref(count)) == nat.EINVAL
    assert lib.cpbus_shard_range(10, 2, 2, C.byref(first), C.byref(count)) == nat.EINVAL
    assert lib.cpbus_shard_range(10, 2, 0, None, C.byref(count)) == nat.EINVAL
    with pytest.raises(ValueError):
        sharding.shard_range(10, 2, 2)
