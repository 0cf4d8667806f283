"""Host logic of dealing one map's cubes over several devices (``CryoEMPredictor(devices=)``): the model calls
the workers make are the one-device calls, and the device list is parsed strictly.  No GPU needed."""
import itertools

import pytest

from mica_b200 import _lib
from mica_b200.pipeline import deal_cubes, worker_batches
from mica_b200.predict import parse_devices


def one_device_calls(n, super_batch, model_batch):
    """(start, end) of every model call of a one-device run, in the visiting order."""
    calls = []
    for s in range(0, n, super_batch):
        e = min(n, s + super_batch)
        calls += [(c, min(e, c + model_batch)) for c in range(s, e, model_batch)]
    return calls


def worker_calls(lo, hi, super_batch, model_batch):
    calls = []
    for b0, b1 in worker_batches(lo, hi, super_batch):
        assert 0 < b1 - b0 <= super_batch
        calls += [(lo + c, lo + min(b1, c + model_batch)) for c in range(b0, b1, model_batch)]
    return calls


@pytest.mark.parametrize('n,super_batch,model_batch,workers',
                         list(itertools.product((0, 1, 5, 216, 1331), (8, 20, 256), (1, 3, 8), (1, 2, 3, 8))))
def test_dealt_model_calls_are_the_one_device_calls(n, super_batch, model_batch, workers):
    ranges = deal_cubes(n, super_batch, model_batch, workers)
    assert len(ranges) == workers
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(ranges[:-1], ranges[1:]))       # contiguous, in order
    got = [c for lo, hi in ranges for c in worker_calls(lo, hi, super_batch, model_batch)]
    assert got == one_device_calls(n, super_batch, model_batch)
    for lo, hi in ranges:                                 # balanced to within one chunk
        assert hi >= lo and abs((hi - lo) - n / workers) <= model_batch


def test_fewer_chunks_than_workers_leave_workers_idle():
    ranges = deal_cubes(5, 20, 8, 3)                      # 5 cubes are one chunk
    assert sorted(hi - lo for lo, hi in ranges) == [0, 0, 5]
    assert deal_cubes(0, 20, 8, 3) == [(0, 0)] * 3
    assert worker_batches(4, 4, 20) == []
    with pytest.raises(_lib.MicaError):
        deal_cubes(10, 20, 8, 0)


def test_chunk_bounds_follow_the_super_batches():
    # model_batch 8 does not divide super_batch 20: chunks start at 0, 8, 16, 20, 28, 36, 40, ...
    ranges = deal_cubes(216, 20, 8, 3)
    starts = {c for c, _ in one_device_calls(216, 20, 8)} | {216}
    assert all(lo in starts and hi in starts for lo, hi in ranges)
    assert ranges == [(0, 68), (68, 140), (140, 216)]    # 72 and 144 lie halfway: the lower start wins
    assert worker_batches(68, 140, 20) == [(0, 12), (12, 32), (32, 52), (52, 72)]
    assert worker_batches(76, 144, 20) == [(0, 4), (4, 24), (24, 44), (44, 64), (64, 68)]


def test_parse_devices():
    assert parse_devices(None, 8) is None
    assert parse_devices('', 8) is None and parse_devices('  ', 8) is None
    assert parse_devices('all', 3) == [0, 1, 2] and parse_devices('ALL', 1) == [0]
    assert parse_devices('0,1', 2) == [0, 1] and parse_devices(' 2, 0 ', 3) == [2, 0]
    assert parse_devices(['cuda:0'] * 3, 1) == [0, 0, 0]
    assert parse_devices([1, 'cuda:0', '2'], 3) == [1, 0, 2]
    for bad in ('garbage', '0,,1', '0;1', 'cpu', 'cuda', '-1', '1.5', '2'):
        with pytest.raises(ValueError):
            parse_devices(bad, 2)
    with pytest.raises(ValueError):
        parse_devices('all', 0)
    with pytest.raises(ValueError):
        parse_devices('0,0', 2, allow_repeats=False)      # MICA_DEVICES: one worker per GPU


def test_peer_enable_rejects_bad_devices_before_touching_the_device():
    lib = _lib.lib
    assert lib.mica_peer_enable(0, 0) == 0                # same device: nothing to enable
    assert lib.mica_peer_enable(-1, 0) == -1
    assert b'device' in lib.mica_last_error()
