"""The recovery policy of the device decode calls (no GPU): which decodes decode_ladder tries, in which order, and when
Engine._decode repeats the series in two-launch mode.  The decodes are scripted: each returns the status words it is given."""
import numpy as np
import pytest

from flac_raster_b200 import _native as nat
from flac_raster_b200.engine import Engine, decode_ladder

T, F = True, False


def words(*names):
    w = np.zeros(8, dtype=np.int64)
    for n in names:
        w[getattr(nat, n)] += 1
    return w


CLEAN = words()
WIDE = words("ST_LPC_ORDER_ABOVE_12")
MISSING = words("ST_FRAMES_MISSING")
CRC = words("ST_CRC16_ERRORS")
PARSE = words("ST_PARSE_ERRORS")


def run(results, has_index=True, allow_scan=True):
    calls = []
    todo = iter(results)

    def attempt(max_order, use_index):
        calls.append((max_order, use_index))
        return next(todo)

    status = decode_ladder(attempt, has_index, allow_scan, "frb_decode_test")
    assert next(todo, None) is None, "an attempt the ladder should have made was not made"
    return calls, status


@pytest.mark.parametrize("results, has_index, allow_scan, expect", [
    ([CLEAN], T, T, [(12, T)]),                                        # clean indexed decode
    ([WIDE, CLEAN], T, T, [(12, T), (32, T)]),                         # LPC order above 12 under the index
    ([MISSING, CLEAN], T, T, [(12, T), (12, F)]),                      # rejected index
    ([CRC, WIDE, CLEAN], T, T, [(12, T), (12, F), (32, F)]),           # rejected index, then wide order
    ([WIDE, PARSE, CLEAN], T, T, [(12, T), (32, T), (12, F)]),         # the wide-order attempt rejects the index
    ([CLEAN], F, T, [(12, F)]),                                        # no index
    ([WIDE, CLEAN], F, T, [(12, F), (32, F)]),
    ([MISSING], F, T, [(12, F)]),                                      # a damaged scan is the answer
    ([PARSE], T, F, [(12, T)]),                                        # scan not allowed, index rejected
    ([WIDE, CLEAN], T, F, [(12, T), (32, T)]),
])
def test_attempt_order(results, has_index, allow_scan, expect):
    calls, status = run(results, has_index, allow_scan)
    assert calls == expect
    assert status is results[-1]


def test_rejected_tiles_raise_naming_the_caller():
    with pytest.raises(nat.NativeError, match="frb_decode_test") as ei:
        run([words("ST_TILES_REJECTED", "ST_TILES_REJECTED")])
    assert ei.value.status == nat.ERR_INVALID_ARG and "2 tile(s)" in str(ei.value)
    with pytest.raises(nat.NativeError):                               # also when the index is damaged at the same time
        run([words("ST_TILES_REJECTED", "ST_FRAMES_MISSING")])


def test_status_damaged():
    assert not nat.status_damaged(CLEAN) and not nat.status_damaged(WIDE)
    assert not nat.status_damaged(words("ST_FRAMES_DECODED", "ST_OFFSET_WAIT_TIMEOUTS"))
    assert all(nat.status_damaged(w) for w in (MISSING, CRC, PARSE))


def engine_with(results, two_launch=False):
    """An Engine without a device whose status downloads return `results` in turn, and the log of its launches."""
    eng = Engine.__new__(Engine)
    eng._two_launch = two_launch
    todo = iter(results)
    launches = []

    def download(t, dtype, count):
        assert t == "d_status" and dtype == np.int32 and count == 8
        return next(todo).astype(np.int32)

    def launch(max_order, use_index):
        launches.append((max_order, use_index, eng._two_launch))

    eng._download = download
    return eng, launch, launches, todo


def test_offset_timeout_switches_to_two_launch_mode_and_repeats_the_ladder_once():
    timeout = words("ST_OFFSET_WAIT_TIMEOUTS")
    eng, launch, launches, todo = engine_with([MISSING, timeout, timeout])
    status = eng._decode(launch, "d_status", True, True, "frb_decode_test")
    assert eng._two_launch
    assert launches == [(12, T, F), (12, F, F), (12, T, T)]            # the repeat starts again with the index
    assert list(status) == list(timeout) and next(todo, None) is None

    eng, launch, launches, _ = engine_with([timeout, WIDE, CLEAN])
    status = eng._decode(launch, "d_status", False, True, "frb_decode_test")
    assert launches == [(12, F, F), (12, F, T), (32, F, T)] and list(status) == list(CLEAN)


def test_no_repeat_in_two_launch_mode_or_without_a_timeout():
    eng, launch, launches, _ = engine_with([words("ST_OFFSET_WAIT_TIMEOUTS")], two_launch=True)
    status = eng._decode(launch, "d_status", False, True, "frb_decode_test")
    assert launches == [(12, F, T)] and status[nat.ST_OFFSET_WAIT_TIMEOUTS] == 1
    eng, launch, launches, _ = engine_with([CLEAN])
    eng._decode(launch, "d_status", True, True, "frb_decode_test")
    assert launches == [(12, T, F)] and not eng._two_launch
