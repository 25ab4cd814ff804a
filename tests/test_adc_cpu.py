"""int16 ADC traces on the host, no GPU: the integer threshold the scan compares with, the AdcTrace type and its
validation, File(current=AdcTrace)."""
import ctypes

import numpy as np
import pytest

from pypore_b200 import _lib, parsers
from pypore_b200.adc import AdcTrace
from pypore_b200.DataTypes import File

COUNTS = np.arange(-32768, 32768, dtype=np.int64)


def key_threshold(scale, offset, threshold):
    L = _lib.load()
    key, kxor = ctypes.c_int32(), ctypes.c_int32()
    assert L.pp_adc16_key_threshold(scale, offset, threshold, ctypes.byref(key), ctypes.byref(kxor)) == _lib.PP_OK
    return key.value, kxor.value


def decode(counts, scale, offset):
    return np.asarray(counts).astype(np.float64) * scale + offset


@pytest.mark.parametrize("scale", [0.0305, 1.0 / 32, -0.0305, -1.0 / 32, 3.1e-4, -7.0])
@pytest.mark.parametrize("offset", [0.0, -0.0, 0.0123, -5.5])
def test_key_threshold_equals_brute_force_over_every_count(scale, offset):
    cur = decode(COUNTS, scale, offset)
    vals = np.unique(cur)
    thresholds = [vals[0], vals[-1], vals[len(vals) // 2], vals[len(vals) // 3],
                  (vals[100] + vals[101]) / 2, np.nextafter(vals[7], np.inf), np.nextafter(vals[7], -np.inf),
                  vals[0] - 1.0, vals[-1] + 1.0, np.nan, np.inf, -np.inf, 0.0, -0.0]
    for thr in thresholds:
        key, kxor = key_threshold(scale, offset, thr)
        assert kxor == (-1 if scale < 0 else 0)
        keys = COUNTS ^ kxor
        assert np.array_equal(keys < key, cur < thr), (scale, offset, thr, key)


def test_key_threshold_ends():
    assert key_threshold(0.5, 0.0, np.nan)[0] == -32768         # nothing is below a NaN threshold
    assert key_threshold(0.5, 0.0, np.inf)[0] == 32768          # everything is below +inf
    assert key_threshold(-0.5, 0.0, -np.inf)[0] == -32768


def test_adc_trace_slicing_and_decode_are_the_numpy_formula():
    rng = np.random.RandomState(5)
    c = rng.randint(-32768, 32768, 10007).astype(np.int16)
    c[:2] = (-32768, 32767)
    for scale, offset in ((0.0305, 0.0123), (-1.0 / 3, 7.25), (1.0 / 32, 0.0)):
        t = AdcTrace(c, scale, offset)
        want = c.astype(np.float64) * scale + offset
        assert len(t) == len(c) and t.shape == c.shape
        assert np.array_equal(t.decode(), want)
        assert t.decode().tobytes() == want.tobytes()
        for sl in (slice(0, 10), slice(100, 5000, 3), slice(-7, None), slice(5, 5)):
            assert t[sl].tobytes() == want[sl].tobytes()
        assert t[17] == want[17] and isinstance(t[17], np.floating)


@pytest.mark.parametrize("scale, offset", [(0.0, 0.0), (np.nan, 0.0), (np.inf, 0.0), (1.0, np.nan), (1.0, -np.inf),
                                           (1e305, 0.0), (-1e305, 1.0), (1e300, 1.7976931348623157e308)])
def test_invalid_decoding_raises_before_any_library_call(scale, offset, monkeypatch):
    monkeypatch.setattr(_lib, "load", lambda: pytest.fail("library called"))
    with pytest.raises(ValueError):
        AdcTrace(np.zeros(4, np.int16), scale, offset)


def test_c_check_agrees():
    L = _lib.load()
    for scale, offset in ((0.0, 0.0), (np.nan, 0.0), (1.0, np.inf), (1e305, 0.0), (1e300, 1.7976931348623157e308)):
        assert L.pp_adc16_check(scale, offset) == _lib.PP_ERR_ARG
    for scale, offset in ((0.0305, 0.0123), (-1.0, 5.0), (1e300, 0.0)):
        assert L.pp_adc16_check(scale, offset) == _lib.PP_OK


@pytest.mark.parametrize("counts", [np.zeros(4, np.int32), np.zeros(4, np.float32), np.zeros((2, 2), np.int16),
                                    np.zeros(8, np.int16)[::2], [1, 2, 3]])
def test_counts_must_be_contiguous_1d_int16(counts):
    with pytest.raises(TypeError):
        AdcTrace(counts, 0.5)


def test_file_with_adc_current_reports_the_decoded_current_without_a_device():
    c = np.arange(-300, 300, dtype=np.int16)
    t = AdcTrace(c, 0.0305, 0.0123)
    f = File(current=t, timestep=1000. / 1e5)
    assert "current" not in f.__dict__                        # nothing decoded until asked
    assert f.current.dtype == np.float64 and np.array_equal(f.current, t.decode())
    assert f.current is f.current                             # decoded once
    f.current = np.zeros(3)                                   # another current replaces the counts
    assert f._samples().shape == (3,) and not isinstance(f._samples(), AdcTrace)
    g = File(current=t, timestep=1000. / 1e5)
    g.to_meta()
    assert not hasattr(g, "current")


def test_plain_integer_arrays_keep_the_float32_route():
    x = np.arange(-100, 100, dtype=np.int16)
    assert parsers._device_trace(x).dtype == np.float32
