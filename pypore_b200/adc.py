"""``AdcTrace``: a trace kept as the int16 ADC counts a nanopore amplifier records, plus the scale and offset that
turn them into current (the reference's loader computes ``counts * scale + offset`` in float64, read_abf.py:208-210).

Every parser and ``File`` accepts one wherever a trace goes.  The counts travel to the device at 2 B per sample --
half of float32, a quarter of the float64 current a non-dyadic scale needs -- and every result is the one the
float64 current ``decode()`` gives.  The parse paths never decode the whole trace on the host.
"""
import math

import numpy as np


def check_decoding(scale, offset):
    """(scale, offset) as floats; ValueError unless scale is finite and non-zero, offset finite and every int16
    count decodes to a finite value (decode is monotone in the count: checking both ends suffices)."""
    scale, offset = float(scale), float(offset)
    if not (math.isfinite(scale) and scale != 0.0 and math.isfinite(offset)):
        raise ValueError("ADC scale must be finite and non-zero and offset finite, got scale=%r offset=%r"
                         % (scale, offset))
    with np.errstate(over="ignore", invalid="ignore"):
        ends = np.array([-32768, 32767], np.float64) * scale + offset
    if not np.all(np.isfinite(ends)):
        raise ValueError("ADC scale %r and offset %r decode some counts to a non-finite current" % (scale, offset))
    return scale, offset


class AdcTrace(object):
    """int16 counts (1-D, C-contiguous) and their decoding ``current = counts * scale + offset`` in float64.

    ``len()``, ``shape``, indexing and slicing (decoded float64) and ``decode()`` (the whole current) behave like
    the float64 array the decoding gives."""

    def __init__(self, counts, scale, offset=0.0):
        if not (isinstance(counts, np.ndarray) and counts.dtype == np.int16 and counts.ndim == 1
                and counts.flags.c_contiguous):
            raise TypeError("AdcTrace counts must be a 1-D C-contiguous int16 numpy array")
        self.scale, self.offset = check_decoding(scale, offset)
        self.counts = counts

    def _decode(self, counts):
        return np.asarray(counts).astype(np.float64) * self.scale + self.offset

    def decode(self):
        """The whole trace as the float64 current."""
        return self._decode(self.counts)

    def __len__(self):
        return self.counts.shape[0]

    @property
    def shape(self):
        return self.counts.shape

    def __getitem__(self, index):
        return self._decode(self.counts[index])

    def __repr__(self):
        return "AdcTrace(%d counts, scale=%r, offset=%r)" % (len(self), self.scale, self.offset)
