"""Tag-count and length limits of the CRF: checked before anything touches the device, so no GPU is needed."""
import pytest


def test_more_than_128_tags_is_an_error():
    from polus_b200 import _lib
    from polus_b200.layers import CRF
    B, Tn = 2, 8
    for K in (0, 129):
        with pytest.raises(ValueError, match=r"K must be in \[1,128\]"):
            _lib.call("polus_crf_nll", None, None, None, None, None, B, Tn, K, None, None, None, None, None)
        with pytest.raises(ValueError, match=r"K must be in \[1,128\]"):
            _lib.call("polus_crf_decode", None, None, None, B, Tn, K, None, None, None)
    crf = CRF(129)
    with pytest.raises(ValueError, match="at most 128 tags"):
        crf.build((B, Tn, 129))
    assert crf.transitions is None and not crf.weights


def test_sequence_length_limits():
    """At K = 128 the loss takes up to 19 904 steps (shared memory: E and m_t, c_t) and the decode up to 1 760 (one byte
    back-pointer per tag and step); every K takes at least 512."""
    import ctypes as C
    from polus_b200 import _lib
    gem = C.c_void_p(256)  # the loss requires an emission-gradient pointer; nothing is dereferenced on these paths
    with pytest.raises(ValueError, match="T = 19905 too long"):
        _lib.call("polus_crf_nll", None, None, None, None, None, 2, 19905, 128, None, None, gem, None, None)
    with pytest.raises(ValueError, match="T = 1761 too long"):
        _lib.call("polus_crf_decode", None, None, None, 2, 1761, 128, None, None, None)
    # accepted shapes get as far as B == 0, which returns before any launch
    _lib.call("polus_crf_nll", None, None, None, None, None, 0, 19904, 128, None, None, gem, None, None)
    _lib.call("polus_crf_decode", None, None, None, 0, 1760, 128, None, None, None)
