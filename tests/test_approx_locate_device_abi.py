"""CPU tests of the device-resident approximate locates (awry_locate_device_hamming[_strands],
awry_locate_device_edit[_strands]): argument errors are reported before any device is touched.  The searches
themselves run in tests/test_gpu_approx_locate_device.py."""
import ctypes as C

import numpy as np

CALLS = ("awry_locate_device_hamming", "awry_locate_device_hamming_strands", "awry_locate_device_edit",
         "awry_locate_device_edit_strands")


def test_bad_arguments_need_no_device():
    from awry_b200 import fm_index as f
    lib = f.native()
    qb = np.frombuffer(b"ACGTACGT", np.uint8).copy()
    qo = np.array([0, 8], np.uint64)
    off = np.zeros(3, np.uint64)
    hits, dist, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
    for name in CALLS:
        call = getattr(lib, name)
        # null index
        assert call(None, 0, qb.ctypes.data, qo.ctypes.data, 1, 1, off.ctypes.data, C.byref(hits), C.byref(dist),
                    C.byref(n), None) == -1, name
        # null outputs and inputs
        assert call(None, 0, qb.ctypes.data, qo.ctypes.data, 1, 1, None, None, None, None, None) == -1, name
        assert call(None, 0, None, None, 1, 1, off.ctypes.data, C.byref(hits), None, C.byref(n), None) == -1, name
        # k > 3
        for k in (4, 7, 1 << 31):
            assert call(None, 0, qb.ctypes.data, qo.ctypes.data, 1, k, off.ctypes.data, C.byref(hits), C.byref(dist),
                        C.byref(n), None) == -1, (name, k)
        # an empty batch still needs an index
        assert call(None, 0, None, None, 0, 1, off.ctypes.data, C.byref(hits), None, C.byref(n), None) == -1, name
        assert b"null" in lib.awry_last_error(), name

