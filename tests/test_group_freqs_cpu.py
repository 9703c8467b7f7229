"""Argument checks of apgk_group_read_freqs_device that need no device."""
import ctypes as C


def test_group_read_freqs_refuses_a_null_group(apgk_lib):
    from allpathslg_b200._lib import E_ARG, GroupFreqStats

    st = GroupFreqStats()
    fb = (C.c_uint64 * 1)(0)
    nb = (C.c_uint64 * 1)(0)
    outs = (C.c_void_p * 1)(None)
    assert apgk_lib.apgk_group_read_freqs_device(None, outs, fb, nb, C.byref(st)) == E_ARG
    assert apgk_lib.apgk_group_read_freqs_device(None, None, None, None, None) == E_ARG
