"""Argument checks of apgk_group_build_occurrences that need no device."""
import ctypes as C


def test_group_build_occurrences_refuses_a_null_group(apgk_lib):
    from allpathslg_b200._lib import E_ARG, GroupOccStats

    st = GroupOccStats()
    assert apgk_lib.apgk_group_build_occurrences(None, C.byref(st)) == E_ARG
    assert apgk_lib.apgk_group_build_occurrences(None, None) == E_ARG
