"""Argument checks of apgk_group_build_affixes that need no device."""
import ctypes as C


def test_group_build_affixes_refuses_a_null_group(apgk_lib):
    from allpathslg_b200._lib import E_ARG, GroupAffixStats

    st = GroupAffixStats()
    assert apgk_lib.apgk_group_build_affixes(None, C.byref(st)) == E_ARG
    assert apgk_lib.apgk_group_build_affixes(None, None) == E_ARG
