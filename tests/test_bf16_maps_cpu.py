"""CPU: the bf16 feature-map surface of the C ABI (CF_IO_BF16, cf_point_gather_bf16) is declared, exported and bound."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    return open(os.path.join(ROOT, "include", "cf_b200.h")).read()


def test_io_bf16_flag_matches_the_header(dcf):
    m = re.search(r"#define CF_IO_BF16 (0x[0-9a-fA-F]+)\b", _header())
    assert m, "CF_IO_BF16 is not defined in include/cf_b200.h"
    assert dcf._lib.IO_BF16 == int(m.group(1), 16)
    # a flag bit: disjoint from the modes and from CF_BWD_DETERMINISTIC
    assert dcf._lib.IO_BF16 & dcf._lib.BWD_DETERMINISTIC == 0
    assert all(dcf._lib.IO_BF16 & m == 0 for m in dcf._lib.MODES.values())


def test_point_gather_bf16_is_declared_exported_and_bound(dcf):
    assert re.search(r"CF_API\s+int\s+cf_point_gather_bf16\s*\(", _header())
    assert os.path.exists(dcf.SO_PATH), "build it: python -c 'import __graft_entry__ as g; g.build()'"
    assert hasattr(ctypes.CDLL(dcf.SO_PATH), "cf_point_gather_bf16")
    # same arguments as cf_point_gather
    assert dcf._lib.SIGNATURES["cf_point_gather_bf16"] == dcf._lib.SIGNATURES["cf_point_gather"]

