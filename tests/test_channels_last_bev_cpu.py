"""CPU: the channels_last BEV-map flag of the C ABI (CF_IO_NHWC) is declared, bound, and ignored by the workspace sizes."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_io_nhwc_flag_matches_the_header(dcf):
    h = open(os.path.join(ROOT, "include", "cf_b200.h")).read()
    m = re.search(r"#define CF_IO_NHWC (0x[0-9a-fA-F]+)\b", h)
    assert m, "CF_IO_NHWC is not defined in include/cf_b200.h"
    L = dcf._lib
    assert L.IO_NHWC == int(m.group(1), 16)
    # a flag bit: disjoint from the modes, CF_IO_BF16 and CF_BWD_DETERMINISTIC
    assert L.IO_NHWC & (L.IO_BF16 | L.BWD_DETERMINISTIC) == 0
    assert all(L.IO_NHWC & m == 0 for m in L.MODES.values())


def test_workspace_sizes_ignore_the_layout_flag(dcf):
    L, lib = dcf._lib, dcf.load()
    for m in L.MODES.values():
        for flags in (0, L.IO_BF16):
            for C, B, H, W in ((32, 2, 350, 300), (128, 4, 88, 75), (256, 1, 22, 19), (48, 3, 37, 53)):
                assert (lib.cf_fusion_workspace_bytes(C, m | flags | L.IO_NHWC, B, H, W)
                        == lib.cf_fusion_workspace_bytes(C, m | flags, B, H, W))
                assert lib.cf_fusion_packed_bytes(C, m | flags | L.IO_NHWC) == lib.cf_fusion_packed_bytes(C, m | flags)
