"""CVG_MATCH_CROSS_CHECK, the cross-check flag of cvg_detect_params.method, as the header defines it against the Python
constant and detect_params(cross_check=...); the struct keeps its 64-byte layout (the library loads without a GPU)."""
import ctypes as C
import os
import subprocess

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))

FLAG_C = r"""
#include <stdio.h>
#include "cvgraft.h"
int main(void)
{
    printf("%d %d %zu\n", CVG_MATCH_CROSS_CHECK, CVG_VERIFY_METHOD_MASK, sizeof(cvg_detect_params));
    return 0;
}
"""


def test_flag_matches_header(tmp_path):
    from computervision_objectdetection_featurematching_b200 import api
    from computervision_objectdetection_featurematching_b200._lib import DetectParams
    src = tmp_path / "flag.c"
    src.write_text(FLAG_C)
    exe = tmp_path / "flag"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           str(src)])
    flag, mask, size = map(int, subprocess.check_output([str(exe)]).split())
    assert flag == api.MATCH_CROSS_CHECK == 0x100
    assert mask == 0xFF and not flag & mask                         # the flag sits above every verify method
    assert size == C.sizeof(DetectParams) == 64


def test_detect_params_sets_the_flag():
    from computervision_objectdetection_featurematching_b200 import api
    for m in (api.VERIFY_HOMOGRAPHY, api.VERIFY_AFFINE, api.VERIFY_AFFINE_PARTIAL):
        assert api.detect_params(method=m).method == m
        p = api.detect_params(method=m, cross_check=True)
        assert p.method == api.MATCH_CROSS_CHECK | m
        assert p.ratio == api.detect_params(method=m).ratio and p.refine_iters == 10
    assert api.detect_params().method == api.VERIFY_HOMOGRAPHY
