"""cvg_detect_params as a C compiler lays it out (include/cvgraft.h) against the ctypes mirror in _lib.py, and the defaults
cvg_detect_params_default hands out (the library loads without a GPU)."""
import ctypes as C
import os
import subprocess

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))

LAYOUT_C = r"""
#include <stdio.h>
#include <stddef.h>
#include "cvgraft.h"
int main(void)
{
    printf("%zu %zu %zu %d %d %d\n", sizeof(cvg_detect_params), offsetof(cvg_detect_params, method),
           offsetof(cvg_detect_params, refine_iters), CVG_VERIFY_HOMOGRAPHY, CVG_VERIFY_AFFINE, CVG_VERIFY_AFFINE_PARTIAL);
    return 0;
}
"""


def test_detect_params_layout_matches_ctypes(tmp_path):
    from computervision_objectdetection_featurematching_b200 import api
    from computervision_objectdetection_featurematching_b200._lib import DetectParams
    src = tmp_path / "layout.c"
    src.write_text(LAYOUT_C)
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                           str(src)])
    size, off_method, off_refine, hom, aff, part = map(int, subprocess.check_output([str(exe)]).split())
    assert size == C.sizeof(DetectParams) == 64
    assert off_method == DetectParams.method.offset == 56                  # the layout before `method`: 56 bytes
    assert off_refine == DetectParams.refine_iters.offset == 60
    assert (hom, aff, part) == (api.VERIFY_HOMOGRAPHY, api.VERIFY_AFFINE, api.VERIFY_AFFINE_PARTIAL) == (0, 1, 2)


def test_detect_params_defaults():
    from computervision_objectdetection_featurematching_b200 import api
    p = api.detect_params()
    assert p.size == 64 and p.method == api.VERIFY_HOMOGRAPHY and p.refine_iters == 10
    assert p.ransac.threshold == 5.0 and p.ransac.max_iters == 2000 and p.ransac.confidence == 0.995 and p.ransac.flags == 0
    q = api.detect_params(method=api.VERIFY_AFFINE_PARTIAL, refine_iters=3, ransac=api.ransac_params(3.0, 2000, 0.99))
    assert q.method == 2 and q.refine_iters == 3 and q.ransac.threshold == 3.0 and q.ransac.confidence == 0.99
