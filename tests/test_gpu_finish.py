"""The warp-cooperative 9x9 eigen-solves of the refit/LM kernel against the serial ones, on the device."""
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from computervision_objectdetection_featurematching_b200 import api
    c = api.Context(0)
    yield c
    c.close()


def test_selftest_warp_jacobi_bit_identical(ctx):
    """jacobi9_warp, solve_eig9_warp and invert_eig_max_diag9_warp against jacobi<9>, solve_eig<9> and
    invert_eig_max_diag<9> on 10 240 seeded matrices (LtL of 4-point samples, DLT systems of 5..4000 points, LM's
    A + lambda D, small-integer matrices with tied pivot candidates, zeros in the upper triangle): 0 differing doubles."""
    assert ctx.selftest(1) == 0


def test_selftest_rejects_unknown_test(ctx):
    from computervision_objectdetection_featurematching_b200 import api
    with pytest.raises(api.CvgError):
        ctx.selftest(2)
