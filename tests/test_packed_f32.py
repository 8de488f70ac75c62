import pytest


@pytest.mark.gpu
def test_packed_f32_pairs_selftest():
    """both halves of the packed f32 pairs (fma / add / mul .rn.f32x2) the carve's filter and box classifier run on ==
    the scalar IEEE operations, bit for bit (NaN-ness for a NaN), over 2^31 cases of 3 x 2 operations: random bit
    patterns, denormal-range exponents, cancellation c = -RN(a b), and +-0 / +-inf / NaN / denormal specials"""
    from ar_voxel_project_b200.engine import selftest
    bad, checked = selftest(2, 1 << 31, seed=12347)
    assert checked == 6 * (1 << 31) and bad == 0, (bad, checked)
