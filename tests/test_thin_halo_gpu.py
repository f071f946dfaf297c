"""GPU parity of the compact thin halo (CisConv.thin: <= 16 input channels staged as 16-byte-per-pixel planes, x-adjacent 8-channel
taps paired in one K=16 MMA, stride-2 layers as four space-to-depth phases) at the shapes of the benchmarked step, against the same
fp32 reference and tolerance as tests/test_conv_engine_gpu.py."""
import pytest

from convref import run_conv_case
from unsupervised_detection_b200._lib import ACT_ELU, ACT_LEAKY

pytestmark = pytest.mark.gpu

THIN_CASES = [
    dict(N=12, H=256, W=448, cins=[8], cout=32, k=7, stride=2, act=ACT_ELU, bn=True),          # recover conv1 (3B, B = 4)
    dict(N=4, H=256, W=448, cins=[8], cout=32, k=5, act=ACT_ELU, bn=True),                     # generator conv1
    dict(N=2, H=384, W=640, cins=[3], cout=16, k=3, stride=2, act=ACT_LEAKY, alpha=0.1, backward=False),   # PWC-Net first layer
    dict(N=2, H=192, W=320, cins=[16], cout=16, k=3, act=ACT_LEAKY, alpha=0.1),
    dict(N=2, H=64, W=96, cins=[32], cout=16, k=3, stride=2, act=ACT_LEAKY),                   # grouped-parity dgrad, 16-ch gradient
    dict(N=3, H=37, W=29, cins=[8], cout=16, k=3),                                            # odd taps per row, ragged last tiles
    dict(N=2, H=40, W=52, cins=[8, 8], cout=32, k=5, act=ACT_ELU, bn=True),                    # two 8-channel sources = two planes
    dict(N=2, H=33, W=47, cins=[16], cout=16, k=4, stride=2, act=ACT_LEAKY),                   # even kernel, stride 2
]


@pytest.mark.parametrize('case', THIN_CASES, ids=lambda c: 'k%d_s%d_c%s_o%d_%dx%d' % (c['k'], c.get('stride', 1), '+'.join(map(str, c['cins'])),
                                                                                      c['cout'], c['H'], c['W']))
def test_thin_halo_conv(case):
    r = run_conv_case(**case)
    tol = lambda ref: 2 ** -7 * ref + 1e-3
    assert r['fwd_err'] <= tol(r['fwd_ref']), r
    if 'dx_err' in r:
        assert r['dx_err'] <= tol(r['dx_ref']), r
        assert r['dw_err'] <= 2 ** -7 * r['dw_ref'] + 1e-3, r
        assert r['db_err'] <= 2 ** -7 * r['db_ref'] + 1e-3, r


@pytest.mark.parametrize('case', [THIN_CASES[1], THIN_CASES[3], THIN_CASES[5]], ids=['k5_c8', 'k3_c16', 'k3_c8_ragged'])
def test_thin_halo_persistent_kernel(case):
    """The persistent weight-resident kernel on the compact halo (persist mode 3): bit-identical to the one-tile-per-CTA kernel."""
    from unsupervised_detection_b200 import _lib
    case = dict(case, backward=False)
    r0 = run_conv_case(**case)
    _lib.load().cis_set_persist_mode(3)
    try:
        r = run_conv_case(**case)
    finally:
        _lib.load().cis_set_persist_mode(-1)
    assert r['fwd_err'] <= 2 ** -7 * r['fwd_ref'] + 1e-3, r
    assert r['fwd_err'] == r0['fwd_err']
