"""CPU: the configuration surface of ELLC_ARITH_REFERENCE.  ellc_create validates it before it looks for a device, so every
rejected combination returns ELLC_ERR_INVALID (-1) here too."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi as m
    return m


def test_constants_and_defaults(capi):
    assert capi.ARITH_FAST == 0 and capi.ARITH_STRICT == 1 and capi.ARITH_REFERENCE == 2
    cfg = capi.default_config(480, 270)
    assert cfg.lc_bands == 2                                   # FLAG_DO_PARALLEL_CONST_WEIGHT_POSE_EST, as the lc_* fixture was made
    assert capi.default_config(480, 270, lc_bands=1, arithmetic=capi.ARITH_REFERENCE).lc_bands == 1


@pytest.mark.parametrize("over", [
    dict(arithmetic=2, jacobian_at_warped=1),
    dict(arithmetic=2, lm_lambda=0.1),
    dict(arithmetic=2, ctas_per_pair=2),
    dict(arithmetic=2, ctas_per_pair=4),
    dict(arithmetic=2, pairs_per_cta=2),
    dict(arithmetic=2, lc_bands=0),
    dict(arithmetic=2, lc_bands=3),
    dict(arithmetic=3),
    dict(arithmetic=-1),
])
def test_invalid_reference_configs_rejected(capi, over):
    h = C.c_void_p()
    cfg = capi.default_config(480, 270, **over)
    assert capi.lib().ellc_create(C.byref(cfg), C.byref(h)) == -1
    assert not h.value


@pytest.mark.parametrize("over", [dict(), dict(ctas_per_pair=1, pairs_per_cta=1, lc_bands=1)])
def test_valid_reference_configs_pass_validation(capi, over):
    """Accepted combinations get as far as the device probe: -1 would be a validation failure, -2 is "no device"."""
    h = C.c_void_p()
    cfg = capi.default_config(480, 270, arithmetic=capi.ARITH_REFERENCE, **over)
    rc = capi.lib().ellc_create(C.byref(cfg), C.byref(h))
    assert rc in (0, -2)
    if rc == 0:
        capi.lib().ellc_destroy(h)
