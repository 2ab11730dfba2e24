"""The paired (float2) forms of the SFU arithmetic (csrc/fb_math.h, "paired SFU arithmetic"), which the SFU kernels issue
as FFMA2 / FADD2 / FMUL2, against the scalar forms that specify them: every output BIT-EXACT.  Inputs are dense grids
across each saturation and clamp boundary, +-0, subnormals and a few million seeded random floats; the elements are
arranged so that the two lanes of many pairs take different branches."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PHI_LO, PHI_HI, SP_THR = np.float32(8.5e-8), np.float32(16.635532), np.float32(13.942385)


def _probe(ctx, fn, x):
    from fbgnn import _ffi
    dx = ctx.asarray(x)
    dy = ctx.empty(x.shape, np.float32)
    _ffi.call("fbgnn_math_probe", ctx.handle, fn.encode(), dx.ptr, dy.ptr, x.size)
    return dy.numpy()


def _around(c, ulps=4096):
    """float32 values within `ulps` steps of c, both sides."""
    c = np.float32(c)
    if c == 0:
        out = np.arange(0, ulps + 1).astype(np.int32).view(np.float32)
        return np.concatenate([out, -out])
    bits = c.view(np.int32).astype(np.int64) + np.arange(-ulps, ulps + 1)
    return bits.astype(np.int32).view(np.float32)


def _specials():
    sub = np.array([1, 2, 3, 0x1234, 0x7fffff], dtype=np.int32).view(np.float32)
    return np.concatenate([np.float32([0.0, -0.0]), sub, -sub, np.finfo(np.float32).tiny * np.float32([1, -1])])


def _inputs(grids, random, seed):
    """Grids + specials + random values, shuffled, then interleaved with a second shuffle so that adjacent elements
    (the two lanes of one paired call) come from independent draws."""
    rng = np.random.default_rng(seed)
    x = np.concatenate([*(g.astype(np.float32) for g in grids), _specials(), random(rng).astype(np.float32)])
    a, b = rng.permutation(x), rng.permutation(x)
    out = np.empty(2 * x.size, np.float32)
    out[0::2], out[1::2] = a, b
    return out


N = 2_000_000
CASES = {
    "exp2s": ("sfu_exp2s", [_around(0.0), _around(1.0), _around(-80.0), _around(80.0)],
              lambda r: r.uniform(-86, 86, N)),
    "phi_open": ("sfu_phi_open", [_around(PHI_LO), _around(PHI_HI), _around(SP_THR), np.linspace(1e-8, 30, 20001)],
                 lambda r: np.exp(r.uniform(np.log(1e-9), np.log(80), N))),
    "softplus": ("sfu_softplus", [_around(SP_THR), _around(-SP_THR), _around(86.0), _around(-86.0), _around(0.0)],
                 lambda r: r.uniform(-110, 110, N)),
    "tanh": ("sfu_tanh", [_around(10.0), _around(-10.0), _around(0.0), np.linspace(-12, 12, 20001)],
             lambda r: r.uniform(-20, 20, N)),
    # two-argument forms: the probe pairs element i with element n-1-i (and i + n/3, i + 2n/3 for vn_msg)
    "logaddexp_open": ("sfu_logaddexp_open", [_around(-17.5), _around(0.0), np.linspace(-20, 0, 20001)],
                       lambda r: np.concatenate([r.uniform(-17.5, 0, N // 2), r.uniform(-60, 60, N // 2)])),
    "vn_corr": ("sfu_vn_corr", [_around(17.5), _around(-17.5), _around(0.0), _around(8.75), _around(-8.75)],
                lambda r: np.concatenate([r.uniform(-20, 20, N // 2), r.uniform(-60, 60, N // 2)])),
    "vn_msg": ("sfu_vn_msg", [_around(0.0), np.linspace(-30, 30, 20001)],
               lambda r: r.uniform(-60, 60, N)),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_paired_form_matches_scalar(name):
    import fbgnn as F
    import test_gpu_parity as P
    scalar, grids, random = CASES[name]
    ctx = F.default_context()
    x = _inputs(grids, random, seed=sorted(CASES).index(name) + 1)
    P.assert_bitexact(_probe(ctx, "sfu2_" + name, x), _probe(ctx, scalar, x), name)
    # an odd count: the last element is evaluated as a pair with itself
    P.assert_bitexact(_probe(ctx, "sfu2_" + name, x[:1001]), _probe(ctx, scalar, x[:1001]), name + " (odd n)")


def test_lanes_take_different_branches():
    """The interleaving puts saturated and unsaturated arguments into the same pair, which the bit comparison above
    then covers for every pair."""
    x = _inputs(CASES["phi_open"][1], CASES["phi_open"][2], seed=1)
    lo, hi = x[0::2], x[1::2]
    sat_lo = (lo <= PHI_LO) | (lo >= PHI_HI)
    sat_hi = (hi <= PHI_LO) | (hi >= PHI_HI)
    assert np.count_nonzero(sat_lo != sat_hi) > 10000
    y = _inputs(CASES["softplus"][1], CASES["softplus"][2], seed=2)
    assert np.count_nonzero((y[0::2] > SP_THR) != (y[1::2] > SP_THR)) > 10000
