"""Constant folds of the step kernel's control loop that must not change a single result bit (fpv_step_kernel.cuh).

The strict build rounds every multiply and add of the reference's torch expressions separately, so a fold of two constants is
only allowed where it gives the same float32 for every input the kernel can feed it.  Each fold is checked here over its whole
input domain, as numpy float32 (round to nearest even, subnormals kept, like the -fmad=false build) against the unfolded form."""
import numpy as np

_CHUNK = 1 << 26


def _all_floats():
    """Every float32 bit pattern, in chunks: +-0, subnormals, normals, +-inf and the NaNs."""
    base = np.arange(_CHUNK, dtype=np.uint32)
    for lo in range(0, 1 << 32, _CHUNK):
        yield (base + np.uint32(lo)).view(np.float32)


def test_rotor_speed_times_two_pi():
    """om * 2 * pi == om * (2 pi) for every float om (mechanical power, fpv_asymmetry.py:614): om * 2 is exact (a subnormal
    doubles exactly; an overflow gives inf on both sides) and 2 * float32(pi) is exact, so both sides round the same real product
    once.  The rotor speeds are unbounded state (a reset may load any value), so the domain is all of float32."""
    two, pi = np.float32(2.0), np.float32(np.pi)
    two_pi = np.float32(6.28318530717958647692)
    assert two_pi == two * pi
    with np.errstate(over="ignore", invalid="ignore"):
        for om in _all_floats():
            a = (om * two) * pi
            b = om * two_pi
            same = (a.view(np.uint32) == b.view(np.uint32)) | ((a != a) & (b != b))
            assert same.all(), om[~same][:4]
