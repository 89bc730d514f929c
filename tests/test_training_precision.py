"""CPU: the arithmetic of riser_conv1d_wgrad_cl (csrc/train.cu) emulated in float64 -- operands split into bf16 hi + lo
planes, the three products hi*hi + hi*lo + lo*hi -- against the exact weight gradient, at the error measure the GPU
test (tests/test_gpu_training.py) bounds: max |dW - exact| / S with S = sum |dZ| |X|.  It shows that the bar BETA
has room over the three-product format and that dropping the lo planes (one bf16 pass) would not meet it."""
import numpy as np

from tests.test_gpu_training import BETA


def _bf16(a):
    """Round float32 values to bf16 (nearest even), returned as float64."""
    u = np.asarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).astype(np.float64)


def _split(a):
    hi = _bf16(a)
    lo = _bf16((a.astype(np.float64) - hi).astype(np.float32))
    return hi, lo


def _ratio(rows=1024, cin=24, cout=16, seed=0):
    rng = np.random.default_rng(seed)
    dz = (rng.standard_normal((rows, cout)) * np.exp(rng.uniform(-8, 8, (rows, 1)))).astype(np.float32)
    x = np.maximum(rng.standard_normal((rows, cin)), 0).astype(np.float32)
    exact = dz.astype(np.float64).T @ x.astype(np.float64)
    s = np.abs(dz.astype(np.float64)).T @ np.abs(x.astype(np.float64))
    (ah, al), (bh, bl) = _split(dz), _split(x)
    three = ah.T @ bh + ah.T @ bl + al.T @ bh
    one = ah.T @ bh
    return np.max(np.abs(three - exact) / s), np.max(np.abs(one - exact) / s)


def test_three_products_meet_beta_and_one_does_not():
    r3, r1 = _ratio()
    print(f"emulated max |err| / S: three products {r3:.2e}, hi only {r1:.2e}, beta {BETA:.1e}")
    assert r3 <= BETA / 4
    assert r1 >= 4 * BETA
