"""Error bounds of the spec exp and sigmoid (DESIGN.md section 4), measured on every fp32 input by tests/test_gpu_spec_math.py.

Errors are in units of the fp32 ulp of the float64 reference value (2^-149 where that value is subnormal)."""
import numpy as np

EXP_MAX_ULP = 1.0104        # exp, wherever the result is finite (measured: 1.010350 at x = -5.8778844)
SIG_MAX_ULP = 2.4808        # sigmoid, wherever the reference is a normal float (measured: 2.480738 at x = -16.635704, where
                            # 1 + exp(-x) lies just above 2^24 and its reciprocal just below 2^-24: one ulp of the sum is two
                            # of the quotient)

# sigmoid(x) = 1 / (1 + exp(-x)) is exactly +0 for x <= SIG_ZERO_EDGE: exp(-x) overflows to +inf there, although the true value is
# a subnormal near 1e-39 (from 2.9e-39 at the edge down to 2^-149 at x = -103.28).  The literal formula, not a defect.
SIG_ZERO_EDGE = np.uint32(0xC2B17218).view(np.float32)      # -88.72284
