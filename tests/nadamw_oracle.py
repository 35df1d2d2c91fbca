"""Test-only numpy restatement of torch.optim.NAdam(decoupled_weight_decay=True) at one step, the update of
stgcn_nadamw_step: float32 arrays and a float32 momentum-cache product ``mu_product``, the step scalars in Python floats
(fp64), as torch's _single_tensor_nadam computes them.  Pinned against torch itself by test_nadamw_oracle.py."""
import numpy as np


def nadamw_step(p, g, m, v, mu_product, t, lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                momentum_decay=4e-3):
    """One step t (1-based).  Returns (p, m, v, mu_product), all float32."""
    f32 = np.float32
    b1, b2 = betas
    p, g, m, v = (np.asarray(a, np.float32) for a in (p, g, m, v))
    p = p * f32(1.0 - lr * weight_decay)
    mu = b1 * (1.0 - 0.5 * 0.96 ** (t * momentum_decay))
    mu_next = b1 * (1.0 - 0.5 * 0.96 ** ((t + 1) * momentum_decay))
    mu_product = f32(f32(mu_product) * f32(mu))
    m = m + f32(1.0 - b1) * (g - m)
    v = v * f32(b2) + f32(1.0 - b2) * g * g
    denom = np.sqrt(v / f32(1.0 - b2 ** t)) + f32(eps)
    c_g = -lr * (1.0 - mu) / (1.0 - float(mu_product))
    c_m = -lr * mu_next / (1.0 - float(mu_product) * mu_next)
    p = p + f32(c_g) * g / denom
    p = p + f32(c_m) * m / denom
    return p, m, v, mu_product
