"""Float64 reference of the input gradients (mrgan_input_grad): the oracle's phase-0 discriminator forward, the seed
e_t - softmax(l) at the logits, and its backward pass down to the input."""
import numpy as np

from oracle import gan_oracle as O


def input_grad(pD, x, target=None, alpha=0.0):
    """d log softmax(l(x))[t] / dx, float64 [n, D]; target None = each row's first maximal logit."""
    pD = [np.asarray(p, dtype=np.float64) for p in pD]
    logits, cache = O.disc_forward(pD, np.asarray(x, dtype=np.float64), None, alpha=alpha)
    t = np.argmax(logits, axis=1) if target is None else np.asarray(target)
    e = np.exp(logits - logits.max(axis=1, keepdims=True))
    seed = -e / e.sum(axis=1, keepdims=True)
    seed[np.arange(len(t)), t] += 1.0
    return O.disc_backward(pD, cache, seed, need_dx=True)[1]


def log_prob(pD, x, t, alpha=0.0):
    """log softmax(l(x))[t] per row, float64 (for finite differences)."""
    logits = O.disc_forward(pD, x, None, alpha=alpha)[0]
    m = logits.max(axis=1, keepdims=True)
    lse = (m + np.log(np.exp(logits - m).sum(axis=1, keepdims=True)))[:, 0]
    return logits[np.arange(len(t)), t] - lse
