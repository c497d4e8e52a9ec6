"""Multi-VAE (daisy/model/VAECFRecommender.py) restated in numpy fp64, with the dropout masks and the reparameterisation
noise as inputs.  The parameter block is packed in module-registration order with the encoder.0 weight transposed to
[item_num, h_1], as the device stores it but without the device's alignment padding (from_device / to_device convert).
TEST INFRASTRUCTURE: the GPU tests and bench compare the kernels against it; tests/test_vae_oracle.py pins it against the
reference's own runs (tests/golden/vae.npz)."""
import numpy as np


def rating_matrix(hid, hval, item_num):
    """get_user_rating_matrix: index_put_ of the padded history, written column by column -> the last write to a cell wins
    (the (0, 0.0) padding erases item 0 from every shorter row)."""
    hid = np.asarray(hid, np.int64)
    hval = np.asarray(hval, np.float32)
    R = np.zeros((hid.shape[0], item_num), np.float32)
    rows = np.arange(hid.shape[0])
    for j in range(hid.shape[1]):
        R[rows, hid[:, j]] = hval[:, j]
    return R


def dims(item_num, hidden, lat):
    E = [item_num] + list(hidden) + [lat]
    D = [lat // 2] + E[::-1][1:]
    return E, D


def _sizes(item_num, hidden, lat):
    """Sizes of the block's parts in order: (weight, bias) per encoder Linear, then per decoder Linear."""
    E, D = dims(item_num, hidden, lat)
    out = []
    for ds in (E, D):
        for a, b in zip(ds[:-1], ds[1:]):
            out += [a * b, b]
    return out


def from_device(net, item_num, hidden, lat):
    """The device block (every part zero-padded to a multiple of 4 floats) -> the packed layout used here."""
    net = np.asarray(net)
    parts, o = [], 0
    for n in _sizes(item_num, hidden, lat):
        parts.append(net[o:o + n])
        o += -(-n // 4) * 4
    return np.concatenate(parts)


def to_device(flat, item_num, hidden, lat):
    """The packed layout -> the device block (zero padding after every part)."""
    flat = np.asarray(flat)
    parts, o = [], 0
    for n in _sizes(item_num, hidden, lat):
        parts += [flat[o:o + n], np.zeros((-n) % 4, flat.dtype)]
        o += n
    return np.concatenate(parts)


def unpack(net, item_num, hidden, lat):
    """flat block -> ([(W [out, in], b)] encoder, [...] decoder), fp64."""
    E, D = dims(item_num, hidden, lat)
    net = np.asarray(net, np.float64)
    out, o = [], 0
    for side, ds in ((0, E), (1, D)):
        layers = []
        for k, (a, b) in enumerate(zip(ds[:-1], ds[1:])):
            w = net[o:o + a * b]
            W = w.reshape(a, b).T if (side == 0 and k == 0) else w.reshape(b, a)
            o += a * b
            layers.append((W, net[o:o + b].copy()))
            o += b
        out.append(layers)
    return out[0], out[1]


def pack(enc, dec):
    parts = []
    for k, (W, b) in enumerate(enc):
        parts += [(W.T if k == 0 else W).reshape(-1), b]
    for W, b in dec:
        parts += [W.reshape(-1), b]
    return np.concatenate(parts)


def anneal(update, cap, total):
    return min(cap, 1.0 * update / total) if total > 0 else cap


def loss_grad(net, R, item_num, hidden, lat, dropout=0.0, mask=None, eps=None, ann=0.2, training=True, want_grad=True):
    """loss (float) and the gradient of the flat block (fp64) for one batch.  mask: [B, item_num] keep (0/1), eps [B, lat//2]."""
    enc, dec = unpack(net, item_num, hidden, lat)
    R = np.asarray(R, np.float64)
    B = R.shape[0]
    half, lvo = lat // 2, lat - lat // 2
    denom = np.maximum(np.sqrt((R * R).sum(1)), 1e-12)
    x0 = R / denom[:, None]
    if training and dropout > 0:
        x0 = x0 * mask / (1 - dropout)
    acts = [x0]
    h = x0
    for k, (W, b) in enumerate(enc):
        h = h @ W.T + b
        if k < len(enc) - 1:
            h = np.tanh(h)
        acts.append(h)
    mu, lv = h[:, :half], h[:, lvo:]
    std = np.exp(0.5 * lv)
    z = eps * std + mu if training else mu.copy()
    dacts = [z]
    y = z
    for k, (W, b) in enumerate(dec):
        y = y @ W.T + b
        if k < len(dec) - 1:
            y = np.tanh(y)
        dacts.append(y)
    logits = y
    m = logits.max(1, keepdims=True)
    lse = m[:, 0] + np.log(np.exp(logits - m).sum(1))
    ce = -((logits - lse[:, None]) * R).sum(1).mean()
    kl = -0.5 * np.mean(np.sum(1 + lv - mu ** 2 - np.exp(lv), 1)) * ann
    loss = ce + kl
    if not want_grad:
        return loss, None
    S = R.sum(1)
    sm = np.exp(logits - lse[:, None])
    g = (sm * S[:, None] - R) / B
    gdec = [None] * len(dec)
    for k in range(len(dec) - 1, -1, -1):
        W, _ = dec[k]
        if k < len(dec) - 1:
            g = g * (1 - dacts[k + 1] ** 2)
        gdec[k] = (g.T @ dacts[k], g.sum(0))
        g = g @ W
    dz = g
    c = ann / B
    dh = np.zeros((B, lat))
    dh[:, :half] = dz + c * mu
    dh[:, lvo:] = (dz * eps * 0.5 * std if training else 0.0) + 0.5 * c * (np.exp(lv) - 1)
    g = dh
    genc = [None] * len(enc)
    for k in range(len(enc) - 1, -1, -1):
        W, _ = enc[k]
        if k < len(enc) - 1:
            g = g * (1 - acts[k + 1] ** 2)
        genc[k] = (g.T @ acts[k], g.sum(0))
        g = g @ W
    return loss, pack(genc, gdec)


def step(net, grad, opt, lr, state, t, beta1=0.9, beta2=0.999, eps=1e-8):
    """SGD, or torch.optim.Adam's single-tensor rule, step number t (1-based), on the flat block (fp64)."""
    net = np.asarray(net, np.float64)
    if opt == 'sgd':
        return net - lr * grad
    m = state.get('m', np.zeros_like(net))
    v = state.get('v', np.zeros_like(net))
    m = beta1 * m + (1 - beta1) * grad
    v = beta2 * v + (1 - beta2) * grad * grad
    state['m'], state['v'] = m, v
    return net - lr / (1 - beta1 ** t) * m / (np.sqrt(v) / np.sqrt(1 - beta2 ** t) + eps)
