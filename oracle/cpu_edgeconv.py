"""Float64 reference of one EdgeConv layer in training and eval mode (models/dgcnn_util.py:114-126: get_graph_feature ->
Conv2d(2C, Co, 1, bias=False) -> BatchNorm2d -> LeakyReLU -> max over the k neighbours), forward and backward, in numpy.
No build step.  Two entry points:

  layer_x  the layer from x (B,C,N), idx (B,N,k) and the weight W (Co,2C): y = W [x_j - x_i; x_i] per edge, batch
           statistics (biased) and running buffers like nn.BatchNorm2d, the output, the selected slot and its margin,
           and dx, dW, dgamma, dbeta with torch's LeakyReLU derivative (x > 0 ? 1 : slope).
  layer_z  the same layer from the fp32 point-major product z = [P | Q] (B,N,ld >= 2co) the GPU forms: y = P[idx] + Q
           (exact in float64), slot selection by the kernels' rule on fp32 sgn * P, everything else float64; returns
           what the kernel entry points expose (statistics, s1, out, jstar, dz, dgamma, dbeta) plus error bounds.

Selection rule of both: ext = max over the k slots where the folded scale gamma * invstd >= 0 (so gamma = -0.0 takes the
max) and min where it is < 0, the lowest slot on ties.  The margin of a selection is its distance to the best slot that
names ANOTHER point (inf when all k slots name one point): duplicates of the selected point cannot change any gradient.
Memory stays at one cloud's (N,k,Co) edge tensor at a time."""
import numpy as np

EPS32 = float(np.finfo(np.float32).eps)
f64 = np.float64


def _act(v, slope):
    return np.where(v >= 0, v, v * slope)


def _dact(v, slope):
    return np.where(v > 0, 1.0, slope)  # torch: leaky_relu'(0) = slope


def _select(key, idx_b):
    """key (N,k,Co): per (i,o) the first slot of the maximum, and the margin to the best slot naming another point"""
    js = np.argmax(key, axis=1)  # first occurrence
    best = np.take_along_axis(key, js[:, None, :], axis=1)[:, 0, :]
    sel_pt = np.take_along_axis(np.broadcast_to(idx_b[:, :, None], key.shape), js[:, None, :], axis=1)
    other = np.where(idx_b[:, :, None] == sel_pt, -np.inf, key)
    alt = np.argmax(other, axis=1)
    margin = best - np.take_along_axis(other, alt[:, None, :], axis=1)[:, 0, :]
    return js, alt, margin


def _running(mean, var, m, running_mean, running_var, momentum, nbt):
    nbt = nbt + 1
    mom = 1.0 / nbt if momentum is None else momentum
    rm = (1 - mom) * np.asarray(running_mean, f64) + mom * mean
    rv = (1 - mom) * np.asarray(running_var, f64) + mom * var * (m / max(m - 1, 1))
    return rm, rv, nbt


def layer_x(x, idx, w, gamma=None, beta=None, running_mean=None, running_var=None, num_batches_tracked=0, momentum=0.1,
            eps=1e-5, slope=0.2, train=True, g=None, kc=8.0, rho=1e-5):
    """x (B,C,N), idx (B,N,k), w (Co,2C); gamma / beta None = affine=False; running_* None = track_running_stats=False
    (batch statistics in both modes, like nn.BatchNorm2d); momentum None = cumulative average.  g (B,Co,N) upstream
    gradient or None.  Returns a dict of float64 arrays.

    Bounds for an fp32 evaluation through z = [P | Q]: P and Q carry kc * eps * (|W1| |x| and |W2 - W1| |x|) of
    rounding, the batch statistics a relative error rho.  A selection whose margin is below the rounding of its two
    candidates is 'ambiguous' (count in 'ambiguous'): the bounds of out and of every gradient entry it reaches include the
    size of the flip to the other candidate.  *_bound hold the bounds, propagated through the absolute values of every
    term, plus rho of those absolute values for the fp32 sums."""
    x = np.asarray(x, f64)
    idx = np.asarray(idx, np.int64)
    w = np.asarray(w, f64)
    b, c, n = x.shape
    k = idx.shape[2]
    co = w.shape[0]
    w1, w2 = w[:, :c], w[:, c:]
    ga = np.ones(co) if gamma is None else np.asarray(gamma, f64)
    be = np.zeros(co) if beta is None else np.asarray(beta, f64)
    m = float(b * n * k)
    xt = np.ascontiguousarray(x.transpose(0, 2, 1))

    def edges(bi):  # y (N,k,Co) = W [x_j - x_i; x_i]
        xi = xt[bi]
        d = xi[idx[bi]] - xi[:, None, :]
        return (d.reshape(n * k, c) @ w1.T).reshape(n, k, co) + (xi @ w2.T)[:, None, :]

    r = {}
    batch = train or running_mean is None
    if batch:
        s = sum(edges(bi).sum(axis=(0, 1)) for bi in range(b))
        mean = s / m
        var = sum(((edges(bi) - mean) ** 2).sum(axis=(0, 1)) for bi in range(b)) / m
        if train and running_mean is not None:
            r["running_mean"], r["running_var"], r["num_batches_tracked"] = _running(
                mean, var, m, running_mean, running_var, momentum, num_batches_tracked)
    else:
        mean, var = np.asarray(running_mean, f64), np.asarray(running_var, f64)
    invstd = 1.0 / np.sqrt(var + eps)
    scale = ga * invstd
    r.update(mean=mean, var=var, invstd=invstd)
    up = scale >= 0
    out = np.empty((b, co, n))
    jstar = np.empty((b, n, co), np.int64)
    alt = np.empty((b, n, co), np.int64)
    margin = np.empty((b, n, co))
    yhat_sel = np.empty((b, n, co))
    for bi in range(b):
        y = edges(bi)
        js, al, mg = _select(np.where(up, y, -y), idx[bi])
        ys = np.take_along_axis(y, js[:, None, :], axis=1)[:, 0, :]
        yhat_sel[bi] = (ys - mean) * invstd
        out[bi] = _act(ga * yhat_sel[bi] + be, slope).T
        jstar[bi], alt[bi], margin[bi] = js, al, mg
    ax = np.abs(xt)
    mag_p, mag_q = ax @ np.abs(w1).T, ax @ np.abs(w2 - w1).T  # (B,N,Co)
    pick = lambda a, j: np.stack([np.take_along_axis(a[bi][idx[bi]], j[bi][:, None, :], axis=1)[:, 0, :]  # noqa: E731
                                  for bi in range(b)])
    ry = kc * EPS32 * (pick(mag_p, jstar) + pick(mag_p, alt) + mag_q)  # y's rounding at either candidate
    r["mean_round"] = kc * EPS32 * (mag_p.max(axis=(0, 1)) + mag_q.max(axis=(0, 1)))  # the batch mean's share of it
    amb = margin < ry
    yerr = ry * invstd + rho * (np.abs(yhat_sel) + 1.0)  # error of yhat at the selected edge
    bn_sel = ga * yhat_sel + be
    out_bound = np.abs(ga) * (yerr + np.where(amb, margin * invstd, 0.0)) + rho * np.abs(be) + EPS32 * np.abs(bn_sel)
    r.update(out=out, jstar=jstar, alt=alt, margin=margin, ambiguous=int(amb.sum()), out_bound=out_bound.transpose(0, 2, 1))
    if g is None:
        return r
    g = np.asarray(g, f64).transpose(0, 2, 1)  # (B,N,Co)
    dbn = g * _dact(bn_sel, slope)
    dbeta = dbn.sum(axis=(0, 1))
    dgamma = (dbn * yhat_sel).sum(axis=(0, 1))
    # the activation's derivative may differ where bn is within its error of 0
    flip = np.where(np.abs(bn_sel) <= np.abs(ga) * yerr + rho * np.abs(be) + EPS32, np.abs(g) * abs(1 - slope), 0.0)
    dbeta_b = (flip + rho * np.abs(dbn)).sum(axis=(0, 1))
    dgamma_b = (flip * np.abs(yhat_sel) + np.abs(dbn) * yerr + rho * np.abs(dbn * yhat_sel)).sum(axis=(0, 1))
    dw_b = np.zeros((co, 2 * c))
    dx_b = np.zeros((b, n, c))
    dw1 = np.zeros((co, c))
    dw2 = np.zeros((co, c))
    dxt = np.zeros((b, n, c))
    for bi in range(b):
        onehot = np.zeros((n, k, co))
        np.put_along_axis(onehot, jstar[bi][:, None, :], 1.0, axis=1)
        dy = onehot * dbn[bi][:, None, :]
        if batch:
            yh = (edges(bi) - mean) * invstd
            dy = dy - dbeta / m - yh * (dgamma / m)
        dy = dy * (ga * invstd)
        # error of every edge's dy: the terms' absolute values times rho, the per-channel terms' bounds, yhat's rounding;
        # an ambiguous selection may move its term to the other candidate's slot
        gi = np.abs(ga * invstd)
        sel_abs = gi * np.abs(dbn[bi])
        e = np.zeros((n, k, co))  # error of dy, then rho of its terms' absolute values
        np.put_along_axis(e, jstar[bi][:, None, :], (gi * flip[bi] + rho * sel_abs)[:, None, :], axis=1)
        amb_add = np.where(amb[bi], sel_abs + gi * flip[bi], 0.0)[:, None, :]
        for js in (alt[bi], jstar[bi]):
            np.put_along_axis(e, js[:, None, :], np.take_along_axis(e, js[:, None, :], axis=1) + amb_add, axis=1)
        if batch:
            yh_abs = np.abs(yh)
            yh_err = kc * EPS32 * (mag_p[bi][idx[bi]] + mag_q[bi][:, None, :]) * invstd + rho * (yh_abs + 1.0)
            e += gi * ((rho * np.abs(dbeta) + dbeta_b) / m + (rho * np.abs(dgamma) + dgamma_b) / m * yh_abs
                       + np.abs(dgamma) / m * yh_err)
        xi = xt[bi]
        d = xi[idx[bi]] - xi[:, None, :]
        dyr = dy.reshape(n * k, co)
        dw1 += dyr.T @ d.reshape(n * k, c)
        dsum = dy.sum(axis=1)
        dw2 += dsum.T @ xi
        np.add.at(dxt[bi], idx[bi].reshape(-1), dyr @ w1)
        dxt[bi] += dsum @ (w2 - w1)
        er, esum = e.reshape(n * k, co), e.sum(axis=1)
        dw_b[:, :c] += er.T @ np.abs(d).reshape(n * k, c)
        dw_b[:, c:] += esum.T @ np.abs(xi)
        np.add.at(dx_b[bi], idx[bi].reshape(-1), er @ np.abs(w1))
        dx_b[bi] += esum @ np.abs(w2 - w1)
    r.update(dx=dxt.transpose(0, 2, 1), dw=np.concatenate([dw1, dw2], axis=1), dgamma=dgamma, dbeta=dbeta,
             dx_bound=dx_b.transpose(0, 2, 1), dw_bound=dw_b, dgamma_bound=dgamma_b, dbeta_bound=dbeta_b)
    return r


# ---------------------------------------------------------------------------------------------------------------- z-level
def _pq(z, co):
    z = np.asarray(z)
    assert z.dtype == np.float32 and z.shape[2] >= 2 * co
    return z[..., :co], z[..., co:2 * co]


def stats_z(z, idx, co):
    """batch mean and biased variance (Co) of y = P[idx] + Q over every edge, float64 two-pass; s1 (B,N,Co) = sum_j P[idx]"""
    p32, q32 = _pq(z, co)
    b, n, k = idx.shape
    m = float(b * n * k)
    s1 = np.stack([p32[bi].astype(f64)[idx[bi]].sum(axis=1) for bi in range(b)])
    mean = (s1 + k * q32.astype(f64)).sum(axis=(0, 1)) / m
    var = sum(((p32[bi].astype(f64)[idx[bi]] + q32[bi].astype(f64)[:, None, :] - mean) ** 2).sum(axis=(0, 1))
              for bi in range(b)) / m
    return mean, var, s1


def forward_z(z, idx, co, scale, shift, slope):
    """out (B,Co,N) float64 from the given fp32 scale / shift, jstar (B,N,Co) uint8 by the kernels' rule on fp32 sgn * P,
    and 'bound' (B,Co,N): the fp32 forward's rounding, 2 eps (|scale| (|P*| + |Q|) + |shift|) + one ulp of the result"""
    p32, q32 = _pq(z, co)
    scale32 = np.asarray(scale, np.float32)
    sgn = np.where(scale32 >= 0, np.float32(1), np.float32(-1))
    sc, sh = scale32.astype(f64), np.asarray(shift, np.float32).astype(f64)
    b, n, k = idx.shape
    out = np.empty((b, co, n))
    bound = np.empty((b, co, n))
    jstar = np.empty((b, n, co), np.uint8)
    for bi in range(b):
        js = np.argmax(p32[bi][idx[bi]] * sgn, axis=1)  # exact in fp32, first slot of the extremum
        ps = np.take_along_axis(p32[bi][idx[bi]], js[:, None, :], axis=1)[:, 0, :].astype(f64)
        q = q32[bi].astype(f64)
        v = sc * (ps + q) + sh
        o = _act(v, slope)
        out[bi] = o.T
        bound[bi] = (2 * EPS32 * (np.abs(sc) * (np.abs(ps) + np.abs(q)) + np.abs(sh)) + EPS32 * np.abs(o)).T
        jstar[bi] = js
    return out, jstar, bound


def backward_z(z, idx, co, jstar, g, scale, shift, mean, invstd, gamma, slope, train):
    """Backward of forward_z with the given fp32 statistics: g (B,N,Co) point-major.  Returns dz (B,N,ld) (dP | dQ, the
    padding columns zero), dgamma, dbeta (float64) and their bounds: fp32 arithmetic with e = eps * (chain length + 8) on
    the sum of the absolute values of every term, where a term's yhat = (P + Q - mean) invstd carries the rounding of
    its fp32 sum, eps (|P| + |Q| + |mean|) invstd."""
    p32, q32 = _pq(z, co)
    ld = z.shape[2]
    b, n, k = idx.shape
    m = float(b * n * k)
    f = lambda a: np.asarray(a, np.float32).astype(f64)  # noqa: E731
    sc, sh, mu, iv, ga = f(scale), f(shift), f(mean), f(invstd), f(gamma)
    g = f(g)
    js = np.asarray(jstar, np.int64)
    dbn = np.empty((b, n, co))
    yh_sel = np.empty((b, n, co))
    ysel_mag = np.empty((b, n, co))
    for bi in range(b):
        pj = p32[bi].astype(f64)[idx[bi]]
        ps = np.take_along_axis(pj, js[bi][:, None, :], axis=1)[:, 0, :]
        q = q32[bi].astype(f64)
        y = ps + q
        dbn[bi] = g[bi] * _dact(sc * y + sh, slope)
        yh_sel[bi] = (y - mu) * iv
        ysel_mag[bi] = (np.abs(ps) + np.abs(q) + np.abs(mu)) * iv
    dbeta = dbn.sum(axis=(0, 1))
    dgamma = (dbn * yh_sel).sum(axis=(0, 1))
    dbeta_b = EPS32 * 8 * np.abs(dbn).sum(axis=(0, 1))
    dgamma_b = EPS32 * 8 * (np.abs(dbn) * (np.abs(yh_sel) + ysel_mag)).sum(axis=(0, 1))
    a_ = ga * dbeta / m if train else np.zeros(co)
    bc = ga * dgamma / m if train else np.zeros(co)
    # the error of A and Bc: their sums' bounds plus one rounding
    a_b = np.abs(ga) * dbeta_b / m + EPS32 * np.abs(a_) if train else np.zeros(co)
    bc_b = np.abs(ga) * dgamma_b / m + EPS32 * np.abs(bc) if train else np.zeros(co)
    dz = np.zeros((b, n, ld))
    bound = np.zeros((b, n, ld))
    for bi in range(b):
        pj = p32[bi].astype(f64)[idx[bi]]  # (N,k,Co)
        q = q32[bi].astype(f64)
        onehot = np.zeros((n, k, co))
        np.put_along_axis(onehot, js[bi][:, None, :], 1.0, axis=1)
        dsel = ga * dbn[bi] * (1.0 if train else iv)  # (N,Co)
        if train:
            yh = (pj + q[:, None, :] - mu) * iv
            yh_mag = (np.abs(pj) + np.abs(q)[:, None, :] + np.abs(mu)) * iv
            dy = iv * (onehot * dsel[:, None, :] - a_ - bc * yh)
            mag = iv * (onehot * np.abs(dsel)[:, None, :] + np.abs(a_) + np.abs(bc) * (np.abs(yh) + yh_mag))
            err = iv * (a_b + bc_b * np.abs(yh))  # from the per-channel terms' own error
        else:
            dy = onehot * dsel[:, None, :]
            mag = onehot * np.abs(dsel)[:, None, :]
            err = np.zeros_like(mag)
        dq = dy.sum(axis=1)
        dq_mag, dq_err = mag.sum(axis=1), err.sum(axis=1)
        dp = np.zeros((n, co))
        dp_mag = np.zeros((n, co))
        dp_err = np.zeros((n, co))
        flat = idx[bi].reshape(-1)
        np.add.at(dp, flat, dy.reshape(n * k, co))
        np.add.at(dp_mag, flat, mag.reshape(n * k, co))
        np.add.at(dp_err, flat, err.reshape(n * k, co))
        deg = np.bincount(flat, minlength=n).astype(f64)[:, None]
        dz[bi, :, :co], dz[bi, :, co:2 * co] = dp, dq
        bound[bi, :, :co] = dp_err + EPS32 * (deg + 8) * dp_mag
        bound[bi, :, co:2 * co] = dq_err + EPS32 * (k + 8) * dq_mag
    return dict(dz=dz, dgamma=dgamma, dbeta=dbeta, dz_bound=bound, dgamma_bound=dgamma_b, dbeta_bound=dbeta_b)


def layer_z(z, idx, co, gamma=None, beta=None, eps=1e-5, slope=0.2, train=True, g=None, running_mean=None,
            running_var=None):
    """The whole layer from fp32 z: float64 statistics (batch statistics when train, else the running buffers), the
    folded scale / shift rounded to fp32 as the kernels use them, forward_z, and backward_z when g (B,N,Co) is given."""
    ga = np.ones(co, np.float32) if gamma is None else np.asarray(gamma, np.float32)
    be = np.zeros(co, np.float32) if beta is None else np.asarray(beta, np.float32)
    mean, var, s1 = stats_z(z, idx, co)
    if not train:
        mean, var = np.asarray(running_mean, f64), np.asarray(running_var, f64)
    invstd = 1.0 / np.sqrt(var + eps)
    mean32, invstd32 = mean.astype(np.float32), invstd.astype(np.float32)
    scale32 = (ga * invstd32).astype(np.float32)
    shift32 = (be - scale32 * mean32).astype(np.float32)
    out, jstar, out_bound = forward_z(z, idx, co, scale32, shift32, slope)
    r = dict(mean=mean, var=var, invstd=invstd, s1=s1, out=out, jstar=jstar, out_bound=out_bound, scale=scale32,
             shift=shift32)
    if g is not None:
        r.update(backward_z(z, idx, co, jstar, g, scale32, shift32, mean32, invstd32, ga, slope, train))
    return r
