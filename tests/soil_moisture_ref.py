"""Plain-Python restatement of the soil-moisture outputs (definitions in include/lgar_b200.h), evaluated on a front
list: scalar IEEE double arithmetic in the library's exact operation order (the library is built without FMA
contraction), so on the same front list the values agree bit for bit."""
import math

import numpy as np


def cumulative(thickness):
    """cum[l] = thickness[0] + ... + thickness[l], summed left to right like the library."""
    cum, c = [], 0.0
    for l, th in enumerate(thickness):
        c = float(th) if l == 0 else c + float(th)
        cum.append(c)
    return cum


def layer_water(depth, theta, counts, thickness):
    """W_l of every layer: `depth`, `theta` in list order, `counts[l]` fronts in the list of layer l."""
    cum = cumulative(thickness)
    out, o = [], 0
    for l, nf in enumerate(counts):
        base = 0.0 if l == 0 else cum[l] - float(thickness[l])
        s = 0.0
        for i in range(o, o + nf - 1):
            s = s + (float(depth[i]) - base) * (float(theta[i]) - float(theta[i + 1]))
        if nf > 0:
            s = s + (float(depth[o + nf - 1]) - base) * float(theta[o + nf - 1])
        out.append(s)
        o += nf
    return out


def theta_at(z, depth, theta, counts, thickness):
    """theta(z): the first front of the list of the layer with cum[l-1] < z <= cum[l] whose depth >= z; NaN below the
    column or when no front of that list qualifies."""
    cum = cumulative(thickness)
    o = 0
    for l, nf in enumerate(counts):
        if z <= cum[l]:
            for i in range(o, o + nf):
                if float(depth[i]) >= z:
                    return float(theta[i])
            return math.nan
        o += nf
    return math.nan


def counts_from_layers(front_layer, n, L):
    """List lengths per layer from the layer_num of the first n fronts (which must be grouped in list order)."""
    lay = np.asarray(front_layer[:n], dtype=np.int64)
    assert np.all(np.diff(lay) >= 0), f"layer numbers not grouped in list order: {lay}"
    return [int((lay == l).sum()) for l in range(L)]


def outputs_of_dump(fronts, front_layer, nfronts, thickness, depths):
    """W[T,L] and theta[T,D] of a front dump fronts[T,16,5] / front_layer[T,16] / nfronts[T]."""
    T, L = len(nfronts), len(thickness)
    W = np.full((T, L), np.nan)
    th = np.full((T, len(depths)), np.nan)
    for t in range(T):
        n = int(nfronts[t])
        cnt = counts_from_layers(front_layer[t], n, L)
        d, q = fronts[t, :n, 0], fronts[t, :n, 1]
        W[t] = layer_water(d, q, cnt, thickness)
        th[t] = [theta_at(float(z), d, q, cnt, thickness) for z in depths]
    return W, th
