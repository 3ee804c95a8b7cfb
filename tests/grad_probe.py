"""Elementwise checks of one training step against a float64 reference (test helper, not a conftest).

Three pieces:

* `reference`: the math of `oracle.ref_model.RefModel.gradients` in float64 with the input block kept sparse
  (`scipy.sparse`) and the decoder evaluated at target entries only, so that catalogues of 2^18 columns cost what
  their batch holds, not B x N. Alongside every gradient it returns a magnitude bound S: the same backward pass
  with every factor replaced by its magnitude (|h|, |W|, |scale * act'|; for the error |mask|(|h||W| + |b|) + |t|
  instead of |e|), so that rho * S bounds what float32 summation can do to that element.
* probes that read the device's gradient back from one optimizer step:
    - SGD(lr=L), L a power of two: the update kernels do w = fmaf(-lr, g, w), so G = (W0 - W1) / L in float64 is
      the device's gradient to within 2^-24 |W1| / L. Every element must satisfy
          |G - g64| <= rho * S + 2^-23 (|W0| + |W1|) / L
      and where S is 0 (columns and arrays the batch does not touch, no L2) W1 must equal W0 bit for bit.
    - Adagrad / RMSprop / Adam with epsilon = E >= 2^10 max|g| and lr = E * L / 16: the rules are then nearly linear
      in g, so a scale error shows instead of being normalised away. Step 1 is checked against the float64 rule
      applied to g64; the optimizer state of step 2 is rebuilt from the device's own step-1 change (the rule
      inverts cleanly in this regime) and step 2 is checked against the rule applied to the float64 gradient at
      the device's W1.
* `row_launches`: which `k_row_update<NV, KIND, WIDE, HEAVY>` instantiations one training step launches.

Error analysis behind rho. Every float32 quantity of the step is a sum of products: the encoder sum over a row's
ratings, the hidden and decoder dot products over H, the gradient sums over the batch's matches (<= B rows) and
the tensor-core contractions (3xTF32: the dropped lo*lo term is 2^-22 relative per product). A sum of n terms in
float32 is off by at most n * 2^-24 * sum|terms| in the worst case; with round-to-nearest the rounding errors are
independent and of either sign, so the error grows like sqrt(n) * 2^-24 * sum|terms| and stays below
c * sqrt(n) * 2^-24 * sum|terms| with c of a few. S carries sum|terms| through every stage (first-order error
propagation: the forward magnitudes include |act'| times the magnitude of the pre-activation, and |act'| includes
max|act''| times it), so the bound is rho(n) * S with
    rho(n) = 2e-5 * max(1, sqrt(n / 128)),     n = the longest sum of the step (max of B and the padded widths)
2e-5 = 335 * 2^-24 at n = 128, i.e. c ~ 30 over sqrt(128) * 2^-24: room for the few stages that compound, not for
a lost or doubled term (which moves an element by its whole share of S). Activations with a kink (relu, and selu
whose slope jumps at 0) are outside this first-order bound: a pre-activation within rounding of 0 may take either
branch. The callers use smooth activations. The MAE loss has the same issue at err = 0; there an entry whose
float64 error is within 4 rho of its magnitude may take either sign, and its full contribution is allowed.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import scipy.sparse as sp

from oracle import philox, ref_model

ULP = 2.0 ** -24

# |act''| bounds of the smooth activations (the error of act'(z) is at most this times the error of z)
ACT2_MAX = {"linear": 0.0, None: 0.0, "sigmoid": 0.1, "tanh": 0.77, "elu": 1.0, "softplus": 0.25}

# ---------------------------------------------------------------------------------------------------------------
# the batch, sparse
# ---------------------------------------------------------------------------------------------------------------


@dataclass
class SparseBatch:
    """One batch as the model sees it: x0 [B, nblk*N] (sparse), target entries (row, column, value, mask)."""
    B: int
    N: int
    nblk: int
    x0: sp.csr_matrix
    t_row: np.ndarray
    t_col: np.ndarray
    t_val: np.ndarray
    t_mask: np.ndarray


def blocks_of(aux_type):
    return {None: 1, "causal": 2, "dropout": 2, "zeros": 2, "both": 3}[aux_type]


def from_dense(feed, targets, aux_type):
    """SparseBatch of a dense feed [x, (aux), mask_out, (observed)] (what `RefModel` takes)."""
    causal = aux_type is not None
    parts = [feed[0], feed[1]] + ([feed[3]] if aux_type == "both" else []) if causal else [feed[0]]
    mask = np.asarray(feed[2] if causal else feed[1], dtype=np.float64)
    t = np.asarray(targets, dtype=np.float64)
    x0 = sp.csr_matrix(np.concatenate([np.asarray(p, dtype=np.float64) for p in parts], axis=1))
    r, c = np.nonzero((mask != 0) | (t != 0))
    return SparseBatch(mask.shape[0], mask.shape[1], len(parts), x0, r, c, t[r, c], mask[r, c])


def _last_writes(r, c, v, width):
    """The last of the writes (r, c, v) to each cell (r, c) of a [*, width] array: the dense fills are
    last-write-wins, so a row that repeats a column keeps one value per array."""
    key = (r * width + c)[::-1]
    _, first = np.unique(key, return_index=True)
    keep = r.size - 1 - first
    return r[keep], c[keep], v[keep]


def from_batch(batch):
    """SparseBatch of a product `data_reader.Batch` of kind "split" (restates data_reader.py:158-169 on arrays;
    the keep flags must be host-drawn: a reader with rng_on_device = False)."""
    assert batch.kind == "split"
    csr = batch.source.csr
    rows = np.asarray(batch.rows, dtype=np.int64)
    rp = csr.rowptr
    lens = rp[rows + 1] - rp[rows]
    ent = np.repeat(rp[rows] - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()), dtype=np.int64)
    b = np.repeat(np.arange(rows.size), lens)
    c = csr.col[ent].astype(np.int64)
    v = csr.val[ent].astype(np.float64)
    f = np.asarray(batch.flags, dtype=bool)
    a = float(batch.aux_value)
    B, N, aux = rows.size, int(batch.n_cols), batch.aux_type
    nblk = blocks_of(aux)
    ri, ci, vi = [b[f]], [c[f]], [v[f]]                                   # block 0: the input ratings
    if aux == "causal" or aux == "both":
        blk = 2 if aux == "both" else 1
        ri.append(b); ci.append(c + blk * N); vi.append(np.full(b.size, a))      # observed
    if aux in ("dropout", "both"):
        ri.append(b[f]); ci.append(c[f] + N); vi.append(np.full(int(f.sum()), a))  # mask_in
    xr, xc, xv = _last_writes(np.concatenate(ri), np.concatenate(ci), np.concatenate(vi), nblk * N)
    x0 = sp.csr_matrix((xv, (xr, xc)), shape=(B, nblk * N))
    tg = ~f | bool(batch.pass_through)
    tr, tc, tv = _last_writes(b[tg], c[tg], v[tg], N)
    return SparseBatch(B, N, nblk, x0, tr, tc, tv, np.full(tr.size, a))


# ---------------------------------------------------------------------------------------------------------------
# float64 reference of one step + its magnitude bound
# ---------------------------------------------------------------------------------------------------------------


@dataclass
class Net:
    """What the reference needs of a model."""
    widths: List[int]
    activation: str
    loss: str = "mean_squared_error"
    l2: Optional[float] = None
    p_drop: Optional[float] = None
    dropout_seed: int = 0


def keep_masks(net, step, B):
    if net.p_drop is None:
        return [None] * len(net.widths)
    return [philox.dropout_keep(net.dropout_seed, step, l, B, w, net.p_drop) for l, w in enumerate(net.widths)]


def _decoder_at(h, Wd, bd, rows, cols, chunk=1 << 16):
    """full[rows[e], cols[e]] = h[rows[e]] . Wd[:, cols[e]] + bd[cols[e]] without forming [B, N]."""
    out = np.empty(rows.size)
    for s in range(0, rows.size, chunk):
        r, c = rows[s:s + chunk], cols[s:s + chunk]
        out[s:s + chunk] = np.einsum("ek,ke->e", h[r], Wd[:, c]) + bd[c]
    return out


def reference(net, sb, weights, keeps, rho):
    """(g64, S) lists aligned with the weight list. `rho` only enters through the MAE sign allowance."""
    L = len(net.widths)
    W = [np.asarray(w, dtype=np.float64) for w in weights]
    aW = [np.abs(w) for w in W]
    act, act2 = net.activation, ACT2_MAX[net.activation]
    B, N = sb.B, sb.N
    x0 = sb.x0
    ax0 = abs(x0)
    hs, hbars, cache = [x0], [ax0], []
    h, hbar = x0, ax0
    for l in range(L):
        z = np.asarray(h @ W[2 * l]) + W[2 * l + 1]
        zbar = np.asarray(hbar @ aW[2 * l]) + aW[2 * l + 1]
        a = ref_model.act_forward(act, z)
        d1 = ref_model.act_backward(act, z, a)
        scale = None
        if keeps[l] is not None:
            scale = keeps[l].astype(np.float64) / (1.0 - net.p_drop)
        s = 1.0 if scale is None else scale
        h = a * s
        hbar = (np.abs(a) + np.abs(d1) * zbar) * np.abs(s)      # |h| plus what the error of z does to it
        hs.append(h); hbars.append(hbar)
        cache.append((s, d1, np.abs(d1) + act2 * zbar))
    r, c, t, m = sb.t_row, sb.t_col, sb.t_val, sb.t_mask
    full = _decoder_at(h, W[-2], W[-1], r, c)
    fbar = _decoder_at(hbar, aW[-2], aW[-1], r, c)
    err = m * full - t
    ebar = np.abs(m) * fbar + np.abs(t)
    if net.loss == "mean_squared_error":
        dy, dybar = err * (2.0 / (B * N)), ebar * (2.0 / (B * N))
    else:
        dy = np.sign(err) / (B * N)
        amb = np.abs(err) <= 4 * rho * ebar                    # either sign is within rounding
        dybar = (1.0 + amb * (2.0 / rho)) / (B * N)
    D = sp.csr_matrix((dy * m, (r, c)), shape=(B, N))
    Dbar = sp.csr_matrix((dybar * np.abs(m), (r, c)), shape=(B, N))
    g = [None] * len(W)
    S = [None] * len(W)
    g[-2] = np.asarray((D.T @ h).T)
    S[-2] = np.asarray((Dbar.T @ hbar).T)
    g[-1] = np.asarray(D.sum(axis=0)).ravel()
    S[-1] = np.asarray(Dbar.sum(axis=0)).ravel()
    dh = np.asarray(D @ W[-2].T)
    dhbar = np.asarray(Dbar @ aW[-2].T)
    for l in reversed(range(L)):
        s, d1, d1bar = cache[l]
        dz = dh * s * d1
        dzbar = dhbar * np.abs(s) * d1bar
        hin, hinbar = hs[l], hbars[l]
        if l == 0:
            g[0] = np.asarray((hin.T @ dz))
            S[0] = np.asarray((hinbar.T @ dzbar))
        else:
            g[2 * l] = hin.T @ dz
            S[2 * l] = hinbar.T @ dzbar
        g[2 * l + 1] = dz.sum(axis=0)
        S[2 * l + 1] = dzbar.sum(axis=0)
        if l > 0:
            dh = dz @ W[2 * l].T
            dhbar = dzbar @ aW[2 * l].T
    if net.l2 is not None:
        for l in range(L + 1):
            g[2 * l] = g[2 * l] + 2.0 * net.l2 * W[2 * l]
            S[2 * l] = S[2 * l] + 2.0 * net.l2 * aW[2 * l]
    return g, S


def rho_for(B, hps):
    return 2e-5 * max(1.0, math.sqrt(max([B] + list(hps)) / 128.0))


def probe_lr(g64):
    """L: a power of two with L * max|g| ~ 1."""
    gmax = max(float(np.max(np.abs(g))) for g in g64 if g.size)
    return 2.0 ** (-math.floor(math.log2(gmax)))


# ---------------------------------------------------------------------------------------------------------------
# probes
# ---------------------------------------------------------------------------------------------------------------


def _report(name, bad, err, bound):
    if not bad.any():
        return None
    i = int(np.argmax(np.where(bad, err / np.maximum(bound, 1e-300), 0)))
    idx = np.unravel_index(i, bad.shape)
    return "%s: %d of %d elements out of bound (worst %s: |diff| %.3g, bound %.3g)" % (
        name, int(bad.sum()), bad.size, tuple(int(k) for k in idx), err.flat[i], bound.flat[i])


def check_sgd(W0, W1, L, g64, S, rho, label=""):
    """Failures (list of strings) of an SGD(lr=L) step W0 -> W1 against g64 / S."""
    out = []
    for k, (w0, w1, g, s) in enumerate(zip(W0, W1, g64, S)):
        a0, a1 = np.asarray(w0, dtype=np.float64), np.asarray(w1, dtype=np.float64)
        G = (a0 - a1) / L
        err = np.abs(G - g)
        bound = rho * s + 2.0 * ULP * (np.abs(a0) + np.abs(a1)) / L
        bad = err > bound
        bad |= (s == 0) & (np.asarray(w0) != np.asarray(w1))     # untouched: bit for bit
        rep = _report("%sarray %d" % (label, k), bad, err, bound)
        if rep:
            out.append(rep)
    return out


RULE_DEFAULTS = {"adagrad": {}, "rmsprop": {"rho": 0.9}, "adam": {"beta_1": 0.9, "beta_2": 0.999}}


class RuleProbe(object):
    """Float64 Adagrad / RMSprop / Adam in the well-conditioned regime (epsilon E >> |g|, lr = E * L)."""

    def __init__(self, kind, E, lr, decay=0.0, rho=0.9, beta_1=0.9, beta_2=0.999):
        self.kind, self.E, self.lr, self.decay = kind, E, lr, decay
        self.rho, self.b1, self.b2 = rho, beta_1, beta_2
        self.it = 0
        self.state = None

    def _lr(self):
        lr = self.lr / (1.0 + self.decay * self.it) if self.decay > 0 else self.lr
        if self.kind == "adam":
            t = self.it + 1
            lr *= math.sqrt(1.0 - self.b2 ** t) / (1.0 - self.b1 ** t)
        return lr

    def _kc(self):
        """D = k g / (c |g| + E) is the first step of every rule from zero state."""
        lr = self._lr()
        if self.kind == "adagrad":
            return lr, 1.0
        if self.kind == "rmsprop":
            return lr, math.sqrt(1.0 - self.rho)
        return lr * (1.0 - self.b1), math.sqrt(1.0 - self.b2)

    def step(self, g, state):
        """(delta = W_before - W_after, new state, d delta / d g bound)."""
        lr, E = self._lr(), self.E
        if self.kind == "adagrad":
            s = (0.0 if state is None else state) + g * g
            return lr * g / (np.sqrt(s) + E), s, lr / E
        if self.kind == "rmsprop":
            s = (1.0 - self.rho) * g * g + (0.0 if state is None else self.rho * state)
            return lr * g / (np.sqrt(s) + E), s, lr / E
        m0, v0 = (0.0, 0.0) if state is None else state
        m = self.b1 * m0 + (1.0 - self.b1) * g
        v = self.b2 * v0 + (1.0 - self.b2) * g * g
        return lr * m / (np.sqrt(v) + E), (m, v), lr * (1.0 - self.b1) / E

    def state_from_first_step(self, D):
        """The state step 1 left, from the observed change D of a step from zero state (at iteration 0)."""
        k, c = self._kc()
        g1 = D * self.E / (k - c * np.abs(D))
        if self.kind == "adagrad":
            return g1 * g1, g1
        if self.kind == "rmsprop":
            return (1.0 - self.rho) * g1 * g1, g1
        return ((1.0 - self.b1) * g1, (1.0 - self.b2) * g1 * g1), g1

    def check(self, W0, W1, g64, S, rho, states=None, g1_err=None, label=""):
        """Failures of one step W0 -> W1 against the rule applied to g64 from `states` (None: zero state)."""
        out = []
        for k, (w0, w1, g, s) in enumerate(zip(W0, W1, g64, S)):
            a0, a1 = np.asarray(w0, dtype=np.float64), np.asarray(w1, dtype=np.float64)
            st = None if states is None else states[k]
            delta, _, sens = self.step(g, st)
            err = np.abs((a0 - a1) - delta)
            bound = sens * rho * s + 2.0 * ULP * (np.abs(a0) + np.abs(a1)) + 8.0 * ULP * np.abs(delta)
            if g1_err is not None:        # state rebuilt from a float32 change: what its rounding can do
                carry = self.b1 if self.kind == "adam" else 2.0 * np.abs(g) / self.E
                bound = bound + sens * carry * g1_err[k]
            bad = err > bound
            if states is None:
                bad |= (s == 0) & (np.asarray(w0) != np.asarray(w1))
            rep = _report("%sarray %d" % (label, k), bad, err, bound)
            if rep:
                out.append(rep)
        self.it += 1
        return out

    def rebuild(self, W0, W1):
        """(states, bound on the recovered step-1 gradients' error) from the device's step-1 change; call after
        `check` of step 1 (the step-1 learning rate is that of iteration 0)."""
        it, self.it = self.it, 0
        k, c = self._kc()
        states, errs = [], []
        for w0, w1 in zip(W0, W1):
            a0, a1 = np.asarray(w0, dtype=np.float64), np.asarray(w1, dtype=np.float64)
            st, _ = self.state_from_first_step(a0 - a1)
            states.append(st)
            errs.append(2.0 * ULP * (np.abs(a0) + np.abs(a1)) * self.E / (k - c * np.abs(a0 - a1)) * 2.0)
        self.it = it
        return states, errs


def rule_params(kind, g64):
    """(epsilon, lr) of the well-conditioned regime for gradients g64: E = 2^k >= 2^10 max|g|, lr = E L / 16 (a
    step moves a weight by at most ~1/16, so the step-2 gradient is taken near the step-1 point)."""
    L = probe_lr(g64)
    gmax = max(float(np.max(np.abs(g))) for g in g64 if g.size)
    E = 2.0 ** math.ceil(math.log2(gmax * 1024.0))
    return E, E * L / 16.0


# ---------------------------------------------------------------------------------------------------------------
# which k_row_update instantiation runs (csrc/ocf_api.cu: launch_rows, heavy_model, phase_update)
# ---------------------------------------------------------------------------------------------------------------
KINDS = {"sgd": 0, "adagrad": 1, "rmsprop": 2, "adam": 3}
KIND_GRAD = 4                      # ocf_kernels.cuh: KIND_GRAD
HPAD = 128


def pad(h):
    return -(-int(h) // HPAD) * HPAD


def row_launches(n_cols, widths, kind, row_parallel=False):
    """(NV, KIND, WIDE, HEAVY) of every k_row_update launch of one training step, mirroring
        wide  = !grad_mode && n_cols * hp_of_the_launch <= 8 Mi                   (launch_rows)
        heavy = n_cols * max(hp[0], hp[L-1]) <= 32 Mi && !grad_mode                (heavy_model, launch_rows)
        WIDE launches the <NV, KIND, true, true> kernel (launch_row_update)
    and one launch when the decoder and encoder rows share a padded width, else one per width (phase_update).
    Row-parallel steps launch <NV, KIND_GRAD, false, false>. NV = hp / 128 capped at 8 (OCF_NV_SWITCH)."""
    hp0, hpt = pad(widths[0]), pad(widths[-1])
    grad = bool(row_parallel)
    heavy = n_cols * max(hp0, hpt) <= (32 << 20) and not grad
    out = []
    for hp in sorted({hpt, hp0}):
        nv = min(hp // 128, 8)
        if grad:
            out.append((nv, KIND_GRAD, False, False))
            continue
        wide = n_cols * hp <= (8 << 20)
        out.append((nv, KINDS[kind], True, True) if wide else (nv, KINDS[kind], False, heavy))
    return out


def all_instantiations():
    """Every k_row_update instantiation the dispatch can reach."""
    out = set()
    for nv in range(1, 9):
        for k in range(4):
            out |= {(nv, k, True, True), (nv, k, False, True), (nv, k, False, False)}
        out.add((nv, KIND_GRAD, False, False))
    return out
