"""A batched Float64 reference of the three ResNet networks (net_type = MZ_NET_RESNET), written from the blob layout of
csrc/mz_rn_host.h and DESIGN §2.4 alone (not from oracle/mz_oracle.c, not from rn_pack).

Activations are held as (batch, x, y, channel) with x along W; the flat Julia (W,H,C) order is index = x + W*(y + H*c).

quant=False  the network in Float64: Conv (true, flipped-kernel convolution, zero padding), BatchNorm in test mode with
             eps = Float64(1f-5), relu / tanh, flatten in Flux order (k = cell + cells*f).
quant=True   the tensor-core kernels' arithmetic contract with exact sums:
             * conv weights rounded RNE to bf16 after the Float32 fold w * (mul * (gamma / sqrtf(var + 1f-5))); dense weights bf16;
             * inputs staged as bf16 (representation: the board values; prediction: h; dynamics: bf16(0.5 * sa), the x2 lives
               in the first convolution's fold, the action plane enters as plane * E, E = w_plane * s in Float32);
             * products exact, sums in Float64, the sum rounded once to Float32 (an ideal fp32 accumulator);
             * epilogue in Float32: acc + fmaf(plane, E, T) (or acc + T), + skip, activation, then RNE to bf16 where the kernel
               stores (tile epilogues, head scatter, pool rows); value, logits and reward stay Float32.
             With c_acc set it also carries, for every stored element, the interval [lo, hi] of bf16 values the kernel may
             produce when every accumulator is within c_acc * 2^-24 * sum|w*x| of its exact value (inputs themselves taken
             from their own intervals).  The epilogue is monotone in the accumulator and the skip, so the interval's ends are
             the epilogue at the ends.  For a network whose other layers are exact identities this is the accepted set of
             one rounding: one bf16 value, or two adjacent ones next to a rounding boundary.

bug=  applies one deliberate kernel-style mistake, to show that a check built on this reference would catch it:
      "swap" (output channels 0 and 1 of every convolution exchanged), "noflip" (cross-correlation), "wrap" (circular padding),
      "filter_fastest" (head flatten k = f + nheads*cell), "drop_mu" (BatchNorm mean ignored), "plane" (action plane one action
      off), "no_x2" (the dynamics input's x2 missing), "pad" (a padded input channel aliasing channel 0 of the tile)."""
import numpy as np

f32 = np.float32
EPS = f32(1e-5)
U24 = 2.0 ** -24


def bf16(x):
    """RNE of Float32 values to bf16, returned as Float32 (mzh::f2bf16, cvt.rn.bf16x2.f32)."""
    u = np.ascontiguousarray(x, f32).view(np.uint32).astype(np.uint64)
    u = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return u.astype(np.uint32).view(f32)


def units(c):
    """Blob order of the three networks: lists of dicts with kind, k, cin, cout, act and parameter offsets."""
    nf, nb, cells, hs = c.rn_num_filters, c.rn_num_blocks, c.W * c.H, c.width_hidden
    planes = c.C * (c.stacked_observations + 1) + c.stacked_observations
    off = [0]

    def conv(k, cin, cout, act):
        u = dict(kind="conv", k=k, cin=cin, cout=cout, act=act, w=off[0]); off[0] += k * k * cin * cout
        for n in ("b", "beta", "gamma", "mu", "var"):
            u[n] = off[0]; off[0] += cout
        return u

    def dense(cin, cout, act):
        u = dict(kind="dense", k=1, cin=cin, cout=cout, act=act, w=off[0]); off[0] += cin * cout
        u["b"] = off[0]; off[0] += cout
        return u

    def tower(k, cin):
        out = [conv(k, cin, nf, "relu")]
        for _ in range(nb):
            out += [conv(k, nf, nf, "relu"), conv(k, nf, nf, "id")]
        return out

    def head(f, first_act, n_out, out_act):
        return [conv(1, nf, f, "relu"), dense(cells * f, hs, first_act)] + [dense(hs, hs, "relu") for _ in range(c.depth_value)] + \
               [dense(hs, n_out, out_act)]
    rep = tower(c.rn_kernel, planes)
    pred = tower(1, nf); pred += head(c.rn_first_head_filters, "relu", 1, "tanh"); pred += head(c.rn_second_head_filters, "id", c.A, "id")
    dyn = tower(1, nf + 1); dyn += tower(1, nf); dyn += head(c.rn_first_head_filters, "relu", 1, "tanh")
    return [rep, pred, dyn], off[0]


def _act(x, a):
    return np.maximum(x, 0) if a == "relu" else np.tanh(x) if a == "tanh" else x


def _fma32(a, b, c):
    """fmaf in Float32, emulated: the product of two floats is exact in Float64, but the sum is rounded to Float64 and then to
    Float32.  That is two roundings, and in rare cases it differs from fmaf's single one by one Float32 ulp of T (BatchNorm shift
    or action-plane term), which can flip a stored bf16 value that sits on a rounding boundary.  Not seen so far: the CPU replay,
    which calls fmaf itself, is bit-identical to this reference on every tested shape."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f32)


class Ref64:
    def __init__(self, c, blob, quant=False, c_acc=None, bug=None):
        self.c, self.quant, self.c_acc, self.bug = c, quant, c_acc, bug
        self.blob = np.asarray(blob, f32)
        self.nets, n = units(c)
        assert self.blob.shape[0] == n, (self.blob.shape, n)
        self.W, self.H, self.cells = c.W, c.H, c.W * c.H
        self.nt = 1 + 2 * c.rn_num_blocks
        self.nh = 3 + c.depth_value
        self.trace = {}            # name -> outputs recorded on the way (head convolutions)
        self.calib = None          # np.random.Generator: set the BatchNorm statistics of every convolution from its inputs
        self.calib_only = None     # ... or only of the units whose weight offsets are in this set

    # ---- layout ----
    def from_flat(self, a, nch):
        a = np.asarray(a).reshape(-1, nch, self.H, self.W)
        return np.ascontiguousarray(a.transpose(0, 3, 2, 1))

    @staticmethod
    def to_flat(a):
        return np.ascontiguousarray(a.transpose(0, 3, 2, 1)).reshape(a.shape[0], -1)

    # ---- parameters ----
    def P(self, u, name, n=None):
        return self.blob[u[name]:u[name] + (n or u["cout"])]

    def conv_w(self, u):
        k, cin, cout = u["k"], u["cin"], u["cout"]
        return self.blob[u["w"]:u["w"] + k * k * cin * cout].reshape((k, k, cin, cout), order="F")

    def dense_w(self, u):
        return self.blob[u["w"]:u["w"] + u["cin"] * u["cout"]].reshape((u["cout"], u["cin"]), order="F").T   # (in, out)

    # ---- the convolution sum, batched over (sample, cell) ----
    def _sum(self, x, w):
        """x (B, W, H, cin) float64, w (k, k, cin, cout) float64 -> (B, W, H, cout): y[i,j] = sum_ab x[i+p-a, j+p-b] . w[a,b]"""
        k = w.shape[0]; p = k // 2; B, W, H, cin = x.shape
        if self.bug == "noflip":
            w = w[::-1, ::-1]
        if self.bug == "pad" and cin < 64:
            x = np.concatenate([x, x[..., :1]], -1); w = np.concatenate([w, w[:, :, :1]], 2)
        if k == 1:
            return (x.reshape(-1, x.shape[-1]) @ w[0, 0]).reshape(B, W, H, -1)
        xp = np.pad(x, ((0, 0), (p, p), (p, p), (0, 0)), mode="wrap" if self.bug == "wrap" else "constant")
        y = np.zeros((B * W * H, w.shape[3]))
        for a in range(k):
            for b in range(k):
                if not w[a, b].any():
                    continue                                   # (identity layers of the surgery networks: one tap)
                sl = np.ascontiguousarray(xp[:, 2 * p - a:2 * p - a + W, 2 * p - b:2 * p - b + H, :]).reshape(-1, x.shape[-1])
                y += sl @ w[a, b]
        return y.reshape(B, W, H, -1)

    # ---- one ConvBN unit ----
    def conv(self, u, x, skip=None, act=None, mul=1.0, plane=None, store=True):
        """x: Float64 array (quant=False) or a triple (nominal, lo, hi) of bf16 arrays (quant=True); plane: (B,) action-plane values
        (dynamics input: the last input channel of the unit is the action plane)."""
        act = act or u["act"]
        cout = u["cout"]
        b, beta, gamma, mu, var = (self.P(u, n) for n in ("b", "beta", "gamma", "mu", "var"))
        if self.bug == "drop_mu":
            mu = np.zeros_like(mu)
        w = self.conv_w(u)
        if not self.quant:
            wx = w[:, :, :-1] if plane is not None else w
            z = self._sum(x, wx.astype(np.float64))
            if plane is not None:
                z = z + plane[:, None, None, None] * w[0, 0, -1].astype(np.float64)
            z = z + b
            if self.calib is not None and (self.calib_only is None or u["w"] in self.calib_only):
                self._calibrate(u, z)
                b, beta, gamma, mu, var = (self.P(u, n) for n in ("b", "beta", "gamma", "mu", "var"))
            y = (gamma.astype(np.float64) * (z - mu) / np.sqrt(var.astype(np.float64) + np.float64(EPS))) + beta
            if skip is not None:
                y = y + skip
            y = _act(y, act)
            return self._swap(y)
        s = (gamma / np.sqrt(var + EPS)).astype(f32)
        fold = (f32(mul) * s).astype(f32)
        wx = w[:, :, :-1] if plane is not None else w
        wq = bf16((wx * fold).astype(f32)).astype(np.float64)
        T = _fma32((b - mu).astype(f32), s, beta)
        if plane is not None:
            E = (w[0, 0, -1] * s).astype(f32)
            add = _fma32(plane[:, None, None, None].astype(f32), E, T)
        else:
            add = T
        return self._epilogue(x, wq, add, skip, act, store, self._sum, swap=True)

    def _swap(self, y, on=True):
        if on and self.bug == "swap" and y.shape[-1] > 1:
            y = y.copy(); y[..., [0, 1]] = y[..., [1, 0]]
        return y

    def _epilogue(self, x, wq, add, skip, act, store, summ, swap=False):
        nom, lo, hi = x
        acc = summ(nom.astype(np.float64), wq)

        def epi(a, sk):
            y = a.astype(f32) + add
            if sk is not None:
                y = (y + sk).astype(f32)
            y = _act(y, act).astype(f32)
            return bf16(y) if store else y
        out = self._swap(epi(acc, None if skip is None else skip[0]), swap)
        if self.c_acc is None:
            return out, out, out
        if lo is nom and hi is nom:
            alo = ahi = acc
        else:
            wp, wn = np.maximum(wq, 0), np.minimum(wq, 0)
            alo = summ(lo.astype(np.float64), wp) + summ(hi.astype(np.float64), wn)
            ahi = summ(hi.astype(np.float64), wp) + summ(lo.astype(np.float64), wn)
        mag = np.maximum(np.abs(lo), np.abs(hi)).astype(np.float64)
        e = self.c_acc * U24 * summ(mag, np.abs(wq))
        # an fp32 accumulator inside [exact - e, exact + e] rounds (monotonically) to a value inside [RN(lo), RN(hi)]
        olo = self._swap(epi(alo - e, None if skip is None else skip[1]), swap)
        ohi = self._swap(epi(ahi + e, None if skip is None else skip[2]), swap)
        return out, olo, ohi

    def _calibrate(self, u, z):
        """mu, var from the Float64 pre-activations of this layer over the calibration batch (var times U(0.5, 2)); gamma, beta
        such that every channel is positive on a substantial fraction of (sample, cell)."""
        rng, cout = self.calib, u["cout"]
        zz = z.reshape(-1, cout)
        self.blob[u["mu"]:u["mu"] + cout] = zz.mean(0)
        self.blob[u["var"]:u["var"] + cout] = np.maximum(zz.var(0), 1e-4) * rng.uniform(0.5, 2.0, cout)
        self.blob[u["gamma"]:u["gamma"] + cout] = rng.uniform(0.5, 1.5, cout)
        self.blob[u["beta"]:u["beta"] + cout] = rng.uniform(0.0, 0.4, cout)

    # ---- dense layers ----
    def dense(self, u, x, store):
        w = self.dense_w(u); b = self.P(u, "b")
        if not self.quant:
            return _act(x @ w.astype(np.float64) + b, u["act"])
        return self._epilogue(x, bf16(w).astype(np.float64), b, None, u["act"], store, lambda a, ww: a @ ww)

    # ---- networks ----
    def _q(self, x):
        return (x, x, x) if self.quant else x

    def tower(self, us, x, mul=1.0, plane=None):
        x = self.conv(us[0], x, mul=mul, plane=plane)
        for i in range(self.c.rn_num_blocks):
            t = self.conv(us[1 + 2 * i], x)
            x = self.conv(us[2 + 2 * i], t, skip=x, act="relu")
        return x

    def head(self, us, t, name):
        f = self.conv(us[0], t)
        self.trace[name] = f
        nf = us[0]["cout"]

        def flat(a):
            if self.bug == "filter_fastest":
                return np.ascontiguousarray(a.transpose(0, 2, 1, 3)).reshape(a.shape[0], -1)   # k = f + nheads * (x + W*y)
            return self.to_flat(a)
        x = tuple(flat(a) for a in f) if self.quant else flat(f)
        for i, u in enumerate(us[1:]):
            x = self.dense(u, x, store=i < len(us) - 2)
        return x

    def representation(self, stacked):
        planes = self.nets[0][0]["cin"]
        x = self.from_flat(np.asarray(stacked, f32 if self.quant else np.float64), planes)
        x = bf16(x) if self.quant else x
        h = self.tower(self.nets[0], self._q(x))
        return self._flat_out(h)

    def _flat_out(self, h):
        return tuple(self.to_flat(a) for a in h) if self.quant else self.to_flat(h)

    def prediction(self, hidden):
        """-> value (B,), logits (B, A)  (nominal outputs; Float32 in quant mode)"""
        nf = self.c.rn_num_filters
        x = self.from_flat(np.asarray(hidden, f32 if self.quant else np.float64), nf)
        x = bf16(x) if self.quant else x
        us = self.nets[1]; nt, nh = self.nt, self.nh
        t = self.tower(us[:nt], self._q(x))
        v = self.head(us[nt:nt + nh], t, "value_conv")
        z = self.head(us[nt + nh:], t, "policy_conv")
        if self.quant:
            self.value_iv, self.logits_iv = v, z
            return v[0][:, 0], z[0]
        return v[:, 0], z

    def dynamics(self, sa):
        """sa = 2*h || action plane (the kernel reads the plane's first cell) -> next hidden (B, hidden), reward (B,)"""
        nf = self.c.rn_num_filters; hid = self.cells * nf
        sa = np.asarray(sa, f32 if self.quant else np.float64).reshape(-1, hid + self.cells)
        plane = sa[:, hid].astype(np.float64)
        if self.bug == "plane":
            plane = plane + 1.0 / self.c.A
        x = self.from_flat(sa[:, :hid], nf)
        us = self.nets[2]; nt = self.nt
        mul = 1.0 if self.bug == "no_x2" else 2.0
        if self.quant:
            x = bf16((x * f32(0.5)).astype(f32))
            t = self.tower(us[:nt], self._q(x), mul=mul, plane=plane.astype(f32))
        else:
            x = x.astype(np.float64) * (0.5 * mul)
            t = self.tower(us[:nt], x, mul=1.0, plane=plane)
        r = self.head(us[2 * nt:], t, "reward_conv")
        s = self.tower(us[nt:2 * nt], t)
        if self.quant:
            self.reward_iv = r
            return self._flat_out(s), r[0][:, 0]
        return self.to_flat(s), r[:, 0]


def policy(logits):
    z = np.asarray(logits, np.float64)
    e = np.exp(z - z.max(1, keepdims=True))
    return e / e.sum(1, keepdims=True)


def calibrated_blob(c, blob, seed, stacked, actions, only=None, hidden=None, sa=None):
    """A copy of `blob` whose convolutions (or the units in `only`) have BatchNorm statistics taken from the Float64
    pre-activations of that layer over a calibration batch (stacked observations + the action taken after each; the
    prediction and dynamics inputs default to the representation's outputs), so that every channel is live."""
    ref = Ref64(c, np.array(blob, f32, copy=True))
    ref.calib = np.random.default_rng(seed)
    ref.calib_only = None if only is None else {u["w"] for u in only}
    h = ref.representation(stacked)
    ref.prediction(h if hidden is None else hidden)
    if sa is None:
        sa = np.concatenate([2 * h, np.repeat((np.asarray(actions, np.float64) / c.A)[:, None], c.W * c.H, 1)], 1)
    ref.dynamics(sa)
    return ref.blob


def liveness(c, blob, stacked, actions):
    """(min over head-convolution channels of the fraction of (sample, cell) where it is non-zero,
        min standard deviation over the inputs of value, reward and every logit)"""
    ref = Ref64(c, blob)
    h = ref.representation(stacked)
    v, z = ref.prediction(h)
    sa = np.concatenate([2 * h, np.repeat((np.asarray(actions, np.float64) / c.A)[:, None], c.W * c.H, 1)], 1)
    _, r = ref.dynamics(sa)
    frac = min(float((ref.trace[n] != 0).reshape(-1, ref.trace[n].shape[-1]).mean(0).min()) for n in ("value_conv", "policy_conv", "reward_conv"))
    std = min(float(v.std()), float(r.std()), float(z.std(0).min()))
    return frac, std


# ---- weight surgery: layers that are exact identities ----
def set_identity_bn(c, blob, u, rng):
    """b = beta = mu = 0, gamma = sqrtf(var + 1f-5) in Float32: the folded scale is exactly 1 and T = 0"""
    n = u["cout"]
    var = rng.uniform(0.5, 2.0, n).astype(f32)
    blob[u["var"]:u["var"] + n] = var
    blob[u["gamma"]:u["gamma"] + n] = np.sqrt(var + EPS).astype(f32)
    for k in ("b", "beta", "mu"):
        blob[u[k]:u[k] + n] = 0.0


def set_dense(blob, u, w):
    """w: (in, out)"""
    blob[u["w"]:u["w"] + u["cin"] * u["cout"]] = np.asarray(w, f32).reshape(-1)


def set_conv(blob, u, w):
    k, cin, cout = u["k"], u["cin"], u["cout"]
    blob[u["w"]:u["w"] + k * k * cin * cout] = np.asarray(w, f32).reshape(-1, order="F")


def centre_select(u, src, scale=1.0):
    """a k x k kernel whose only non-zero entries are the centre tap, output channel co <- input channel src[co]"""
    k = u["k"]; w = np.zeros((k, k, u["cin"], u["cout"]), f32)
    for co, ci in enumerate(src):
        if ci is not None:
            w[k // 2, k // 2, ci, co] = scale
    return w


def bf16_weights(blob, u):
    """round a unit's weights to bf16 in place (its fold by an identity BatchNorm is then exact)"""
    n = u["k"] * u["k"] * u["cin"] * u["cout"]
    blob[u["w"]:u["w"] + n] = bf16(blob[u["w"]:u["w"] + n])
