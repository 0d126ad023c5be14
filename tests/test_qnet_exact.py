"""The Q-network bit for bit: forward, gradients and Adam steps on inputs chosen so that no f32 sum of the network rounds.

When every term of a sum is an integer multiple of one power-of-two unit u and the magnitudes of the terms add up to less
than 2^24 u, every partial sum, in any order and however the adder aligns its operands, is an integer number of units
below 2^24 and so an f32 value: the result does not depend on the order of the sum. Products of two bf16 values are
exact, the library is built with -fmad=false, and its divisions and square roots are IEEE. Then every bf16 rounding the
device makes is the rounding of a value the reference knows exactly, and the reference predicts every output with zero
tolerance, at every batch size.

The inputs:
* the replay's frame ring is overwritten with seeded random pixels (0/1, or 0..15) through a checkpoint round trip, so
  that neighbouring pixels differ and an index error reads another value; the records stay real, so episode starts
  (zero-filled stack slots) and partial stacks are still there;
* sparse weights of +-1 times a power of two per layer, about three non-zeros per output unit; across the N_DRAWS draws
  every kernel row of every layer is non-zero at least once;
* biases on the grid, set from quantiles of each layer's pre-activations so that every ReLU mask is non-trivial;
* loss weights B * 2^-M, so that dL/dQ = clip(Q_a - y) * 2^-M exactly at any batch size B, and targets that put items
  on the quadratic and on the saturated side of the Huber loss.

The reference is float64 torch (exact below 2^53, so the order of its own sums does not matter either) with the
convolutions written as unfold / fold and matrix products. It rounds to bf16 (round to nearest even, restated on the
bits) exactly where the device rounds, and checks its own premise at every accumulation it computes: a construction that
breaks it fails loudly instead of passing by luck.

Equality is numeric (np.array_equal): +0.0 and -0.0 count as equal, every other bit must match. The Adam restatement
compares the bits of the f32 master weights."""
import math
import os

import numpy as np
import pytest

gpu = pytest.mark.gpu

BIG = 32768              # the largest minibatch DESIGN §11 reports
CHUNK = 512              # items per reference chunk of the forward (conv1's unfolded input of a chunk: 420 MB of f64)
GRAD_CHUNK = 256         # ... of the backward (which holds more per item)
N_DRAWS = 3              # weight draws; their non-zeros cover every kernel row
NNZ = 3                  # non-zeros per output unit of a kernel (at least)
SCALE = (-2, -1, -1, -1, -1)   # log2 of the weight unit of conv1, conv2, conv3, dense 1, dense 2
M_WEIGHT = 6             # loss weights B * 2^-M: dL/dQ = clip(d) * 2^-M
LIMIT = 2.0 ** 24
# minibatch sizes (tests/test_qnet_batch_edges.py _sizes, plus 2, 3 and 7: conv2 packs 2 items per batch, conv3 3)
SIZES = ["1", "2", "3", "7", "127", "128", "129", "last_narrow", "last_narrow+1", "last_narrow+3", "first_wide_tile", str(BIG)]
KERAS = ("conv1_kernel", "conv1_bias", "conv2_kernel", "conv2_bias", "conv3_kernel", "conv3_bias", "dense1_kernel", "dense1_bias",
         "dense2_kernel", "dense2_bias")


# ---- bf16 rounding and units ----
def _bf16(t):
    """Round a float64 tensor that holds f32 values to the nearest bf16 (ties to even), restated on the f32 bits."""
    import torch
    a = t.abs().to(torch.float32)
    assert torch.equal(a.to(torch.float64), t.abs()), "a value to be rounded to bf16 is not an f32 value: the premise is broken"
    u = a.view(torch.int32)                                   # finite, non-negative: < 0x7F800000
    u = (u + 0x7FFF + ((u >> 16) & 1)) & -0x10000
    return torch.copysign(u.view(torch.float32).to(torch.float64), t)


def _unit(t):
    """The largest power of two that divides every non-zero element of t (inf if there is none)."""
    import torch
    nz = t[t != 0].abs()
    if nz.numel() == 0:
        return math.inf
    m, e = torch.frexp(nz)
    mi = (m * 2.0 ** 53).to(torch.int64)
    return float(torch.ldexp((mi & -mi).to(torch.float64), e - 53).min())


class _Premise:
    """Checks sum |terms| < 2^24 * unit for an accumulation and keeps the worst ratio per accumulation."""

    def __init__(self):
        self.worst = {}

    def __call__(self, what, abs_sum, unit):
        r = float(abs_sum.max()) / (LIMIT * unit) if abs_sum.numel() else 0.0
        assert r < 1.0, "premise broken at %s: sum |terms| = %.6g is not below 2^24 units of %g" % (what, float(abs_sum.max()), unit)
        self.worst[what] = max(self.worst.get(what, 0.0), r)


def _no_check(what, abs_sum, unit):
    pass


# ---- the reference ----
def _torch_weights(torch, w, dev, bf):
    """Keras f32 arrays -> f64 tensors: conv kernels [co][ci][kx][ky] and the dense-1 kernel rounded by bf (the device's bf16
    operand copies), the head kernel [512][3] and the biases as they are (f32 on the device)."""
    W = {}
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), device=dev)
    for i in (1, 2, 3):
        W["k%d" % i] = bf(t(w["conv%d_kernel" % i]).permute(3, 2, 0, 1).contiguous())
        W["b%d" % i] = t(w["conv%d_bias" % i])
    W["k4"], W["b4"] = bf(t(w["dense1_kernel"])), t(w["dense1_bias"])
    W["k5"], W["b5"] = t(w["dense2_kernel"]), t(w["dense2_bias"])
    return W


STRIDES = (4, 2, 1)


def _forward(torch, W, x, chk, bf=_bf16):
    """x f64 [n][4][84(x)][84(y)] -> (Q [n][3], [x, a1, a2, a3, h]): the activations after bias, ReLU and the rounding bf,
    where the device rounds them to bf16."""
    F = torch.nn.functional
    acts = [x]
    for i in (1, 2, 3):
        k, b = W["k%d" % i], W["b%d" % i]
        cols = F.unfold(x, k.shape[2:], stride=STRIDES[i - 1])               # [n][ci*kx*ky][pixels]; x >= 0
        km = k.reshape(k.shape[0], -1)
        chk("conv%d" % i, km.abs() @ cols + b.abs()[:, None], min(_unit(x) * _unit(k), _unit(b)))
        side = (x.shape[2] - k.shape[2]) // STRIDES[i - 1] + 1
        x = bf(torch.relu(km @ cols + b[:, None])).reshape(x.shape[0], k.shape[0], side, side)
        del cols
        acts.append(x)
    flat = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)                     # Keras Flatten of [7(x)][7(y)][64]
    chk("dense1", flat @ W["k4"].abs() + W["b4"].abs(), min(_unit(flat) * _unit(W["k4"]), _unit(W["b4"])))
    h = bf(torch.relu(flat @ W["k4"] + W["b4"]))
    chk("head", h @ W["k5"].abs() + W["b5"].abs(), min(_unit(h) * _unit(W["k5"]), _unit(W["b5"])))
    acts.append(h)
    return h @ W["k5"] + W["b5"], acts


class _GradSums:
    """Weight- and bias-gradient sums over chunks, with the sums of |terms| and the common unit of the terms."""

    def __init__(self):
        self.g, self.a, self.u = {}, {}, {}

    def add(self, name, g, a, u):
        self.g[name] = self.g[name] + g if name in self.g else g
        self.a[name] = self.a[name] + a if name in self.a else a
        self.u[name] = min(self.u.get(name, math.inf), u)

    def keras(self, chk):
        out = {}
        for name in KERAS:
            chk(name, self.a[name], self.u[name])
            g = self.g[name]
            if name.startswith("conv") and name.endswith("kernel"):
                g = g.permute(2, 3, 1, 0)                                      # [co][ci][kx][ky] -> Keras [kx][ky][ci][co]
            out[name] = g.cpu().numpy()
        return out


def _backward(torch, W, acts, q, action, y, c, chk, sums, bf=_bf16):
    """The backward of sum_i c * Huber(Q(s_i)[a_i] - y_i) for one chunk, rounded where the device rounds (dQ is
    clip(d) * c). Adds to the gradient sums and returns the TD errors d."""
    F = torch.nn.functional
    x, a1, a2, a3, h = acts
    n = x.shape[0]
    ar = torch.arange(n, device=x.device)
    d = q[ar, action] - y
    chk("td", q[ar, action].abs() + y.abs(), min(_unit(q), _unit(y)))
    dqa = d.clamp(-1.0, 1.0) * c
    dq = torch.zeros_like(q)
    dq[ar, action] = dqa
    w5a = W["k5"][:, action].T                                               # [n][512]
    chk("dH", (dqa[:, None] * w5a).abs(), _unit(dqa) * _unit(W["k5"]))
    dh = (h > 0) * (dqa[:, None] * w5a)                                      # f32 on the device
    dhb = bf(dh)
    sums.add("dense2_kernel", h.T @ dq, h.T @ dq.abs(), _unit(h) * _unit(dq))
    sums.add("dense2_bias", dq.sum(0), dq.abs().sum(0), _unit(dq))
    sums.add("dense1_bias", dh.sum(0), dh.abs().sum(0), _unit(dh))
    flat = a3.permute(0, 2, 3, 1).reshape(n, -1)
    sums.add("dense1_kernel", flat.T @ dhb, flat.T @ dhb.abs(), _unit(flat) * _unit(dhb))
    chk("dA3", dhb.abs() @ W["k4"].abs().T, _unit(dhb) * _unit(W["k4"]))
    dz = (dhb @ W["k4"].T) * (flat > 0)
    dz = dz.reshape(n, 7, 7, 64).permute(0, 3, 1, 2)                         # NCHW
    for i, a_in in ((3, a2), (2, a1), (1, x)):
        k, s = W["k%d" % i], STRIDES[i - 1]
        co = k.shape[0]
        dzb = bf(dz)
        sums.add("conv%d_bias" % i, dz.sum((0, 2, 3)), dz.abs().sum((0, 2, 3)), _unit(dz))
        cols = F.unfold(a_in, k.shape[2:], stride=s)                         # [n][ci*kx*ky][pixels]; a_in >= 0
        dzm = dzb.reshape(n, co, -1)
        sums.add("conv%d_kernel" % i, torch.einsum("nol,nkl->ok", dzm, cols).reshape(k.shape),
                 torch.einsum("nol,nkl->ok", dzm.abs(), cols).reshape(k.shape), _unit(a_in) * _unit(dzb))
        del cols
        if i == 1:
            break
        km = k.reshape(co, -1)
        ga = F.fold(km.abs().T @ dzm.abs(), a_in.shape[2:], k.shape[2:], stride=s)
        chk("dA%d" % (i - 1), ga, _unit(dzb) * _unit(k))
        dz = F.fold(km.T @ dzm, a_in.shape[2:], k.shape[2:], stride=s) * (a_in > 0)
    return d


# ---- seeded weights on the grid ----
def _draw_weights(qlb, draw):
    """Kernels of +-1 times 2^SCALE: the rows (kernel positions) of a layer are split over the N_DRAWS draws by one fixed
    permutation, each draw spreads its rows over the output units and tops every unit up to NNZ non-zeros. The head is
    dense in {-1, 0, 1} * 2^SCALE[4]. Biases are zero here (_calibrate sets them)."""
    rng = np.random.default_rng([7, draw])
    w = {}
    for li, name in enumerate(("conv1_kernel", "conv2_kernel", "conv3_kernel", "dense1_kernel")):
        shape = qlb.QNET_SHAPES[name]
        rows, cols = int(np.prod(shape[:-1])), shape[-1]
        mine = np.random.default_rng([7, li]).permutation(rows)[draw::N_DRAWS]
        m = np.zeros((rows, cols))
        m[mine, rng.permutation(np.resize(np.arange(cols), mine.size))] = rng.choice([-1.0, 1.0], size=mine.size)
        for c in range(cols):
            short = NNZ - np.count_nonzero(m[:, c])
            if short > 0:
                m[rng.choice(np.flatnonzero(m[:, c] == 0), size=short, replace=False), c] = rng.choice([-1.0, 1.0], size=short)
        w[name] = (m * 2.0 ** SCALE[li]).reshape(shape).astype(np.float32)
        w[name.replace("kernel", "bias")] = np.zeros(cols, np.float32)
    w["dense2_kernel"] = (rng.choice([-1.0, 0.0, 1.0], size=(512, 3)) * 2.0 ** SCALE[4]).astype(np.float32)
    w["dense2_bias"] = (rng.integers(-8, 9, size=3) * 2.0 ** sum(SCALE)).astype(np.float32)
    return w


def _calibrate(torch, w, x, seed):
    """Sets the conv and dense-1 biases, layer by layer on the stacks x: bias_c = -(a quantile, drawn from 0.35..0.65, of
    unit c's pre-activations), an element of the grid. Returns the fraction of positive activations per layer."""
    rng = np.random.default_rng(seed)
    W = _torch_weights(torch, w, x.device, _bf16)
    n, a, frac = x.shape[0], x, []
    for i, name in enumerate(("conv1", "conv2", "conv3", "dense1")):
        if i < 3:
            k = W["k%d" % (i + 1)]
            z = k.reshape(k.shape[0], -1) @ torch.nn.functional.unfold(a, k.shape[2:], stride=STRIDES[i])    # [n][units][pixels]
            zs = z.permute(1, 0, 2).reshape(k.shape[0], -1).T                                           # [samples][units]
        else:
            z = zs = a.permute(0, 2, 3, 1).reshape(n, -1) @ W["k4"]
        srt = torch.sort(zs, dim=0).values
        pick = torch.from_numpy((rng.uniform(0.35, 0.65, size=zs.shape[1]) * (zs.shape[0] - 1)).astype(np.int64)).to(x.device)
        b = -srt[pick, torch.arange(zs.shape[1], device=x.device)]
        w[name + "_bias"][:] = b.cpu().numpy().astype(np.float32)
        frac.append(float((zs + b > 0).double().mean()))
        if i < 3:
            side = (a.shape[2] - k.shape[2]) // STRIDES[i] + 1
            a = _bf16(torch.relu(z + b[:, None])).reshape(n, k.shape[0], side, side)
    return frac


# ---- the world: a replay with random pixels, one network, the reference outputs ----
class _World:
    def __init__(self, qlb, torch, pmax, tmpdir):
        self.qlb, self.torch, self.pmax = qlb, torch, pmax
        self.n_envs = n = 1024
        env = self.env = qlb.BreakoutEnvironment(n_envs=n, seed=5, replay_capacity=n * 64)
        rng = np.random.default_rng(5)
        env.step_many(rng.integers(0, 3, size=(50, n), dtype=np.uint8))
        env.reset(mask=(np.arange(n) % 7 == 0).astype(np.uint8))
        env.step_many(rng.integers(0, 3, size=(30, n), dtype=np.uint8))
        env.reset(mask=(np.arange(n) % 5 == 0).astype(np.uint8))
        env.step_many(rng.integers(0, 3, size=(3, n), dtype=np.uint8))
        self.time_slots = env.state_view().time_slots
        assert env.time() > self.time_slots                                 # the ring has wrapped
        # the frame ring is the last array of a checkpoint: overwrite it with seeded random pixels
        path = str(tmpdir / ("ring_p%d.ckpt" % pmax))
        env.save(path)
        nbytes = self.time_slots * n * 7056
        self.frames = np.random.default_rng(100 + pmax).integers(0, pmax + 1, size=nbytes, dtype=np.uint8)
        assert os.path.getsize(path) > nbytes
        with open(path, "r+b") as f:
            f.seek(-nbytes, os.SEEK_END)
            f.write(memoryview(self.frames))
        env.load(path)
        os.remove(path)
        self.rb = qlb.ReplayBuffer(env)
        assert self.rb.len() >= BIG
        self.perm = rng.permutation(self.rb.len())[:BIG].astype(np.uint32)
        sm = torch.cuda.get_device_properties(0).multi_processor_count
        self.last_narrow = 128 * ((sm - 1) // 2)                             # dense_tc_kernel<128> while m_tiles * 2 < sm
        assert self.last_narrow + 128 < BIG
        self.dev = torch.device("cuda")
        self._w, self._frac, self._qref = {}, {}, {}
        self.net, self._net_draw = None, None

    def stacks(self, idx, which, chunk=CHUNK):
        """(offset, f64 CUDA [n][4][84(x)][84(y)]) per chunk of the replay transitions idx."""
        for o in range(0, idx.size, chunk):
            smp = self.rb.get_many(idx[o:o + chunk], self.qlb.LAYOUT_U8_BXYH, want_state=which == 0, want_next=which == 1)
            st = smp.state if which == 0 else smp.state_next
            yield o, self.torch.from_numpy(st).to(self.dev).permute(0, 3, 1, 2).to(self.torch.float64)

    def weights(self, draw):
        if draw not in self._w:
            w = _draw_weights(self.qlb, draw)
            _, x = next(self.stacks(self.perm[:512], 0))
            self._frac[draw] = _calibrate(self.torch, w, x, 1000 * self.pmax + draw)
            self._w[draw] = w
        return self._w[draw]

    def use(self, draw):
        """The world's network, holding the weights of `draw`."""
        w = self.weights(draw)
        if self.net is None:
            self.net = self.qlb.QNetwork(self.env, w)
        elif self._net_draw != draw:
            self.net.set_weights(w)
        self._net_draw = draw
        return self.net

    def W(self, draw):
        return _torch_weights(self.torch, self.weights(draw), self.dev, _bf16)

    def q_ref(self, draw, which):
        """The reference Q of every item of the permutation (state or state_next), and the premise check's worst ratios."""
        if (draw, which) not in self._qref:
            W, chk = self.W(draw), _Premise()
            with self.torch.no_grad():
                q = np.concatenate([_forward(self.torch, W, x, chk)[0].cpu().numpy() for _, x in self.stacks(self.perm, which)])
            self._qref[(draw, which)] = q, chk.worst
            self.torch.cuda.empty_cache()
        return self._qref[(draw, which)]

    def size(self, name):
        ln = self.last_narrow
        return {"last_narrow": ln, "last_narrow+1": ln + 1, "last_narrow+3": ln + 3, "first_wide_tile": (ln + 1 + 127) // 128 * 128}.get(name) or int(name)

    def window(self, n):
        o = (n * 7919) % (BIG - n + 1)
        return o, self.perm[o:o + n]

    def release(self):
        """Closes the network (its buffers grow with the largest batch it ran); use() makes a new one."""
        if self.net is not None:
            self.net.close()
        self.net, self._net_draw = None, None

    def close(self):
        self.release()
        self.env.close()


@pytest.fixture(scope="module")
def lab(qlb, tmp_path_factory):
    """World(pmax) for pixel ranges 0..pmax, built on first use and kept for the module; only the world last asked for
    keeps a network."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    worlds = {}

    def get(pmax):
        for p, w in worlds.items():
            if p != pmax:
                w.release()
        if pmax not in worlds:
            worlds[pmax] = _World(qlb, torch, pmax, tmp_path_factory.mktemp("ring"))
        return worlds[pmax]
    yield get
    for w in worlds.values():
        w.close()


def _report(what, worst):
    k = max(worst, key=worst.get)
    print("\n[premise] %-44s largest sum |terms| / 2^24 units: %.3g (%s)" % (what, worst[k], k))


def _assert_equal(got, ref, what):
    got = np.asarray(got, dtype=np.float64)
    bad = got != ref
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: %d of %d elements differ; first at %s: got %r, expected %r"
                             % (what, int(bad.sum()), bad.size, i, float(got[i]), float(ref[i])))


def _first_argmax(q):
    return np.argmax(q, axis=1).astype(np.uint8)                            # numpy takes the first maximum, like tf.argmax


# ---- self-checks of the harness ----
def test_bf16_rounding_matches_torch():
    """_bf16 is torch's float -> bfloat16 conversion (round to nearest, ties to even) on random values of every magnitude
    and sign, on exact ties with an even and with an odd bf16 neighbour below, and one ulp either side of a tie."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(0)
    r = (rng.standard_normal(100000) * np.exp2(rng.integers(-60, 60, size=100000))).astype(np.float32)
    base = rng.integers(0x00800000, 0x7F000000, size=20000, dtype=np.int64) & ~0xFFFF
    ties = np.concatenate([base | 0x8000, base | 0x18000, base | 0x7FFF, base | 0x8001, base | 0x18001, base | 0x17FFF])
    t = np.concatenate([ties.astype(np.uint32).view(np.float32), r, np.float32([0.0, 1.0, 1.5, 255.0, 257.0, 259.0])])
    t = np.concatenate([t, -t])
    x = torch.from_numpy(t).to(torch.float64)
    want = x.to(torch.float32).to(torch.bfloat16).to(torch.float64)
    got = _bf16(x)
    assert torch.equal(got, want)
    assert torch.equal(_bf16(torch.tensor([257.0, 259.0, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8], dtype=torch.float64)),
                       torch.tensor([256.0, 260.0, 1.0, 1.0 + 2.0 ** -6], dtype=torch.float64))


def test_unit_is_the_largest_dividing_power_of_two():
    torch = pytest.importorskip("torch")
    t = torch.tensor([0.0, 3.0 * 2.0 ** -5, -12.0, 2.0 ** 20], dtype=torch.float64)
    assert _unit(t) == 2.0 ** -5 and _unit(t[1:2]) == 2.0 ** -5 and _unit(t[2:]) == 4.0 and _unit(t[:1]) == math.inf


def test_reference_backward_matches_autograd(qlb):
    """With the bf16 rounding replaced by the identity, the reference's forward and hand-written backward equal torch
    autograd through F.conv2d on the Keras model (float64, random weights and pixels; rel. 1e-9): the unfold / fold index
    maps, the Flatten order, the masks and the Keras layouts of the reference are right."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.default_rng(1)
    n = 3
    w = {k: (rng.standard_normal(s) / np.sqrt(np.prod(s[:-1]) if len(s) > 1 else 10)).astype(np.float32) for k, s in qlb.QNET_SHAPES.items()}
    x = torch.from_numpy(rng.integers(0, 256, size=(n, 4, 84, 84)).astype(np.float64))
    x[1, :2] = 0                                                             # a partial stack
    action = torch.tensor([2, 0, 1])
    ident = lambda t: t
    W = _torch_weights(torch, w, "cpu", ident)
    q, acts = _forward(torch, W, x, _no_check, bf=ident)
    y = q[torch.arange(n), action] - torch.tensor([0.4, -3.0, 0.7], dtype=torch.float64)     # quadratic and saturated items
    sums = _GradSums()
    scale = 0.25
    _backward(torch, W, acts, q, action, y, scale, _no_check, sums, bf=ident)
    got = sums.keras(_no_check)
    P = {k: torch.tensor(v.astype(np.float64), requires_grad=True) for k, v in w.items()}
    h = x
    for i in (1, 2, 3):
        h = torch.relu(F.conv2d(h, P["conv%d_kernel" % i].permute(3, 2, 0, 1), P["conv%d_bias" % i], stride=STRIDES[i - 1]))
    h = torch.relu(h.permute(0, 2, 3, 1).reshape(n, -1) @ P["dense1_kernel"] + P["dense1_bias"])
    qq = h @ P["dense2_kernel"] + P["dense2_bias"]
    assert torch.allclose(q, qq.detach(), rtol=1e-12, atol=1e-9)
    (scale * F.huber_loss(qq[torch.arange(n), action], y, reduction="sum", delta=1.0)).backward()
    for k in KERAS:
        ref = P[k].grad.numpy()
        assert np.abs(ref).max() > 0, k
        assert np.allclose(got[k], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max()), (k, np.abs(got[k] - ref).max())


@gpu
@pytest.mark.parametrize("pmax", [1, 15])
def test_checkpoint_patch_reaches_the_frame_ring(lab, qlb, pmax):
    """After the load, the current stacks hold the injected bytes: slot h of env e is frame (T - d) mod time_slots of e,
    d = ((k - h - 1) mod 4) + 1, where the episode has that frame (d <= k), and zeros where it does not."""
    world = lab(pmax)
    env, n, ts = world.env, world.n_envs, world.time_slots
    obs = env.obs(qlb.LAYOUT_U8_BHYX)
    ks = env.read_state()["episode_step"].astype(np.int64)
    k = np.where(ks < 4, ks, 4 + (ks & 3))
    frames = world.frames.reshape(ts * n, 84, 84)
    T = env.time()
    present = np.zeros((n, 4), bool)
    for h in range(4):
        d = ((k - h - 1) & 3) + 1
        present[:, h] = d <= k
        exp = np.where(present[:, h, None, None], frames[((T - d) % ts) * n + np.arange(n)], 0)
        assert np.array_equal(obs[:, h], exp), h
    assert present.all(axis=1).any() and (~present).any(axis=1).any() and present.any(axis=1).any()
    assert obs.max() == pmax


@gpu
@pytest.mark.parametrize("pmax", [1, 15])
def test_weight_draws_cover_every_kernel_row_and_masks_are_mixed(lab, pmax):
    """Across the draws every kernel row (kernel position x input channel) of every layer is non-zero, every draw has
    20-80 % positive activations in each ReLU layer, and the replay holds all-zero and partial stacks."""
    world = lab(pmax)
    ws = [world.weights(dr) for dr in range(N_DRAWS)]
    for name in ("conv1_kernel", "conv2_kernel", "conv3_kernel", "dense1_kernel"):
        rows = np.any([w[name].reshape(-1, w[name].shape[-1]) != 0 for w in ws], axis=0).any(axis=1)
        assert rows.all(), name
    for dr in range(N_DRAWS):
        assert all(0.2 <= f <= 0.8 for f in world._frac[dr]), (dr, world._frac[dr])
    st = world.rb.get_many(world.perm[:4096], world.qlb.LAYOUT_U8_BXYH, want_next=False).state
    per_slot = st.reshape(4096, -1, 4).max(axis=1)
    assert (per_slot.max(axis=1) == 0).any() and ((per_slot.min(axis=1) == 0) & (per_slot.max(axis=1) > 0)).any()


# ---- forward ----
@gpu
@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("draw", range(N_DRAWS))
@pytest.mark.parametrize("pmax", [1, 15])
def test_forward_is_exact(lab, pmax, draw, size, which):
    """Q, the greedy action (first maximum) and max Q of every item equal the reference, for state (0) and state_next (1),
    at every size where a kernel changes shape. Integer-grid Q values tie often, so the tie rule is checked on every item."""
    world = lab(pmax)
    n = world.size(size)
    o, idx = world.window(n)
    q_all, worst = world.q_ref(draw, which)
    q_ref = q_all[o:o + n]
    q, action, max_q = world.use(draw).forward(idx, which)
    what = "forward pmax=%d draw=%d n=%d which=%d" % (pmax, draw, n, which)
    _assert_equal(q, q_ref, what + " Q")
    assert np.array_equal(action, _first_argmax(q_ref)), what
    _assert_equal(max_q, q_ref.max(axis=1), what + " max Q")
    if n == BIG:
        srt = np.sort(q_ref, axis=1)
        assert (srt[:, 2] == srt[:, 1]).sum() > 10, "degenerate test: no ties at the maximum"
        assert len(np.unique(q_ref)) > 50, "degenerate test: too few distinct Q values"
        _report(what, worst)


@gpu
@pytest.mark.parametrize("draw", range(N_DRAWS))
@pytest.mark.parametrize("pmax", [1, 15])
def test_forward_current_observation_is_exact(lab, qlb, pmax, draw):
    """forward() with no indices (the actor's path: the current stacks of all 1,024 envs, some just reset)."""
    world = lab(pmax)
    q, action, max_q = world.use(draw).forward()
    obs = world.env.obs(qlb.LAYOUT_U8_BXYH)
    x = world.torch.from_numpy(obs).to(world.dev).permute(0, 3, 1, 2).to(world.torch.float64)
    chk = _Premise()
    with world.torch.no_grad():
        q_ref = _forward(world.torch, world.W(draw), x, chk)[0].cpu().numpy()
    _assert_equal(q, q_ref, "current observation")
    assert np.array_equal(action, _first_argmax(q_ref))
    _assert_equal(max_q, q_ref.max(axis=1), "current observation max Q")


# ---- gradients ----
def _targets(q_ref, action, seed):
    """y = Q_a - d with d on the grid: 40 % in the quadratic branch (|d| <= 3/4), 50 % saturated (|d| >= 1), 10 % zero."""
    rng = np.random.default_rng(seed)
    b = q_ref.shape[0]
    kind = rng.integers(0, 10, size=b)
    quad = rng.choice([-0.75, -0.5, -0.25, 0.25, 0.5, 0.75], size=b)
    sat = rng.choice([-1.0, 1.0], size=b) * rng.choice([1.0, 1.25, 1.5, 2.0, 3.0], size=b)
    d = np.where(kind < 4, quad, np.where(kind < 9, sat, 0.0))
    y = q_ref[np.arange(b), action.astype(np.int64)] - d
    assert np.array_equal(y.astype(np.float32), y), "targets off the f32 grid"
    return y


def _reference_grads(world, draw, idx, action, y, c):
    torch = world.torch
    W, chk, sums = world.W(draw), _Premise(), _GradSums()
    td = []
    with torch.no_grad():
        for o, x in world.stacks(idx, 0, GRAD_CHUNK):
            q, acts = _forward(torch, W, x, chk)
            a = torch.from_numpy(action[o:o + GRAD_CHUNK].astype(np.int64)).to(world.dev)
            yy = torch.from_numpy(y[o:o + GRAD_CHUNK]).to(world.dev)
            td.append(_backward(torch, W, acts, q, a, yy, c, chk, sums).cpu().numpy())
            del acts
        out = sums.keras(chk), np.concatenate(td), chk.worst
    torch.cuda.empty_cache()
    return out


def _check_grads(qlb, g, ref, what):
    for name in KERAS:
        assert np.abs(ref[name]).max() > 0, (what, name, "degenerate test: zero gradient")
        _assert_equal(g[name], ref[name], "%s %s" % (what, name))


GRAD_CASES = [(15, "1"), (15, "3"), (15, "32"), (15, "129"), (15, "300"), (15, "2000"), (15, "last_narrow+1"), (1, "2000"),
              (1, "last_narrow+1"), (1, str(BIG))]


@gpu
@pytest.mark.parametrize("pmax,size", GRAD_CASES)
def test_weighted_gradients_are_exact(lab, qlb, pmax, size):
    """All ten gradients element by element and the TD errors, with loss weights b * 2^-M (dL/dQ = clip(d) * 2^-M
    exactly), from one item to 32,768 (every K slice of the split weight gradients, every split of the column sums). The
    longest sum is conv1's weight gradient, 400 b products: 0..15 pixels keep it below 2^24 units up to last_narrow + 1
    items, binary pixels at 32,768."""
    world = lab(pmax)
    b = world.size(size)
    draw = GRAD_CASES.index((pmax, size)) % N_DRAWS
    net = world.use(draw)
    o, idx = world.window(b)
    action = world.rb.get_many(idx, want_state=False, want_next=False).action
    y = _targets(world.q_ref(draw, 0)[0][o:o + b], action, b)
    wb = b * 2.0 ** -M_WEIGHT
    assert np.float32(wb) == wb
    g, td = net.debug_grads_weighted(idx, y.astype(np.float32), np.full(b, wb, np.float32))
    ref, td_ref, worst = _reference_grads(world, draw, idx, action, y, 2.0 ** -M_WEIGHT)
    what = "gradients pmax=%d b=%d" % (pmax, b)
    _assert_equal(td, td_ref, what + " td")
    _check_grads(qlb, g, ref, what)
    _report(what, worst)


@gpu
def test_unweighted_gradients_are_exact(lab, qlb):
    """debug_grads (no loss weights) at b = 256, a power of two: dL/dQ = clip(d) / b is exact."""
    world = lab(15)
    b = 256
    net = world.use(1)
    o, idx = world.window(b)
    action = world.rb.get_many(idx, want_state=False, want_next=False).action
    y = _targets(world.q_ref(1, 0)[0][o:o + b], action, 11)
    g = net.debug_grads(idx, y.astype(np.float32))
    ref, _, worst = _reference_grads(world, 1, idx, action, y, 1.0 / b)
    _check_grads(qlb, g, ref, "unweighted gradients b=%d" % b)
    _report("unweighted gradients b=%d" % b, worst)


# ---- Adam ----
def _blocks(qlb):
    out, off = [], 0
    for name in KERAS:
        size = int(np.prod(qlb.QNET_SHAPES[name]))
        out.append((off, size))
        off += size
    return out


def _flat(w):
    return np.concatenate([np.asarray(w[k], np.float32).ravel() for k in KERAS])


def _norms(qlb, g):
    """sumsq_partial_kernel + the norm of adam_kernel, in their order: per variable 32 chunks of ceil(n / 32); in a chunk 256
    thread-strided running sums of squares, then the shared-memory halving tree; the 32 chunk partials in order; sqrtf."""
    out = []
    for off, n in _blocks(qlb):
        per = -(-n // 32)
        rows = -(-per // 256)
        sq = np.zeros(32 * per, np.float32)
        p = g[off:off + n]
        sq[:n] = p * p
        x = np.zeros((32, rows * 256), np.float32)
        x[:, :per] = sq.reshape(32, per)
        x = x.reshape(32, rows, 256)
        acc = np.zeros((32, 256), np.float32)
        for r in range(rows):
            acc = acc + x[:, r, :]
        w = 128
        while w:
            acc[:, :w] = acc[:, :w] + acc[:, w:2 * w]
            w >>= 1
        t = np.float32(0.0)
        for c in range(32):
            t = np.float32(t + acc[c, 0])
        out.append(np.sqrt(t))
    return out


def _adam_step(qlb, w, m, v, g, t, cfg):
    """One update of the flat f32 blocks w, m, v (in place) as adam_kernel computes it; alpha formed in double and cast,
    1 - beta in double and cast, as qnet_train_step does."""
    lr, b1, b2, eps, clip = (float(np.float32(cfg[k])) for k in ("lr", "beta1", "beta2", "epsilon", "clipnorm"))
    alpha = np.float32(lr * math.sqrt(1.0 - b2 ** float(t)) / (1.0 - b1 ** float(t)))
    one_b1, one_b2, eps, clip = np.float32(1.0 - b1), np.float32(1.0 - b2), np.float32(eps), np.float32(clip)
    norms = _norms(qlb, g)
    for (off, n), nrm in zip(_blocks(qlb), norms):
        s = slice(off, off + n)
        gi = g[s]
        if clip > 0:
            gi = (gi * clip) / np.maximum(nrm, clip)
        mi = m[s] + (gi - m[s]) * one_b1
        vi = v[s] + (gi * gi - v[s]) * one_b2
        m[s], v[s] = mi, vi
        w[s] = w[s] - (mi * alpha) / (np.sqrt(vi) + eps)
    return norms


def _adam_world(world, seed):
    """A Q-network with Glorot-uniform weights (any weights do: the update is checked on the library's own gradients)."""
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in world.qlb.QNET_SHAPES.items():
        if name.endswith("kernel"):
            lim = np.sqrt(6.0 / (np.prod(shape[:-1]) + shape[-1]))
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        else:
            w[name] = rng.uniform(-0.1, 0.1, size=shape).astype(np.float32)
    return w


def _assert_same_bits(got, exp, what):
    bad = got.view(np.uint32) != exp.view(np.uint32)
    if bad.any():
        i = int(np.argmax(bad))
        ulp = np.abs(got.view(np.int32).astype(np.int64) - exp.view(np.int32).astype(np.int64)).max()
        raise AssertionError("%s: %d of %d weights differ (up to %d ulp); first at %d: got %r, expected %r" % (what, int(bad.sum()), bad.size, ulp, i, got[i], exp[i]))


@gpu
@pytest.mark.parametrize("config", ["no_clip", "clip_between_norms", "beta2_0.95"])
def test_adam_steps_are_bit_exact(lab, qlb, config):
    """50 updates of one minibatch (32 items, fixed targets): after each, the f32 master weights equal, bit for bit, the
    update restated in float32 in the kernels' own operation order from the library's own gradients (debug_grads on the
    same weights: the update is deterministic, so these are the gradients it used). clip_between_norms sets clipnorm
    between the variables' gradient norms so that some variables are clipped and others are not."""
    world = lab(15)
    net = qlb.QNetwork(world.env, _adam_world(world, 7))
    idx = world.perm[:32]
    smp = world.rb.get_many(idx, qlb.LAYOUT_U8_BXYH, want_state=False, want_next=False)
    y = (smp.reward + np.float32(0.5)).astype(np.float32)
    cfg = dict(lr=2.5e-4, beta1=0.9, beta2=0.999, epsilon=1e-7, clipnorm=0.0)
    if config == "clip_between_norms":
        g0 = net.debug_grads(idx, y)
        nrm = sorted(float(np.linalg.norm(g0[k].astype(np.float64))) for k in g0)
        cfg["clipnorm"] = float(np.float32((nrm[4] + nrm[5]) / 2))
    if config == "beta2_0.95":
        cfg.update(lr=1e-3, beta2=0.95, clipnorm=1.0)
    net.set_adam(**cfg)
    w = _flat(net.get_weights())
    m, v = np.zeros_like(w), np.zeros_like(w)
    clipped = set()
    for t in range(1, 51):
        g = _flat(net.debug_grads(idx, y))
        norms = _adam_step(qlb, w, m, v, g, t, cfg)
        clipped |= {k for k, nv in zip(KERAS, norms) if cfg["clipnorm"] > 0 and nv > cfg["clipnorm"]}
        net.train(idx, y)
        _assert_same_bits(_flat(net.get_weights()), w, "%s step %d" % (config, t))
    if config == "clip_between_norms":
        assert 0 < len(clipped) < 10, clipped
    net.close()


@gpu
def test_three_minibatches_in_one_call_are_three_restated_steps(lab, qlb):
    """train(n_batches=3) equals three restated updates on the gradients of each minibatch at the weights it meets
    (taken from a second network that steps one minibatch at a time)."""
    world = lab(15)
    w0 = _adam_world(world, 8)
    cfg = dict(lr=5e-4, beta1=0.9, beta2=0.999, epsilon=1e-7, clipnorm=1.0)
    one, step = qlb.QNetwork(world.env, w0), qlb.QNetwork(world.env, w0)
    one.set_adam(**cfg)
    step.set_adam(**cfg)
    idx = world.perm[100:196]
    smp = world.rb.get_many(idx, qlb.LAYOUT_U8_BXYH, want_state=False, want_next=False)
    y = (smp.reward - np.float32(0.25)).astype(np.float32)
    w = _flat(w0)
    m, v = np.zeros_like(w), np.zeros_like(w)
    for j in range(3):
        s = slice(32 * j, 32 * (j + 1))
        _adam_step(qlb, w, m, v, _flat(step.debug_grads(idx[s], y[s])), j + 1, cfg)
        step.train(idx[s], y[s])
        _assert_same_bits(_flat(step.get_weights()), w, "single step %d" % (j + 1))
    one.train(idx, y, n_batches=3)
    _assert_same_bits(_flat(one.get_weights()), w, "n_batches=3")
    one.close()
    step.close()
