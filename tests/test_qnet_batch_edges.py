"""The Q-network at the batch sizes where its kernels change shape: the dense layer's N tile of 256 (dense_tc_kernel<256>,
taken once (M tiles x 2) CTAs fill the SMs), the tails of every 128-item tile, and the split-K weight gradients and split
column sums of training at 9,345 and 32,768 items.

One reference throughout: the Keras model in float64 torch on the GPU, with weights and the activations between layers
rounded straight from f64 to bf16 at the points where the tensor-core path rounds them (accumulation in f64, the head in
f32 weights like the device's), rounding passed through unchanged by autograd. Errors are bounded per item (forward) or on
sets of a few items (gradients), so one wrong row at a tile tail or a K-slice boundary cannot hide in a batch-wide norm."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BIG = 32768          # the largest minibatch DESIGN §11 reports
CHUNK = 2048         # items per reference chunk (f64 activations of one chunk: about 1 GB with autograd)
KC = 64              # K elements per weight-gradient pipeline step (qnet.cuh KC)


def _random_weights(qlb, seed):
    rng = np.random.default_rng(seed)
    w = {}
    for name, shape in qlb.QNET_SHAPES.items():
        if name.endswith("kernel"):
            fan_in = int(np.prod(shape[:-1])); fan_out = shape[-1]
            lim = np.sqrt(6.0 / (fan_in + fan_out))                      # Keras default glorot_uniform
            w[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        else:
            w[name] = rng.uniform(-0.1, 0.1, size=shape).astype(np.float32)
    return w


# ---- restatement of the split choices in qlc_api.cu (pick_splits, wgrad_shapes, colsum_rows_per_split) ----
def _pick_splits(k_valid, mn_tiles):
    chunks = (k_valid + KC - 1) // KC
    sp = max(1, min((296 + mn_tiles - 1) // mn_tiles, 64, (chunks + 1) // 2))
    per = (chunks + sp - 1) // sp
    return (chunks + per - 1) // per, per * KC


WGRAD = {"dense1": (1, 50), "conv3": (49, 5), "conv2": (81, 4), "conv1": (400, 2)}     # K rows per item, M x N tiles


def _colsum_rows_per_split(rows):
    return max(256, (rows + 63) // 64)


def _straddling_items(boundaries, per_item):
    """Items holding K (or row) indices z - 1 and z of every slice boundary z."""
    out = set()
    for z in boundaries:
        out |= {(z - 1) // per_item, z // per_item}
    return out


def _boundary_sets(b):
    """Positions in a minibatch of b whose items sit on a slice boundary: of each weight-gradient GEMM (K = item * pixels +
    pixel, slices of kc) and of each split column sum (rows = item * pixels + pixel, splits of rows_per_split)."""
    sets = {}
    for name, (per, mn) in WGRAD.items():
        splits, kc = _pick_splits(b * per, mn)
        sets["wgrad_" + name] = _straddling_items([z * kc for z in range(1, splits)], per)
    for name, per in (("head", 1), ("conv3", 49), ("conv2", 81), ("conv1", 400)):
        rps = _colsum_rows_per_split(b * per)
        sets["colsum_" + name] = _straddling_items(list(range(rps, b * per, rps)), per)
    return {k: np.array(sorted(v), np.int64) for k, v in sets.items()}


# ---- the f64 reference ----
def _bf(torch, t):
    """Round f64 to the nearest bf16 value (ties to even), kept in f64, straight-through for autograd: r - t is exact
    (Sterbenz), so t + (r - t) is r."""
    u = t.detach().contiguous().view(torch.int64)
    r = ((u + ((1 << 44) - 1) + ((u >> 45) & 1)) & ~((1 << 45) - 1)).view(torch.float64)
    return t + (r - t.detach())


def _forward(torch, W, x):
    """Keras model on x [B][4][84(x)][84(y)] f64; returns (Q [B][3], the bf16-rounded dense-1 activations [B][512])."""
    F = torch.nn.functional
    for i in (1, 2, 3):
        k = _bf(torch, W["conv%d_kernel" % i].permute(3, 2, 0, 1))
        x = _bf(torch, torch.relu(F.conv2d(x, k, W["conv%d_bias" % i], stride={1: 4, 2: 2, 3: 1}[i])))
    x = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)                        # Flatten of [7][7][64]
    h = _bf(torch, torch.relu(x @ _bf(torch, W["dense1_kernel"]) + W["dense1_bias"]))
    return h @ W["dense2_kernel"] + W["dense2_bias"], h


def _weights64(torch, w, grad=False):
    return {k: torch.tensor(v, dtype=torch.float64, device="cuda", requires_grad=grad) for k, v in w.items()}


def _stacks(torch, qlb, rb, idx, which):
    """(offset, f64 CUDA [n][4][84(x)][84(y)]) per chunk of the replay transitions idx (state or state_next), u8 on the host."""
    for o in range(0, idx.size, CHUNK):
        smp = rb.get_many(idx[o:o + CHUNK], qlb.LAYOUT_U8_BXYH, want_state=which == 0, want_next=which == 1)
        st = smp.state if which == 0 else smp.state_next
        yield o, torch.from_numpy(st).cuda().permute(0, 3, 1, 2).to(torch.float64)


def _reference_q(torch, w, chunks):
    """(Q [n][3], hw [n][3] = sum_j |h_j w5_ja|, s [n] = max_a (|b5_a| + hw_a)) over (offset, stack chunk) pairs."""
    W = _weights64(torch, w)
    qs, hws = [], []
    with torch.no_grad():
        for _, x in chunks:
            q, h = _forward(torch, W, x)
            qs.append(q.cpu().numpy()); hws.append((h.abs() @ W["dense2_kernel"].abs()).cpu().numpy())
    q, hw = np.concatenate(qs), np.concatenate(hws)
    return q, hw, (np.abs(w["dense2_bias"].astype(np.float64)) + hw).max(axis=1)


def _reference_grads(torch, qlb, rb, w, idx, action, y, b):
    """f64 gradients of (1/b) sum_i Huber(Q(s_i)[a_i] - y_i) over the items idx, accumulated chunk by chunk."""
    W = _weights64(torch, w, grad=True)
    for o, x in _stacks(torch, qlb, rb, idx, 0):
        q, _ = _forward(torch, W, x)
        a = torch.from_numpy(action[o:o + CHUNK].astype(np.int64)).cuda()
        d = q.gather(1, a.unsqueeze(1)).squeeze(1) - torch.from_numpy(y[o:o + CHUNK].astype(np.float64)).cuda()
        ad = d.abs()
        (torch.where(ad <= 1, 0.5 * d * d, ad - 0.5).sum() / b).backward()
    return {k: W[k].grad.cpu().numpy() for k in W}


def _report(what, ratio):
    print("\n[margin] %-58s worst error / tolerance = %.3g" % (what, ratio))


def _check_forward(q, action, max_q, q_ref, s, what):
    """|q - ref| <= 1e-2 * s_i + 1e-6 for every item and action; action and max_q exactly the first argmax / max of q."""
    err = np.abs(q.astype(np.float64) - q_ref)
    ratio = err / (1e-2 * s[:, None] + 1e-6)
    i = int(ratio.max(axis=1).argmax())
    assert ratio.max() <= 1.0, (what, "item", i, q[i], q_ref[i], s[i])
    assert np.array_equal(action, q.argmax(axis=1).astype(np.uint8)), what
    assert np.array_equal(max_q, q.max(axis=1)), what
    _report(what, ratio.max())


def _check_grads(qlb, g, ref, what, tol=2e-2):
    worst = (0.0, None)
    for name in qlb.QNET_SHAPES:
        assert np.all(np.isfinite(g[name])), (what, name)
        nref = np.linalg.norm(ref[name])
        assert nref > 0, (what, name)
        e = np.linalg.norm(g[name].astype(np.float64) - ref[name]) / nref
        assert e <= tol, (what, name, e)
        worst = max(worst, (e / tol, name))
    _report("%s, %s" % (what, worst[1]), worst[0])


def _saturating_targets(q, action, seed):
    """Targets at least 2 from the library's Q(s)[a]: the Huber gradient is then +-1/b on both sides, so forward rounding
    differences do not reach dL/dq."""
    qa = q[np.arange(q.shape[0]), action.astype(np.int64)]
    rng = np.random.default_rng(seed)
    return (qa + rng.choice([-1.0, 1.0], size=qa.size) * (2.0 + rng.uniform(0, 1, size=qa.size))).astype(np.float32)


class _World:
    """A replay of 40,960 transitions (1,024 envs) holding episode starts and partially filled stacks, one network, and a
    fixed permutation of the replay whose windows give the minibatches."""

    def __init__(self, qlb, torch):
        self.qlb, self.torch = qlb, torch
        n_envs = 1024
        self.env = qlb.BreakoutEnvironment(n_envs=n_envs, seed=5, replay_capacity=n_envs * 64)
        rng = np.random.default_rng(5)
        self.env.step_many(rng.integers(0, 3, size=(30, n_envs), dtype=np.uint8))
        self.env.reset(mask=(np.arange(n_envs) % 7 == 0).astype(np.uint8))
        self.env.step_many(rng.integers(0, 3, size=(10, n_envs), dtype=np.uint8))
        self.rb = qlb.ReplayBuffer(self.env)
        assert self.rb.len() >= BIG
        self.perm = rng.permutation(self.rb.len())[:BIG].astype(np.uint32)
        self.w = _random_weights(qlb, 3)
        self.net = qlb.QNetwork(self.env, self.w)
        sm = torch.cuda.get_device_properties(0).multi_processor_count
        self.last_narrow = 128 * ((sm - 1) // 2)         # dense_tc_kernel<128> while m_tiles * 2 < sm
        assert self.last_narrow + 128 < BIG
        self._ref = {}

    def window(self, n):
        """n distinct replay indices: a window of the permutation, at an offset that depends on n."""
        o = (n * 7919) % (BIG - n + 1)
        return o, self.perm[o:o + n]

    def reference(self, which):
        """The f64 reference (Q, hw, s) of every item of the permutation, state (0) or state_next (1)."""
        if which not in self._ref:
            self._ref[which] = _reference_q(self.torch, self.w, _stacks(self.torch, self.qlb, self.rb, self.perm, which))
        return self._ref[which]

    def close(self):
        self.net.close(); self.env.close()


@pytest.fixture(scope="module")
def world(qlb):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    w = _World(qlb, torch)
    yield w
    w.close()


def _sizes():
    return ["1", "127", "128", "129", "last_narrow", "last_narrow+1", "last_narrow+3", "first_wide_tile", str(BIG)]


def _size(world, name):
    ln = world.last_narrow
    return {"last_narrow": ln, "last_narrow+1": ln + 1, "last_narrow+3": ln + 3, "first_wide_tile": (ln + 1 + 127) // 128 * 128}.get(name) or int(name)


def test_replay_holds_episode_starts_and_partial_stacks(qlb, world):
    """The permutation the tests draw from holds stacks with every frame zero (episode starts: Q from the biases alone) and
    stacks with some zero frames."""
    st = world.rb.get_many(world.perm[:4096], qlb.LAYOUT_U8_BXYH, want_next=False).state
    per_slot = st.reshape(4096, -1, 4).max(axis=1)
    assert (per_slot.max(axis=1) == 0).any()
    assert ((per_slot.min(axis=1) == 0) & (per_slot.max(axis=1) > 0)).any()


def test_wide_dense_kernel_runs_past_the_boundary(qlb, world):
    """The boundary comes from the device's SM count: last_narrow items run dense_tc_kernel<128>, one more runs
    dense_tc_kernel<256> (checked on the profiler's kernel names, so the wide-path tests cannot silently stop covering it)."""
    torch = world.torch
    from torch.profiler import ProfilerActivity, profile

    def kernels(n):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            world.net.forward(world.window(n)[1], 0)
            torch.cuda.synchronize()
        return " ".join(e.key for e in prof.key_averages())
    narrow, wide = kernels(world.last_narrow), kernels(world.last_narrow + 1)
    assert "dense_tc_kernel<128>" in narrow and "dense_tc_kernel<256>" not in narrow, narrow
    assert "dense_tc_kernel<256>" in wide and "dense_tc_kernel<128>" not in wide, wide


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("size", _sizes())
def test_forward_per_item_bound(qlb, world, size, which):
    """Every item and action: |q - ref| <= 1e-2 * s_i + 1e-6 with s_i = max_a (|b5_a| + sum_j |h_ij w5_ja|) from the
    reference, at the tails of the 128-item tile (conv2 packs 2 items per CTA and conv3 3, so odd sizes and sizes not a
    multiple of 3 leave partial conv batches too), on both sides of the narrow / wide boundary and at 32,768 items.
    Tolerance: s_i bounds every partial sum of the head, so an error of each activation relative to itself maps to at most
    that relative error of s_i. The device and the reference round at the same four points; where the f32 and the f64
    accumulation fall on opposite sides of a bf16 rounding boundary an activation moves by one bf16 ulp (<= 2^-8
    relative, 3.9e-3), and a flip in a conv layer reaches the dense sums through weights of both signs. 1e-2 is the
    batch-wide tolerance of test_qnet.py, now per item: an item whose Q is small (an episode start) is held to its own
    scale. The 1e-6 floor covers items whose head sums are all near zero."""
    n = _size(world, size)
    o, idx = world.window(n)
    q, action, max_q = world.net.forward(idx, which)
    q_ref, _, s = world.reference(which)
    _check_forward(q, action, max_q, q_ref[o:o + n], s[o:o + n], "forward n=%d which=%d" % (n, which))


def test_forward_current_observation_wide(qlb, world):
    """forward() with no indices (the actor's path, reading the current stacks) on last_narrow + 1 envs, some of them just
    reset: the per-item bound of test_forward_per_item_bound."""
    torch = world.torch
    n = world.last_narrow + 1
    env = qlb.BreakoutEnvironment(n_envs=n, seed=17, replay_capacity=n * 8)
    rng = np.random.default_rng(17)
    env.step_many(rng.integers(0, 3, size=(6, n), dtype=np.uint8))
    env.reset(mask=(np.arange(n) % 5 == 0).astype(np.uint8))
    env.step_many(rng.integers(0, 3, size=(2, n), dtype=np.uint8))
    net = qlb.QNetwork(env, world.w)
    q, action, max_q = net.forward()
    obs = env.obs(qlb.LAYOUT_U8_BXYH)
    chunks = ((o, torch.from_numpy(obs[o:o + CHUNK]).cuda().permute(0, 3, 1, 2).to(torch.float64)) for o in range(0, n, CHUNK))
    q_ref, _, s = _reference_q(torch, world.w, chunks)
    _check_forward(q, action, max_q, q_ref, s, "current observation n=%d" % n)
    net.close(); env.close()


def _permuted_runs(world, base, seed):
    """base indices plus 24 repeats of some of them, in two random orders: each item's Q must be the same bits in both
    orders and in every copy."""
    rng = np.random.default_rng(seed)
    items = np.concatenate([base, rng.choice(base, size=24, replace=False)])
    pa, pb = rng.permutation(items.size), rng.permutation(items.size)
    qa, aa, ma = world.net.forward(items[pa], 0)
    qb, ab, mb = world.net.forward(items[pb], 0)
    qa_u, qb_u = np.empty_like(qa), np.empty_like(qb)
    qa_u[pa], qb_u[pb] = qa, qb                        # back to the order of `items`
    assert np.array_equal(qa_u.view(np.uint32), qb_u.view(np.uint32))
    ma_u, aa_u = np.empty_like(ma), np.empty_like(aa)
    ma_u[pa], aa_u[pa] = ma, aa
    mb_u, ab_u = np.empty_like(mb), np.empty_like(ab)
    mb_u[pb], ab_u[pb] = mb, ab
    assert np.array_equal(ma_u.view(np.uint32), mb_u.view(np.uint32)) and np.array_equal(aa_u, ab_u)
    first = {int(v): i for i, v in reversed(list(enumerate(items)))}
    dup = np.arange(base.size, items.size)
    orig = np.array([first[int(v)] for v in items[dup]])
    assert np.array_equal(qa_u[dup].view(np.uint32), qa_u[orig].view(np.uint32))


def test_forward_is_independent_of_position_and_duplicates(qlb, world):
    """Bit-exact: every output row accumulates over K in an order fixed by the kernels alone (conv rows, dense rows, the head's
    partials in tile order), so an item's Q may not depend on where it sits in the batch or who its neighbours are. 1,000
    items plus 24 repeats in two orders (narrow), and the same within one wide batch of last_narrow + 1,000 items."""
    _permuted_runs(world, world.window(1000)[1], 1)
    base = world.window(world.last_narrow + 1000 - 24)[1]
    assert base.size + 24 > world.last_narrow
    _permuted_runs(world, base, 2)


def test_narrow_and_wide_agree(qlb, world):
    """The same last_narrow + 1 items in one wide call and in two narrow calls. The conv layers are the same kernels and the
    dense layer multiplies the same bf16 operands, so a hidden unit can at most move by one bf16 ulp (2^-7 relative at the
    top, 2^-8 typical); the head sums 512 products in 2 tiles of 256 (wide) or 4 of 128 (narrow), each sum of at most
    256 + 2 + 1 rounded f32 terms, so the two differ by at most 2 * 259 * 2^-24 * s_i. Bound:
    |dq_a| <= 2^-7 * sum_j |h_j w5_ja| + 3.1e-5 * s_i."""
    n = world.last_narrow + 1
    o, idx = world.window(n)
    qw, _, _ = world.net.forward(idx, 0)
    half = n // 2
    qn = np.concatenate([world.net.forward(idx[:half], 0)[0], world.net.forward(idx[half:], 0)[0]])
    _, hw, s = world.reference(0)
    hw, s = hw[o:o + n], s[o:o + n]
    d = np.abs(qw.astype(np.float64) - qn)
    ratio = d / (2.0 ** -7 * hw + 3.1e-5 * s[:, None])
    assert ratio.max() <= 1.0, float(ratio.max())
    print("\n[observed] narrow vs wide: max |dq| / s_i = %.3g, items differing: %d of %d" % ((d / s[:, None]).max(), int((d > 0).any(axis=1).sum()), n))
    _report("narrow vs wide", ratio.max())


def test_small_calls_are_independent_of_history(qlb, world):
    """A network that ran a 32,768-item forward and update gives the same bits on a later 300-item forward and 32-item
    gradient as a fresh network with the same weights: its buffers (cap_items, rows_padded of the head, the head's per-row
    tickets, stale rows of the dense operand, training scratch sized for 32,768) leave no trace."""
    idx300, idx32 = world.window(300)[1], world.window(32)[1]
    y32 = np.random.default_rng(32).uniform(-3, 3, size=32).astype(np.float32)
    fresh, used = qlb.QNetwork(world.env, world.w), qlb.QNetwork(world.env, world.w)
    qa = fresh.forward(idx300, 0)
    ga = fresh.debug_grads(idx32, y32)
    big = world.window(BIG)[1]
    used.forward(big, 0)
    used.debug_grads(big, np.zeros(BIG, np.float32))
    qb = used.forward(idx300, 0)
    gb = used.debug_grads(idx32, y32)
    for x, z in zip(qa, qb):
        assert np.array_equal(x.view(np.uint8), z.view(np.uint8))
    for k in ga:
        assert np.array_equal(ga[k].view(np.uint32), gb[k].view(np.uint32)), k
    fresh.close(); used.close()


def test_wide_forward_uses_the_trained_weights(qlb, world):
    """Three train() steps (batch 32, lr 1e-2 so the weights move far) re-derive every operand copy, the dense layer's N-256
    planes included: a wide forward then meets the per-item bound against the reference built from get_weights() - and the
    reference of the old weights misses it, so the check can tell stale operands from fresh ones."""
    torch = world.torch
    net = qlb.QNetwork(world.env, world.w)
    net.set_adam(lr=1e-2)
    idx32 = world.window(32)[1]
    y32 = np.random.default_rng(7).uniform(-3, 3, size=96).astype(np.float32)
    net.train(np.tile(idx32, 3), y32, n_batches=3)
    w2 = net.get_weights()
    n = world.last_narrow + 1
    o, idx = world.window(n)
    q, action, max_q = net.forward(idx, 0)
    q_ref, _, s = _reference_q(torch, w2, _stacks(torch, qlb, world.rb, idx, 0))
    _check_forward(q, action, max_q, q_ref, s, "wide forward after 3 updates")
    q_old, _, s_old = world.reference(0)
    stale = np.abs(q.astype(np.float64) - q_old[o:o + n]) > 1e-2 * s_old[o:o + n, None] + 1e-6
    assert stale.any(axis=1).mean() > 0.5, "degenerate test: the updates hardly moved Q"
    net.close()


def test_head_ties_take_the_first_maximum(qlb, world):
    """Equal dense-2 columns and biases make Q bitwise equal across actions: the action is 0 (the first maximum, like
    tf.argmax), on the narrow and the wide path. With columns and biases 1 and 2 equal and above 0, the action is 1. max_q
    is that common value, bit for bit."""
    w = {k: v.copy() for k, v in world.w.items()}
    net = qlb.QNetwork(world.env, w)
    for n in (300, world.last_narrow + 1):
        idx = world.window(n)[1]
        w["dense2_kernel"][:, 1] = w["dense2_kernel"][:, 2] = w["dense2_kernel"][:, 0]
        w["dense2_bias"][:] = w["dense2_bias"][0]
        net.set_weights(w)
        q, action, max_q = net.forward(idx, 0)
        assert np.array_equal(q[:, 0].view(np.uint32), q[:, 1].view(np.uint32)) and np.array_equal(q[:, 0].view(np.uint32), q[:, 2].view(np.uint32))
        assert np.all(action == 0), n
        assert np.array_equal(max_q.view(np.uint32), q[:, 0].view(np.uint32))
        w["dense2_bias"][0] = w["dense2_bias"][1] - 1.0
        net.set_weights(w)
        q, action, max_q = net.forward(idx, 0)
        assert np.array_equal(q[:, 1].view(np.uint32), q[:, 2].view(np.uint32)) and np.all(q[:, 1] > q[:, 0])
        assert np.all(action == 1), n
        assert np.array_equal(max_q.view(np.uint32), q[:, 1].view(np.uint32))
    net.close()


def _train_sizes():
    return ["last_narrow+1", str(BIG)]


def _minibatch(world, size):
    b = _size(world, size)
    _, idx = world.window(b)
    action = world.rb.get_many(idx, want_state=False, want_next=False).action
    q, _, _ = world.net.forward(idx, 0)
    return b, idx, action, q


@pytest.mark.parametrize("size", _train_sizes())
def test_full_batch_gradients(qlb, world, size):
    """All gradients finite, and per variable ||g - g_ref|| <= 2e-2 * ||g_ref|| against the f64 reference over the whole
    minibatch. Tolerance (as test_qnet_train.py): the backward rounds its GEMM operands (the back-propagated gradients) to
    bf16, 2^-9 relative each, through up to four layers, plus f32 accumulation order."""
    b, idx, action, q = _minibatch(world, size)
    y = _saturating_targets(q, action, b)
    g = world.net.debug_grads(idx, y)
    ref = _reference_grads(world.torch, qlb, world.rb, world.w, idx, action, y, b)
    _check_grads(qlb, g, ref, "full-batch gradients b=%d" % b)


@pytest.mark.parametrize("size", _train_sizes())
def test_weighted_gradients_isolate_items(qlb, world, size):
    """Loss weight 1 on a set S of positions and 0 elsewhere: a zero-weight item adds exact zeros to every GEMM and sum, so
    the library computes (1/b) sum_{i in S} grad L_i with the full-size machinery (every K slice, every column-sum split).
    Compared per variable with the f64 reference on S alone, scaled by 1/b, at 2e-2 (test_full_batch_gradients). One set
    holds positions 0, 1, 127, 128, 129, b-2, b-1 and 17 random ones; each other set holds the items straddling every slice
    boundary of one weight-gradient GEMM or one split column sum. With at most ~130 items per set one item is several
    per cent of a variable's norm, above the tolerance."""
    b, idx, action, q = _minibatch(world, size)
    y = _saturating_targets(q, action, b + 1)
    rng = np.random.default_rng(b)
    edges = np.array([0, 1, 127, 128, 129, b - 2, b - 1])
    sets = {"edges": np.unique(np.concatenate([edges, rng.choice(np.setdiff1d(np.arange(b), edges), size=17, replace=False)]))}
    for name, S in _boundary_sets(b).items():
        if not any(np.array_equal(S, T) for T in sets.values()):       # at 32,768 most boundaries fall on multiples of 512
            sets[name] = S
    for name, S in sets.items():
        assert S.size and S.max() < b, name
        wt = np.zeros(b, np.float32)
        wt[S] = 1.0
        g, _ = world.net.debug_grads_weighted(idx, y, wt)
        ref = _reference_grads(world.torch, qlb, world.rb, world.w, idx[S], action[S], y[S], b)
        _check_grads(qlb, g, ref, "item set %s (%d items) b=%d" % (name, S.size, b))


@pytest.mark.parametrize("size", _train_sizes())
def test_training_forward_equals_inference_forward(qlb, world, size):
    """The TD errors of debug_grads_weighted are q[i, a_i] - y_i bit for bit, with q from forward(idx, 0) at the same size:
    keeping the hidden activations for the backward does not change Q."""
    b, idx, action, q = _minibatch(world, size)
    y = np.random.default_rng(b).uniform(-4, 4, size=b).astype(np.float32)
    wt = np.random.default_rng(b + 1).uniform(0, 1, size=b).astype(np.float32)
    _, td = world.net.debug_grads_weighted(idx, y, wt)
    exp = q[np.arange(b), action.astype(np.int64)] - y
    assert np.array_equal(td.view(np.uint32), exp.view(np.uint32))


def test_mean_huber_loss_at_32768(qlb, world):
    """train()'s loss at b = 32,768 is mean Huber(q_a - y) in f64 on the library's own Q, about half the items on each branch.
    Tolerance: every term is >= 0 and carries <= 3 f32 roundings (q - y, d * d); the device sums them in a fixed two-level
    order (rows_per_split rows in 8 sequential lanes, the 8 lanes, then the splits in order) and divides once, so the
    relative error is at most (ceil(rows_per_split / 8) + 8 + splits + 4) * 2^-24 (test_huber_quadratic_and_linear_branches
    at 64 items: 1e-6)."""
    b = BIG
    _, idx = world.window(b)
    action = world.rb.get_many(idx, want_state=False, want_next=False).action
    net = qlb.QNetwork(world.env, world.w)
    q, _, _ = net.forward(idx, 0)
    qa = q[np.arange(b), action.astype(np.int64)]
    y = (qa - np.random.default_rng(3).uniform(-2.5, 2.5, size=b)).astype(np.float32)
    d = qa.astype(np.float64) - y
    assert 0.3 < np.mean(np.abs(d) < 1) < 0.5
    exp = np.mean(np.where(np.abs(d) <= 1, 0.5 * d * d, np.abs(d) - 0.5))
    loss = float(net.train(idx, y)[0])
    rps = _colsum_rows_per_split(b)
    tol = (-(-min(rps, b) // 8) + 8 + -(-b // rps) + 4) * 2.0 ** -24 * exp
    assert abs(loss - exp) <= tol, (loss, exp, tol)
    _report("mean Huber loss b=%d" % b, abs(loss - exp) / tol)
    net.close()
