"""The lean fkine / Jacobian kernels and the DH-like general kernels at every joint count, 1..10, fp64 and fp32.

fkj_launch_n sends a call to the lean kernels (k_fkj_fast, k_fkj_back_fast) when the chain is DH-like (unflipped Rz
joints, Rx-form or pure-translation inter-joint constants), jindex is dense, ldq == n, q is 16-byte aligned and there
are at least 32 rows; the ragged last rows go to the general kernel's DH-like form (PROF 1).  Which code runs then
depends on n and the dtype: the shared-memory Jacobian stash (fp64, odd n <= 7, fused call), padded J stages written
with one bulk copy per row (fp64 n = 4, 8; fp32 n = 8), 8-byte stage units (fp32, odd n).  The chains here come from
oracle.chains.dh_like_chain, which tests/test_dhlike_reference_cpu.py pins against an extended-precision restatement.

Every call goes through the C ABI directly, so that the tests choose q's row stride and the alignment of q, T and J,
and count the kernel launches a call costs: two (lean kernel + ragged tail) is the proof that the lean kernel ran.
Comparisons run on the device: some outputs are a quarter of a gigabyte.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import b2kin as rtb  # noqa: E402
from oracle import chains as ch  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from test_gpu_parity import TOL, dev, ets_from_desc, ref_inputs  # noqa: E402

NS = list(range(1, 11))
DTS = [np.float64, np.float32]
# 32 (4k + 1) rows: the last block of the lean grid has one live warp and three that return at once
ROWS = [1, 31, 32, 33, 32 * 5, 4099]
BIG = 2**19 + 17  # more tiles than one resident grid: the lean kernels' one-grid-ahead L2 prefetch fires
ENTRIES = ("fkine", "jacob0", "jacobe", "fkine_jacob0", "fkine_jacobe")
WT = {"fkine", "fkine_jacob0", "fkine_jacobe"}


@pytest.fixture(scope="module", autouse=True)
def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def tdt(dt):
    return torch.float64 if dt == np.float64 else torch.float32


class Chain:
    """One chain description as the kernels (an ETS) and the CPU oracle see it."""

    def __init__(self, desc):
        self.desc = desc
        self.n = int(desc["n"])
        self.ets = ets_from_desc(desc)
        self.C = orc.Chain(desc)

    def reach(self, base=None, tool=None):
        return ch.chain_reach(self.desc, base, tool)

    def ref(self, Q, base=None, tool=None):
        """{entry: (T, J)} from the oracle: T with base and tool, J0 / Je with the tool only."""
        T, J0, Je = self.C.fkine(Q, base, tool), self.C.jacob0(Q, tool), self.C.jacobe(Q, tool)
        return {"fkine": (T, None), "jacob0": (None, J0), "jacobe": (None, Je), "fkine_jacob0": (T, J0),
                "fkine_jacobe": (T, Je)}


def dh_chain(n, tail, seed):
    return Chain(ch.dh_like_chain(np.random.default_rng(seed), n, tail=tail))


def base_tool(seed):
    rng = np.random.default_rng(seed)
    return ch.random_se3(rng), ch.random_se3(rng)


def call(chain, entry, q, rows, ldq=None, base=None, tool=None, T=None, J=None):
    """One C-ABI entry point on the current stream.  q is a device tensor whose data_ptr() is row 0; T / J (allocated
    NaN-filled when not given, so that a row no kernel wrote cannot pass) may be views at any address.
    Returns (T, J, kernel launches the call cost)."""
    n = chain.n
    dt = q.dtype
    ldq = n if ldq is None else ldq
    if entry in WT and T is None:
        T = torch.full((rows, 4, 4), float("nan"), dtype=dt, device="cuda")
    if entry != "fkine" and J is None:
        J = torch.full((rows, 6, n), float("nan"), dtype=dt, device="cuda")
    if entry not in WT:
        T = None
    if entry == "fkine":
        J = None
    L = rtb._lib.lib()
    code = rtb._lib.F64 if dt == torch.float64 else rtb._lib.F32
    b = None if base is None else np.ascontiguousarray(base, dtype=np.float64)
    t = None if tool is None else np.ascontiguousarray(tool, dtype=np.float64)
    bp, tp = rtb._lib.dptr(b), rtb._lib.dptr(t)
    st = torch.cuda.current_stream().cuda_stream
    h, qp = chain.ets._chain, q.data_ptr()
    c0 = rtb.launch_count()
    if entry == "fkine":
        rc = L.b2k_fkine(h, code, qp, rows, ldq, bp, tp, T.data_ptr(), st)
    elif entry == "jacob0":
        rc = L.b2k_jacob0(h, code, qp, rows, ldq, tp, J.data_ptr(), st)
    elif entry == "jacobe":
        rc = L.b2k_jacobe(h, code, qp, rows, ldq, tp, J.data_ptr(), st)
    elif entry == "fkine_jacob0":
        rc = L.b2k_fkine_jacob0(h, code, qp, rows, ldq, bp, tp, T.data_ptr(), J.data_ptr(), st)
    else:
        rc = L.b2k_fkine_jacobe(h, code, qp, rows, ldq, bp, tp, T.data_ptr(), J.data_ptr(), st)
    rtb._lib.check(rc)
    return T, J, rtb.launch_count() - c0


def lean_launches(rows, lean=True):
    """Launches of one call: the lean kernel and the general one for the ragged rest, or the general kernel alone."""
    return 2 if lean and rows >= 32 and rows % 32 else 1


def tol_for(dt, reach):
    tol = dict(TOL[dt])
    # absolute floor scaled with the chain's reach, as test_gpu_parity.py::test_fixture_random_chains does; the fp32 bar
    # (rtol 1e-4, atol 1e-5 per unit of reach) is the project's fp32 parity bar, not fitted to these chains.  On an
    # NVIDIA B200 (1000 W power limit) the worst entry of any (n, dtype) used 0.04 % of the fp64 bar and 4.8 % of the fp32 bar.
    tol["atol"] *= max(1.0, reach)
    return tol


# worst error against the oracle per (n, dtype): the largest |got - want|, and the largest fraction of the bar it used
WORST = {}


def check(got, want, tol, what, key=None):
    """assert_allclose on the device (NaN in got fails), recording the worst error under `key`."""
    w = torch.from_numpy(np.ascontiguousarray(want)).cuda()
    g = got.double()
    err = (g - w).abs()
    bar = tol["atol"] + tol["rtol"] * w.abs()
    bad = ~(err <= bar)
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} entries outside rtol {tol['rtol']:g} atol "
                             f"{tol['atol']:.3g}; first at {idx}: got {float(g[idx])!r}, want {float(w[idx])!r}")
    if key is not None:
        e, r = float(err.max()), float((err / bar).max())
        old = WORST.get(key, (0.0, 0.0))
        WORST[key] = (max(old[0], e), max(old[1], r))


def report(key):
    e, r = WORST.get(key, (0.0, 0.0))
    print(f"\n[worst vs oracle] n={key[0]} {key[1]}: max |err| {e:.3g}, {r:.3g} of the bar")


def q_rows(n, rows, seed):
    """Mostly U(-pi, pi).  Inside a full tile, in the ragged tail and scattered (so that lanes of one warp take
    different sincos paths): rows with every angle in [8, 100) -- fp32 leaves the special-function unit for the
    Cody-Waite + polynomial path above B2K_MUFU_LIMIT -- and rows with one joint beyond 1.1e5, past the fast
    reduction's range, which take b2k_sincos_batch's per-element slow path in both precisions."""
    rng = np.random.default_rng(seed)
    Q = rng.uniform(-np.pi, np.pi, (rows, n))
    if rows < 31:
        return Q
    full = rows // 32 * 32
    mid, huge = [], []
    if full:
        mid.append(5)
        huge.append(9)
    if rows > full:
        mid.append(rows - 1)
        if rows - full >= 2:
            huge.append(full)
    scat = rng.choice(rows, max(2, rows // 64), replace=False)
    mid += list(scat[0::2])
    huge += list(scat[1::2])
    for r in mid:
        Q[r] = rng.uniform(8, 100, n) * rng.choice([-1, 1], n)
    for r in huge:
        Q[r, rng.integers(n)] = rng.uniform(1.1e5, 1e6) * rng.choice([-1, 1])
    return Q


def run_and_check(chain, dt, Q, base, tool, key, what, launches):
    """All five entry points on Q against the oracle; each call must cost `launches` kernel launches."""
    want = chain.ref(ref_inputs(Q, dt) if dt == np.float32 else Q, base, tool)
    tol = tol_for(dt, chain.reach(base, tool))
    q = dev(Q, dt)
    out = {}
    for entry in ENTRIES:
        T, J, k = call(chain, entry, q, Q.shape[0], base=base, tool=tool)
        assert k == launches, f"{what} {entry}: {k} kernel launches, expected {launches}"
        wT, wJ = want[entry]
        if T is not None:
            check(T, wT, tol, f"{what} {entry} T", key)
        if J is not None:
            check(J, wJ, tol, f"{what} {entry} J", key)
        out[entry] = (T, J)
    return q, out


# ------------------------------------------------------------------ oracle sweep
@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_oracle_sweep(n, dt):
    """Both tail forms, with and without base and tool, every edge row count: the lean kernels' full tiles, the
    general DH-like kernel's ragged tails and small batches, each call proven to have taken the intended path."""
    key = (n, np.dtype(dt).name)
    base, tool = base_tool(n)
    for tail in (False, True):
        chain = dh_chain(n, tail, 100 * n + tail)
        for b, t in ((None, None), (base, tool)):
            for rows in ROWS:
                Q = q_rows(n, rows, 7 * rows + n)
                run_and_check(chain, dt, Q, b, t, key, f"n={n} tail={tail} base/tool={b is not None} rows={rows}",
                              lean_launches(rows))
    report(key)


@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_controls_take_the_generic_walk(n, dt):
    """The same geometry with one joint flipped, or one joint about y: not DH-like, so every call is one launch of the
    generic (PROF 0) kernel, and it agrees with the oracle too."""
    key = (n, np.dtype(dt).name)
    base, tool = base_tool(n)
    d = ch.dh_like_chain(np.random.default_rng(100 * n + 1), n, tail=True)
    for what, desc in (("flip", ch.perturb_joint(d, n // 2, flip=True)), ("Ry", ch.perturb_joint(d, n - 1, axis=ch.RY))):
        chain = Chain(desc)
        for rows in (33, 4099):
            Q = q_rows(n, rows, 3 * rows + n)
            run_and_check(chain, dt, Q, base, tool, key, f"n={n} {what} rows={rows}", 1)
    report(key)


# ------------------------------------------------------------------ one large batch: oracle, variant 4, slices
@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_large_batch(n, dt):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    # more 32-row tiles than any lean grid keeps resident (4 warps a block, at most 16 blocks an SM)
    assert BIG > 32 * 4 * sms * 16
    key = (n, np.dtype(dt).name)
    base, tool = base_tool(n)
    chain = dh_chain(n, True, 100 * n + 1)
    Q = q_rows(n, BIG, n)
    q, out = run_and_check(chain, dt, Q, base, tool, key, f"n={n} rows={BIG}", lean_launches(BIG))
    report(key)

    # Variant 4 runs the persistent general kernel in its DH-like form, several tiles per warp, and no lean kernel.
    # Both forms evaluate the same chain_forward<..., PROF = 1> / jacob0_row / backward_walk_dh expressions.
    rtb.set_variant(4)
    try:
        for entry in ENTRIES:
            T, J, k = call(chain, entry, q, BIG, base=base, tool=tool)
            assert k == 1, f"variant 4 {entry}: {k} launches"
            if T is not None:
                assert torch.equal(T, out[entry][0]), f"{entry}: T of the lean and the persistent kernel differ"
            if J is not None:
                assert torch.equal(J, out[entry][1]), f"{entry}: J of the lean and the persistent kernel differ"
    finally:
        rtb.set_variant(0)

    # a 32-row-aligned slice evaluated on its own reproduces its rows of the full call (its ragged end now goes
    # through the general kernel)
    r0, m = 32 * 1000 + 32 * (n % 3), 32 * 37 + 5
    for entry in ENTRIES:
        T, J, k = call(chain, entry, q[r0:r0 + m], m, base=base, tool=tool)
        assert k == 2
        if T is not None:
            assert torch.equal(T, out[entry][0][r0:r0 + m]), f"{entry}: T of the slice differs"
        if J is not None:
            assert torch.equal(J, out[entry][1][r0:r0 + m]), f"{entry}: J of the slice differs"


# ------------------------------------------------------------------ bit-identities at 4099 rows
@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_fused_equals_separate(n, dt):
    """Without a base the fused calls return exactly what the single-output calls return: fkine_jacob0 T == fkine T
    and J == jacob0 J (at fp64 odd n <= 7 the fused kernel keeps its stash in shared memory, jacob0 in registers),
    fkine_jacobe J == jacobe J."""
    _, tool = base_tool(n)
    for tail in (False, True):
        chain = dh_chain(n, tail, 100 * n + tail)
        q = dev(q_rows(n, 4099, 11 * n), dt)
        for t in (None, tool):
            out = {e: call(chain, e, q, 4099, tool=t)[:2] for e in ENTRIES}
            assert torch.equal(out["fkine_jacob0"][0], out["fkine"][0])
            assert torch.equal(out["fkine_jacob0"][1], out["jacob0"][1])
            assert torch.equal(out["fkine_jacobe"][1], out["jacobe"][1])


@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_nan_row_stays_in_its_row(n, dt):
    """A NaN configuration inside a full tile and one in the ragged tail leave every other row bit-identical: staged
    and bulk-copied outputs land in their own rows."""
    base, tool = base_tool(n)
    chain = dh_chain(n, True, 100 * n + 1)
    Q = q_rows(n, 4099, 13 * n)
    clean = dev(Q, dt)
    Q[[100, 4097]] = np.nan
    dirty = dev(Q, dt)
    keep = torch.ones(4099, dtype=torch.bool, device="cuda")
    keep[[100, 4097]] = False
    for entry in ENTRIES:
        a = call(chain, entry, clean, 4099, base=base, tool=tool)[:2]
        b = call(chain, entry, dirty, 4099, base=base, tool=tool)[:2]
        for x, y in zip(a, b):
            if x is not None:
                assert torch.equal(x[keep], y[keep]), f"{entry}: a NaN row changed other rows"
        # the pose and the base-frame Jacobian of a NaN configuration are NaN (Je of a one-joint chain is constant)
        for y in (b[0], b[1] if entry == "jacob0" else None):
            if y is not None:
                assert bool(torch.isnan(y[~keep].reshape(2, -1)).any(dim=1).all()), f"{entry}: a NaN row came out finite"


# ------------------------------------------------------------------ layouts of q
@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_q_layouts(n, dt):
    """q one row into its buffer (16-byte aligned, hence lean, only when a row is a multiple of 16 bytes) and q as the
    first n columns of (rows, n + 1) rows (ldq != n: the general kernel, exact-image or padded q tile)."""
    key = (n, np.dtype(dt).name)
    base, tool = base_tool(n)
    chain = dh_chain(n, True, 100 * n + 1)
    rows = 4099
    Q = q_rows(n, rows, 17 * n)
    want = chain.ref(ref_inputs(Q, dt) if dt == np.float32 else Q, base, tool)
    tol = tol_for(dt, chain.reach(base, tool))
    es = np.dtype(dt).itemsize
    shifted = dev(np.vstack([np.zeros((1, n)), Q]), dt)[1:]
    wide = dev(np.hstack([Q, np.full((rows, 1), 1e3)]), dt)
    cases = (("one row in", shifted, n, lean_launches(rows, (n * es) % 16 == 0)), ("ldq = n + 1", wide, n + 1, 1))
    for what, q, ldq, launches in cases:
        for entry in ENTRIES:
            T, J, k = call(chain, entry, q, rows, ldq=ldq, base=base, tool=tool)
            assert k == launches, f"{what} {entry}: {k} launches, expected {launches}"
            if T is not None:
                check(T, want[entry][0], tol, f"{what} {entry} T", key)
            if J is not None:
                check(J, want[entry][1], tol, f"{what} {entry} J", key)
    report(key)


# ------------------------------------------------------------------ output alignment
def offset_view(shape, dt, nbytes, align):
    """An uninitialised (NaN) tensor of `shape` starting `nbytes` past an `align`-byte boundary."""
    es = np.dtype(dt).itemsize
    k = nbytes // es
    flat = torch.full((int(np.prod(shape)) + align // es,), float("nan"), dtype=tdt(dt), device="cuda")
    v = flat[k:k + int(np.prod(shape))].view(shape)
    assert v.data_ptr() % align == nbytes
    return v


@pytest.mark.parametrize("dt", DTS, ids=["f64", "f32"])
@pytest.mark.parametrize("n", NS)
def test_output_alignment_contract(n, dt):
    """J 8 bytes past a 16-byte boundary: fine for fp32 with odd n (its J stage moves 8-byte units), refused with a
    ValueError for fp64 and for fp32 with even n (16-byte units).  T 16 bytes past a 32-byte boundary: refused."""
    key = (n, np.dtype(dt).name)
    base, tool = base_tool(n)
    chain = dh_chain(n, True, 100 * n + 1)
    rows = 4099
    Q = q_rows(n, rows, 19 * n)
    q = dev(Q, dt)
    want = chain.ref(ref_inputs(Q, dt) if dt == np.float32 else Q, base, tool)
    tol = tol_for(dt, chain.reach(base, tool))
    units8 = dt == np.float32 and n % 2 == 1
    for entry in ENTRIES[1:]:
        J = offset_view((rows, 6, n), dt, 8, 16)
        if units8:
            T, J, k = call(chain, entry, q, rows, base=base, tool=tool, J=J)
            assert k == 2
            check(J, want[entry][1], tol, f"J 8 bytes off, {entry}", key)
        else:
            c0 = rtb.launch_count()
            with pytest.raises(ValueError, match="16-byte aligned"):
                call(chain, entry, q, rows, base=base, tool=tool, J=J)
            assert rtb.launch_count() == c0
    for entry in ("fkine", "fkine_jacob0", "fkine_jacobe"):
        T = offset_view((rows, 4, 4), dt, 16, 32)
        c0 = rtb.launch_count()
        with pytest.raises(ValueError, match="32-byte aligned"):
            call(chain, entry, q, rows, base=base, tool=tool, T=T)
        assert rtb.launch_count() == c0
    report(key)


# ------------------------------------------------------------------ chained calls, no synchronisation
CHAIN_ROWS = 262144  # 8192 tiles: many more blocks than are resident at once, so consecutive grids do overlap


def _fkj(chain, q):
    """fkine_jacob0 into torch.empty outputs: no fill kernel between two fkj kernels on the stream."""
    rows = q.shape[0]
    T = torch.empty((rows, 4, 4), dtype=q.dtype, device=q.device)
    J = torch.empty((rows, 6, chain.n), dtype=q.dtype, device=q.device)
    T, J, _ = call(chain, "fkine_jacob0", q, rows, T=T, J=J)
    return T, J


def _tail_rows(J, rows, n):
    flat = J.view(-1)
    return flat[flat.numel() - rows * n:].view(rows, n)


@pytest.mark.parametrize("n", [5, 4], ids=["stash", "padded"])
def test_chained_calls_without_sync(n):
    """tests/test_gpu_fkj_chained.py's check at fp64 n = 5 (shared-memory stash) and n = 4 (padded J stage): q written
    by the kernel right before -- the previous call's J, or a torch kernel -- gives what synchronised calls give."""
    chain = dh_chain(n, True, 100 * n + 1)
    g = torch.Generator(device="cuda").manual_seed(n)
    q0 = (torch.rand((CHAIN_ROWS, n), generator=g, device="cuda", dtype=torch.float64) * 2 - 1).mul_(math.pi)
    rows = [CHAIN_ROWS, CHAIN_ROWS + 6, CHAIN_ROWS - 26]  # even counts keep the tail slice 16-byte aligned
    torch.cuda.synchronize()
    chained, q = [], q0
    for r in rows:
        T, J = _fkj(chain, q)
        chained.append((T, J))
        q = _tail_rows(J, r, n)
    torch.cuda.synchronize()
    q = q0
    for k, r in enumerate(rows):
        q = q.clone()
        torch.cuda.synchronize()
        T, J = _fkj(chain, q)
        torch.cuda.synchronize()
        assert torch.equal(T, chained[k][0]) and torch.equal(J, chained[k][1]), f"call {k} differs"
        q = _tail_rows(J, r, n)

    src = [torch.rand((CHAIN_ROWS, n), generator=g, device="cuda", dtype=torch.float64) * 6 - 3 for _ in range(4)]
    qbuf = torch.empty((CHAIN_ROWS, n), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    chained = []
    for s in src:
        torch.sin(s, out=qbuf)
        chained.append(_fkj(chain, qbuf))
    torch.cuda.synchronize()
    for k, s in enumerate(src):
        q = torch.sin(s)
        torch.cuda.synchronize()
        T, J = _fkj(chain, q)
        torch.cuda.synchronize()
        assert torch.equal(T, chained[k][0]) and torch.equal(J, chained[k][1]), f"torch-written q, call {k} differs"


# ------------------------------------------------------------------ DHRobot round trip
@pytest.mark.parametrize("mdh", [False, True], ids=["dh", "mdh"])
@pytest.mark.parametrize("n", NS)
def test_dhrobot_round_trip(n, mdh):
    """Random standard / modified DH robots (revolute, zero offsets: DH-like) through DHRobot's own ETS against the
    oracle on the reference's DH -> ETS expansion."""
    rng = np.random.default_rng(50 + n + 20 * mdh)
    links = []
    for j in range(n):
        alpha = ch.DH_ALPHAS[(j + n) % len(ch.DH_ALPHAS)]
        alpha = float(rng.uniform(-np.pi, np.pi)) if alpha is None else alpha
        d = float(rng.uniform(-0.5, 0.5)) if j % 3 else 0.0
        links.append(dict(d=d, a=float(rng.uniform(-0.5, 0.5)), alpha=alpha))
    cls = rtb.RevoluteMDH if mdh else rtb.RevoluteDH
    rob = rtb.DHRobot([cls(**L) for L in links])
    desc = ch.dh_to_ets(links, mdh)
    C = orc.Chain(desc)
    rows = 4099
    Q = q_rows(n, rows, 23 * n + mdh)
    for dt in DTS:
        Qr = ref_inputs(Q, dt) if dt == np.float32 else Q
        tol = tol_for(dt, ch.chain_reach(desc))
        q = dev(Q, dt)
        for what, fn, want in (("fkine", rob.eval, C.fkine(Qr)), ("jacob0", rob.jacob0, C.jacob0(Qr)),
                               ("jacobe", rob.jacobe, C.jacobe(Qr))):
            c0 = rtb.launch_count()
            got = fn(q)
            assert rtb.launch_count() - c0 == 2, f"{what}: the DH robot did not take the lean kernel"
            check(got, want, tol, f"{'MDH' if mdh else 'DH'} {what} {np.dtype(dt).name}")
