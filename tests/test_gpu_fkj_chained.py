"""Back-to-back fkine_jacob0 calls on one stream with no synchronisation in between.

The fkj kernels are launched with programmatic stream serialization: a call's blocks may become resident while the
previous kernel on the stream is still running, and each kernel waits for that kernel's writes before it reads q.
These tests feed a call q that the immediately preceding kernel wrote -- the previous call's own J output, or a torch
kernel -- and check the results bit for bit against the same calls with a device synchronise between each pair.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import b2kin as rtb  # noqa: E402

ROWS = 262144  # 8192 tiles: many more blocks than are resident at once, so consecutive grids do overlap


@pytest.fixture(scope="module")
def panda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return rtb.models.Panda().ets()


def _fkj(ets, q):
    """One fkine_jacob0 call through the C ABI on the current stream: no allocation or copy that could synchronise."""
    L = rtb._lib.lib()
    n = q.shape[0]
    T = torch.empty((n, 4, 4), dtype=q.dtype, device=q.device)
    J = torch.empty((n, 6, 7), dtype=q.dtype, device=q.device)
    code = rtb._lib.F64 if q.dtype == torch.float64 else rtb._lib.F32
    rtb._lib.check(L.b2k_fkine_jacob0(ets._chain, code, q.data_ptr(), n, 7, None, None, T.data_ptr(), J.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
    return T, J


def _tail_rows(J, rows):
    """The last `rows` x 7 values of J's storage as a q array: the rows the previous grid's last blocks wrote."""
    flat = J.view(-1)
    return flat[flat.numel() - rows * 7:].view(rows, 7)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_q_is_previous_jacobian(panda, dtype):
    g = torch.Generator(device="cuda").manual_seed(7)
    q0 = (torch.rand((ROWS, 7), generator=g, device="cuda", dtype=torch.float64) * 2 - 1).mul_(np.pi).to(dtype)
    # rows: a whole number of tiles, then ragged counts (even, so the tail slice stays 16-byte aligned) whose last
    # rows go through the general kernel right behind the lean one
    rows = [ROWS, ROWS + 6, ROWS - 26]
    torch.cuda.synchronize()
    chained = []
    q = q0
    for r in rows:
        T, J = _fkj(panda, q)
        chained.append((T, J))
        q = _tail_rows(J, r)
    torch.cuda.synchronize()

    q = q0
    for k, r in enumerate(rows):
        q = q.clone()
        torch.cuda.synchronize()
        T, J = _fkj(panda, q)
        torch.cuda.synchronize()
        assert torch.equal(T, chained[k][0]), f"call {k}: T differs from the synchronised evaluation"
        assert torch.equal(J, chained[k][1]), f"call {k}: J differs from the synchronised evaluation"
        q = _tail_rows(J, r)


def test_q_written_by_torch_kernel(panda):
    g = torch.Generator(device="cuda").manual_seed(11)
    src = [torch.rand((ROWS, 7), generator=g, device="cuda", dtype=torch.float64) * 6 - 3 for _ in range(4)]
    qbuf = torch.empty((ROWS, 7), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    chained = []
    for s in src:  # the same q buffer every call: a torch kernel overwrites it between two fkj kernels that read it
        torch.sin(s, out=qbuf)
        chained.append(_fkj(panda, qbuf))
    torch.cuda.synchronize()

    for k, s in enumerate(src):
        q = torch.sin(s)
        torch.cuda.synchronize()
        T, J = _fkj(panda, q)
        torch.cuda.synchronize()
        assert torch.equal(T, chained[k][0]), f"call {k}: T differs from the synchronised evaluation"
        assert torch.equal(J, chained[k][1]), f"call {k}: J differs from the synchronised evaluation"
