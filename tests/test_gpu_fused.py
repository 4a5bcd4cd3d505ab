"""GPU parity of the fused aggregate+project tcgen05 kernel (gnnml3_fused_agg_proj) against a float64 restatement
of the reference's message passing (libs/spect_conv.py:70-80,93-94: index_select, scale by edge_attr[:, k],
scatter-add, matmul with W_k, sum, bias) and of the ML3Layer node branch (:208-212).  FP32 bar: rtol 1e-5."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_kernels import assert_close, dev, np_csr  # noqa: E402


def _graph(N, deg, seed, blk=40):
    g = torch.Generator().manual_seed(seed)
    E = N * deg
    src = torch.randint(0, N, (E,), generator=g)
    dst = ((src // blk) * blk + torch.randint(0, blk, (E,), generator=g)).clamp(max=N - 1)
    return torch.stack([src, dst]), g


def _ref_main(x, ei, ea, W, bias):
    """sum_k scatter_add(ea[:, k] * x[src]) @ W_k (+ bias) in float64; ea in ORIGINAL edge order."""
    x, ea, W = x.double(), ea.double(), W.double()
    N = x.size(0)
    out = torch.zeros(N, W.size(2), dtype=torch.float64)
    for k in range(W.size(0)):
        h = torch.zeros(N, x.size(1), dtype=torch.float64).index_add_(0, ei[1], ea[:, k:k + 1] * x[ei[0]])
        out += h @ W[k]
    if bias is not None:
        out += bias.double()
    return out


CASES = [  # N, deg, K, F, Nc, G
    (3000, 6, 8, 32, 30, 2),      # ZINC layers 2-4
    (3001, 6, 8, 25, 30, 2),      # ZINC layer 1 (x rows need padding)
    (1000, 5, 6, 2, 32, 16),      # graph8c / EXP layer 1
    (2000, 6, 12, 32, 16, 16),    # counting (two K passes)
    (1500, 4, 10, 64, 64, 0),     # sweep shape: two feature blocks per support, BN = 64
    (700, 3, 5, 17, 9, 0),
    (900, 9, 7, 40, 33, 4),
    (95, 2, 4, 8, 8, 1),          # less than one tile
    (97, 0, 8, 32, 30, 2),        # no edges at all in the rows (E = 0 is handled by the host fallback; here deg 0 -> E = 0)
]


@pytest.fixture(params=["ts-window", "ts-global", "planes-gather", "planes-slots"])
def fused_mode(request):
    """Every variant of the fused kernel: the tensor-memory generation (fused_layer_ts.cu) with the tile's source rows staged
    in shared memory (tile windows given) or gathered from global memory, and the shared-memory-plane generation
    (fused_layer.cu) in both aggregator modes (gnnml3_fused_set_ts / gnnml3_fused_set_mode)."""
    from gnn_matlang_b200 import _lib
    lib = _lib.load()
    ts = request.param.startswith("ts")
    old_ts = lib.gnnml3_fused_set_ts(1 if ts else 0)
    old = lib.gnnml3_fused_set_mode(1 if request.param == "planes-slots" else 0)
    yield request.param
    lib.gnnml3_fused_set_mode(old)
    lib.gnnml3_fused_set_ts(old_ts)


def _win(mode, rowptr, col):
    from gnn_matlang_b200 import ops
    return ops.tile_windows(rowptr, col) if mode == "ts-window" else None


def _check_path(mode, K, F, before):
    """The variant under test is the one that ran (no silent fall-through to the other generation)."""
    from gnn_matlang_b200 import ops
    ts, planes = ops.fused_path_counts()
    if mode.startswith("ts") and F <= 32 and K % 2 == 0:
        assert ts > before[0] and planes == before[1], "tensor-memory kernel did not run"
    else:
        assert planes > before[1] and ts == before[0], "shared-memory-plane kernel did not run"


@pytest.mark.parametrize("N,deg,K,F,Nc,G", CASES)
def test_fused_forward_ml3(N, deg, K, F, Nc, G, fused_mode):
    from gnn_matlang_b200 import ops
    if deg == 0:
        pytest.skip("E == 0 takes the unfused host path")
    ei, g = _graph(N, deg, N + K)
    E = ei.size(1)
    x = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    bias = torch.randn(Nc, generator=g) * 0.3
    csr = np_csr(ei.numpy(), N)
    perm = torch.from_numpy(csr["perm"])
    ea_s = ea[perm].contiguous()                       # dst-sorted order, as the modules keep it
    d = dev()
    i32 = lambda a: torch.from_numpy(a.astype(np.int32)).to(d)
    xa = ops.aligned_rows(x.to(d))
    ref = _ref_main(x, ei, ea, W, bias)
    win = _win(fused_mode, i32(csr["rowptr"]), i32(csr["col"]))
    before = ops.fused_path_counts()
    if G > 0 and F <= 32:
        w11 = torch.randn(G, F, generator=g) / np.sqrt(F)
        w12 = torch.randn(G, F, generator=g) / np.sqrt(F)
        b11, b12 = torch.randn(G, generator=g) * 0.2, torch.randn(G, generator=g) * 0.2
        wg = torch.cat([w11.t(), w12.t()], 1).contiguous().to(d)
        y, aux = ops.fused_agg_proj(i32(csr["rowptr"]), i32(csr["col"]), None, ea_s.to(d), xa, W.view(K * F, Nc).to(d),
                                    bias=bias.to(d), S=xa, self_mode=1, Bself=wg, bias_s=torch.cat([b11, b12]).to(d), G=G,
                                    epilogue=1, win=win)
        t1 = torch.tanh(x.double() @ w11.double().t() + b11.double())
        t2 = torch.tanh(x.double() @ w12.double().t() + b12.double())
        assert_close(y[:, :Nc], torch.relu(ref), name="relu(conv)")
        assert_close(y[:, Nc:], t1 * t2, name="gate")
        assert_close(aux, torch.cat([t1, t2], 1), name="aux")
    else:
        out, aux = ops.fused_agg_proj(i32(csr["rowptr"]), i32(csr["col"]), None, ea_s.to(d), xa, W.view(K * F, Nc).to(d),
                                      bias=bias.to(d), epilogue=0, win=win)
        assert aux is None
        assert_close(out, ref, name="conv")
    _check_path(fused_mode, K, F, before)


@pytest.mark.parametrize("N,deg,K,F,Nc,Fs", [(3000, 6, 8, 30, 32, 4), (2000, 5, 6, 32, 2, 32), (1200, 4, 10, 64, 64, 0),
                                              (1000, 6, 12, 16, 32, 32)])
def test_fused_transposed_with_self_block(N, deg, K, F, Nc, Fs, fused_mode):
    """The dx form: transposed CSR, edge weights through permT, a self block accumulating into the main columns."""
    from gnn_matlang_b200 import ops
    ei, g = _graph(N, deg, 7 * N + K)
    E = ei.size(1)
    gout = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    csr = np_csr(ei.numpy(), N)
    ea_s = ea[torch.from_numpy(csr["perm"])].contiguous()
    d = dev()
    i32 = lambda a: torch.from_numpy(a.astype(np.int32)).to(d)
    # transposed aggregation: row s sums over edges with src == s, gathering rows dst  -> swap the roles of src/dst
    ref = _ref_main(gout, torch.stack([ei[1], ei[0]]), ea, W, None)
    F4 = (F + 3) // 4 * 4
    buf = torch.zeros(N, F4 + (Fs + 3) // 4 * 4)
    buf[:, :F] = gout
    S = Bs = None
    if Fs:
        sv = torch.randn(N, Fs, generator=g)
        Bs = torch.randn(Fs, Nc, generator=g) / np.sqrt(Fs)
        buf[:, F4:F4 + Fs] = sv
        ref = ref + sv.double() @ Bs.double()
    bufd = buf.to(d)
    out, _ = ops.fused_agg_proj(i32(csr["rowptrT"]), i32(csr["colT"]), i32(csr["permT"]), ea_s.to(d), bufd[:, :F],
                                W.view(K * F, Nc).to(d), S=bufd[:, F4:F4 + Fs] if Fs else None, self_mode=2 if Fs else 0,
                                Bself=Bs.to(d) if Fs else None, epilogue=0,
                                win=_win(fused_mode, i32(csr["rowptrT"]), i32(csr["colT"])))
    assert_close(out, ref, name="dx form")


def test_fused_large_batch_matches_two_kernel_path(fused_mode):
    """ZINC bench shape (many tiles per SM): fused result == SpMM + GEMM of the same library."""
    from gnn_matlang_b200 import ops
    N, deg, K, F, Nc = 150000, 6, 8, 32, 30
    ei, g = _graph(N, deg, 11, blk=23)
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    x = torch.randn(N, F, generator=g).to(d)
    ea_s = torch.randn(ei.size(1), K, generator=g).to(d)
    W = (torch.randn(K * F, Nc, generator=g) / 16).to(d)
    out, _ = ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, x, W, epilogue=0,
                                win=plan["win"] if fused_mode == "ts-window" else None)
    H = ops.spmm_k(plan["rowptr"], plan["col"], None, ea_s, x)
    ref = ops.gemm_nn(H, W)
    assert_close(out, ref, rtol=2e-6, name="fused vs two-kernel")


def test_tile_windows_are_exact():
    """gnnml3_tile_windows: {min, max + 1} source row over each 128-row tile's CSR slots ({0, 0} for an empty tile) -- integer
    work, bit-exact against numpy."""
    from gnn_matlang_b200 import _lib, ops
    rows = _lib.load().gnnml3_tile_rows()
    for N, deg, blk in [(1000, 5, 40), (4097, 3, 700), (130, 1, 13)]:
        ei, _ = _graph(N, deg, N, blk=blk)
        ei = ei[:, ei[1] >= 300] if N == 1000 else ei          # rows 0..299 without any slot: tiles 0 and 1 are empty
        csr = np_csr(ei.numpy(), N)
        d = dev()
        win = ops.tile_windows(torch.from_numpy(csr["rowptr"].astype(np.int32)).to(d),
                               torch.from_numpy(csr["col"].astype(np.int32)).to(d)).cpu().numpy()
        nt = (N + rows - 1) // rows
        assert win.shape == (nt, 2)
        for t in range(nt):
            e0, e1 = csr["rowptr"][t * rows], csr["rowptr"][min((t + 1) * rows, N)]
            c = csr["col"][e0:e1]
            exp = (0, 0) if e1 == e0 else (int(c.min()), int(c.max()) + 1)
            assert tuple(win[t]) == exp, (N, t, tuple(win[t]), exp)


def test_fused_ts_mixed_windows_and_side_output():
    """Tensor-memory kernel on a graph whose first half has local edges (tiles staged in shared memory) and whose second half
    has long-range edges (windows wider than the TMA box: those tiles gather from global memory) -- one launch, both
    aggregator paths; plus the aggregate side output `hout` the backward's weight gradient consumes."""
    from gnn_matlang_b200 import ops
    N, deg, K, F, Nc = 6000, 5, 8, 30, 32
    g = torch.Generator().manual_seed(99)
    E = N * deg
    src = torch.randint(0, N, (E,), generator=g)
    near = ((src // 40) * 40 + torch.randint(0, 40, (E,), generator=g)).clamp(max=N - 1)
    far = torch.randint(N // 2, N, (E,), generator=g)
    dst = torch.where(src < N // 2, near, far)
    ei = torch.stack([src, dst])
    x = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    win = plan["win"].cpu().numpy()
    width = win[:, 1] - win[:, 0]
    assert (width <= 256).any() and (width > 256).any(), "the case must contain staged and unstaged tiles"
    ea_s = ea.to(d)[plan["perm"].long()].contiguous()
    xa = ops.aligned_rows(x.to(d))
    hout = torch.full((N, K * 32), float("nan"), device=d)
    before = ops.fused_path_counts()
    out, _ = ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), epilogue=0, hout=hout,
                                win=plan["win"])
    assert ops.fused_path_counts()[0] == before[0] + 1
    assert_close(out, _ref_main(x, ei, ea, W, None), name="conv (mixed windows)")
    H = torch.zeros(N, K, 32, dtype=torch.float64)
    for k in range(K):
        H[:, k, :F] = torch.zeros(N, F, dtype=torch.float64).index_add_(0, ei[1], ea[:, k:k + 1].double() * x.double()[ei[0]])
    assert_close(hout, H.view(N, K * 32), name="aggregate side output")


@pytest.mark.parametrize("staged", [True, False])
@pytest.mark.parametrize("N,deg,K,Fi,Fo", [(3000, 6, 8, 32, 30), (3001, 5, 8, 25, 30), (1000, 7, 6, 2, 32), (60, 3, 2, 8, 8),
                                           (100000, 6, 8, 32, 30), (2000, 4, 4, 17, 9)])
def test_fused_sddmm(N, deg, K, Fi, Fo, staged):
    """d ea[p, k] = <x[col[p]], gc[t] W_k^T> against float64; with the plan's source windows (source rows staged in shared
    memory by TMA) and without (every edge gathers from global memory)."""
    from gnn_matlang_b200 import ops
    ei, g = _graph(N, deg, 3 * N + K, blk=25)
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    x = torch.randn(N, Fi, generator=g)
    gc = torch.randn(N, Fo, generator=g)
    W = torch.randn(K, Fi, Fo, generator=g) / np.sqrt(Fo)
    dea = ops.fused_sddmm(plan["rowptr"], plan["col"], ops.aligned_rows(x.to(d)), ops.aligned_rows(gc.to(d)), W.to(d), ei.size(1),
                          win=plan["win"] if staged else None)
    rowptr = plan["rowptr"].cpu().long()
    col = plan["col"].cpu().long()
    dst = torch.repeat_interleave(torch.arange(N), rowptr[1:] - rowptr[:-1])
    dH = torch.einsum("no,kio->nki", gc.double(), W.double())              # [N, K, Fi]
    ref = torch.einsum("ei,eki->ek", x.double()[col], dH[dst])
    assert_close(dea, ref, name="fused sddmm")


def test_fused_sddmm_mixed_windows_and_crowded_tiles():
    """One launch with all three kinds of tiles: local edges (staged), long-range edges (window wider than the TMA box: global
    gathers) and rows with more CSR slots than the staging buffer holds (global gathers); staged and unstaged results must be
    bit-identical (same arithmetic, same order)."""
    from gnn_matlang_b200 import ops
    N, deg, K, Fi, Fo = 6000, 5, 8, 30, 32
    g = torch.Generator().manual_seed(17)
    E = N * deg
    src = torch.randint(0, N, (E,), generator=g)
    near = ((src // 40) * 40 + torch.randint(0, 40, (E,), generator=g)).clamp(max=N - 1)
    far = torch.randint(N // 2, N, (E,), generator=g)
    dst = torch.where(src < N // 2, near, far)
    # rows 0..63 receive 40 extra local edges each: 2560 + slots in one 64-row tile (> 1024)
    xs = torch.randint(0, 64, (64 * 40,), generator=g)
    xd = torch.arange(64).repeat_interleave(40)
    ei = torch.stack([torch.cat([src, xs]), torch.cat([dst, xd])])
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    win = plan["win"].cpu().numpy()
    width = win[:, 1] - win[:, 0]
    assert (width <= 256).any() and (width > 256).any()
    rowptr = plan["rowptr"].cpu().long()
    assert int(rowptr[64] - rowptr[0]) > 1024
    x = torch.randn(N, Fi, generator=g)
    gc = torch.randn(N, Fo, generator=g)
    W = torch.randn(K, Fi, Fo, generator=g) / np.sqrt(Fo)
    args = (plan["rowptr"], plan["col"], ops.aligned_rows(x.to(d)), ops.aligned_rows(gc.to(d)), W.to(d), ei.size(1))
    a = ops.fused_sddmm(*args, win=plan["win"])
    b = ops.fused_sddmm(*args, win=None)
    assert torch.equal(a, b)
    col = plan["col"].cpu().long()
    dstv = torch.repeat_interleave(torch.arange(N), rowptr[1:] - rowptr[:-1])
    dH = torch.einsum("no,kio->nki", gc.double(), W.double())
    assert_close(a, torch.einsum("ei,eki->ek", x.double()[col], dH[dstv]), name="fused sddmm (mixed tiles)")


def test_act_bwd_y_layout_and_sums():
    from gnn_matlang_b200 import ops
    g = torch.Generator().manual_seed(5)
    N, Fo, G = 1000, 30, 2
    pre = torch.randn(N, Fo + 2 * G, generator=g)
    gy = torch.randn(N, Fo + G, generator=g)
    y = torch.cat([torch.relu(pre[:, :Fo]), torch.tanh(pre[:, Fo:Fo + G]) * torch.tanh(pre[:, Fo + G:])], 1)
    aux = torch.tanh(pre[:, Fo:])
    d = dev()
    gpre, csum = ops.ml3_act_bwd_y(y.to(d), aux.to(d), gy.to(d), Fo, G)
    pr = pre.double().requires_grad_(True)
    yr = torch.cat([torch.relu(pr[:, :Fo]), torch.tanh(pr[:, Fo:Fo + G]) * torch.tanh(pr[:, Fo + G:])], 1)
    yr.backward(gy.double())
    Fo4 = 32
    assert gpre.shape == (N, 36)
    assert_close(gpre[:, :Fo], pr.grad[:, :Fo], name="gc")
    assert_close(gpre[:, Fo4:Fo4 + 2 * G], pr.grad[:, Fo:], name="gates")
    assert float(gpre[:, Fo:Fo4].abs().max()) == 0.0
    assert_close(csum, pr.grad.sum(0), name="bias sums")


@pytest.mark.parametrize("precision,rtol", [("tf32", 2e-3), ("bf16", 2e-2)])
@pytest.mark.parametrize("N,deg,K,F,Nc,G", [(3000, 6, 8, 32, 30, 2), (1000, 5, 6, 2, 32, 16), (2000, 6, 12, 32, 16, 16), (1500, 4, 8, 30, 48, 0)])
def test_fused_flagged_precisions(N, deg, K, F, Nc, G, precision, rtol):
    """north_star "(TF32, or bf16 when flagged)": the tensor-memory kernel with ONE tensor-core product per k-step on TF32-
    truncated / BF16-rounded inputs, FP32 accumulation.  Stated tolerances relative to the result's scale: TF32 2e-3 (10-bit
    mantissa, inputs truncated), BF16 2e-2 (8-bit mantissa, 256-term contractions)."""
    from gnn_matlang_b200 import _lib, ops
    prec = {"tf32": _lib.PREC_TF32, "bf16": _lib.PREC_BF16}[precision]
    ei, g = _graph(N, deg, N + K)
    E = ei.size(1)
    x = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    bias = torch.randn(Nc, generator=g) * 0.3
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    ea_s = ea.to(d)[plan["perm"].long()].contiguous()
    xa = ops.aligned_rows(x.to(d))
    ref = _ref_main(x, ei, ea, W, bias)
    before = ops.fused_path_counts()
    if G > 0:
        w11 = torch.randn(G, F, generator=g) / np.sqrt(F)
        w12 = torch.randn(G, F, generator=g) / np.sqrt(F)
        b11, b12 = torch.randn(G, generator=g) * 0.2, torch.randn(G, generator=g) * 0.2
        wg = torch.cat([w11.t(), w12.t()], 1).contiguous().to(d)
        y, aux = ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), bias=bias.to(d), S=xa, self_mode=1,
                                    Bself=wg, bias_s=torch.cat([b11, b12]).to(d), G=G, epilogue=1, win=plan["win"], precision=prec)
        t1 = torch.tanh(x.double() @ w11.double().t() + b11.double())
        t2 = torch.tanh(x.double() @ w12.double().t() + b12.double())
        assert_close(y[:, :Nc], torch.relu(ref), rtol=rtol, name="relu(conv) " + precision)
        assert_close(y[:, Nc:], t1 * t2, rtol=rtol, name="gate " + precision)
        assert_close(aux, torch.cat([t1, t2], 1), rtol=rtol, name="aux " + precision)
        err = (y[:, :Nc].cpu().double() - torch.relu(ref)).abs().max() / ref.abs().max()
    else:
        out, _ = ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), bias=bias.to(d), epilogue=0,
                                    win=plan["win"], precision=prec)
        assert_close(out, ref, rtol=rtol, name="conv " + precision)
        err = (out.cpu().double() - ref).abs().max() / ref.abs().max()
    assert ops.fused_path_counts()[0] == before[0] + 1
    # the flagged modes must really be reduced precision (a silent fall-through to 3xTF32 would sit at ~1e-7)
    assert float(err) > 1e-5, "suspiciously exact for %s: %.2e" % (precision, float(err))
    # an unknown precision, and anything but 0 or 1 as the epilogue, is GNNML3_ERR_INVALID
    with pytest.raises(RuntimeError, match=r"code 1\).*unknown precision"):
        ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), epilogue=0, precision=3)
    with pytest.raises(RuntimeError, match=r"code 1\).*unknown epilogue"):
        ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), epilogue=0x101, precision=prec)


@pytest.mark.parametrize("precision,rtol", [("tf32", 5e-3), ("bf16", 5e-2)])
def test_ml3layer_module_in_flagged_precision(precision, rtol):
    """ML3Layer(precision=...) forward + backward through the fused tensor-memory kernels in the flagged modes vs the oracle."""
    from gnn_matlang_b200.libs.spect_conv import ML3Layer
    from oracle import gnnml3_oracle as O
    g = torch.Generator().manual_seed(3)
    N, deg, K = 2000, 5, 8
    ei, _ = _graph(N, deg, 5)
    x = torch.randn(N, 32, generator=g)
    ea = torch.randn(ei.size(1), K, generator=g)
    torch.manual_seed(1)
    ref = O.OracleML3Layer(True, K, K, 32, 30, 2)
    lay = ML3Layer(True, K, K, 32, 30, 2, precision=precision)
    lay.load_state_dict(ref.state_dict())
    lay = lay.to(dev())
    xr = x.clone().requires_grad_(True)
    yr = ref(xr, ei, ea)
    gy = torch.randn(yr.shape, generator=g)
    yr.backward(gy)
    xd = x.to(dev()).requires_grad_(True)
    y = lay(xd, ei.to(dev()), ea.to(dev()))
    y.backward(gy.to(dev()))
    assert_close(y, yr, rtol=rtol, name="layer out")

    def close_in_norm(a, ref, name):
        """Reduced precision flips the ReLU mask of pre-activations within ~rtol of zero, which changes single gradient entries
        by O(1): gradients are held to the tolerance in the Frobenius norm and entry-wise for at least 99 % of the entries."""
        a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
        rel = float((a - ref).norm() / ref.norm())
        frac_bad = float(((a - ref).abs() > rtol * ref.abs() + rtol * ref.abs().max()).double().mean())
        assert rel <= 4 * rtol, "%s: relative Frobenius error %.3e" % (name, rel)
        if ref.numel() >= 10000:          # (small weight tensors are sums over all nodes: the norm bound is the meaningful one)
            assert frac_bad <= 0.01, "%s: %.2f %% entries off" % (name, 100 * frac_bad)

    close_in_norm(xd.grad, xr.grad, "dx")
    for (k, p), (_, pr) in zip(lay.named_parameters(), ref.named_parameters()):
        close_in_norm(p.grad, pr.grad, "grad " + k)
