"""GPU parity tests of the individual sm_100a kernels, called through the C ABI (ctypes), against the CPU oracle."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from replay_b200 import ops as _ops

    return _ops


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, 5])
def test_umma_operand_modes(ops, mode):
    """tcgen05 descriptor encodings: K-major / MN-major smem operands, A from TMEM."""
    g = torch.Generator().manual_seed(mode)
    a = torch.randn(128, 128, generator=g).to(torch.bfloat16)
    b = torch.randn(128, 128, generator=g).to(torch.bfloat16)
    ref = a.double() @ b.double().T
    a_in = a.T.contiguous() if mode & 4 else a
    b_in = b.T.contiguous() if mode & 1 else b
    d = ops.selftest_umma(mode, a_in.cuda(), b_in.cuda()).cpu().double()
    err = (d - ref).abs().max().item()
    assert err < 1e-3, f"mode {mode}: max err {err}"


def _topk_case(ops, B, I, d, K, S, seed, with_seen=True):
    from oracle import sasrec as osr

    g = torch.Generator().manual_seed(seed)
    hq = (torch.randn(B, d, generator=g) * 0.5).to(torch.bfloat16)
    table = (torch.randn(I, d, generator=g) * 0.5).to(torch.bfloat16)
    seen = torch.randint(0, I + 5, (B, S), generator=g) if with_seen else None  # ids >= I are padding
    if with_seen:
        seen[0, :] = I  # a user with nothing seen
        seen[1, : S // 2] = seen[1, 0]  # duplicates
    ids_ref, sc_ref = osr.score_topk(hq.float(), table.float(), seen, K, acc_dtype=torch.float64)
    seen_sorted = ops.seen_prepare(seen.cuda(), I) if with_seen else None
    ids, sc = ops.score_topk(hq.cuda(), table.cuda(), K, seen_sorted)
    ids, sc = ids.cpu(), sc.cpu()
    torch.testing.assert_close(sc.double(), sc_ref, rtol=1e-4, atol=1e-4)
    mism = ids != ids_ref
    if mism.any():
        # adjudicate in fp64: a swap is only acceptable between scores closer than fp32 accumulation noise
        full = hq.double() @ table.double().T
        gap = (torch.gather(full, 1, ids.clamp_min(0)) - torch.gather(full, 1, ids_ref)).abs()
        assert (gap[mism] < 1e-5).all(), f"{int(mism.sum())} index mismatches beyond fp32 noise"
        assert mism.float().mean() < 1e-3
    return ids, sc


@pytest.mark.parametrize("B,I,d,K,S", [(6, 300, 64, 10, 16), (128, 4000, 64, 10, 50), (300, 50000, 128, 10, 200),
                                       (512, 20001, 128, 20, 64), (130, 9000, 256, 5, 32), (64, 5000, 512, 10, 32)])
def test_score_topk_matches_oracle(ops, B, I, d, K, S):
    _topk_case(ops, B, I, d, K, S, seed=B + I)


def test_score_topk_no_filter(ops):
    _topk_case(ops, 200, 10000, 128, 10, 0, seed=5, with_seen=False)


def test_score_topk_golden_reference(ops, golden_dir):
    """End of the reference chain on the golden vectors generated from the real reference: eval hidden (bf16-rounded)
    x item table -> SeenItemsFilter -> torch.topk.  The hidden/table are rounded to bf16 for the kernel, so compare against
    the oracle on the same rounded inputs, and check the reference's own top-k set overlaps almost entirely."""
    import os

    import numpy as np

    from oracle import golden
    from oracle import sasrec as osr

    z = golden.load(os.path.join(golden_dir, "sasrec_new_small.npz"))
    n_items, d = int(z["n_items"]), int(z["d"])
    table = torch.from_numpy(z["sd::body.embedder.feature_embedders.item_id.emb.weight"])[:n_items]
    hq = torch.from_numpy(z["eval_hidden_last"])
    seen = torch.from_numpy(z["seen_ids"])
    hq16, tb16 = hq.to(torch.bfloat16), table.to(torch.bfloat16)
    ids_ref, _ = osr.score_topk(hq16.float(), tb16.float(), seen, 10)
    ids, sc = ops.score_topk(hq16.cuda(), tb16.cuda(), 10, ops.seen_prepare(seen.cuda(), n_items))
    assert torch.equal(ids.cpu(), ids_ref)
    ref_ids = torch.from_numpy(z["topk_ids"])
    overlap = np.mean([len(set(a.tolist()) & set(b.tolist())) / 10 for a, b in zip(ids.cpu(), ref_ids)])
    assert overlap > 0.9


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("T,n_valid,I,d", [(256, 256, 1000, 64), (300, 217, 5000, 128), (1024, 1000, 20001, 128),
                                           (384, 300, 3000, 256)])
def test_ce_head_fwd_bwd_matches_oracle(ops, T, n_valid, I, d, fused):
    """Fused CE head vs the oracle's logsumexp CE (nn/loss/ce.py:49-81) and its autograd gradients."""
    g = torch.Generator().manual_seed(T + I)
    hc = (torch.randn(T, d, generator=g) * 1.0).to(torch.bfloat16)
    hc[n_valid:] = 0
    table = (torch.randn(I, d, generator=g) * 0.3).to(torch.bfloat16)
    labels = torch.randint(0, I, (T,), generator=g, dtype=torch.int64)
    # oracle in fp64 on the same bf16-rounded inputs
    h64 = hc[:n_valid].double().requires_grad_(True)
    e64 = table.double().requires_grad_(True)
    logits = h64 @ e64.T
    lse = torch.logsumexp(logits, -1)
    loss = (lse - logits.gather(1, labels[:n_valid, None])[:, 0]).mean()
    loss.backward()

    st = ops.CEHeadState(T, I, d, "cuda")
    nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
    d_hc = torch.zeros(T, d, device="cuda", dtype=torch.bfloat16)
    out = ops.ce_head_fwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc=d_hc if fused else None,
                          n_valid_hint=n_valid)
    torch.cuda.synchronize()
    assert abs(out[0].item() - loss.item()) < 2e-4 * max(1.0, abs(loss.item())), (out[0].item(), loss.item())
    assert abs(out[1].item() - 1.0 / n_valid) < 1e-9
    torch.testing.assert_close(st.lse[:n_valid].cpu().double(), lse.detach(), rtol=1e-5, atol=1e-4)

    d_tab = torch.full((I + 1, d), 7.0, device="cuda", dtype=torch.float32)  # must be overwritten, pad row untouched
    ops.ce_head_bwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc, d_tab)
    torch.cuda.synchronize()
    gh, ge = h64.grad, e64.grad
    # softmax probabilities travel through bf16 (8 bit mantissa): compare with a norm-relative tolerance
    eh = (d_hc[:n_valid].cpu().double() - gh).norm() / gh.norm()
    ee = (d_tab[:I].cpu().double() - ge).norm() / ge.norm()
    assert eh < 1e-2, f"dH rel err {eh}"
    assert ee < 1e-2, f"dE rel err {ee}"
    assert (d_tab[I] == 7.0).all()
    assert (d_hc[n_valid:] == 0).all()


def test_ce_head_fused_falls_back_when_logits_are_unbounded(ops):
    """The single-reference-max trick is guarded by a device-side bound on |logit|; huge logits must take the two-pass
    path (and still give the right loss / gradients) without any host-side decision."""
    T, n_valid, I, d = 256, 200, 2000, 64
    g = torch.Generator().manual_seed(1)
    hc = (torch.randn(T, d, generator=g) * 6.0).to(torch.bfloat16)  # ||h|| ~ 48, ||e|| ~ 16 -> bound far above 100/log2e
    hc[n_valid:] = 0
    table = (torch.randn(I, d, generator=g) * 2.0).to(torch.bfloat16)
    labels = torch.randint(0, I, (T,), generator=g, dtype=torch.int64)
    h64, e64 = hc[:n_valid].double().requires_grad_(True), table.double().requires_grad_(True)
    logits = h64 @ e64.T
    loss = (torch.logsumexp(logits, -1) - logits.gather(1, labels[:n_valid, None])[:, 0]).mean()
    loss.backward()
    st = ops.CEHeadState(T, I, d, "cuda")
    nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
    d_hc = torch.zeros(T, d, device="cuda", dtype=torch.bfloat16)
    d_tab = torch.zeros(I + 1, d, device="cuda")
    out = ops.ce_head_fwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc=d_hc, n_valid_hint=n_valid)
    ops.ce_head_bwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc, d_tab)
    torch.cuda.synchronize()
    assert abs(out[0].item() - loss.item()) < 1e-3 * abs(loss.item()), (out[0].item(), loss.item())
    assert (d_hc[:n_valid].cpu().double() - h64.grad).norm() / h64.grad.norm() < 1e-2
    assert (d_tab[:I].cpu().double() - e64.grad).norm() / e64.grad.norm() < 1e-2


@pytest.mark.parametrize("M,N,K,b_mn", [(2048, 128, 128, False), (5000, 256, 128, False), (3000, 128, 256, True),
                                        (1500, 384, 64, True), (2048, 128, 128, True), (4096, 512, 128, False),
                                        (300, 128, 128, False), (257, 192, 128, True)])
def test_gemm_matches_matmul(ops, M, N, K, b_mn, monkeypatch):
    """rp_gemm (tile kernel and the weight-stationary persistent kernel, forced on here for M >= 1024) with the fused
    epilogue: bias + ReLU + residual, K-major and MN-major weights."""
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, generator=g) * 0.2).to(torch.bfloat16)
    bias = torch.randn(N, generator=g)
    R = torch.randn(M, N, generator=g).to(torch.bfloat16)
    ref = torch.relu(A.double() @ W.double().T + bias.double()) + R.double()
    Bop = W.T.contiguous() if b_mn else W  # MN-major: stored [K, N]
    C = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
    ops.gemm(A.cuda(), Bop.cuda(), C, M, N, K, b_mn=b_mn, bias=bias.cuda(), act=1, residual=R.cuda())
    torch.cuda.synchronize()
    err = (C.cpu().double() - ref).abs().max().item()
    assert err < 0.08, err  # bf16 output rounding of O(10) values
    # fp32 output, no epilogue: tight tolerance
    C32 = torch.zeros(M, N, device="cuda", dtype=torch.float32)
    ops.gemm(A.cuda(), Bop.cuda(), C32, M, N, K, b_mn=b_mn, out_mode=2)
    torch.cuda.synchronize()
    assert (C32.cpu().double() - A.double() @ W.double().T).abs().max().item() < 2e-3


def test_gemm_exp2_epilogue_dynamic_limits_and_accumulate(ops):
    """The additions behind the d = 512 CE backward: act 3 (exp2 with a per-row offset), device-side M / K limits and the
    non-atomic accumulate store."""
    g = torch.Generator().manual_seed(5)
    M, N, K = 700, 1000, 512
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16)
    W = (torch.randn(N, K, generator=g) * 0.1).to(torch.bfloat16)
    off = torch.randn(M, generator=g) - 3.0
    n_rows = torch.tensor([533], dtype=torch.int32, device="cuda")
    C = torch.full((M, 1024), 9.0, device="cuda", dtype=torch.bfloat16)  # pitch 1024 > N
    ops.gemm(A.cuda(), W.cuda(), C, M, N, K, act=3, row_exp2_offset=off.cuda(), m_limit=n_rows)
    torch.cuda.synchronize()
    ref = torch.exp2((A.double() @ W.double().T) * 1.4426950408889634 + off.double()[:, None])
    got = C[:, :N].cpu().double()
    assert ((got[:533] - ref[:533]).abs() / (ref[:533].abs() + 1e-6)).max() < 1.5e-2      # bf16 output
    assert (C[640:, :N] == 9.0).all() and (C[:, N:] == 9.0).all()                          # skipped tiles / pitch untouched
    # K limit + accumulate: D (+)= A^T . B over the first *k rows only
    Kt, Mo, No = 900, 304, 512
    X = (torch.randn(Kt, Mo, generator=g) * 0.3).to(torch.bfloat16)   # stored [K, M]  (A read MN-major)
    Y = (torch.randn(Kt, No, generator=g) * 0.3).to(torch.bfloat16)   # stored [K, N]  (B read MN-major)
    for kl in (0, 1, 450, 900, 5000):
        klim = torch.tensor([kl + 100], dtype=torch.int32, device="cuda")
        D = torch.full((Mo, No), 2.0, device="cuda")
        ops.gemm(X.cuda(), Y.cuda(), D, Mo, No, Kt, a_mn=True, b_mn=True, out_mode=4, k_limit=klim, k_limit_base=100)
        E = torch.full((Mo, No), 2.0, device="cuda")
        ops.gemm(X.cuda(), Y.cuda(), E, Mo, No, Kt, a_mn=True, b_mn=True, out_mode=2, k_limit=klim, k_limit_base=100)
        torch.cuda.synchronize()
        k = min((kl + 63) // 64 * 64, Kt)  # the limit acts on whole 64-row contraction chunks
        refd = X[:k].double().T @ Y[:k].double()
        assert (E.cpu().double() - refd).abs().max() < 5e-3, kl
        assert (D.cpu().double() - 2.0 - refd).abs().max() < 5e-3, kl


@pytest.mark.parametrize("T,n_valid,I,budget", [(700, 533, 3000, None), (700, 533, 3000, 256 * 3008 * 2), (384, 384, 1001, 1),
                                                (512, 0, 640, None)])
def test_ce_head_wide_hidden_matches_oracle(ops, T, n_valid, I, budget, monkeypatch):
    """d = 512 (config 5): two-pass forward + chunked materialised-G backward, several chunk sizes (budget env)."""
    d = 512
    if budget is not None:
        monkeypatch.setenv("RP_CE_WIDE_G_BYTES", str(budget))
    g = torch.Generator().manual_seed(T + I)
    hc = (torch.randn(T, d, generator=g) * 0.7).to(torch.bfloat16)
    hc[n_valid:] = 0
    table = (torch.randn(I, d, generator=g) * 0.15).to(torch.bfloat16)
    labels = torch.randint(0, I, (T,), generator=g, dtype=torch.int64)
    st = ops.CEHeadState(T, I, d, "cuda")
    nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
    d_hc = torch.zeros(T, d, device="cuda", dtype=torch.bfloat16)
    d_tab = torch.full((I + 1, d), 7.0, device="cuda", dtype=torch.float32)
    out = ops.ce_head_fwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc=d_hc, n_valid_hint=n_valid)
    ops.ce_head_bwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc, d_tab)
    torch.cuda.synchronize()
    if n_valid == 0:
        assert (d_tab[:I] == 0).all() and (d_tab[I] == 7.0).all()
        return
    h64, e64 = hc[:n_valid].double().requires_grad_(True), table.double().requires_grad_(True)
    logits = h64 @ e64.T
    lse = torch.logsumexp(logits, -1)
    loss = (lse - logits.gather(1, labels[:n_valid, None])[:, 0]).mean()
    loss.backward()
    assert abs(out[0].item() - loss.item()) < 2e-4 * max(1.0, abs(loss.item())), (out[0].item(), loss.item())
    torch.testing.assert_close(st.lse[:n_valid].cpu().double(), lse.detach(), rtol=1e-5, atol=1e-4)
    eh = (d_hc[:n_valid].cpu().double() - h64.grad).norm() / h64.grad.norm()
    ee = (d_tab[:I].cpu().double() - e64.grad).norm() / e64.grad.norm()
    assert eh < 1e-2 and ee < 1e-2, (eh, ee)
    assert (d_tab[I] == 7.0).all()


def test_activation_dropout_generator_statistics(ops):
    """The counter hash behind the activation dropout (rp_philox.cuh drop_row_key / drop_col_key / drop_mix), observed through rp_dropout_bwd on an all-ones
    input: keep rate, no row / column / lag structure, different masks for different sites, seeds and step counters."""
    from replay_b200._lib import check, lib
    rows, cols, p = 8192, 128, 0.2
    x = torch.ones(rows, cols, device="cuda", dtype=torch.bfloat16)
    st = torch.cuda.current_stream().cuda_stream

    def mask(seed, off, counter=None):
        out = torch.empty_like(x)
        cptr = None if counter is None else counter.data_ptr()
        check(lib().rp_dropout_bwd(x.data_ptr(), out.data_ptr(), rows, cols, None, p, seed, off, cptr, st), "rp_dropout_bwd")
        return (out.float() > 0)

    m = mask(1234, 3 << 40)
    n = rows * cols
    sig = (p * (1 - p) / n) ** 0.5
    assert abs(m.float().mean().item() - (1 - p)) < 5 * sig
    assert (m.float().mean(0) - (1 - p)).abs().max() < 6 * (p * (1 - p) / rows) ** 0.5      # columns
    assert (m.float().mean(1) - (1 - p)).abs().max() < 6 * (p * (1 - p) / cols) ** 0.5      # rows
    f = m.float().flatten() - (1 - p)
    for lag in (1, 2, 3, 4, 5, 8, 128, 129):                                                 # serial correlation
        c = (f[:-lag] * f[lag:]).mean().item() / (p * (1 - p))
        assert abs(c) < 6 / n ** 0.5, (lag, c)
    assert torch.equal(m, mask(1234, 3 << 40))                                               # regenerable
    for other in (mask(1235, 3 << 40), mask(1234, 4 << 40), mask(1234, 3 << 40, torch.tensor([7], device="cuda", dtype=torch.int64))):
        agree = (m == other).float().mean().item()                                           # independent masks agree 68 %
        assert abs(agree - (p * p + (1 - p) ** 2)) < 0.005, agree


@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, False), (True, True)])
def test_persistent_streaming_gemm(ops, a_mn, b_mn):
    """gemm_ps_kernel (tiles >= #SMs, K = 512 so the weight-stationary kernel does not take it): all four operand layouts,
    fused epilogue (bias + GELU + residual, bf16 out), fp32 store and accumulate, N not a multiple of the tile."""
    g = torch.Generator().manual_seed(int(a_mn) * 2 + int(b_mn))
    M, N, K = 2504, 1184, 512          # 20 x 10 tiles, ragged last M and N tile (pitches stay 16-byte multiples)
    A = (torch.randn(M, K, generator=g) * 0.5).to(torch.bfloat16)
    W = (torch.randn(N, K, generator=g) * 0.1).to(torch.bfloat16)
    bias = torch.randn(N, generator=g)
    R = torch.randn(M, N, generator=g).to(torch.bfloat16)
    Aop = (A.T.contiguous() if a_mn else A).cuda()
    Bop = (W.T.contiguous() if b_mn else W).cuda()
    z = A.double() @ W.double().T
    ref = torch.nn.functional.gelu(z + bias.double()) + R.double()
    C = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
    ops.gemm(Aop, Bop, C, M, N, K, a_mn=a_mn, b_mn=b_mn, bias=bias.cuda(), act=2, residual=R.cuda())
    torch.cuda.synchronize()
    assert (C.cpu().double() - ref).abs().max().item() < 0.06
    C32 = torch.full((M, N), 1.5, device="cuda")
    ops.gemm(Aop, Bop, C32, M, N, K, a_mn=a_mn, b_mn=b_mn, out_mode=2)
    ops.gemm(Aop, Bop, C32, M, N, K, a_mn=a_mn, b_mn=b_mn, out_mode=4, alpha=0.5)
    torch.cuda.synchronize()
    assert (C32.cpu().double() - 1.5 * z).abs().max().item() < 5e-3
    # dynamic limits on the device
    lim = torch.tensor([1000], dtype=torch.int32, device="cuda")
    Cm = torch.full((M, N), 9.0, device="cuda")
    ops.gemm(Aop, Bop, Cm, M, N, K, a_mn=a_mn, b_mn=b_mn, out_mode=2, m_limit=lim)
    klim = torch.tensor([200], dtype=torch.int32, device="cuda")
    Ck = torch.full((M, N), 9.0, device="cuda")
    ops.gemm(Aop, Bop, Ck, M, N, K, a_mn=a_mn, b_mn=b_mn, out_mode=2, k_limit=klim)
    torch.cuda.synchronize()
    assert (Cm[:1000].cpu().double() - z[:1000]).abs().max().item() < 5e-3 and (Cm[1024:] == 9.0).all()
    zk = A[:, :256].double() @ W[:, :256].double().T      # the limit acts on whole 64-element chunks: 200 -> 256
    assert (Ck.cpu().double() - zk).abs().max().item() < 5e-3


def test_ce_head_wide_hidden_large_enough_for_the_persistent_gemm(ops):
    """d = 512 CE backward at a size whose G / dE GEMMs run on gemm_ps_kernel (exp2 epilogue + device-side row limit, MN-major
    operands + device-side contraction limit)."""
    T, n_valid, I, d = 1536, 1300, 5000, 512
    g = torch.Generator().manual_seed(11)
    hc = (torch.randn(T, d, generator=g) * 0.7).to(torch.bfloat16)
    hc[n_valid:] = 0
    table = (torch.randn(I, d, generator=g) * 0.15).to(torch.bfloat16)
    labels = torch.randint(0, I, (T,), generator=g, dtype=torch.int64)
    st = ops.CEHeadState(T, I, d, "cuda")
    nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
    d_hc = torch.zeros(T, d, device="cuda", dtype=torch.bfloat16)
    d_tab = torch.full((I + 1, d), 7.0, device="cuda", dtype=torch.float32)
    out = ops.ce_head_fwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc=d_hc, n_valid_hint=n_valid)
    ops.ce_head_bwd(st, hc.cuda(), table.cuda(), labels.int().cuda(), nv, d_hc, d_tab, n_valid_hint=n_valid)
    torch.cuda.synchronize()
    h64, e64 = hc[:n_valid].double().requires_grad_(True), table.double().requires_grad_(True)
    logits = h64 @ e64.T
    loss = (torch.logsumexp(logits, -1) - logits.gather(1, labels[:n_valid, None])[:, 0]).mean()
    loss.backward()
    assert abs(out[0].item() - loss.item()) < 2e-4 * abs(loss.item())
    eh = (d_hc[:n_valid].cpu().double() - h64.grad).norm() / h64.grad.norm()
    ee = (d_tab[:I].cpu().double() - e64.grad).norm() / e64.grad.norm()
    assert eh < 1e-2 and ee < 1e-2, (eh, ee)


@pytest.mark.parametrize("T,d,mask", [(3000, 128, False), (20000, 128, True), (777, 64, True), (40000, 64, False)])
def test_fused_ffn_matches_reference_formula(ops, T, d, mask):
    """rp_ffn_fused (inference): relu(y W1^T + b1) W2^T + b2 + y in one pass, ragged last tile, optional row mask."""
    from replay_b200._lib import check, lib
    g = torch.Generator().manual_seed(T + d)
    y = torch.randn(T, d, generator=g).to(torch.bfloat16)
    w1 = (torch.randn(d, d, generator=g) * 0.15).to(torch.bfloat16)
    w2 = (torch.randn(d, d, generator=g) * 0.15).to(torch.bfloat16)
    b1, b2 = torch.randn(d, generator=g) * 0.3, torch.randn(d, generator=g) * 0.3
    rm = (torch.rand(T, generator=g) > 0.3) if mask else None
    u = torch.relu(y.double() @ w1.double().T + b1.double()).to(torch.bfloat16).double()   # the hidden activation is bf16
    ref = u @ w2.double().T + b2.double() + y.double()
    if mask:
        ref = ref * rm[:, None].double()
    out = torch.full((T + 5, d), 3.0, device="cuda", dtype=torch.bfloat16)
    yc, w1c, w2c, b1c, b2c = y.cuda(), w1.cuda(), w2.cuda(), b1.cuda(), b2.cuda()
    rmc = rm.to(torch.uint8).cuda() if mask else None
    check(lib().rp_ffn_fused(yc.data_ptr(), w1c.data_ptr(), b1c.data_ptr(), w2c.data_ptr(), b2c.data_ptr(),
                             None if rmc is None else rmc.data_ptr(), T, d, out.data_ptr(), torch.cuda.current_stream().cuda_stream),
          "rp_ffn_fused")
    torch.cuda.synchronize()
    err = (out[:T].cpu().double() - ref).abs().max().item()
    assert err < 0.06, err            # bf16 output rounding of O(5) values
    assert (out[T:] == 3.0).all()     # nothing written beyond T


@pytest.mark.parametrize("T,d,mask", [(3000, 128, False), (20000, 128, True), (777, 64, True), (33000, 64, False)])
def test_fused_post_attention_block_matches_reference_formula(ops, T, d, mask):
    """rp_post_attn_fused (inference): h = o Wo^T + bo + q ; y = LN(h) ; out = relu(y W1^T + b1) W2^T + b2 + y."""
    from replay_b200._lib import check, lib
    g = torch.Generator().manual_seed(T * 3 + d)
    o = torch.randn(T, d, generator=g).to(torch.bfloat16)
    qin = torch.randn(T, d, generator=g).to(torch.bfloat16)
    wo, w1, w2 = ((torch.randn(d, d, generator=g) * 0.15).to(torch.bfloat16) for _ in range(3))
    bo, b1, b2, lb = (torch.randn(d, generator=g) * 0.3 for _ in range(4))
    lw = 1 + torch.randn(d, generator=g) * 0.1
    rm = (torch.rand(T, generator=g) > 0.3) if mask else None
    h = o.double() @ wo.double().T + bo.double() + qin.double()
    y = torch.nn.functional.layer_norm(h, (d,), lw.double(), lb.double(), 1e-8)
    yb = y.to(torch.bfloat16).double()                          # y feeds the FFN (and its residual) as bf16
    u = torch.relu(yb @ w1.double().T + b1.double()).to(torch.bfloat16).double()
    ref = u @ w2.double().T + b2.double() + yb
    if mask:
        ref = ref * rm[:, None].double()
    out = torch.full((T + 3, d), 3.0, device="cuda", dtype=torch.bfloat16)
    t = [x.cuda() for x in (o, qin, wo, bo, lw, lb, w1, b1, w2, b2)]
    rmc = rm.to(torch.uint8).cuda() if mask else None
    check(lib().rp_post_attn_fused(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(), t[5].data_ptr(),
                                   1e-8, t[6].data_ptr(), t[7].data_ptr(), t[8].data_ptr(), t[9].data_ptr(),
                                   None if rmc is None else rmc.data_ptr(), T, d, out.data_ptr(), 0, torch.cuda.current_stream().cuda_stream),
          "rp_post_attn_fused")
    torch.cuda.synchronize()
    err = (out[:T].cpu().double() - ref).abs().max().item()
    assert err < 0.08, err
    assert (out[T:] == 3.0).all()


@pytest.mark.parametrize("T,shapes", [(1000, [(128, 128), (128, 128), (256, 128)]), (4096 + 37, [(64, 64), (128, 64)]),
                                      (700, [(1024, 256), (256, 1024), (768, 256)])])
def test_wgrad_group_matches_matmul(ops, T, shapes):
    """rp_wgrad_group: every dW_i (+)= dY_i^T X_i and db_i (+)= colsum(dY_i) of a block in one launch, operands read in place
    (column views with a row pitch), against fp64 matmuls; accumulate semantics; bit-identical across runs (no float atomics)."""
    import ctypes

    from replay_b200._lib import WgradPair, check, lib

    g = torch.Generator().manual_seed(T)
    L = lib()
    pairs, keep = [], []
    arr = (WgradPair * len(shapes))()
    for k, (n_out, n_in) in enumerate(shapes):
        # dY is a column view of a wider array (as dK / dV inside dKV), X has its natural pitch
        wide = (torch.randn(T, n_out + 64, generator=g) * 0.5).to(torch.bfloat16).cuda()
        dY = wide[:, 64:]
        X = (torch.randn(T, n_in, generator=g) * 0.5).to(torch.bfloat16).cuda()
        dW = torch.full((n_out, n_in), 0.25, device="cuda")
        db = torch.full((n_out,), -1.0, device="cuda")
        arr[k].dY, arr[k].dy_ld, arr[k].n_out = dY.data_ptr(), dY.stride(0), n_out
        arr[k].X, arr[k].x_ld, arr[k].n_in = X.data_ptr(), X.stride(0), n_in
        arr[k].dW, arr[k].dw_ld, arr[k].db = dW.data_ptr(), dW.stride(0), db.data_ptr()
        pairs.append((dY, X, dW, db))
        keep.append(wide)
    need = L.rp_wgrad_group_workspace(arr, len(shapes))
    assert need > 0
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    check(L.rp_wgrad_group(arr, len(shapes), T, 1, ws.data_ptr(), need, st), "rp_wgrad_group")
    torch.cuda.synchronize()
    first = [(dW.clone(), db.clone()) for _, _, dW, db in pairs]
    for (dY, X, dW, db) in pairs:
        ref = dY.double().T @ X.double() + 0.25
        refb = dY.double().sum(0) - 1.0
        assert (dW.double() - ref).abs().max() < 2e-3 * max(1.0, ref.abs().max().item())
        assert (db.double() - refb).abs().max() < 2e-3 * max(1.0, refb.abs().max().item())
    # overwrite mode + determinism
    check(L.rp_wgrad_group(arr, len(shapes), T, 0, ws.data_ptr(), need, st), "rp_wgrad_group")
    torch.cuda.synchronize()
    for (dY, X, dW, db), (w1, b1) in zip(pairs, first):
        assert torch.equal(dW + 0.25, w1) or (dW + 0.25 - w1).abs().max() < 1e-5  # same partial sums, only the +0.25 differs
        torch.testing.assert_close(db - 1.0, b1, rtol=0, atol=1e-5)
    again = [(dW.clone(), db.clone()) for _, _, dW, db in pairs]
    check(L.rp_wgrad_group(arr, len(shapes), T, 0, ws.data_ptr(), need, st), "rp_wgrad_group")
    torch.cuda.synchronize()
    for (_, _, dW, db), (w2, b2) in zip(pairs, again):
        assert torch.equal(dW, w2) and torch.equal(db, b2)


@pytest.mark.parametrize("T,d", [(1000, 128), (517, 64), (128 * 150 + 5, 128)])
def test_ln_qkv_fused_matches_formula(ops, T, d):
    """rp_ln_qkv_fused: q_in = LN(x), Q = q_in Wq^T + bq, [K|V] = x Wkv^T + bkv in one pass, vs fp64 on the same bf16 inputs
    (transformer.py:99-106: the query is the NORMALISED x, keys / values the un-normalised one)."""
    from replay_b200._lib import check, lib

    g = torch.Generator().manual_seed(T + d)
    x = (torch.randn(T, d, generator=g) * 1.3 + 0.2).to(torch.bfloat16)
    w_in = (torch.randn(3 * d, d, generator=g) / d ** 0.5).to(torch.bfloat16)
    b_in = torch.randn(3 * d, generator=g) * 0.1
    ln_w, ln_b = 1 + 0.1 * torch.randn(d, generator=g), 0.1 * torch.randn(d, generator=g)
    xd = x.double()
    mean, var = xd.mean(-1, keepdim=True), xd.var(-1, unbiased=False, keepdim=True)
    q_ref = (xd - mean) / torch.sqrt(var + 1e-8) * ln_w.double() + ln_b.double()
    dev = dict(device="cuda")
    q_in, Q = torch.zeros(T, d, dtype=torch.bfloat16, **dev), torch.zeros(T, d, dtype=torch.bfloat16, **dev)
    KV = torch.zeros(T, 2 * d, dtype=torch.bfloat16, **dev)
    mo, ro = torch.zeros(T, **dev), torch.zeros(T, **dev)
    xc, wc, bc, lw, lb = x.cuda(), w_in.cuda(), b_in.cuda(), ln_w.cuda(), ln_b.cuda()
    check(lib().rp_ln_qkv_fused(xc.data_ptr(), lw.data_ptr(), lb.data_ptr(), 1e-8, wc.data_ptr(), bc.data_ptr(), T, d,
                                q_in.data_ptr(), Q.data_ptr(), KV.data_ptr(), mo.data_ptr(), ro.data_ptr(), 0,
                                torch.cuda.current_stream().cuda_stream), "rp_ln_qkv_fused")
    torch.cuda.synchronize()
    assert (q_in.cpu().double() - q_ref).abs().max() < 3e-2
    torch.testing.assert_close(mo.cpu().double(), mean[:, 0], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(ro.cpu().double(), 1 / torch.sqrt(var[:, 0] + 1e-8), rtol=1e-3, atol=1e-4)
    q16 = q_in.cpu().double()  # the Q GEMM consumes the bf16 q_in the kernel itself produced
    Q_ref = q16 @ w_in[:d].double().T + b_in[:d].double()
    KV_ref = xd @ w_in[d:].double().T + b_in[d:].double()
    assert (Q.cpu().double() - Q_ref).abs().max() < 3e-2 * max(1.0, Q_ref.abs().max().item())
    assert (KV.cpu().double() - KV_ref).abs().max() < 3e-2 * max(1.0, KV_ref.abs().max().item())
    assert (Q.cpu().double() - Q_ref).norm() / Q_ref.norm() < 5e-3 and (KV.cpu().double() - KV_ref).norm() / KV_ref.norm() < 5e-3


@pytest.mark.parametrize("T,d", [(1000, 128), (517, 64), (128 * 150 + 5, 128)])
def test_pre_attn_bwd_matches_formula(ops, T, d):
    """rp_pre_attn_bwd: dq_in = dQ Wq + dh ; LayerNorm backward ; dx = dKV Wkv + t ; dln_w, dln_b - vs fp64 autograd-free formulas."""
    from replay_b200._lib import check, lib

    g = torch.Generator().manual_seed(T * 3 + d)
    bf = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).to(torch.bfloat16)  # noqa: E731
    dQ, dKV, dh, x = bf(T, d, sc=0.3), bf(T, 2 * d, sc=0.3), bf(T, d, sc=0.3), bf(T, d, sc=1.2)
    w_in = bf(3 * d, d, sc=1 / d ** 0.5)
    ln_w = 1 + 0.1 * torch.randn(d, generator=g)
    xd = x.double()
    mean, var = xd.mean(-1), xd.var(-1, unbiased=False)
    rstd = 1 / torch.sqrt(var + 1e-8)
    xhat = (xd - mean[:, None]) * rstd[:, None]
    dq = dQ.double() @ w_in[:d].double() + dh.double()
    gg = dq * ln_w.double()
    t = rstd[:, None] * (gg - gg.mean(-1, keepdim=True) - xhat * (gg * xhat).mean(-1, keepdim=True))
    dx_ref = dKV.double() @ w_in[d:].double() + t
    dw_ref, db_ref = (dq * xhat).sum(0), dq.sum(0)
    dx = torch.zeros(T, d, dtype=torch.bfloat16, device="cuda")
    dw, db = torch.full((d,), 2.0, device="cuda"), torch.full((d,), -3.0, device="cuda")
    args = [t_.cuda() for t_ in (dQ, dKV, dh, x, mean.float(), rstd.float(), ln_w, w_in)]
    check(lib().rp_pre_attn_bwd(*[a.data_ptr() for a in args], T, d, dx.data_ptr(), dw.data_ptr(), db.data_ptr(), 0,
                                torch.cuda.current_stream().cuda_stream), "rp_pre_attn_bwd")
    torch.cuda.synchronize()
    assert (dx.cpu().double() - dx_ref).norm() / dx_ref.norm() < 6e-3
    assert (dx.cpu().double() - dx_ref).abs().max() < 3e-2 * max(1.0, dx_ref.abs().max().item())
    assert ((dw.cpu().double() - 2.0) - dw_ref).norm() / dw_ref.norm() < 5e-3   # accumulated on top of the preset values
    assert ((db.cpu().double() + 3.0) - db_ref).norm() / db_ref.norm() < 5e-3


@pytest.mark.parametrize("T,d,drop,masked", [(1000, 128, 0.0, False), (900, 128, 0.25, True), (517, 64, 0.1, False),
                                             (128 * 150 + 5, 128, 0.2, False)])
def test_post_attn_bwd_matches_formula(ops, T, d, drop, masked):
    """rp_post_attn_bwd (dropout' -> FFN backward -> LayerNorm2 backward -> out-projection backward in one pass) vs fp64
    formulas; the site-2 dropout mask is taken from rp_dropout_bwd (the same stream), site 1 is encoded in the zeros of u."""
    from replay_b200._lib import check, lib

    L = lib()
    g = torch.Generator().manual_seed(T * 7 + d)
    bf = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).to(torch.bfloat16)  # noqa: E731
    dz, h = bf(T, d, sc=0.5), bf(T, d, sc=1.5)
    u = torch.relu(bf(T, d))  # ~half zeros, like relu + dropout output
    w2, w1, wo = bf(d, d, sc=1 / d ** 0.5), bf(d, d, sc=1 / d ** 0.5), bf(d, d, sc=1 / d ** 0.5)
    ln_w = 1 + 0.1 * torch.randn(d, generator=g)
    rowmask = (torch.rand(T, generator=g) > 0.3).to(torch.uint8) if masked else None
    seed, off2 = 1234567, 5 << 40
    st = torch.cuda.current_stream().cuda_stream
    ctr = torch.tensor([99], dtype=torch.int64, device="cuda")
    # reference mask of site 2: d_t_ref = dropout_bwd(dz * rowmask)
    dzc = dz.cuda()
    ones = torch.ones(T, d, dtype=torch.bfloat16, device="cuda")
    keep = torch.empty_like(ones)
    check(L.rp_dropout_bwd(ones.data_ptr(), keep.data_ptr(), T, d, None, drop, seed, off2, ctr.data_ptr(), st), "rp_dropout_bwd")
    keep = keep.cpu().double()  # 0 or 1/(1-p) (bf16-rounded scale: divide it out)
    keep = (keep > 0).double() / (1.0 - drop)
    rm = rowmask.double()[:, None] if masked else 1.0
    dzm = dz.double() * rm
    d_t = dzm * keep
    hd = h.double()
    mean, var = hd.mean(-1), hd.var(-1, unbiased=False)
    rstd = 1 / torch.sqrt(var + 1e-8)
    xhat = (hd - mean[:, None]) * rstd[:, None]
    d_t16 = d_t.to(torch.bfloat16).double()
    du = (d_t16 @ w2.double()) * (u.double() != 0) / (1.0 - drop)
    du16 = du.to(torch.bfloat16).double()
    dy = du16 @ w1.double() + dzm
    gg = dy * ln_w.double()
    dh = rstd[:, None] * (gg - gg.mean(-1, keepdim=True) - xhat * (gg * xhat).mean(-1, keepdim=True))
    d_o = dh.to(torch.bfloat16).double() @ wo.double()
    o = {k: torch.zeros(T, d, dtype=torch.bfloat16, device="cuda") for k in ("d_t", "du", "dh", "d_o")}
    dw, db = torch.full((d,), 1.0, device="cuda"), torch.full((d,), -1.0, device="cuda")
    need_dt = masked or drop > 0
    args = [dzc, u.cuda(), h.cuda(), mean.float().cuda(), rstd.float().cuda(), ln_w.cuda(), w2.cuda(), w1.cuda(), wo.cuda()]
    rmc = rowmask.cuda() if masked else None
    check(L.rp_post_attn_bwd(*[a.data_ptr() for a in args], None if rmc is None else rmc.data_ptr(), T, d, drop, seed, off2,
                             ctr.data_ptr(), o["d_t"].data_ptr() if need_dt else None, o["du"].data_ptr(), o["dh"].data_ptr(),
                             o["d_o"].data_ptr(), dw.data_ptr(), db.data_ptr(), 0, st), "rp_post_attn_bwd")
    torch.cuda.synchronize()
    rel = lambda a, b: float((a.cpu().double() - b).norm() / b.norm())  # noqa: E731
    if need_dt:
        assert rel(o["d_t"], d_t) < 5e-3
    assert rel(o["du"], du) < 8e-3, rel(o["du"], du)
    assert rel(o["dh"], dh) < 1e-2, rel(o["dh"], dh)
    assert rel(o["d_o"], d_o) < 1.2e-2, rel(o["d_o"], d_o)
    assert float(((dw.cpu().double() - 1.0) - (dy * xhat).sum(0)).norm() / (dy * xhat).sum(0).norm()) < 1e-2
    assert float(((db.cpu().double() + 1.0) - dy.sum(0)).norm() / dy.sum(0).norm()) < 1e-2


def test_gemm_weight_stationary_wide_tile_matches_matmul(ops):
    """The predict body's K | V projection shape (M >= 131072 rows, N = 256, K = 128, bias): gemm_ws_kernel<256> keeps both
    128-column halves of the weight in one CTA so the activations are read once; against a fp32 matmul of the same bf16 data."""
    cuda = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(5)
    M, N, K = 131072 + 300, 256, 128
    A = (torch.randn(M, K, device=cuda, generator=g) * 0.5).bfloat16()
    W = (torch.randn(N, K, device=cuda, generator=g) * 0.2).bfloat16()
    b = torch.randn(N, device=cuda, generator=g)
    C = torch.zeros(M, N, device=cuda, dtype=torch.bfloat16)
    ops.gemm(A, W, C, M, N, K, bias=b)
    torch.cuda.synchronize()
    rows = torch.cat([torch.arange(0, 4096, device=cuda), torch.arange(M - 4096, M, device=cuda)])
    ref = A[rows].float() @ W.float().T + b
    assert torch.allclose(C[rows].float(), ref, atol=3e-2, rtol=2e-2)
    assert float((C[rows].float() - ref).abs().mean()) < 4e-3
