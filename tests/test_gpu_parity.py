"""GPU parity: the sm_100a kernels (through the C ABI) vs the oracle and vs the committed
fixtures of the executed reference.  Tolerances: floats <= 1e-4 relative (north_star), integer
outputs bit-exact.  bf16/fp16 storage is compared against the fp32 oracle at the storage type's
own precision and reported separately."""
import math

import pytest
import torch

from conftest import load_golden, rel_err
from oracle import pooling_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4


def dev(t):
    return t.cuda() if isinstance(t, torch.Tensor) else t


def ragged_ptr(gen, n, mean, p_empty=0.15, max_count=None):
    counts = torch.poisson(torch.full((n,), float(mean)), generator=gen).long()
    if max_count is not None:
        counts = counts.clamp(max=max_count)
    counts[torch.rand(n, generator=gen) < p_empty] = 0
    return torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)])


def close(a, b, tol=TOL, what=""):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = max(float(b.abs().max()), 1e-30) if b.numel() else 1.0
    err = float((a - b).abs().max()) / scale if b.numel() else 0.0
    assert err <= tol, f"{what}: rel err {err:.3e} > {tol}"


# ------------------------------------------------------------------------------------------------
# segment primitives vs the reference fixtures
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["k7", "k32"])
def test_segment_ops_vs_reference_fixture(tag):
    from deepviewagg_b200 import ops
    g = load_golden("segment_ops_" + tag)
    x, ptr = g["src"].cuda(), g["ptr"].cuda()
    for red in ("sum", "mean", "max", "min"):
        xr = x.clone().requires_grad_(True)
        o = ops.segment_csr(xr, ptr, reduce=red)
        close(o, g[f"out_{red}"], 1e-6, f"segment_csr {red}")
        gr = torch.autograd.grad((o * g["w"].cuda()).sum(), xr)[0]
        close(gr, g[f"grad_{red}"], 1e-6, f"segment_csr grad {red}")
        close(ops.segment_gather_csr(x, ptr, reduce=red), g[f"seg_gather_{red}"], 1e-6)
    for s in (0, 1):
        xr = x.clone().requires_grad_(True)
        o = ops.segment_softmax_csr(xr, ptr, scaling=bool(s))
        close(o, g[f"softmax_{s}"], 1e-5, "segment_softmax")
        gr = torch.autograd.grad((o * g["wv"].cuda()).sum(), xr)[0]
        assert (gr.cpu() - g[f"softmax_grad_{s}"]).abs().max() < 1e-5
    sr = g["gather_src"].cuda().requires_grad_(True)
    o = ops.gather_csr(sr, ptr)
    assert torch.equal(o.cpu(), g["gather_out"])
    gr = torch.autograd.grad((o * g["wv"].cuda()).sum(), sr)[0]
    close(gr, g["gather_grad"], 1e-5, "gather_csr grad")


def test_kat_softmax_gpu():
    from deepviewagg_b200 import ops
    g = load_golden("kat_softmax")
    out = ops.segment_softmax_csr(g["src"].cuda(), g["csr"].cuda())
    close(out, g["out"], 1e-6)
    out = ops.segment_softmax_csr(g["src"].cuda(), g["csr"].cuda(), scaling=True)
    close(out, g["out_scaled"], 1e-6)
    em = ops.segment_softmax_csr(torch.tensor([[1.], [2.], [3.]]).cuda(), torch.tensor([0, 2, 2, 3]).cuda())
    close(em, g["empty_mid"], 1e-6)
    assert torch.equal(ops.gather_csr(torch.tensor([[1.], [2.], [3.]]).cuda(),
                                      torch.tensor([0, 2, 2, 5]).cuda()).cpu(), g["gather"])


def test_segment_edge_cases():
    from deepviewagg_b200 import ops
    # all-empty, single huge segment, first-arg ties, 1D source, zero segments
    ptr = torch.tensor([0, 0, 0, 0]).cuda()
    x = torch.zeros(0, 5).cuda()
    for red in ("sum", "mean", "max", "min"):
        assert torch.equal(ops.segment_csr(x, ptr, reduce=red).cpu(), torch.zeros(3, 5))
    x = torch.tensor([1., 3., 3., 2., 3.]).cuda().requires_grad_(True)
    ptr = torch.tensor([0, 5]).cuda()
    o = ops.segment_csr(x, ptr, reduce="max")
    o.sum().backward()
    assert x.grad.tolist() == [0, 1, 0, 0, 0]          # first arg-max only (torch_scatter)
    vals, arg = ops.segment_csr_arg(torch.tensor([[2.], [2.], [5.]]).cuda(), torch.tensor([0, 2, 2, 3]).cuda(), "min")
    assert arg.view(-1).tolist() == [0, 3, 2] and vals.view(-1).tolist() == [2, 0, 5]
    big = torch.randn(100000, 3).cuda()
    close(ops.segment_csr(big, torch.tensor([0, 100000]).cuda(), reduce="mean"), big.mean(0, keepdim=True), 1e-4)
    with pytest.raises(TypeError):
        ops.segment_csr(big, torch.tensor([0, 100000], dtype=torch.int32).cuda())


@pytest.fixture(params=["stream", "ring", "lane"])
def va_path(request):
    """Run the test once per kernel pair of the fused view attention (dva_view_attention_set_path):
    'stream' = streaming kernels for both passes, 'ring' = ring forward + lane-per-view backward, 'lane' =
    streaming forward + lane-per-view backward (ring / lane wherever they apply); the default 'auto' choice
    is restored afterwards."""
    from deepviewagg_b200 import _lib
    lib = _lib.load()
    assert lib.dva_view_attention_set_path({"stream": 1, "ring": 2, "lane": 3}[request.param]) == 0
    yield request.param
    assert lib.dva_view_attention_set_path(0) == 0


# ------------------------------------------------------------------------------------------------
# the fused kernel vs the oracle
# ------------------------------------------------------------------------------------------------
def _run_va(N, mean_v, C, G, seed, dtype=torch.float32, use_idx=None, gating=True, scaling=True,
            p_empty=0.15, tol=TOL, perm=True):
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(seed)
    ptr = ragged_ptr(gen, N, mean_v, p_empty)
    V = int(ptr[-1])
    R = V if (use_idx is None or perm) else V + 13
    x = torch.randn(R, C, generator=gen)
    if dtype != torch.float32:
        x = x.to(dtype).float()  # the oracle sees exactly the stored values
    compat = torch.randn(V, G, generator=gen) * 2
    if V > 3:
        compat[1] = compat[0]  # ties on the arg-max path
    idx = None
    if use_idx is not None:
        idx = torch.randperm(R, generator=gen)[:V] if perm else torch.randint(0, R, (V,), generator=gen)
        idx = idx.to(use_idx)
    gw = (torch.randn(1, G, generator=gen) * 0.7 + 1) if gating else None
    gb = (torch.randn(1, G, generator=gen) * 0.3) if gating else None
    w = torch.randn(N, C, generator=gen)

    xo, co = x.clone().requires_grad_(True), compat.clone().requires_grad_(True)
    gwo = gw.clone().requires_grad_(True) if gating else None
    gbo = gb.clone().requires_grad_(True) if gating else None
    ref_out, ref_att = O.view_attention(xo, co, ptr, G, idx=idx, gate_weight=gwo, gate_bias=gbo,
                                        group_scaling=scaling)
    leaves = [xo, co] + ([gwo, gbo] if gating else [])
    ref_g = torch.autograd.grad((ref_out * w).sum(), leaves)

    xg = x.to(dtype).cuda().requires_grad_(True)
    cg = compat.cuda().requires_grad_(True)
    gwg = gw.cuda().requires_grad_(True) if gating else None
    gbg = gb.cuda().requires_grad_(True) if gating else None
    out, att, seg_max = ops.view_attention(xg, cg, ptr.cuda(), G, idx=dev(idx), gate_weight=gwg,
                                           gate_bias=gbg, group_scaling=scaling, idx_is_permutation=perm)
    gl = [xg, cg] + ([gwg, gbg] if gating else [])
    got_g = torch.autograd.grad((out.float() * w.cuda()).sum(), gl)
    torch.cuda.synchronize()
    close(out.float(), ref_out, tol, "out")
    close(att, ref_att, 1e-5 if dtype == torch.float32 else 1e-4, "attentions")
    # unseen points: exact zeros (SURVEY D.1)
    empty = (ptr[1:] == ptr[:-1])
    assert (out[empty.cuda()] == 0).all()
    names = ["grad_x", "grad_compat", "grad_gate_w", "grad_gate_b"]
    # half storage: out and the upstream gradient are rounded to the storage type before the
    # backward pass, so gradients carry ~2 storage-ulps of relative error
    gtol = tol if dtype == torch.float32 else 3 * tol
    for n, a, b in zip(names, got_g, ref_g):
        close(a.float(), b, gtol, n)


@pytest.mark.parametrize("C,G", [(128, 4), (64, 4), (32, 4), (16, 2), (512, 4), (256, 8), (8, 8),
                                 (10, 4), (20, 1), (96, 32), (1024, 4), (7, 1), (130, 2), (36, 4)])
def test_view_attention_shapes(C, G, va_path):
    _run_va(300, 6, C, G, seed=C * 7 + G)


@pytest.mark.parametrize("kw", [dict(gating=False), dict(scaling=False), dict(use_idx=torch.int32),
                                dict(use_idx=torch.int64), dict(use_idx=torch.int64, perm=False),
                                dict(gating=False, scaling=False, use_idx=torch.int32)])
def test_view_attention_variants(kw, va_path):
    _run_va(257, 5, 128, 4, seed=5, **kw)
    _run_va(120, 9, 48, 4, seed=6, **kw)


def test_view_attention_long_segments_and_empties(va_path):
    _run_va(40, 90, 128, 4, seed=1)                 # segments > 32 views (multi-chunk path)
    _run_va(9, 300, 64, 4, seed=2, use_idx=torch.int32)
    _run_va(64, 3, 128, 4, seed=3, p_empty=0.9)     # mostly unseen points
    _run_va(50, 4, 128, 4, seed=4, p_empty=1.0)     # no view at all (V == 0)
    _run_va(1, 1, 128, 4, seed=8, p_empty=0.0)
    # ring forward: segments cut into several pieces at arbitrary batch offsets, 16/32-row batches
    _run_va(40, 90, 64, 4, seed=13)
    _run_va(700, 21, 32, 4, seed=14, use_idx=torch.int32)
    _run_va(500, 40, 128, 8, seed=15, dtype=torch.float32)
    _run_va(33, 70, 16, 4, seed=16)


def test_view_attention_many_ranges(va_path):
    # more point ranges than resident warps: every warp walks several ranges (ring refill between them)
    _run_va(60000, 3, 64, 4, seed=21, use_idx=torch.int32)
    _run_va(45000, 2, 128, 4, seed=22, p_empty=0.5)


@pytest.mark.parametrize("dtype,tol", [(torch.bfloat16, 1.6e-2), (torch.float16, 2e-3)])
def test_view_attention_half_storage(dtype, tol, va_path):
    # storage-precision parity (fp32 accumulate): reported separately from the 1e-4 fp32 bar
    _run_va(300, 8, 128, 4, seed=10, dtype=dtype, tol=tol)
    _run_va(200, 8, 64, 4, seed=11, dtype=dtype, tol=tol, use_idx=torch.int32)
    _run_va(100, 8, 12, 4, seed=12, dtype=dtype, tol=tol)   # non-vectorisable C


def test_view_attention_zero_points(va_path):
    from deepviewagg_b200 import ops
    out, att, _ = ops.view_attention(torch.zeros(0, 16).cuda(), torch.zeros(0, 4).cuda(),
                                     torch.zeros(1, dtype=torch.long).cuda(), 4)
    assert out.shape == (0, 16) and att.shape == (0, 4)


def test_qk_scores_vs_oracle():
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(3)
    for (N, G, D, ds) in ((200, 4, 8, True), (77, 1, 3, False), (50, 8, 2, True), (3001, 4, 8, True),
                         (500, 4, 4, True), (333, 2, 16, False), (100, 8, 16, True)):
        ptr = ragged_ptr(gen, N, 5)
        V = int(ptr[-1])
        k = torch.randn(V, G * D, generator=gen)
        q = torch.randn(N, G * D, generator=gen)
        w = torch.randn(V, G, generator=gen)
        ko, qo = k.clone().requires_grad_(True), q.clone().requires_grad_(True)
        ref = O.qk_compatibilities(ko, qo, ptr, G, ds)
        rg = torch.autograd.grad((ref * w).sum(), [ko, qo])
        kg, qg = k.cuda().requires_grad_(True), q.cuda().requires_grad_(True)
        got = ops.qk_scores(kg, qg, ptr.cuda(), G, ds)
        gg = torch.autograd.grad((got * w.cuda()).sum(), [kg, qg])
        close(got, ref, 1e-5, "qk compat")
        close(gg[0], rg[0], 1e-5, "grad keys")
        close(gg[1], rg[1], 1e-5, "grad queries")


def test_gather_pool_vs_oracle():
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(9)
    B, C, H, W, Vw = 3, 24, 20, 31, 400
    aptr = ragged_ptr(gen, Vw, 2, p_empty=0.1)
    P = int(aptr[-1])
    img = torch.randint(0, B, (Vw,), generator=gen)
    pix = torch.stack([torch.randint(0, W, (P,), generator=gen), torch.randint(0, H, (P,), generator=gen)], 1)
    fmap = torch.randn(B, C, H, W, generator=gen).relu()
    w = torch.randn(Vw, C, generator=gen)
    for red in ("max", "mean", "sum", "min"):
        fo = fmap.clone().requires_grad_(True)
        ref = O.segment_csr(O.feature_map_gather(fo, img, pix, aptr), aptr, reduce=red)
        rg = torch.autograd.grad((ref * w).sum(), fo)[0]
        for cl in (False, True):
            for pdt in (torch.int16, torch.int32):
                fg = (fmap.permute(0, 2, 3, 1).contiguous() if cl else fmap).cuda().requires_grad_(True)
                got = ops.gather_pool(fg, img.cuda(), pix.to(pdt).cuda(), aptr.cuda(), red, channels_last=cl)
                gg = torch.autograd.grad((got * w.cuda()).sum(), fg)[0]
                gg = gg.permute(0, 3, 1, 2) if cl else gg
                close(got, ref, 1e-6, f"gather_pool {red}")
                close(gg, rg, 1e-5, f"gather_pool grad {red}")


@pytest.mark.parametrize("C,dtype", [(64, torch.float32), (160, torch.float32), (64, torch.bfloat16),
                                     (8, torch.float32), (12, torch.float32)])
def test_gather_pool_channels_last_vector_path(C, dtype):
    """The 16-byte-chunk kernels of the channels-last layout: mostly one pixel per view (exact
    splatting: no arg table traffic), some views with several pixels and some with none; rows wider
    than one warp pass (C = 160) and narrower than a sub-warp (C = 8); C = 12 is the scalar path."""
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(C)
    B, H, W, Vw = 4, 33, 47, 3000
    counts = torch.ones(Vw, dtype=torch.long)
    counts[torch.rand(Vw, generator=gen) < 0.15] = 0
    counts[torch.rand(Vw, generator=gen) < 0.15] = 3
    aptr = torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)])
    P = int(aptr[-1])
    img = torch.randint(0, B, (Vw,), generator=gen)
    pix = torch.stack([torch.randint(0, W, (P,), generator=gen), torch.randint(0, H, (P,), generator=gen)], 1)
    fmap = torch.randn(B, C, H, W, generator=gen).relu().to(dtype).float()
    w = torch.randn(Vw, C, generator=gen).to(dtype).float()
    tol, gtol = (1e-6, 1e-5) if dtype == torch.float32 else (8e-3, 1e-5)
    for red in ("max", "mean", "sum", "min"):
        fo = fmap.clone().requires_grad_(True)
        ref = O.segment_csr(O.feature_map_gather(fo, img, pix, aptr), aptr, reduce=red)
        rg = torch.autograd.grad((ref * w).sum(), fo)[0]
        fg = fmap.permute(0, 2, 3, 1).contiguous().to(dtype).cuda().requires_grad_(True)
        got = ops.gather_pool(fg, img.cuda(), pix.to(torch.int16).cuda(), aptr.cuda(), red, channels_last=True)
        gg = torch.autograd.grad(got, fg, w.to(dtype).cuda())[0].float().permute(0, 3, 1, 2)
        close(got.float(), ref, tol, f"gather_pool(cl) {red}")
        close(gg, rg, gtol if dtype == torch.float32 else 8e-3, f"gather_pool(cl) grad {red}")


@pytest.mark.parametrize("interp", [False, True])
def test_gather_pool_nchw_through_transposition(interp):
    """NCHW maps of which a large share is gathered are transposed once to channels-last
    (dva_transpose_last2) and pooled by the vector kernels; same values and map gradient as the
    direct NCHW kernels (sparse gather of the same map: below the share threshold)."""
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(77)
    B, C, H, W = 3, 32, 37, 53
    fmap = torch.randn(B, C, H, W, generator=gen).relu().cuda()
    for Vw in (40, 4000):                              # 40 views: direct NCHW kernels; 4000: transposed
        counts = torch.randint(0, 3, (Vw,), generator=gen)
        aptr = torch.cat([torch.zeros(1, dtype=torch.long), counts.cumsum(0)])
        P = int(aptr[-1])
        img = torch.randint(0, B, (Vw,), generator=gen)
        msz = (2 * W, 2 * H) if interp else (W, H)
        pix = torch.stack([torch.randint(0, msz[0], (P,), generator=gen), torch.randint(0, msz[1], (P,), generator=gen)], 1)
        w = torch.randn(Vw, C, generator=gen).cuda()
        res = []
        for cl in (False, True):
            f = (fmap.permute(0, 2, 3, 1).contiguous() if cl else fmap.clone()).requires_grad_(True)
            args = (f, img.cuda(), pix.to(torch.int16).cuda(), aptr.cuda())
            out = ops.interp_pool(*args, msz, "max", channels_last=cl) if interp else ops.gather_pool(*args, "max", channels_last=cl)
            g = torch.autograd.grad(out, f, w)[0]
            res.append((out, g.permute(0, 3, 1, 2) if cl else g))
        assert torch.equal(res[0][0], res[1][0])
        close(res[0][1], res[1][1], 1e-6, "map gradient")
        assert res[0][1].shape == fmap.shape and res[0][1].is_contiguous()


# ------------------------------------------------------------------------------------------------
# the drop-in modules vs the executed reference (state_dict interchange)
# ------------------------------------------------------------------------------------------------
def _module_from_fixture(g, cls):
    kw = dict(g["kw"])
    m = cls(save_last=True, **kw)
    missing = m.load_state_dict(g["sd"], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m.cuda(), kw


@pytest.mark.parametrize("name", ["group_pool_toy", "group_pool_c64", "group_pool_usemod",
                                  "group_pool_g1_nogate", "group_pool_oddgroups", "group_pool_minmax"])
def test_group_pool_module_vs_reference(name, va_path):
    from deepviewagg_b200.modules.multimodal.pooling import GroupBimodalCSRPool
    g = load_golden(name)
    m, kw = _module_from_fixture(g, GroupBimodalCSRPool)
    m.train()
    x_mod = g["x_mod"].cuda().requires_grad_(True)
    x_map = g["x_map"].cuda().requires_grad_(True)
    out = m(None, x_mod, x_map, g["ptr"].cuda())
    params = dict(m.named_parameters())
    grads = torch.autograd.grad((out * g["w"].cuda()).sum(), [x_mod, x_map] + list(params.values()),
                                allow_unused=True)
    close(out, g["out"], TOL, "out")
    close(m._last_C, g["last_C"], TOL, "compatibilities")
    close(m._last_A, g["last_A"], TOL, "attentions")
    if m.G is not None:
        close(m._last_G, g["last_G"], TOL, "gating")
    for n, gr in zip(["x_mod", "x_map"] + ["param/" + k for k in params], grads):
        ref = g["grad"][n]
        gr = torch.zeros_like(ref) if gr is None else gr.cpu()
        assert (gr - ref).abs().max() <= 2e-4 * max(1.0, float(ref.abs().max())), (name, n)
    # running statistics were updated like the reference's (momentum 0.1)
    ge = load_golden(name + "_eval")
    for k, v in m.state_dict().items():
        if "running_" in k:
            close(v, ge["sd"][k], 1e-4, k)
    me, _ = _module_from_fixture(ge, GroupBimodalCSRPool)
    me.eval()
    with torch.no_grad():
        close(me(None, ge["x_mod"].cuda(), ge["x_map"].cuda(), ge["ptr"].cuda()), ge["out"], TOL, "eval out")


@pytest.mark.parametrize("name", ["qkv_pool_base", "qkv_pool_modqk"])
def test_qkv_pool_module_vs_reference(name, va_path):
    from deepviewagg_b200.modules.multimodal.pooling import QKVBimodalCSRPool
    g = load_golden(name)
    m, kw = _module_from_fixture(g, QKVBimodalCSRPool)
    m.train()
    x_main = g["x_main"].cuda().requires_grad_(True)
    x_mod = g["x_mod"].cuda().requires_grad_(True)
    x_map = g["x_map"].cuda().requires_grad_(True)
    out = m(x_main, x_mod, x_map, g["ptr"].cuda())
    params = dict(m.named_parameters())
    grads = torch.autograd.grad((out * g["w"].cuda()).sum(), [x_main, x_mod, x_map] + list(params.values()),
                                allow_unused=True)
    close(out, g["out"], TOL, "out")
    close(m._last_C, g["last_C"], TOL, "compatibilities")
    close(m._last_A, g["last_A"], TOL, "attentions")
    for n, gr in zip(["x_main", "x_mod", "x_map"] + ["param/" + k for k in params], grads):
        ref = g["grad"][n]
        gr = torch.zeros_like(ref) if gr is None else gr.cpu()
        assert (gr - ref).abs().max() <= 2e-4 * max(1.0, float(ref.abs().max())), (name, n)


def test_simple_pools_and_fusion_modules():
    from deepviewagg_b200.modules.multimodal.pooling import BimodalCSRPool, HeuristicBimodalCSRPool
    from deepviewagg_b200.modules.multimodal.fusion import BimodalFusion
    g = load_golden("simple_pools")
    x_mod, x_map, ptr = g["x_mod"].cuda(), g["x_map"].cuda(), g["ptr"].cuda()
    for mode in ("max", "mean", "min", "sum"):
        close(BimodalCSRPool(mode=mode)(None, x_mod, None, ptr), g["bimodal_" + mode], 1e-6)
    for mode in ("max", "min"):
        for feat in (0, 5):
            got = HeuristicBimodalCSRPool(mode=mode, feat=feat)(None, x_mod, x_map, ptr)
            assert torch.equal(got.cpu(), g[f"heuristic_{mode}_{feat}"])
    a, b = g["fusion_a"].cuda(), g["fusion_b"].cuda()
    for mode in BimodalFusion.MODES:
        assert torch.equal(BimodalFusion(mode)(a, b).cpu(), g["fusion_" + mode])
    assert BimodalFusion("residual")(None, b) is b and BimodalFusion("residual")(a, None) is a


def test_row_index_fusion_equals_materialised_gather(va_path):
    """GroupBimodalCSRPool(row_index=perm) == GroupBimodalCSRPool on x_mod[perm] (modules.py:518)."""
    from deepviewagg_b200.modules.multimodal.pooling import GroupBimodalCSRPool
    g = load_golden("group_pool_c64")
    m, kw = _module_from_fixture(g, GroupBimodalCSRPool)
    m.eval()
    x_mod, x_map, ptr = g["x_mod"].cuda(), g["x_map"].cuda(), g["ptr"].cuda()
    perm = torch.randperm(x_mod.shape[0], generator=torch.Generator().manual_seed(0)).cuda()
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(perm.numel(), device="cuda")
    with torch.no_grad():
        a = m(None, x_mod, x_map, ptr)
        b = m(None, x_mod[inv], x_map, ptr, row_index=perm)  # x_mod[inv][perm] == x_mod
    close(b, a, 1e-6, "row_index fusion")


# ------------------------------------------------------------------------------------------------
# BASELINE-size properties (no oracle can run at 1M x 32 x 128 in seconds)
# ------------------------------------------------------------------------------------------------
def test_full_size_properties(va_path):
    from deepviewagg_b200 import ops
    N, v, C, G = 1_000_000, 32, 128, 4
    V = N * v
    gen = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.randn(V, C, device="cuda", generator=gen)
    ptr = torch.arange(0, V + 1, v, device="cuda")
    # (1) constant scores -> attention 1/v -> plain mean over the point's views
    out, att, _ = ops.view_attention(x, torch.zeros(V, G, device="cuda"), ptr, G, group_scaling=True)
    close(att[:1000], torch.full((1000, G), 1.0 / v), 1e-6, "uniform attention")
    ref = x.view(N, v, C)[:50000].mean(1)
    close(out[:50000], ref, 1e-5, "mean property")
    del out, att
    # (2) attention rows sum to one per (point, group); linear in x
    compat = torch.randn(V, G, device="cuda", generator=gen)
    out1, att, _ = ops.view_attention(x, compat, ptr, G, group_scaling=True)
    s = att.view(N, v, G).sum(1)
    assert (s - 1).abs().max() < 1e-5
    out2, _, _ = ops.view_attention(x * 2.0, compat, ptr, G, group_scaling=True)
    close(out2, out1 * 2.0, 1e-6, "linearity")
    del out2
    # (3) a permuted table read through idx gives the same result (gather correctness at scale)
    perm = torch.randperm(V, device="cuda", generator=gen).int()
    xp = torch.empty_like(x)
    xp[perm.long()] = x
    out3, _, _ = ops.view_attention(xp, compat, ptr, G, idx=perm, group_scaling=True)
    assert torch.equal(out3, out1)
    del xp, out3
    # (4) backward: d(sum(out*w))/dx rows = a * w  (no gating) -- checked on a slice
    xr = x.requires_grad_(True)
    out, att, _ = ops.view_attention(xr, compat, ptr, G, group_scaling=True)
    w = torch.randn(N, C, device="cuda", generator=gen)
    (gx,) = torch.autograd.grad((out * w).sum(), xr)
    k = 2000
    exp = att[:k * v].repeat_interleave(C // G, dim=1) * w[:k].repeat_interleave(v, dim=0)
    close(gx[:k * v], exp, 1e-6, "grad_x property")


# ------------------------------------------------------------------------------------------------
# fused BatchNorm + LeakyReLU vs torch (base_modules.py:38-48 semantics)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("R,C", [(5000, 128), (777, 64), (3000, 32), (100, 8), (1, 16), (4099, 33), (20000, 512)])
def test_bn_act_vs_torch(R, C):
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(R + C)
    z = (torch.randn(R, C, generator=gen) * 2 + 3).cuda()          # non-zero mean: exercises the shift
    w = torch.randn(R, C, generator=gen).cuda()
    for training in (True, False):
        if R == 1 and training:
            continue                                              # torch refuses 1 value per channel
        bn_a = torch.nn.BatchNorm1d(C, momentum=0.1).cuda()
        bn_b = torch.nn.BatchNorm1d(C, momentum=0.1).cuda()
        with torch.no_grad():
            bn_a.weight.copy_(torch.rand(C, generator=gen) + 0.5)
            bn_a.bias.copy_(torch.randn(C, generator=gen) * 0.3)
            bn_a.running_mean.copy_(torch.randn(C, generator=gen))
            bn_a.running_var.copy_(torch.rand(C, generator=gen) + 0.5)
        bn_b.load_state_dict(bn_a.state_dict())
        bn_a.train(training), bn_b.train(training)
        za, zb = z.clone().requires_grad_(True), z.clone().requires_grad_(True)
        ya = torch.nn.functional.leaky_relu(bn_a(za), 0.2)
        yb = ops.batch_norm_act(zb, bn_b, negative_slope=0.2)
        ga = torch.autograd.grad((ya * w).sum(), [za, bn_a.weight, bn_a.bias])
        gb = torch.autograd.grad((yb * w).sum(), [zb, bn_b.weight, bn_b.bias])
        close(yb, ya, 2e-5, "bn_act y")
        for n, a, b in zip(("dz", "dgamma", "dbeta"), gb, ga):
            # LeakyReLU'(a) is decided by the sign of a ~ 0 for a handful of elements (torch keeps the
            # sign of its own rounded output): allow isolated flips, bound everything else tightly
            bad = (a - b).abs() > 2e-4 * max(1.0, float(b.abs().max()))
            assert int(bad.sum()) <= 4 + a.numel() // 100000, (n, training, int(bad.sum()))
        close(bn_b.running_mean, bn_a.running_mean, 1e-5, "running_mean")
        close(bn_b.running_var, bn_a.running_var, 1e-5, "running_var")
        assert int(bn_b.num_batches_tracked) == int(bn_a.num_batches_tracked)


# ------------------------------------------------------------------------------------------------
# tcgen05 projection GEMM vs an fp64 matmul
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N", [(4096, 128, 128), (1000, 64, 64), (37, 8, 32), (50000, 128, 64), (3000, 512, 512),
                                   (129, 32, 4), (1, 16, 16),
                                   # skinny kernels (K, N <= 64): the DeepSetFeat layers 8->32, 32->32, 33->32, 64->32
                                   (70001, 8, 32), (100000, 32, 32), (64123, 33, 32), (30000, 64, 32), (5000, 64, 64),
                                   (999, 33, 33), (4, 5, 7), (200000, 32, 64), (1500, 3, 1)])
def test_tc_linear_vs_fp64(M, K, N):
    from deepviewagg_b200 import ops
    gen = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=gen).cuda().requires_grad_(True)
    w = (torch.randn(N, K, generator=gen) / math.sqrt(K)).cuda().requires_grad_(True)
    g = torch.randn(M, N, generator=gen).cuda()
    ref = x.double() @ w.double().t()
    ref_gx = g.double() @ w.double()
    ref_gw = g.double().t() @ x.double()
    # 3xTF32 on the tensor cores: ~1e-6 of the result's max at K <= 128, growing with the length of the
    # fp32 accumulation (K for y / grad_x, the M rows for grad_w); cuBLAS' own fp32 SIMT GEMM is 4e-7 .. 2e-6
    tol_k = 2e-6 if K <= 128 else 6e-6
    tol_m = 2e-6 * max(1.0, math.sqrt(M / 4096.0))
    for mode, tol in (("fp32", tol_k), ("tf32", 2e-3)):
        ops.set_gemm_precision(mode)
        try:
            y = ops.linear(x, w)
            gx, gw = torch.autograd.grad((y * g).sum(), [x, w])
        finally:
            ops.set_gemm_precision("fp32")
        close(y, ref, tol, f"linear {mode}")
        close(gx, ref_gx, tol, f"linear grad_x {mode}")
        close(gw, ref_gw, max(tol, tol_m), f"linear grad_w {mode}")
    # widths that are not a multiple of 4 are zero-padded onto the same kernels (no library GEMM)
    x2 = torch.randn(100, 130, generator=gen).cuda()
    w2 = torch.randn(66, 130, generator=gen).cuda()
    close(ops.linear(x2, w2).double(), x2.double() @ w2.double().t(), 3e-6, "padded widths")


# ------------------------------------------------------------------------------------------------
# one narrow MLP layer as a single autograd node (fused backward: dz on chip, dX and dW from one tile) vs fp64 torch
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N,need_dx", [(5000, 32, 32, True), (70001, 8, 32, False), (30000, 64, 32, True),
                                           (777, 12, 16, True), (33, 32, 32, True), (100000, 32, 32, True),
                                           (15, 64, 32, True), (4099, 16, 32, False), (2000, 32, 8, True)])
def test_mlp_layer_fused_backward_vs_fp64(M, K, N, need_dx):
    from deepviewagg_b200 import ops, _lib
    assert _lib.load().dva_mlp_layer_bwd_supported(M, N, K)
    gen = torch.Generator().manual_seed(M + K + N)
    x0 = torch.randn(M, K, generator=gen) * 1.5 + 0.3
    w0 = torch.randn(N, K, generator=gen) / math.sqrt(K)
    g = torch.randn(M, N, generator=gen).cuda()
    bn_a = torch.nn.BatchNorm1d(N, momentum=0.1).double().cuda()
    bn_b = torch.nn.BatchNorm1d(N, momentum=0.1).cuda()
    with torch.no_grad():
        bn_b.weight.copy_(torch.rand(N, generator=gen) + 0.5)
        bn_b.bias.copy_(torch.randn(N, generator=gen) * 0.3)
        bn_a.weight.copy_(bn_b.weight.double()), bn_a.bias.copy_(bn_b.bias.double())
    xa = x0.double().cuda().requires_grad_(need_dx)
    wa = w0.double().cuda().requires_grad_(True)
    xb = x0.cuda().requires_grad_(need_dx)
    wb = w0.cuda().requires_grad_(True)
    ya = torch.nn.functional.leaky_relu(bn_a(xa @ wa.t()), 0.2)
    if not _lib.load().dva_linear_bnstats_supported(M, N, K):
        pytest.skip("the forward of this shape takes the unfused route")
    old_max_k = ops._MLP_LAYER_FUSED["max_k"]
    ops._MLP_LAYER_FUSED["max_k"] = 64            # the routing prefers the unfused chain above K = 32; test the kernel anyway
    try:
        yb = ops.linear_bn_act(xb, wb, bn_b, negative_slope=0.2)
    finally:
        ops._MLP_LAYER_FUSED["max_k"] = old_max_k
    assert type(yb.grad_fn).__name__.startswith("_MLPLayer"), type(yb.grad_fn).__name__
    # the unfused chain on the same inputs: same forward kernels, hence the same LeakyReLU slope decisions
    bn_c = torch.nn.BatchNorm1d(N, momentum=0.1).cuda()
    bn_c.load_state_dict({k: v.float() for k, v in bn_a.state_dict().items()})
    with torch.no_grad():
        bn_c.running_mean.zero_(), bn_c.running_var.fill_(1.0), bn_c.num_batches_tracked.zero_()
    xc = x0.cuda().requires_grad_(need_dx)
    wc = w0.cuda().requires_grad_(True)
    ops._MLP_LAYER_FUSED["on"] = False
    try:
        yc = ops.linear_bn_act(xc, wc, bn_c, negative_slope=0.2)
    finally:
        ops._MLP_LAYER_FUSED["on"] = True
    gc = torch.autograd.grad((yc * g).sum(), ([xc] if need_dx else []) + [wc, bn_c.weight, bn_c.bias])
    ins_a = ([xa] if need_dx else []) + [wa, bn_a.weight, bn_a.bias]
    ins_b = ([xb] if need_dx else []) + [wb, bn_b.weight, bn_b.bias]
    ga = torch.autograd.grad((ya * g.double()).sum(), ins_a)
    gb = torch.autograd.grad((yb * g).sum(), ins_b)
    close(yb, ya, 2e-5, "mlp layer y")
    names = (["dx"] if need_dx else []) + ["dw", "dgamma", "dbeta"]
    assert torch.equal(yb, yc)
    for n, a, c, b in zip(names, gb, gc, ga):
        scale = max(1.0, float(b.abs().max()))
        # fused vs unfused: same slope decisions, different fp32 summation orders only
        assert float((a - c).abs().max()) <= 2e-5 * scale * max(1.0, math.sqrt(M / 4096.0)), \
            (n, float((a - c).abs().max()), scale)
        # vs fp64: an activation within rounding of the LeakyReLU kink may take the other slope -- isolated elements
        # of dx, and O(|dA| |x|) per flipped element in the sums over the rows (dw, dgamma, dbeta)
        bad = (a.double() - b).abs() > 5e-5 * scale
        if n == "dx":
            assert int(bad.sum()) <= 4 + a.numel() // 100000, (n, int(bad.sum()))
        else:
            assert float((a.double() - b).abs().max()) <= 1e-3 * scale, (n, float((a.double() - b).abs().max()), scale)
    close(bn_b.running_mean, bn_a.running_mean.float(), 1e-5, "running_mean")
    close(bn_b.running_var, bn_a.running_var.float(), 1e-5, "running_var")
