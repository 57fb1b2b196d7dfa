"""Oracle parity AT THE SIZE of the BASELINE.json configs (VERDICT r1: the largest oracle-checked case
was 60 000 points x 3 views; the 1 M test is property-only).

  config #1  S3DIS step: 4 x 40 k-point spheres = 160 000 points, ragged views (mean 8, 15 % unseen),
             C = 64, fp32 and bf16 storage
  config #3  KITTI-360 cylinder per GPU: 80 000 points, ragged views (mean 20), C = 128

Both the fused operator (ops.view_attention: forward, attentions, every gradient) and the whole
GroupBimodalCSRPool module (DeepSetFeat map encoder, E_mod, E_score, gating; forward + gradients of
inputs and of every parameter, train-mode BatchNorm over all rows) are compared with the CPU oracle
(oracle/pooling_oracle.py, pinned on reference-executed fixtures; run in fp64 for the module) on the same
seeded inputs.
Tolerance: 1e-4 relative (north_star) for fp32; storage precision for bf16, stated below."""
import pytest
import torch

from oracle import pooling_oracle as O
from test_gpu_parity import TOL, _run_va, close, ragged_ptr

pytestmark = pytest.mark.gpu

CONFIGS = {"config1_s3dis": dict(N=160_000, mean_v=8, C=64), "config3_kitti360": dict(N=80_000, mean_v=20, C=128)}


@pytest.fixture(params=["auto", "stream", "ring", "lane"])
def path(request):
    """Kernel pair of the fused view attention (dva_view_attention_set_path): 'auto' = the library's per-shape
    choice, 'stream' = streaming kernels for both passes, 'ring' = ring forward + lane-per-view backward, 'lane' =
    streaming forward + lane-per-view backward; 'auto' is restored afterwards."""
    from deepviewagg_b200 import _lib
    lib = _lib.load()
    assert lib.dva_view_attention_set_path({"auto": 0, "stream": 1, "ring": 2, "lane": 3}[request.param]) == 0
    yield request.param
    assert lib.dva_view_attention_set_path(0) == 0


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_view_attention_at_config_size_fp32(cfg, path):
    c = CONFIGS[cfg]
    _run_va(c["N"], c["mean_v"], c["C"], 4, seed=101, use_idx=torch.int32)          # rows through a permutation
    _run_va(c["N"], c["mean_v"], c["C"], 4, seed=102)                                # rows in place


def test_view_attention_config2_bf16_storage(path):
    """config #2 (config #1's shape, bf16 I/O, fp32 accumulate): storage-precision parity, tolerance
    1.6e-2 relative to the tensor's max (2 bf16 ulps), reported separately from the fp32 bar."""
    c = CONFIGS["config1_s3dis"]
    _run_va(c["N"], c["mean_v"], c["C"], 4, seed=103, dtype=torch.bfloat16, tol=1.6e-2, use_idx=torch.int32)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_group_pool_module_at_config_size(cfg):
    from deepviewagg_b200.modules.multimodal.pooling import GroupBimodalCSRPool
    c = CONFIGS[cfg]
    N, C, G = c["N"], c["C"], 4
    gen = torch.Generator().manual_seed(7 + N)
    ptr = ragged_ptr(gen, N, c["mean_v"])
    V = int(ptr[-1])
    torch.manual_seed(11)
    m = GroupBimodalCSRPool(in_map=8, in_mod=C, num_groups=G, use_mod=False, gating=True, group_scaling=True,
                            map_encoder="DeepSetFeat", use_num=True)
    with torch.no_grad():                                   # non-trivial BN affine / gate parameters
        for n_, p in m.named_parameters():
            if "batch_norm" in n_ or n_.startswith("G."):
                p.add_(torch.randn(p.shape, generator=gen) * 0.2)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    x_mod = torch.randn(V, C, generator=gen).relu()         # post-ReLU CNN features: exact-zero ties
    x_map = torch.rand(V, 8, generator=gen)
    w = torch.randn(N, C, generator=gen)

    # oracle (CPU, fp64, on the same fp32 inputs): parameters as leaves.  torch's fp32 CPU batch_norm is off by
    # ~1.6e-5 relative over a million rows (its mean and var alone are good to 1e-7); that alone puts hundreds of
    # rows of an fp32 oracle's x_mod gradient past the bound below, so in fp64 the comparison measures the kernels.
    sd64 = {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd64.items() if v.is_floating_point() and "running" not in k}
    sd_o = {**sd64, **leaves}
    xo, mo = x_mod.double().requires_grad_(True), x_map.double().requires_grad_(True)
    ref = O.group_pool(sd_o, xo, mo, ptr, G, use_mod=False, gating_on=True, group_scaling=True,
                       map_encoder_name="DeepSetFeat", training=True, use_num=True)
    names = list(leaves)
    ref_g = torch.autograd.grad((ref["out"] * w.double()).sum(), [xo, mo] + [leaves[k] for k in names], allow_unused=True)

    m = m.cuda().train()
    xg, mg = x_mod.cuda().requires_grad_(True), x_map.cuda().requires_grad_(True)
    out = m(None, xg, mg, ptr.cuda())
    params = dict(m.named_parameters())
    got_g = torch.autograd.grad((out * w.cuda()).sum(), [xg, mg] + [params[k] for k in names], allow_unused=True)
    torch.cuda.synchronize()
    close(out, ref["out"], TOL, f"{cfg} out")
    empty = (ptr[1:] == ptr[:-1])
    assert (out[empty.cuda()] == 0).all()                   # unseen points: exact zeros
    # Gradients: LeakyReLU has a kink at 0.  Among the ~1e8 pre-activations of this size a handful land
    # within float rounding of 0 (|a| ~ 1e-7), where two correct implementations may take either slope
    # (1 or 0.2); each such element perturbs ONE row of the input gradients and adds an O(1) term to the
    # parameter sums.  So: input gradients must agree to 2e-4 on all but <= 5e-5 of the rows (and on every
    # row of a point without such an element), parameter gradients to 5e-3 in relative L2 norm (2e-2 of their max
    # element-wise).
    for n_, a, b in zip(["x_mod", "x_map"] + names, got_g, ref_g):
        b = torch.zeros_like(leaves[n_]) if b is None and n_ in leaves else b
        a = torch.zeros_like(b) if a is None else a.cpu()
        scale = max(1.0, float(b.abs().max()))
        if n_ in ("x_mod", "x_map"):
            # x_map additionally flows through DeepSetFeat's segment MAX (pooling.py:628): two views of a point
            # whose encoded features agree to the last bits may swap the arg-max (5e6 such decisions here)
            bad = ((a - b).abs() > 2e-4 * scale).any(dim=1)
            frac = 5e-5 if n_ == "x_mod" else 1e-3
            assert int(bad.sum()) <= max(8, int(frac * a.shape[0])), (cfg, n_, int(bad.sum()), a.shape[0])
        else:
            rel_l2 = float((a - b).norm() / b.norm().clamp(min=1e-12))
            assert rel_l2 <= 5e-3 and (a - b).abs().max() <= 2e-2 * scale, (cfg, n_, rel_l2, float((a - b).abs().max()), scale)
