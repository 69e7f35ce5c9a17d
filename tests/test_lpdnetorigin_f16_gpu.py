"""The "f16" precision mode for featnet=lpdnetorigin (LPDNetOrign, the reference CLI's default feature network): the 64-channel
fp16 double edge layer (lpd_edgeconv_dg64_f16), the C = 64 gather-only max (lpd_edge_gather_max_f16), their argument checks, and
the whole model against the reference golden, the CPU oracle and the embedding driver.  Runs on the B200 box (-m gpu)."""
import numpy as np
import pytest
import torch

from lpdnet_b200 import _lib, evaluate, ops, synth
from lpdnet_b200.util import PointNetVlad as PNV
from oracle import model_numpy

pytestmark = pytest.mark.gpu

F16_TOL = 5e-5    # the featnet=lpdnet f16 gate (tests/test_model_gpu.py)
DESC_TOL = 1e-4   # strict descriptor gate
TF32_TOL = 2e-4


def build(golden_file, **kw):
    shapes = {k: eval(s) for k, s in zip(golden_file["keys"].tolist(), golden_file["shapes"].tolist())}
    sd = synth.fill_state_dict(shapes)
    model = PNV.PointNetVlad(**kw)
    model.load_state_dict(sd, strict=True)
    return model.cuda().eval(), sd


def run_profiled(model, x, mode):
    prev = ops.set_precision(mode)
    try:
        ops.profile(True)
        with torch.no_grad():
            out = model(x).cpu().numpy()
        labels = [l for l, _, _ in ops.profile(False)]
        with torch.no_grad():
            again = model(x).cpu().numpy()
    finally:
        ops.set_precision(prev)
    return out, again, labels


def f16_compute_labels(labels):
    return [l for l in labels if "f16" in l and l != "lpd_f32_to_f16"]    # the weight conversion is not a compute kernel


def problem(B, N, k, seed):
    """fp16 pre-scaled projections p' | q' [B*N, 128], W2 fp16 [64, 64], s2 of both signs, xyz-kNN indices"""
    g = torch.Generator().manual_seed(seed)
    pq = torch.randn(B * N, 128, generator=g).half().cuda()
    w2 = (torch.randn(64, 64, generator=g) / 8).half().cuda()
    s2 = torch.randn(64, generator=g).cuda()
    t2 = (0.5 * torch.randn(64, generator=g)).cuda()
    assert (s2 < 0).any() and (s2 > 0).any()
    idx = ops.knn(synth.clouds(B, N, seed=seed)[:, 0].contiguous().cuda(), k)
    return pq, w2, s2, t2, idx


def reference(pq, w2, s2, t2, idx, B, N, k, act, slope):
    """y1 = fp16(act(p'_j + q'_i)) in fp16 arithmetic (as the kernel forms it), then z = y1 W2^T, BN, act, max over k in float64"""
    P, Q = pq[:, :64].view(B, N, 64), pq[:, 64:].view(B, N, 64)
    Pj = P[torch.arange(B, device="cuda")[:, None, None], idx.long()]                  # [B, N, k, 64]
    z1 = Pj + Q[:, :, None, :]
    y1 = torch.maximum(z1, z1 * torch.tensor(slope, dtype=torch.float16, device="cuda"))
    z = y1.double() @ w2.double().T
    v = s2.double() * z + t2.double()
    v = torch.where(v > 0, v, v * slope)
    return v.amax(2).reshape(B * N, 64)


@pytest.mark.parametrize("act", ["leaky", "relu"])
@pytest.mark.parametrize("B,N", [(1, 64), (3, 64), (1, 1000), (3, 1000), (1, 4096), (3, 4096)])
@pytest.mark.parametrize("k", [20, 32])
def test_edgeconv_dg64_f16_matches_materialised_reference(cuda, k, B, N, act):
    """within one fp16 ulp of the float64 reference rounded to fp16 (or, next to zero where an ulp is finer than fp32 accumulation
    order, 2^-16 of the layer's output scale); two calls give the same bits.  N = 1000 leaves a ragged last tile."""
    code, slope = (ops.ACT_LEAKY, 0.01) if act == "leaky" else (ops.ACT_RELU, 0.0)
    pq, w2, s2, t2, idx = problem(B, N, k, seed=B * 100 + N + k)
    ref = reference(pq, w2, s2, t2, idx, B, N, k, act, slope)
    ld2 = 72                                                                            # strided output: columns 64..71 untouched
    out = torch.full((B * N, ld2), 7.0, device="cuda", dtype=torch.float16)
    ops.profile(True)
    ops.edgeconv_dg64_f16(pq, 128, pq[:, 64:], 128, idx, B, N, w2, s2, t2, code, slope, out, ld2)
    labels = [l for l, _, _ in ops.profile(False)]
    assert labels == ["lpd_edgeconv_dg_f16[64x64]"]
    again = torch.zeros_like(out)
    ops.edgeconv_dg64_f16(pq, 128, pq[:, 64:], 128, idx, B, N, w2, s2, t2, code, slope, again, ld2)
    assert torch.equal(out[:, :64], again[:, :64]), "the kernel must be deterministic"
    assert (out[:, 64:] == 7.0).all()
    got = out[:, :64].double().cpu().numpy()
    ref16 = ref.half().double().cpu().numpy()
    ulp = np.spacing(np.abs(ref16).astype(np.float16)).astype(np.float64)
    tol = np.maximum(ulp, 2.0 ** -16 * np.abs(ref16).max())
    err = np.abs(got - ref16)
    assert (err <= tol).all(), f"max err {err.max():.3e}, worst excess {(err - tol).max():.3e}"


@pytest.mark.parametrize("B,N,k,ld", [(2, 300, 20, 64), (1, 1000, 32, 64), (3, 64, 7, 128), (1, 257, 1, 64), (2, 4096, 20, 64)])
def test_edge_gather_max_f16_c64_is_exact(cuda, B, N, k, ld):
    """C = 64, q = None, ACT_NONE: out[i] = max_m g[j(i,m)], bit-identical to torch gather + amax (a max of fp16 values is exact)"""
    gen = torch.Generator().manual_seed(N + k)
    g = torch.randn(B * N, ld, generator=gen).half().cuda()
    idx = torch.randint(0, N, (B, N, k), generator=gen, dtype=torch.int32).cuda()
    want = g[:, :64].view(B, N, 64)[torch.arange(B, device="cuda")[:, None, None], idx.long()].amax(2).reshape(B * N, 64)
    out = torch.zeros(B * N, 72, device="cuda", dtype=torch.float16)
    ops.edge_gather_max_f16(g, ld, None, 0, idx, B, N, k, 64, ops.ACT_NONE, 0.0, out, 72)
    assert torch.equal(out[:, :64], want)
    assert (out[:, 64:] == 0).all()


def test_f16_entry_points_reject_unsupported_arguments(cuda):
    """k other than 20 / 32, a leading dimension that breaks the 16-byte row alignment, and a gather width other than 64 / 256
    return LPD_EINVAL (the wrapper raises LpdError) and launch nothing"""
    lib = _lib.load()
    B, N = 1, 256
    pq, w2, s2, t2, idx = problem(B, N, 20, seed=3)
    out = torch.full((B * N, 64), 7.0, device="cuda", dtype=torch.float16)
    _, _, _, _, idx16 = problem(B, N, 16, seed=3)

    def dg(p, ldp, q, ldq, ix, k, ld2=64):
        return lib.lpd_edgeconv_dg64_f16(p.data_ptr(), ldp, q.data_ptr(), ldq, ix.data_ptr(), B, N, k, w2.data_ptr(), s2.data_ptr(),
                                         t2.data_ptr(), ops.ACT_LEAKY, 0.01, out.data_ptr(), ld2, torch.cuda.current_stream().cuda_stream)

    wide = torch.zeros(B * N, 136, device="cuda", dtype=torch.float16)
    for k in (16, 1, 33, 24):
        assert dg(pq, 128, pq[:, 64:], 128, idx16, k) == -1, k
    assert dg(wide, 132, wide[:, 64:], 136, idx, 20) == -1                                  # ldp % 8 != 0
    assert dg(wide, 136, wide[:, 64:], 132, idx, 20) == -1                                  # ldq % 8 != 0
    assert dg(pq, 128, pq[:, 64:], 128, idx, 20, ld2=65) == -1                              # odd ld2
    assert dg(pq, 128, pq[:, 4:], 128, idx, 20) == -1                                       # q not 16-byte aligned
    with pytest.raises(_lib.LpdError):
        ops.edgeconv_dg64_f16(pq, 128, pq[:, 64:], 128, idx16, B, N, w2, s2, t2, ops.ACT_LEAKY, 0.01, out, 64)
    g = torch.zeros(B * N, 256, device="cuda", dtype=torch.float16)
    for C in (128, 32, 512):
        with pytest.raises(_lib.LpdError):
            ops.edge_gather_max_f16(g, 256, None, 0, idx, B, N, 20, C, ops.ACT_NONE, 0.0, out, 256)
    with pytest.raises(_lib.LpdError):
        ops.edge_gather_max_f16(g, 100, None, 0, idx, B, N, 20, 64, ops.ACT_NONE, 0.0, out, 64)   # ldp % 8 != 0
    torch.cuda.synchronize()
    assert (out == 7.0).all(), "a rejected call must not launch"


def test_f16_mode_lpdnetorigin_matches_reference_golden(cuda, golden):
    """c2_lpdnetorigin_eval (B = 2, N = 4096) in f16 mode: the fp16 kernels run, the error is inside the lpdnet f16 gate, and the
    output is deterministic"""
    g = golden("c2_lpdnetorigin_eval")
    model, _ = build(g, num_points=4096, emb_dims=1024, featnet="lpdnetorigin")
    out, again, labels = run_profiled(model, synth.clouds(2, 4096).cuda(), "f16")
    for want in ("lpd_edgeconv_dg_f16[64x64]", "lpd_gemm_f16[", "lpd_edge_gather_ext[C=64]", "lpd_gemm_f16_tn["):
        assert any(l.startswith(want) for l in labels), (want, labels)
    assert not any(l.startswith("lpd_edgeconv_dg_tf32") for l in labels), labels
    err = np.abs(out - g["out"]).max()
    print(f"\n[f16] c2_lpdnetorigin_eval: max-abs descriptor error {err:.3e} (|out|max {np.abs(g['out']).max():.3f})")
    assert np.array_equal(out, again), "f16 mode must be deterministic"
    assert err <= F16_TOL, f"{err:.3e}"


def test_f16_mode_lpdnetorigin_k32_matches_cpu_oracle(cuda, golden):
    g = golden("c2_lpdnetorigin_eval")
    model, sd = build(g, num_points=2048, emb_dims=1024, featnet="lpdnetorigin")
    model.emb_nn.k = 32
    x = synth.clouds(1, 2048, seed=11)
    out, _, labels = run_profiled(model, x.cuda(), "f16")
    assert any(l.startswith("lpd_edgeconv_dg_f16[64x64]") for l in labels), labels
    ref = model_numpy.pointnetvlad_forward(sd, x.numpy(), featnet="lpdnetorigin", k=32)
    err = np.abs(out - ref).max()
    print(f"\n[f16] lpdnetorigin k = 32, N = 2048: max-abs descriptor error vs the fp32 oracle {err:.3e}")
    assert err <= DESC_TOL, f"{err:.3e}"


def test_lpdnetorigin_other_k_and_other_modes_keep_their_path(cuda, golden):
    """k = 16 in f16 mode keeps the tf32 path (no fp16 kernel, tf32 error bound); fp32 and tf32 modes run no fp16 kernel"""
    g = golden("c2_lpdnetorigin_eval")
    model, sd = build(g, num_points=2048, emb_dims=1024, featnet="lpdnetorigin")
    x = synth.clouds(1, 2048, seed=12)
    model.emb_nn.k = 16
    out, _, labels = run_profiled(model, x.cuda(), "f16")
    assert f16_compute_labels(labels) == [], labels
    assert any(l.startswith("lpd_edgeconv_dg_tf32[64x64]") for l in labels), labels
    err = np.abs(out - model_numpy.pointnetvlad_forward(sd, x.numpy(), featnet="lpdnetorigin", k=16)).max()
    print(f"\n[f16] lpdnetorigin k = 16 (tf32 path): max-abs descriptor error vs the fp32 oracle {err:.3e}")
    assert err <= TF32_TOL, f"{err:.3e}"
    model.emb_nn.k = 20
    for mode in ("fp32", "tf32"):
        _, _, labels = run_profiled(model, x.cuda(), mode)
        assert f16_compute_labels(labels) == [], (mode, labels)


def test_f16_mode_lpdnetorigin_through_the_embedding_driver(cuda, golden):
    """get_latent_vectors with an lpdnetorigin model in f16 mode: the captured-graph replay gives the eager driver's bits"""
    g = golden("c2_lpdnetorigin_eval")
    model, _ = build(g, num_points=1024, emb_dims=1024, featnet="lpdnetorigin")
    x = synth.clouds(10, 1024, seed=6)[:, 0].numpy()                          # the driver captures a graph for >= 3 full batches
    prev = ops.set_precision("f16")
    try:
        ops.profile(True)
        with torch.no_grad():
            want = model(torch.from_numpy(x[:3, None]).cuda()).cpu().numpy()
        labels = [l for l, _, _ in ops.profile(False)]
        got = evaluate.get_latent_vectors(model, x, batch_num=3)                 # 3 graph replays + eager tail of 1
        eager = evaluate.get_latent_vectors(model, x, batch_num=3, use_graph=False)
    finally:
        ops.set_precision(prev)
    assert any(l.startswith("lpd_edgeconv_dg_f16[64x64]") for l in labels), labels
    assert hasattr(model, "_lpd_embed_graph")
    assert got.shape == (10, 256) and np.array_equal(got, eager)
    assert np.array_equal(got[:3], want)
