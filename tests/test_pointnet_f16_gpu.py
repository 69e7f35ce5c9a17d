"""The "f16" precision mode for featnet=pointnet (PointNetVLAD): the fused GEMM + per-cloud column max of the STN layers
(lpd_gemm_f16_colmax), its argument checks, and the whole model against the reference goldens, the CPU oracle and the embedding
driver.  Runs on the B200 box (-m gpu)."""
import numpy as np
import pytest
import torch

from lpdnet_b200 import _lib, evaluate, ops, synth
from lpdnet_b200.util import PointNetVlad as PNV
from oracle import model_numpy

pytestmark = pytest.mark.gpu

DESC_TOL = 1e-4   # strict descriptor gate
TF32_TOL = 2e-4

ACTS = {"none": (ops.ACT_NONE, 0.0), "relu": (ops.ACT_RELU, 0.0), "leaky": (ops.ACT_LEAKY, 0.2)}


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


def problem(M, N, K, seed, affine):
    g = torch.Generator().manual_seed(seed)
    A = torch.randn(M, K, generator=g).half().cuda()
    W = (torch.randn(N, K, generator=g) / K ** 0.5).half().cuda()
    scale = shift = None
    if affine:
        scale = torch.randn(N, generator=g).cuda()                       # both signs
        shift = (0.5 * torch.randn(N, generator=g)).cuda()
        assert (scale < 0).any() and (scale > 0).any()
    return A, W, scale, shift


@pytest.mark.parametrize("affine", [False, True])
@pytest.mark.parametrize("act", ["none", "relu", "leaky"])
@pytest.mark.parametrize("K,N", [(64, 256), (128, 256), (64, 1024), (128, 1024)])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("R", [32, 96, 1024, 4096])
def test_gemm_f16_colmax_equals_colmax_of_the_materialised_product(cuda, R, B, K, N, act, affine):
    """lpd_gemm_f16 (fp32 output: the same single-CTA BN = 256 kernel and per-element epilogue) followed by lpd_colmax gives the
    same bits, because a max is exact; two calls agree.  R = 32 and 96 leave ragged last 128-row tiles."""
    code, slope = ACTS[act]
    M = B * R
    A, W, scale, shift = problem(M, N, K, seed=R + 7 * B + K + N, affine=affine)
    full = ops.gemm_f16(A, W, M=M, N=N, K=K, scale=scale, shift=shift, act=code, slope=slope)
    want = ops.colmax(full, B, R, N)
    ops.profile(True)
    got = ops.gemm_f16_colmax(A, W, M=M, N=N, K=K, R=R, scale=scale, shift=shift, act=code, slope=slope)
    labels = [l for l, _, _ in ops.profile(False)]
    assert labels == [f"lpd_gemm_f16_colmax[{M}x{N}x{K}]"]
    again = ops.gemm_f16_colmax(A, W, M=M, N=N, K=K, R=R, scale=scale, shift=shift, act=code, slope=slope)
    assert got.shape == (B, N)
    assert torch.equal(got, want)
    assert torch.equal(got, again), "the kernel must be deterministic"


@pytest.mark.parametrize("R,B", [(32, 3), (96, 1), (160, 1), (32, 5)])
def test_gemm_f16_colmax_ignores_rows_past_m(cuda, R, B):
    """every true output is negative and act is none, so a zero-filled row past M (0 after the epilogue) would win the max;
    M is not a multiple of 128"""
    M, N, K = B * R, 256, 64
    assert M % 128 != 0
    g = torch.Generator().manual_seed(R * B)
    A = (torch.rand(M, K, generator=g) + 0.1).half().cuda()
    W = (-torch.rand(N, K, generator=g) - 0.1).half().cuda()
    got = ops.gemm_f16_colmax(A, W, M=M, N=N, K=K, R=R, act=ops.ACT_NONE, slope=0.0)
    ref = (A.double() @ W.double().T).view(B, R, N).amax(1)
    assert (ref < 0).all() and (got < 0).all()
    assert torch.equal(got, ops.colmax(ops.gemm_f16(A, W, M=M, N=N, K=K), B, R, N))
    assert torch.allclose(got.double(), ref, rtol=1e-5, atol=0)


def test_gemm_f16_colmax_rejects_unsupported_arguments(cuda):
    """R % 32 != 0, M % R != 0, N % 256 != 0, lda % 8 != 0, a misaligned A and a bad act / slope return LPD_EINVAL and launch
    nothing"""
    lib = _lib.load()
    M, N, K = 192, 256, 64
    A, W, _, _ = problem(M, N, K, seed=5, affine=False)
    wide = torch.zeros(M, K + 4, device="cuda", dtype=torch.float16)
    buf = torch.zeros(M * K + 64, device="cuda", dtype=torch.float16)
    part = torch.full((M // 32, 1024), 7.0, device="cuda")
    out = torch.full((M, 1024), 7.0, device="cuda")

    def call(a, lda, m=M, n=N, R=96, act=ops.ACT_RELU, slope=0.0):
        return lib.lpd_gemm_f16_colmax(a.data_ptr(), lda, W.data_ptr(), K, m, n, K, R, None, None, act, slope, part.data_ptr(),
                                       out.data_ptr(), torch.cuda.current_stream().cuda_stream)

    assert call(A, K, R=48, m=96) == -1                                                     # R % 32 != 0
    assert call(A, K, R=64, m=96) == -1                                                     # M % R != 0
    assert call(A, K, n=128) == -1                                                          # N % 256 != 0
    assert call(wide, K + 4) == -1                                                          # lda % 8 != 0
    assert call(buf[4:], K) == -1                                                           # A not 16-byte aligned
    assert call(A, K, act=ops.ACT_LEAKY, slope=2.0) == -1                                   # slope outside [0, 1]
    assert call(A, K, act=ops.ACT_SIGMOID) == -1
    with pytest.raises(_lib.LpdError):
        ops.gemm_f16_colmax(A, W, M=M, N=N, K=K, R=80, act=ops.ACT_NONE, slope=0.0)
    torch.cuda.synchronize()
    assert (part == 7.0).all() and (out == 7.0).all(), "a rejected call must not launch"
    assert call(A, K) == 0                                                                  # the same arguments, valid
    want = ops.colmax(ops.gemm_f16(A, W, M=M, N=N, K=K, act=ops.ACT_RELU), M // 96, 96, N)
    assert torch.equal(out.view(-1)[: 2 * N].view(2, N), want)


@pytest.mark.parametrize("name,N,ft", [("c1_pointnet_eval", 4096, False), ("c1_pointnet_ft_eval", 1024, True)])
def test_f16_mode_pointnet_matches_reference_golden(cuda, golden, name, N, ft):
    """B = 2 in f16 mode: the fp16 kernels run, no STN conv3 map is materialised, the output is deterministic and inside the strict
    descriptor gate"""
    g = golden(name)
    model, _ = build(g, num_points=N, emb_dims=1024, featnet="pointnet", feature_transform=ft)
    out, again, labels = run_profiled(model, synth.clouds(2, N).cuda(), "f16")
    for want in ("lpd_gemm_f16_colmax[", "lpd_gemm_f16[", "lpd_gemm_f16_tn["):
        assert any(l.startswith(want) for l in labels), (want, labels)
    assert sum(l.startswith("lpd_gemm_f16_colmax[") for l in labels) == (2 if ft else 1), labels
    assert not any(l.startswith("lpd_gemm_tf32[") and l.endswith("x1024x128]") for l in labels), labels
    assert "lpd_colmax" not in labels, labels
    err = np.abs(out - g["out"]).max()
    print(f"\n[f16] {name}: max-abs descriptor error {err:.3e} (|out|max {np.abs(g['out']).max():.3f})")
    assert np.array_equal(out, again), "f16 mode must be deterministic"
    assert err <= DESC_TOL, f"{err:.3e}"


@pytest.mark.parametrize("ft", [False, True])
@pytest.mark.parametrize("B,N", [(3, 2048), (2, 192)])
def test_f16_mode_pointnet_matches_cpu_oracle(cuda, golden, B, N, ft):
    """N = 192: B*N is not a multiple of the 128-row GEMM tile"""
    g = golden("c1_pointnet_ft_eval")
    model, sd = build(g, num_points=N, emb_dims=1024, featnet="pointnet", feature_transform=ft)
    x = synth.clouds(B, N, seed=13)
    out, _, labels = run_profiled(model, x.cuda(), "f16")
    assert any(l.startswith("lpd_gemm_f16_colmax[") for l in labels), labels
    ref = model_numpy.pointnetvlad_forward(sd, x.numpy(), featnet="pointnet", feature_transform=ft)
    err = np.abs(out - ref).max()
    print(f"\n[f16] pointnet B = {B}, N = {N}, feature_transform={ft}: max-abs descriptor error vs the fp32 oracle {err:.3e}")
    assert err <= DESC_TOL, f"{err:.3e}"


@pytest.mark.parametrize("N", [1000, 96, 160])
def test_pointnet_other_shapes_and_other_modes_keep_their_path(cuda, golden, N):
    """B = 2 clouds of N points, N not a multiple of 64 (the fp16 NetVLAD aggregate contracts 64-row blocks of each cloud), in
    f16 mode keep the tf32 path (no fp16 kernel, tf32 error bound); fp32 and tf32 modes run no fp16 kernel"""
    g = golden("c1_pointnet_ft_eval")
    model, sd = build(g, num_points=N, emb_dims=1024, featnet="pointnet", feature_transform=True)
    x = synth.clouds(2, N, seed=14)
    out, _, labels = run_profiled(model, x.cuda(), "f16")
    assert f16_compute_labels(labels) == [], labels
    assert "lpd_colmax" in labels, labels
    err = np.abs(out - model_numpy.pointnetvlad_forward(sd, x.numpy(), featnet="pointnet", feature_transform=True)).max()
    print(f"\n[f16] pointnet B = 2, N = {N} (tf32 path): max-abs descriptor error vs the fp32 oracle {err:.3e}")
    assert err <= TF32_TOL, f"{err:.3e}"
    model, _ = build(g, num_points=1024, emb_dims=1024, featnet="pointnet", feature_transform=True)
    for mode in ("fp32", "tf32"):
        _, _, labels = run_profiled(model, synth.clouds(2, 1024, seed=15).cuda(), mode)
        assert f16_compute_labels(labels) == [], (mode, labels)


def test_f16_mode_pointnet_through_the_embedding_driver(cuda, golden):
    """get_latent_vectors with a pointnet model in f16 mode: the captured-graph replay gives the eager driver's bits"""
    g = golden("c1_pointnet_ft_eval")
    model, _ = build(g, num_points=1024, emb_dims=1024, featnet="pointnet", feature_transform=True)
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
    assert any(l.startswith("lpd_gemm_f16_colmax[") for l in labels), labels
    assert hasattr(model, "_lpd_embed_graph")
    assert got.shape == (10, 256) and np.array_equal(got, eager)
    assert np.array_equal(got[:3], want)
