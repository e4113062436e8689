"""Per-kernel numerics on the B200: every CUDA kernel (called through the C ABI) against a plain PyTorch fp32
reference of the same op on the same fp16-rounded inputs.

Tolerance.  Outputs are fp16 with fp32 accumulation.  Two bounds are asserted per kernel:
  * max-norm (SURVEY §7 "Numerics"): max|err| <= 3e-3 * max|ref| + 1e-3;
  * the north-star's literal elementwise tolerance against the fp32 result: |out - ref| <= 1e-4 + 1e-3 |ref|
    (rtol 1e-3 / atol 1e-4).  One fp16 ulp is 9.8e-4 relative at worst, so an output that is the correctly rounded
    fp32 result passes, and so does a one-ulp rounding flip; the fraction of elements outside the tolerance is
    printed and bounded by NS_MAX_VIOL (default 0: none) — kernels whose arithmetic is not a single fp32-accumulated
    contraction pass their own measured bound explicitly (ns_max=...), with the reason at the call site.
"""
import math
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"


NS_RTOL, NS_ATOL = 1e-3, 1e-4
NS_MAX_VIOL = float(os.environ.get("TC_NS_MAX_VIOL", "0"))   # survey runs set 1 to collect the fractions
NS_LOG = os.environ.get("TC_NS_LOG")          # optional: append "what<TAB>violating fraction<TAB>max err" lines


def _close(out, ref, what, rel=3e-3, abs_=1e-3, ns_max=None):
    out = out.float()
    ref = ref.float()
    assert out.shape == ref.shape, f"{what}: shape {out.shape} vs {ref.shape}"
    assert torch.isfinite(out).all(), f"{what}: non-finite output"
    diff = (out - ref).abs()
    err = diff.max().item()
    bound = rel * ref.abs().max().item() + abs_
    viol = (diff > NS_ATOL + NS_RTOL * ref.abs()).float().mean().item()
    print(f"{what}: max err {err:.3e} (bound {bound:.3e}); outside rtol 1e-3/atol 1e-4: {100 * viol:.4f} %")
    if NS_LOG:
        with open(NS_LOG, "a") as f:
            f.write(f"{what}\t{viol:.3e}\t{err:.3e}\n")
    assert err <= bound, f"{what}: max err {err:.4e} > bound {bound:.4e} (ref max {ref.abs().max().item():.3e})"
    lim = NS_MAX_VIOL if ns_max is None else ns_max
    assert viol <= lim, f"{what}: {100 * viol:.4f} % of the outputs outside rtol 1e-3 / atol 1e-4 (allowed {100 * lim:.4f} %)"
    return err


def _viol_frac(out, ref):
    out, ref = out.float(), ref.float()
    return ((out - ref).abs() > NS_ATOL + NS_RTOL * ref.abs()).float().mean().item()


def _autocast_ln_linear(x16, ln, w, b, geglu, n_half):
    """Yardstick for the LayerNorm-folded GEMM: what the reference computes under torch.autocast — LayerNorm in fp32
    rounded to fp16, then an fp16 Linear (fp32 accumulation) rounded to fp16, then GEGLU on fp16 values."""
    n16 = F.layer_norm(x16.float(), (x16.shape[1],), ln.weight, ln.bias, ln.eps).half()
    h = (F.linear(n16.float(), w.half().float(), b)).half().float()
    return (h[:, :n_half] * F.gelu(h[:, n_half:])).half() if geglu else h.half()


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _pack_conv_w(w):
    """[Cout, Cin, KH, KW] -> [Cout, KH*KW*Cin] (tap-major, channel-minor), fp16."""
    co, ci, kh, kw = w.shape
    return w.permute(0, 2, 3, 1).reshape(co, kh * kw * ci).contiguous().half()


@pytest.fixture(scope="module")
def ops():
    from tooncrafter_b200 import ops as _ops
    torch.backends.cuda.matmul.allow_tf32 = False     # the torch references below must be true fp32
    torch.backends.cudnn.allow_tf32 = False
    # first cuDNN/cuBLAS use on a fresh box pages in ~1 GB of libraries: do it outside the per-test timeouts
    F.conv2d(torch.zeros(1, 8, 8, 8, device=DEV), torch.zeros(8, 8, 3, 3, device=DEV), padding=1)
    F.conv3d(torch.zeros(1, 8, 4, 8, 8, device=DEV), torch.zeros(8, 8, 3, 1, 1, device=DEV), padding=(1, 0, 0))
    (torch.zeros(8, 8, device=DEV) @ torch.zeros(8, 8, device=DEV)).sum().item()
    torch.cuda.synchronize()
    return _ops


@pytest.mark.parametrize("rows,K,N", [(300, 320, 320), (4096, 1280, 1280), (128, 64, 16), (2560, 640, 160),
                                       (77, 1024, 640), (1000, 512, 4)])
def test_linear_bias_residual(ops, rows, K, N):
    x = _rand(rows, K, seed=1).half()
    w = _rand(N, K, scale=K ** -0.5, seed=2).half()
    bias = _rand(N, seed=3).float()
    ld = (N + 7) // 8 * 8                      # row strides must be multiples of 8 halfs (16-byte stores)
    res = _rand(rows, ld, seed=4).half()
    out = torch.zeros(rows, ld, dtype=torch.float16, device=DEV)
    ops.linear(x, w, out, rows=rows, K=K, n_cols=N, bias=bias, res=res, ldc=ld, ldr=ld)
    ref = x.float() @ w.float().t() + bias + res[:, :N].float()
    _close(out[:, :N], ref, f"linear {rows}x{K}x{N}")
    assert (out[:, N:] == 0).all()


@pytest.mark.parametrize("K,N,res", [(320, 320, True), (320, 960, False), (640, 640, True)])
def test_linear_skinny_weight_resident(ops, K, N, res):
    """M >> N with a short K loop: enough M tiles per SM that tc_conv_gemm keeps the weight N-tile resident in shared
    memory (reloaded only when the N tile changes) and adds the residual through the tensor core."""
    rows = 81920 if K == 320 else 61440
    x = _rand(rows, K, seed=71).half()
    w = _rand(N, K, scale=K ** -0.5, seed=72).half()
    bias = _rand(N, seed=73).float()
    r = _rand(rows, N, seed=74).half() if res else None
    out = torch.zeros(rows, N, dtype=torch.float16, device=DEV)
    ops.linear(x, w, out, rows=rows, K=K, n_cols=N, bias=bias, res=r)
    ref = x.float() @ w.float().t() + bias
    if res:
        ref = ref + r.float()
    _close(out, ref, f"skinny linear {rows}x{K}x{N}")


def test_linear_strided_slices(ops):
    """A read from / output written into channel slices of wider tensors (concat-by-construction)."""
    rows, K, N = 640, 128, 192
    xw = _rand(rows, 256, seed=5).half()
    w = _rand(N, K, scale=K ** -0.5, seed=6).half()
    outw = torch.full((rows, 512), 7.0, dtype=torch.float16, device=DEV)
    ops.linear(xw, w, outw, rows=rows, K=K, n_cols=N, ldx=256, ldc=512, a_offset=128, out_offset=64)
    ref = xw[:, 128:256].float() @ w.float().t()
    _close(outw[:, 64:64 + N], ref, "linear slices")
    assert (outw[:, :64] == 7.0).all() and (outw[:, 64 + N:] == 7.0).all(), "wrote outside the slice"


def test_linear_geglu(ops):
    rows, K, inner = 1000, 320, 1280
    x = _rand(rows, K, seed=7).half()
    w = _rand(2 * inner, K, scale=K ** -0.5, seed=8).half()   # reference layout: [a ; gate]
    b = _rand(2 * inner, seed=9).float()
    BN = 256
    hb = BN // 2
    # pack per N tile: [a rows of tile | gate rows of tile]
    wa, wg = w[:inner], w[inner:]
    ba, bg = b[:inner], b[inner:]
    wp = torch.cat([torch.cat([wa[i:i + hb], wg[i:i + hb]]) for i in range(0, inner, hb)]).contiguous()
    bp = torch.cat([torch.cat([ba[i:i + hb], bg[i:i + hb]]) for i in range(0, inner, hb)]).contiguous()
    out = torch.zeros(rows, inner, dtype=torch.float16, device=DEV)
    ops.linear(x, wp, out, rows=rows, K=K, n_cols=2 * inner, bias=bp, geglu=True, block_n=BN)
    h = x.float() @ w.float().t() + b
    ref = h[:, :inner] * F.gelu(h[:, inner:])
    _close(out, ref, "geglu")


@pytest.mark.parametrize("rows,C,N,geglu", [(1000, 320, 960, False), (300, 640, 640, False), (2560, 320, 2560, True)])
def test_linear_with_folded_layernorm(ops, rows, C, N, geglu):
    """tc_row_stats + GEMM epilogue  ==  Linear(LayerNorm(x))  (attention.py:243-245 with norm folded into the GEMM)."""
    from tooncrafter_b200 import engine
    x = (_rand(rows, C, seed=55) * 3 + 0.7).half()
    ln = torch.nn.LayerNorm(C).to(DEV)
    with torch.no_grad():
        ln.weight.copy_(_rand(C, seed=56) * 0.2 + 1.0)
        ln.bias.copy_(_rand(C, seed=57) * 0.2)
    w = _rand(N, C, scale=C ** -0.5, seed=58)
    b = _rand(N, seed=59)
    perm = engine.geglu_perm(N).to(DEV) if geglu else None
    f = engine.fold_layernorm(w, b, ln, torch.device(DEV), perm=perm)
    stats = torch.zeros(rows, 2, device=DEV)
    ops.row_stats(x, stats, rows=rows, C=C)
    ref_mean = x.float().mean(1)
    assert (stats[:, 0] - ref_mean).abs().max().item() < 1e-4
    out = torch.zeros(rows, N // 2 if geglu else N, dtype=torch.float16, device=DEV)
    ops.linear(x, f.w, out, rows=rows, K=C, n_cols=N, bias=f.c, ln_stats=stats, ln_u=f.u, geglu=geglu,
               block_n=256 if geglu else 0)
    h = F.linear(F.layer_norm(x.float(), (C,), ln.weight, ln.bias, 1e-5), w, b)
    ref = h[:, :N // 2] * F.gelu(h[:, N // 2:]) if geglu else h
    # not a single contraction (fp16-rounded W*gamma, rstd * (acc - mean * u)): held to the reference's own autocast
    # arithmetic (fp16 LayerNorm output, fp16 weights) as the yardstick for the north-star fraction
    v16 = _viol_frac(_autocast_ln_linear(x, ln, w, b, geglu, N // 2), ref)
    _close(out, ref, f"linear with folded LayerNorm (autocast path: {100 * v16:.3f} % outside)", rel=4e-3, abs_=2e-3,
           ns_max=1.5 * v16 + 0.005)


@pytest.mark.parametrize("rows,C,bn,N2,geglu", [(4196, 320, 160, 960, False), (1000, 640, 160, 640, False),
                                                 (3000, 1280, 256, 2560, True), (70000, 320, 160, 320, False)])
def test_row_stats_from_producer_epilogue(ops, rows, C, bn, N2, geglu):
    """The GEMM that writes an activation also writes per-row {sum, sumsq} partials of its fp16 outputs; the consuming
    LayerNorm-folded GEMM finishes them in its epilogue  ==  Linear(LayerNorm(Linear(x) + res))."""
    from tooncrafter_b200 import engine
    x0 = _rand(rows, C, seed=81).half()
    w0 = _rand(C, C, scale=C ** -0.5, seed=82).half()
    b0 = _rand(C, seed=83).float()
    res = (_rand(rows, C, seed=84) * 2 + 0.5).half()
    slots = -(-C // bn)
    mid = torch.zeros(rows, C, dtype=torch.float16, device=DEV)
    part = torch.full((rows, slots, 2), float("nan"), device=DEV)
    ops.linear(x0, w0, mid, rows=rows, K=C, n_cols=C, bias=b0, res=res, block_n=bn, row_stats=part, row_stats_slots=slots)
    _close(mid, x0.float() @ w0.float().t() + b0 + res.float(), "producer output")
    tot = part.sum(1)
    m32 = mid.float()
    assert (tot[:, 0] - m32.sum(1)).abs().max().item() <= 2e-3 * m32.abs().sum(1).max().item() / 10 + 1e-3
    assert ((tot[:, 1] - (m32 * m32).sum(1)).abs() / (m32 * m32).sum(1)).max().item() < 1e-5
    ln = torch.nn.LayerNorm(C).to(DEV)
    with torch.no_grad():
        ln.weight.copy_(_rand(C, seed=85) * 0.2 + 1.0)
        ln.bias.copy_(_rand(C, seed=86) * 0.2)
    w = _rand(N2, C, scale=C ** -0.5, seed=87)
    b = _rand(N2, seed=88)
    f = engine.fold_layernorm(w, b, ln, torch.device(DEV), perm=engine.geglu_perm(N2).to(DEV) if geglu else None)
    out = torch.zeros(rows, N2 // 2 if geglu else N2, dtype=torch.float16, device=DEV)
    ops.linear(mid, f.w, out, rows=rows, K=C, n_cols=N2, bias=f.c, ln_stats=part, ln_u=f.u, ln_nslots=slots, ln_eps=1e-5,
               geglu=geglu, block_n=256 if geglu else 0)
    h = F.linear(F.layer_norm(m32, (C,), ln.weight, ln.bias, 1e-5), w, b)
    ref = h[:, :N2 // 2] * F.gelu(h[:, N2 // 2:]) if geglu else h
    v16 = _viol_frac(_autocast_ln_linear(mid, ln, w, b, geglu, N2 // 2), ref)
    _close(out, ref, f"consumer of producer-side row statistics (autocast path: {100 * v16:.3f} % outside)", rel=4e-3,
           abs_=2e-3, ns_max=1.5 * v16 + 0.005)


@pytest.mark.parametrize("N,H,W,Cin,Cout", [(4, 20, 32, 128, 192), (6, 5, 8, 256, 320), (2, 40, 64, 64, 320),
                                             (3, 10, 16, 320, 4), (1, 16, 256, 128, 128)])
def test_conv3x3(ops, N, H, W, Cin, Cout):
    x = _rand(N, H, W, Cin, seed=11).half()            # channels-last
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=12)
    bias = _rand(Cout, seed=13).float()
    ld = (Cout + 7) // 8 * 8
    out = torch.zeros(N, H, W, ld, dtype=torch.float16, device=DEV)
    ops.conv_gemm(x, (N, H, W, Cin), (H * W * Cin, W * Cin, Cin), _pack_conv_w(w), ops.TAPS_3x3, out, (N, H, W),
                  Cout, bias=bias, ldc=ld)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.half().float(), bias, padding=1).permute(0, 2, 3, 1)
    _close(out[..., :Cout], ref, f"conv3x3 {N}x{H}x{W} {Cin}->{Cout}")


def test_conv3x3_emb_bias_and_skip(ops):
    """ResBlock-style epilogue: + per-sample embedding vector (bias2) + residual."""
    B, T, H, W, C = 2, 4, 10, 16, 128
    N = B * T
    x = _rand(N, H, W, C, seed=14).half()
    w = _rand(C, C, 3, 3, scale=(9 * C) ** -0.5, seed=15)
    bias = _rand(C, seed=16).float()
    emb = _rand(B, C, seed=17).half()
    res = _rand(N, H, W, C, seed=18).half()
    out = torch.zeros(N, H, W, C, dtype=torch.float16, device=DEV)
    ops.conv_gemm(x, (N, H, W, C), (H * W * C, W * C, C), _pack_conv_w(w), ops.TAPS_3x3, out, (N, H, W), C,
                  bias=bias, bias2=emb, bias2_rows_per=T * H * W, res=res)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.half().float(), bias, padding=1).permute(0, 2, 3, 1)
    ref = ref + emb.float().repeat_interleave(T, 0)[:, None, None, :] + res.float()
    _close(out, ref, "conv3x3 + emb + skip")


@pytest.mark.parametrize("N,H,W,Cin,Cout,res", [(32, 5, 8, 1280, 1280, True), (32, 10, 16, 640, 640, False),
                                                 (8, 5, 8, 2560, 1280, False), (3, 10, 16, 512, 96, True)])
def test_conv3x3_split_k(ops, N, H, W, Cin, Cout, res):
    """Few output tiles and a long K loop (the 1280- and 640-channel UNet levels): the launch splits K over otherwise idle
    SMs; slices park fp32 partial tiles and the last one to finish sums them in slice order — the result must be
    deterministic, identical run to run, and leave the ticket words ready for the next launch."""
    x = _rand(N, H, W, Cin, seed=41).half()
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=42)
    bias = _rand(Cout, seed=43).float()
    emb = _rand(N, Cout, seed=44).half()
    r = _rand(N, H, W, Cout, seed=45).half() if res else None
    wp = _pack_conv_w(w)
    outs = []
    for rep in range(3):
        out = torch.zeros(N, H, W, Cout, dtype=torch.float16, device=DEV)
        ops.conv_gemm(x, (N, H, W, Cin), (H * W * Cin, W * Cin, Cin), wp, ops.TAPS_3x3, out, (N, H, W), Cout,
                      bias=bias, bias2=emb, bias2_rows_per=H * W, res=r)
        cfg = ops.last_gemm_config()
        outs.append(out)
        if rep == 0:
            # another geometry in between: must find zeroed tickets and leave them zeroed
            y = torch.zeros(1280, 640, dtype=torch.float16, device=DEV)
            xa = _rand(1280, 10240, seed=46).half()
            wa = _rand(640, 10240, scale=10240 ** -0.5, seed=47).half()
            ops.linear(xa, wa, y, rows=1280, K=10240, n_cols=640)
            cfg_lin = ops.last_gemm_config()
            _close(y, xa.float() @ wa.float().t(), f"split-K linear 1280x10240x640 {cfg_lin}")
    print("conv launch config:", cfg)
    assert cfg["ksplit"] > 1 and cfg_lin["ksplit"] > 1, f"expected split-K launches: {cfg} {cfg_lin}"
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "split-K result differs run to run"
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.half().float(), bias, padding=1).permute(0, 2, 3, 1)
    ref = ref + emb.float()[:, None, None, :]
    if res:
        ref = ref + r.float()
    _close(outs[0], ref, f"split-K conv3x3 {N}x{H}x{W} {Cin}->{Cout} ksplit={cfg['ksplit']}")


@pytest.mark.parametrize("B,T,H,W,C", [(2, 16, 5, 8, 128), (1, 16, 20, 32, 64), (1, 14, 10, 16, 128)])
def test_temporal_conv(ops, B, T, H, W, C):
    """(3,1,1) Conv3d == 3-tap conv over T on the [B][T][HW][C] view."""
    x = _rand(B, T, H * W, C, seed=21).half()
    w = _rand(C, C, 3, 1, 1, scale=(3 * C) ** -0.5, seed=22)
    bias = _rand(C, seed=23).float()
    res = _rand(B, T, H * W, C, seed=24).half()
    out = torch.zeros_like(x)
    wp = w[:, :, :, 0, 0].permute(0, 2, 1).reshape(C, 3 * C).contiguous().half()
    ops.conv_gemm(x, (B, T, H * W, C), (T * H * W * C, H * W * C, C), wp, ops.TAPS_T3, out, (B, T, H * W), C,
                  bias=bias, res=res, acc_scale=0.5)
    xr = x.float().reshape(B, T, H, W, C).permute(0, 4, 1, 2, 3)
    ref = F.conv3d(xr, w.half().float(), bias, padding=(1, 0, 0)).permute(0, 2, 3, 4, 1).reshape(B, T, H * W, C)
    ref = ref * 0.5 + res.float()
    _close(out, ref, "temporal conv")


def test_conv3x3_stride2(ops):
    N, H, W, C, Cout = 4, 20, 32, 64, 128
    x = _rand(N, H, W, C, seed=31).half()
    w = _rand(Cout, C, 3, 3, scale=(9 * C) ** -0.5, seed=32)
    bias = _rand(Cout, seed=33).float()
    ph = torch.zeros(4, N, H // 2, W // 2, C, dtype=torch.float16, device=DEV)
    ops.phase_split2(x, ph, N=N, H=H, W=W, C_=C)
    out = torch.zeros(N, H // 2, W // 2, Cout, dtype=torch.float16, device=DEV)
    H2, W2 = H // 2, W // 2
    ops.conv_gemm(ph, (4 * N, H2, W2, C), (H2 * W2 * C, W2 * C, C), _pack_conv_w(w), ops.taps_3x3_stride2(N), out,
                  (N, H2, W2), Cout, bias=bias)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), w.half().float(), bias, stride=2, padding=1).permute(0, 2, 3, 1)
    _close(out, ref, "conv3x3 stride 2")


@pytest.mark.parametrize("frames,fps,hw,C,silu,eps", [(8, 1, 160, 320, True, 1e-5), (8, 4, 40, 1280, True, 1e-5),
                                                      (4, 1, 2560, 640, False, 1e-6), (16, 16, 640, 128, True, 1e-5),
                                                      (2, 1, 20480, 256, True, 1e-6), (4, 2, 64, 1920, True, 1e-5),
                                                      # the UNet's shapes: group sizes 10 / 20 / 30 / 40 / 80 channels, ragged pixel counts
                                                      (32, 16, 40, 1280, True, 1e-5), (32, 1, 160, 1280, True, 1e-5),
                                                      (32, 16, 160, 1280, False, 1e-5), (8, 1, 2560, 320, True, 1e-5),
                                                      (16, 1, 640, 640, True, 1e-5), (6, 1, 333, 960, True, 1e-5),
                                                      (4, 2, 77, 2560, True, 1e-5), (16, 1, 2560, 512, True, 1e-6)])
def test_groupnorm(ops, frames, fps, hw, C, silu, eps):
    x = (_rand(frames, hw, C, seed=41) * 1.5 + 0.3).half()
    gamma = (_rand(C, seed=42) * 0.2 + 1.0).float()
    beta = (_rand(C, seed=43) * 0.2).float()
    y = torch.zeros_like(x)
    ops.groupnorm(x, y, gamma, beta, frames=frames, frames_per_stat=fps, hw=hw, C=C, eps=eps, silu=silu)
    xr = x.float().reshape(frames // fps, fps * hw, C).permute(0, 2, 1)   # (n_stat, C, L)
    ref = F.group_norm(xr, 32, gamma, beta, eps)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1).reshape(frames, hw, C)
    _close(y, ref, "groupnorm")


@pytest.mark.parametrize("frames,fps,hw,C", [
    (1, 1, 1021, 1280),      # single-pass kernel, one CTA per (statistics group, norm group), ragged vector count
    (2, 1, 1501, 1280),      # cluster of 2 CTAs per unit
    (1, 1, 5003, 1280),      # cluster of 5
    (1, 1, 6000, 1280),      # cluster of 6 (15.4 MB: the largest tensor the single-pass path takes)
    (4, 2, 333, 2560),       # 80-channel groups (ten 16-byte vectors per pixel)
    (64, 1, 40, 512),        # many small units (2048 of them): fuller threads, small blocks
    (2, 2, 1280, 256),       # 8-channel groups: one vector per pixel
])
def test_groupnorm_single_pass_cluster_shapes(ops, frames, fps, hw, C):
    """Shapes that reach gn_fused_kernel with different cluster sizes (partial sums through distributed shared memory,
    added in rank order): against torch, in place as well, and identical run to run."""
    x = (_rand(frames, hw, C, seed=141) * 1.5 + 0.3).half()
    gamma = (_rand(C, seed=142) * 0.2 + 1.0).float()
    beta = (_rand(C, seed=143) * 0.2).float()
    outs = []
    for rep in range(2):
        y = torch.zeros_like(x)
        ops.groupnorm(x, y, gamma, beta, frames=frames, frames_per_stat=fps, hw=hw, C=C, silu=True)
        outs.append(y)
    z = x.clone()
    ops.groupnorm(z, z, gamma, beta, frames=frames, frames_per_stat=fps, hw=hw, C=C, silu=True)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], z), "single-pass GroupNorm differs run to run / in place"
    xr = x.float().reshape(frames // fps, fps * hw, C).permute(0, 2, 1)
    ref = F.silu(F.group_norm(xr, 32, gamma, beta, 1e-5)).permute(0, 2, 1).reshape(frames, hw, C)
    _close(outs[0], ref, f"single-pass groupnorm {frames}x{fps}x{hw}x{C}")


@pytest.mark.parametrize("frames,fps,hw,C,slice_ld,inplace", [
    (32, 16, 2560, 320, 0, False),      # 52 MB, per-clip statistics
    (32, 1, 2560, 320, 0, True),        # per-frame statistics, in place
    (32, 16, 640, 640, 0, False),
    (32, 1, 640, 640, 0, False),
    (32, 16, 160, 1280, 2560, False),   # reads a channel slice of a wider tensor
    (32, 16, 40, 1280, 0, True),
    (3, 1, 7, 128, 0, False), (300, 1, 64, 64, 0, False),   # tiny rows / more stat groups than SMs
])
def test_groupnorm_full_size(ops, frames, fps, hw, C, slice_ld, inplace):
    """GroupNorm + SiLU at the sizes the benchmark runs (both guidance branches of a 16-frame clip): strided input, in
    place, repeated launches, results identical run to run (the cross-CTA reductions have a fixed order)."""
    ldx = slice_ld or C
    xw = (_rand(frames, hw, ldx, seed=51) * 1.5 + 0.3).half()
    off = ldx - C
    gamma = (_rand(C, seed=52) * 0.2 + 1.0).float()
    beta = (_rand(C, seed=53) * 0.2).float()
    xin = xw[..., off:].float()
    outs = []
    for rep in range(3):
        if inplace:
            y = xw.clone()
            ops.groupnorm(y, y, gamma, beta, frames=frames, frames_per_stat=fps, hw=hw, C=C, silu=True, ldx=ldx, ldy=ldx,
                          x_offset=off, y_offset=off)
            outs.append(y[..., off:].clone())
        else:
            y = torch.zeros(frames, hw, C, dtype=torch.float16, device=DEV)
            ops.groupnorm(xw, y, gamma, beta, frames=frames, frames_per_stat=fps, hw=hw, C=C, silu=True, ldx=ldx, x_offset=off)
            outs.append(y)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "GroupNorm differs run to run"
    xr = xin.reshape(frames // fps, fps * hw, C).permute(0, 2, 1)
    ref = F.silu(F.group_norm(xr, 32, gamma, beta, 1e-5)).permute(0, 2, 1).reshape(frames, hw, C)
    _close(outs[0], ref, f"groupnorm {frames}/{fps} x {hw} x {C}")


def test_gelu2d(ops):
    """Exact-erf GELU on a strided matrix, in place (Resampler feed-forward, resampler.py:27-34)."""
    rows, cols, ld = 300, 1024, 1280
    buf = (_rand(rows, ld, seed=91) * 3).half()
    ref = F.gelu(buf[:, :cols].float())
    keep = buf[:, cols:].clone()
    ops.gelu2d(buf, buf, rows=rows, cols=cols, ldx=ld, ldy=ld)
    _close(buf[:, :cols], ref, "gelu2d")
    assert torch.equal(buf[:, cols:], keep), "wrote outside the column range"


@pytest.mark.parametrize("rows,C", [(1000, 320), (333, 640), (77, 1280), (64, 512)])
def test_layernorm(ops, rows, C):
    x = (_rand(rows, C, seed=51) * 2 + 0.5).half()
    gamma = (_rand(C, seed=52) * 0.2 + 1.0).float()
    beta = (_rand(C, seed=53) * 0.2).float()
    y = torch.zeros_like(x)
    ops.layernorm(x, y, gamma, beta, rows=rows, C=C)
    ref = F.layer_norm(x.float(), (C,), gamma, beta, 1e-5)
    _close(y, ref, "layernorm")


def _sdpa_ref(q, k, v, heads):
    """q [B, Lq, h*64], k/v [B, Lk, h*64] fp16 -> fp32 attention output [B, Lq, h*64]."""
    B, Lq, _ = q.shape
    qh = q.float().reshape(B, Lq, heads, 64).transpose(1, 2)
    kh = k.float().reshape(B, -1, heads, 64).transpose(1, 2)
    vh = v.float().reshape(B, -1, heads, 64).transpose(1, 2)
    s = (qh @ kh.transpose(-1, -2)) * 64 ** -0.5
    o = s.softmax(-1) @ vh
    return o.transpose(1, 2).reshape(B, Lq, heads * 64)


@pytest.mark.parametrize("B,L,heads", [(2, 300, 2), (3, 128, 1), (2, 2560, 5), (4, 40, 3), (1, 640, 10)])
def test_attention_self(ops, B, L, heads):
    C = heads * 64
    q = _rand(B, L, C, seed=61).half()
    k = _rand(B, L, C, seed=62).half()
    v = _rand(B, L, C, seed=63).half()
    out = torch.zeros_like(q)
    ops.attention(q, [dict(k=k, v=v, ldk=C, ldv=C, Lk=L)], out, q_batches=B, Lq=L, heads=heads, scale=64 ** -0.5,
                  ldq=C, ldo=C)
    # P is rounded to fp16 for the PV product (as the reference's autocast bmm does); with few keys (L = 40) the
    # rounding is averaged less: measured <= 0.033 % of the outputs outside the literal tolerance
    _close(out, _sdpa_ref(q, k, v, heads), f"self attention L={L}", ns_max=1e-3)


@pytest.mark.parametrize("single", ["0", "1"])
@pytest.mark.parametrize("B,L,Lk,heads", [(2, 300, 300, 2), (1, 640, 640, 3), (2, 257, 1100, 1)])
def test_attention_both_cta_modes(ops, monkeypatch, single, B, L, Lk, heads):
    """tc_attn3_kernel with two query tiles per CTA (one CTA per SM) and with one tile per CTA (two CTAs per SM): the
    dispatch picks by key count, TC_ATTN_SINGLE forces either — both must agree with the fp32 reference at every shape."""
    monkeypatch.setenv("TC_ATTN_SINGLE", single)
    C = heads * 64
    q = _rand(B, L, C, seed=161).half()
    k = _rand(B, Lk, C, seed=162).half()
    v = _rand(B, Lk, C, seed=163).half()
    out = torch.zeros_like(q)
    ops.attention(q, [dict(k=k, v=v, ldk=C, ldv=C, Lk=Lk)], out, q_batches=B, Lq=L, heads=heads, scale=64 ** -0.5,
                  ldq=C, ldo=C)
    _close(out, _sdpa_ref(q, k, v, heads), f"attention L={L} Lk={Lk} single={single}", ns_max=1e-3)


def test_attention_fused_qkv_layout(ops):
    """q/k/v as column slices of one [tokens][3C] projection output."""
    B, L, heads = 2, 200, 2
    C = heads * 64
    qkv = _rand(B, L, 3 * C, seed=64).half()
    out = torch.zeros(B, L, C, dtype=torch.float16, device=DEV)
    ops.attention(qkv, [dict(k=qkv, v=qkv, ldk=3 * C, ldv=3 * C, Lk=L, k_offset=C, v_offset=2 * C)], out,
                  q_batches=B, Lq=L, heads=heads, scale=64 ** -0.5, ldq=3 * C, ldo=C)
    ref = _sdpa_ref(qkv[..., :C].contiguous(), qkv[..., C:2 * C].contiguous(), qkv[..., 2 * C:].contiguous(), heads)
    _close(out, ref, "attention on fused qkv", ns_max=1e-3)


def test_attention_cross_text_plus_image(ops):
    """Two-segment cross attention: text K/V shared by the T frames of a sample, image K/V per frame."""
    Bs, T, L, heads = 2, 4, 160, 5
    C = heads * 64
    N = Bs * T
    q = _rand(N, L, C, seed=65).half()
    kt = _rand(Bs, 77, C, seed=66).half()
    vt = _rand(Bs, 77, C, seed=67).half()
    ki = _rand(N, 16, C, seed=68).half()
    vi = _rand(N, 16, C, seed=69).half()
    out = torch.zeros_like(q)
    ops.attention(q, [dict(k=kt, v=vt, ldk=C, ldv=C, Lk=77, kv_div=T), dict(k=ki, v=vi, ldk=C, ldv=C, Lk=16)], out,
                  q_batches=N, Lq=L, heads=heads, scale=64 ** -0.5, ldq=C, ldo=C)
    ref = _sdpa_ref(q, kt.repeat_interleave(T, 0), vt.repeat_interleave(T, 0), heads) + _sdpa_ref(q, ki, vi, heads)
    # the resident-K/V kernel splits the normalised P into fp16 hi + lo parts, so only the output rounding is left
    _close(out, ref, "cross attention text+image", ns_max=1e-3)


@pytest.mark.parametrize("Bs,T,L,heads,n_txt,n_img", [(2, 16, 2560, 5, 77, 16), (1, 3, 333, 2, 77, 16), (2, 2, 128, 1, 64, 32),
                                                       (1, 4, 640, 10, 77, 0)])
def test_attention_cross_resident_kv_shapes(ops, Bs, T, L, heads, n_txt, n_img):
    """The short-K/V cross-attention kernel at the UNet level-0 shape and with ragged query tiles; with one segment
    (n_img = 0) the dispatch runs tc_attn3_kernel instead."""
    C = heads * 64
    N = Bs * T
    q = _rand(N, L, C, seed=171).half()
    kt, vt = _rand(Bs, n_txt, C, seed=172).half(), _rand(Bs, n_txt, C, seed=173).half()
    segs = [dict(k=kt, v=vt, ldk=C, ldv=C, Lk=n_txt, kv_div=T)]
    ref = _sdpa_ref(q, kt.repeat_interleave(T, 0), vt.repeat_interleave(T, 0), heads)
    if n_img:
        ki, vi = _rand(N, n_img, C, seed=174).half(), _rand(N, n_img, C, seed=175).half()
        segs.append(dict(k=ki, v=vi, ldk=C, ldv=C, Lk=n_img))
        ref = ref + _sdpa_ref(q, ki, vi, heads)
    out = torch.zeros_like(q)
    ops.attention(q, segs, out, q_batches=N, Lq=L, heads=heads, scale=64 ** -0.5, ldq=C, ldo=C)
    _close(out, ref, f"cross attention resident kv L={L} {n_txt}+{n_img}", ns_max=1e-3)


def test_attention_long_kv(ops):
    """VAE dual-reference style: Lq != Lk, all query batches share kv batch 0."""
    N, Lq, Lk, heads = 3, 512, 1100, 2
    C = heads * 64
    q = _rand(N, Lq, C, seed=70).half()
    k = _rand(1, Lk, C, seed=71).half()
    v = _rand(1, Lk, C, seed=72).half()
    out = torch.zeros_like(q)
    ops.attention(q, [dict(k=k, v=v, ldk=C, ldv=C, Lk=Lk, kv_div=N)], out, q_batches=N, Lq=Lq, heads=heads,
                  scale=64 ** -0.5, ldq=C, ldo=C)
    _close(out, _sdpa_ref(q, k.expand(N, -1, -1), v.expand(N, -1, -1), heads), "attention long kv")


@pytest.mark.parametrize("B,T,P,heads", [(2, 16, 40, 5), (1, 16, 640, 10), (1, 14, 33, 2), (1, 20, 10, 1)])
def test_temporal_attention(ops, B, T, P, heads):
    C = heads * 64
    qkv = _rand(B, T, P, 3 * C, seed=81).half()
    out = torch.zeros(B, T, P, C, dtype=torch.float16, device=DEV)
    ops.temporal_attention(qkv, qkv, qkv, out, ld=3 * C, ldo=C, B=B, T=T, P=P, heads=heads, scale=64 ** -0.5,
                           k_offset=C, v_offset=2 * C)
    x = qkv.float().permute(0, 2, 1, 3).reshape(B * P, T, 3 * C)   # (b p) t c
    ref = _sdpa_ref(x[..., :C].half(), x[..., C:2 * C].half(), x[..., 2 * C:].half(), heads)
    ref = ref.reshape(B, P, T, C).permute(0, 2, 1, 3)
    # 14-20 keys per query; P is split into fp16 hi + lo parts for the PV product, so only the output rounding is left
    _close(out, ref, "temporal attention", ns_max=0.002)


@pytest.mark.parametrize("N,L,D", [(2, 2560, 512), (3, 300, 512), (2, 256, 256), (1, 1000, 128), (2, 64, 64), (1, 130, 384)])
def test_attention_wide(ops, N, L, D):
    """VAE mid-block AttnBlock core (autoencoder_dualref.py:186-200): one head of D channels, q/k/v slices of a fused
    qkv tensor; D = 512 (two CTAs per query tile, each half of the value channels) and the single-CTA widths, with ragged
    query / key tiles.  Scores have the spread of the real layer (q, k ~ N(0, 1), scale D^-0.5)."""
    qkv = _rand(N, L, 3 * D, seed=91).half()
    out = torch.zeros(N, L, D, dtype=torch.float16, device=DEV)
    ops.attention_wide(qkv, out, batches=N, L=L, D=D, scale=D ** -0.5, ld=3 * D, ldo=D, q_offset=0, k_offset=D, v_offset=2 * D)
    q, k, v = (qkv[..., i * D:(i + 1) * D].float() for i in range(3))
    ref = ((q @ k.transpose(-1, -2)) * D ** -0.5).softmax(-1) @ v
    # P is rounded to fp16 for the PV product (as the reference's autocast bmm does): same bound as the d = 64 kernels
    _close(out, ref, f"wide attention N={N} L={L} D={D}", ns_max=1e-3)


def test_attention_wide_growing_maximum(ops):
    """Keys whose scores grow along the sequence force the lazy O rescale (and its wait on the previous PV MMA)."""
    N, L, D = 2, 1024, 512
    qkv = _rand(N, L, 3 * D, seed=92)
    qkv[..., D:2 * D] *= torch.linspace(0.2, 3.0, L, device=DEV)[None, :, None]
    qkv = qkv.half()
    out = torch.zeros(N, L, D, dtype=torch.float16, device=DEV)
    ops.attention_wide(qkv, out, batches=N, L=L, D=D, scale=D ** -0.5, ld=3 * D, ldo=D, q_offset=0, k_offset=D, v_offset=2 * D)
    q, k, v = (qkv[..., i * D:(i + 1) * D].float() for i in range(3))
    ref = ((q @ k.transpose(-1, -2)) * D ** -0.5).softmax(-1) @ v
    _close(out, ref, "wide attention, growing row maximum", ns_max=2e-3)


def test_softmax_rows(ops):
    s = _rand(300, 2560, scale=3.0, seed=85).half()
    ref = (s.float() * 0.125).softmax(-1)
    ops.softmax_rows(s, rows=300, cols=2560, scale=0.125)
    _close(s, ref, "softmax rows", rel=2e-3, abs_=1e-5)


def test_ncthw_to_cl_wide_channels(ops):
    """Tiled transpose used for the decoder's reference feature maps (C % 64 == 0): ragged pixel count, channel slice."""
    B, Cc, T, H, W, Cpad, coff = 2, 128, 3, 7, 9, 256, 64
    x = _rand(B, Cc, T, H, W, seed=131)
    y = torch.zeros(B, T, H, W, Cpad, dtype=torch.float16, device=DEV)
    ops.ncthw_to_cl(x, y, B=B, C_=Cc, T=T, H=H, W=W, Cpad=Cpad, coff=coff, scale=0.25)
    ref = (x * 0.25).permute(0, 2, 3, 4, 1).half()
    assert torch.equal(y[..., coff:coff + Cc], ref), "tiled ncthw_to_cl differs from the reference layout change"
    assert (y[..., :coff] == 0).all() and (y[..., coff + Cc:] == 0).all(), "channels outside the slice were touched"


def test_layout_and_elementwise(ops):
    B, Cc, T, H, W = 2, 4, 3, 6, 8
    x = _rand(B, Cc, T, H, W, seed=91)
    y = torch.zeros(B, T, H, W, 64, dtype=torch.float16, device=DEV)
    ops.ncthw_to_cl(x, y, B=B, C_=Cc, T=T, H=H, W=W, Cpad=64, coff=4, scale=0.5)
    ref = (x * 0.5).permute(0, 2, 3, 4, 1)
    _close(y[..., 4:8], ref, "ncthw_to_cl")
    assert (y[..., :4] == 0).all() and (y[..., 8:] == 0).all()
    back = torch.zeros(B, Cc, T, H, W, dtype=torch.float32, device=DEV)
    ops.cl_to_ncthw(y, back, B=B, C_=Cc, T=T, H=H, W=W, ldx=64, x_offset=4)
    _close(back, (x * 0.5).half().float(), "cl_to_ncthw", rel=0, abs_=0)

    a = _rand(3, 5, 7, 64, seed=92).half()
    up = torch.zeros(3, 10, 14, 64, dtype=torch.float16, device=DEV)
    ops.upsample2x(a, up, N=3, H=5, W=7, C_=64)
    ref = F.interpolate(a.float().permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1)
    _close(up, ref, "upsample2x", rel=0, abs_=0)

    src = _rand(100, 128, seed=93).half()
    dst = torch.zeros(100, 256, dtype=torch.float16, device=DEV)
    ops.copy2d(src, dst, rows=100, cols=128, lds=128, ldd=256, dst_offset=64)
    assert torch.equal(dst[:, 64:192], src) and (dst[:, :64] == 0).all()
    ops.add2d(src, dst, rows=100, cols=128, ldx=128, ldy=256, y_offset=64)
    _close(dst[:, 64:192], 2 * src.float(), "add2d", rel=1e-3, abs_=0)


def test_time_embed_and_small_linear(ops):
    B, dim, hidden = 2, 320, 1280
    t = torch.tensor([999.0, 19.0], device=DEV)
    w1 = _rand(hidden, dim, scale=dim ** -0.5, seed=101).half()
    b1 = _rand(hidden, seed=102).float()
    w2 = _rand(hidden, hidden, scale=hidden ** -0.5, seed=103).half()
    b2 = _rand(hidden, seed=104).float()
    out = torch.zeros(B, hidden, device=DEV)
    ws = torch.zeros(B * (dim + hidden), device=DEV)
    ops.time_embed(t, w1, b1, w2, b2, out, ws, dim=dim, hidden=hidden, accumulate=False)
    half = dim // 2
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device=DEV) / half)
    args = t[:, None] * freqs[None]
    emb = torch.cat([torch.cos(args), torch.sin(args)], -1)
    ref = F.linear(F.silu(F.linear(emb, w1.float(), b1)), w2.float(), b2)
    _close(out, ref, "time_embed", rel=1e-3, abs_=1e-3)
    ops.time_embed(t, w1, b1, w2, b2, out, ws, dim=dim, hidden=hidden, accumulate=True)
    _close(out, 2 * ref, "time_embed accumulate", rel=1e-3, abs_=2e-3)

    J = 2240
    w = _rand(J, hidden, scale=hidden ** -0.5, seed=105).half()
    b = _rand(J, seed=106).float()
    y = torch.zeros(B, J, dtype=torch.float16, device=DEV)
    ops.small_linear(ref.contiguous(), w, b, y, silu_in=True)
    _close(y, F.linear(F.silu(ref), w.float(), b), "small_linear")


def _ddim_ref(e_c, e_uc, x, noise, coef):
    s, phi, sqrt_ac, sqrt_1mac, rescale, sqrt_aprev, dir_coef, sigma = coef
    v = e_uc + s * (e_c - e_uc)                                   # fp16 tensor arithmetic, as ddim.py:226
    if phi > 0:
        dims = list(range(1, v.ndim))
        std_text = e_c.std(dim=dims, keepdim=True)
        std_cfg = v.std(dim=dims, keepdim=True)
        v = phi * (v * (std_text / std_cfg)) + (1 - phi) * v
    v = v.float()      # the reference multiplies by fp32 schedule tensors (ddpm3d.py:240-252): fp16 v promotes to fp32
    eps = sqrt_ac * v + sqrt_1mac * x
    x0 = (sqrt_ac * x - sqrt_1mac * v) * rescale
    return sqrt_aprev * x0 + dir_coef * eps + sigma * noise, x0


@pytest.mark.parametrize("phi", [0.7, 0.0])
def test_ddim_step(ops, phi):
    B, shape = 2, (4, 16, 40, 64)
    n = 4 * 16 * 40 * 64
    e_c = _rand(B, *shape, seed=111).half()
    e_uc = (e_c.float() + 0.3 * _rand(B, *shape, seed=112)).half()
    x = _rand(B, *shape, seed=113)
    noise = _rand(B, *shape, seed=114)
    coef_l = [7.5, phi, 0.6, 0.8, 0.98, 0.7, 0.3, 0.5]
    coef = torch.tensor(coef_l, device=DEV)
    x_prev = torch.zeros_like(x)
    x0 = torch.zeros_like(x)
    ws = torch.zeros(4 * B * 64, dtype=torch.float64, device=DEV)
    ops.ddim_step(e_c, e_uc, x, noise, x_prev, x0, coef, ws, B=B, n=n)
    ref_prev, ref_x0 = _ddim_ref(e_c, e_uc, x, noise, coef_l)
    # the CFG mix is the same fp16 op sequence in both; with guidance rescale the two may round std_text / std_cfg to
    # neighbouring fp16 values (fp64 vs fp32 accumulation of the 655k-element variance): one ulp of the factor moves
    # every v by <= 2^-11 |v| (|v| ~ 8 here), so the literal tolerance is only demanded without the rescale
    ns = 0.0 if phi == 0.0 else 0.10
    _close(x0, ref_x0, f"ddim pred_x0 phi={phi}", rel=2e-3, abs_=2e-3, ns_max=ns)
    _close(x_prev, ref_prev, f"ddim x_prev phi={phi}", rel=2e-3, abs_=2e-3, ns_max=ns)
