"""Attention kernels under sharp and growing scores, against a float64 reference of the same operation.

The kernel tests in test_kernels_gpu.py draw q, k ~ N(0, 1) at scale 1/8: scores of unit spread, whose row maximum
never grows by 2^8 after the first 128-key block, so the lazy O rescale of tc_attn3_kernel and tc_attn_wide_kernel
(the only place the softmax warps read, scale and write back the PV accumulator between MMAs) is never taken there.
This file feeds the attention kernels score distributions where an online softmax goes wrong:

  ramp        k scaled by linspace(0.5, 2.0) along the keys, q x {1, 4, 12}: the row maximum grows along the sequence;
  sharp       q x 25: near-argmax rows;
  staircase   scores built per block: one channel per head carries a per-block offset (q = A there, k = d_block), the
              other channels are small noise, so every block's maximum climbs by exactly delta log2 units
              (8.5: O is rescaled at every block; 7.5: at every second block, with P up to ~2^7.5 in fp16 in between);
  descending  the maximum sits in block 0, later P underflow to fp16 subnormals or 0 (no rescale may happen);
  tail        the maximum sits in the ragged last block (Lk = 128 n + 5): the rescale meets the -inf masking.

The CPU tests check that each generator produces the coverage it claims (a later edit to a generator must not
silently bring the suite back to rows that never rescale); every GPU test asserts its own input's coverage again
before it calls the kernel.  Outputs are also written into wider buffers pre-filled with a sentinel, and nothing
outside the output slice may change.
"""
import math
import re

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda"
LOG2E = 1.4426950408889634
SCALE = 64 ** -0.5
BLOCK = 128                 # key block of the tcgen05 kernels
THR = 8.0                   # kRescaleThreshold of tc_attn3.cu / tc_attn_wide.cu (log2 units)
NS_RTOL, NS_ATOL = 1e-3, 1e-4
FLASH_NS = 1e-3             # P rounded to fp16 before the PV product (test_kernels_gpu.py: attention tests)
XS_NS = 1e-3                # resident-K/V cross attention, P = fp16 hi + lo (test_kernels_gpu.py)
TEMPORAL_NS = 0.002         # temporal attention, P = fp16 hi + lo (test_kernels_gpu.py)
SENTINEL = 1234.0           # exact in fp16
NOISE = 0.2                 # std of the non-offset channels of staircase data: score noise ~0.04 nats, far below the
                            # 0.5 log2-unit margin between the staircase steps and the rescale threshold

# name -> (kind, parameter): q multiplier for ramp / sharp, per-block step (log2 units) for the staircases
DATA = {
    "ramp1": ("ramp", 1.0), "ramp4": ("ramp", 4.0), "ramp12": ("ramp", 12.0), "sharp": ("sharp", 25.0),
    "stair8.5": ("stair", 8.5), "stair7.5": ("stair", 7.5), "descending": ("stair", -4.0), "tail": ("tail", 12.0),
}


# ----------------------------------------------------------------------------------------------------- data
def _offsets(kind, x, Lk, device):
    """Per-key score offset in log2 units."""
    blk = (torch.arange(Lk, device=device) // BLOCK).double()
    if kind == "stair":
        return blk * x
    return torch.where(blk == blk[-1], x, 0.0)          # tail: only the last (ragged) block is lifted


def _gen(data, Bq, Lq, Bk, Lk, heads, *, D=64, scale=SCALE, seed=0, device=None):
    """Seeded fp16 q [Bq, Lq, heads*D], k / v [Bk, Lk, heads*D] with the score distribution `data`."""
    kind, x = DATA[data]
    device = device or DEV
    g = torch.Generator(device=device).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=device)
    C = heads * D
    if kind == "ramp":
        q = rn(Bq, Lq, C) * x
        k = rn(Bk, Lk, C) * torch.linspace(0.5, 2.0, Lk, device=device)[:, None]
    elif kind == "sharp":
        q = rn(Bq, Lq, C) * x
        k = rn(Bk, Lk, C)
    else:
        A = 8.0
        q = rn(Bq, Lq, C) * NOISE
        k = rn(Bk, Lk, C) * NOISE
        q.view(Bq, Lq, heads, D)[..., 0] = A
        k.view(Bk, Lk, heads, D)[..., 0] = (_offsets(kind, x, Lk, device) / (A * scale * LOG2E)).float()[:, None]
    v = rn(Bk, Lk, C)
    return q.half(), k.half(), v.half()


# ----------------------------------------------------------------------------------------------------- references
def _segs(k, v, kv_div):
    if isinstance(k, (list, tuple)):
        return list(zip(k, v, kv_div))
    return [(k, v, kv_div)]


def _scores64(q, k, heads, kv_div=1):
    """Raw scores q.k (unscaled) in float64 from the fp16 inputs, one query batch at a time: (b, [heads, Lq, Lk])."""
    B, Lq, C = q.shape
    D = C // heads
    for b in range(B):
        qh = q[b].double().reshape(Lq, heads, D).transpose(0, 1)
        kh = k[b // kv_div].double().reshape(-1, heads, D).transpose(0, 1)
        yield b, qh @ kh.transpose(1, 2)


def _heads_v(v, b, kv_div, heads):
    return v[b // kv_div].double().reshape(v.shape[1], heads, -1).transpose(0, 1)


def _attn_ref64(q, k, v, heads, scale, kv_div=1):
    """softmax(q k^T * scale) v in float64 from the fp16-rounded inputs; q [B, Lq, C], k / v [B / kv_div, Lk, C].
    k, v and kv_div may be sequences of two segments: the result is then the sum of the two softmax results (text +
    image cross attention, lvdm/modules/attention.py:126-142)."""
    B, Lq, C = q.shape
    out = torch.zeros(B, heads, Lq, C // heads, dtype=torch.float64, device=q.device)
    for ks, vs, div in _segs(k, v, kv_div):
        for b, s in _scores64(q, ks, heads, div):
            out[b] += (s * scale).softmax(-1) @ _heads_v(vs, b, div, heads)
    return out.transpose(1, 2).reshape(B, Lq, C)


def _attn_emulated(q, k, v, heads, scale, kv_div=1, thr=THR):
    """The flash-style kernels' arithmetic: per 128-key block, P = fp16(2^((s - m_use) c)) with the lazy reference
    maximum m_use of tc_attn3.cu:344-367 (thr = 0: the eager rescale of tc_attn_kernel), row sums of the unrounded P,
    O accumulated from the fp16 P and rescaled when m_use moves, fp16 output.  Sums are in float64 here (fp32 in the
    kernels): what this models is the rounding of P and the lazy maximum."""
    B, Lq, C = q.shape
    c = scale * LOG2E
    out = torch.zeros(B, heads, Lq, C // heads, dtype=torch.float64, device=q.device)
    for ks, vs, div in _segs(k, v, kv_div):
        for b, s in _scores64(q, ks, heads, div):
            t = s.float().double() * c                  # fp32 scores, log2 units
            vh = _heads_v(vs, b, div, heads)
            m = torch.full(t.shape[:-1], -math.inf, dtype=torch.float64, device=q.device)
            l = torch.zeros_like(m)
            o = torch.zeros(out.shape[1:], dtype=torch.float64, device=q.device)
            for g0 in range(0, t.shape[-1], BLOCK):
                tb = t[..., g0:g0 + BLOCK]
                m_new = torch.maximum(m, tb.amax(-1))
                m_use = torch.where(m_new - m > thr, m_new, m)
                alpha = torch.exp2(m - m_use)
                p = torch.exp2(tb - m_use[..., None])
                l = l * alpha + p.sum(-1)
                o = o * alpha[..., None] + p.half().double() @ vh[:, g0:g0 + BLOCK]
                m = m_use
            out[b] += o / l[..., None]
    return out.transpose(1, 2).reshape(B, Lq, C).half()


def _lazy_rescales(scores, scale, block=BLOCK, thr=THR):
    """The lazy rescale rule of tc_attn3.cu:344-347 (and tc_attn_wide.cu:275-277) restated in torch.  scores: raw
    q.k [..., Lk].  Per row: the number of key blocks g > 0 at which O is rescaled, i.e. at which the running maximum
    grew by more than 2^thr since the reference maximum m_use was last moved, and the largest P = 2^((s - m_use) c)
    the block exponentials reach (P is rounded to fp16: it must stay far below 65504)."""
    c = scale * LOG2E
    t = scores.double() * c
    m = torch.full(t.shape[:-1], -math.inf, dtype=torch.float64, device=t.device)
    n = torch.zeros(t.shape[:-1], dtype=torch.int64, device=t.device)
    pmax = torch.zeros_like(m)
    for g0 in range(0, t.shape[-1], block):
        bm = t[..., g0:g0 + block].amax(-1)
        m_new = torch.maximum(m, bm)
        grow = m_new - m > thr                           # first block: m = -inf, always grows
        if g0 > 0:
            n += grow
        m = torch.where(grow, m_new, m)
        pmax = torch.maximum(pmax, torch.exp2(bm - m))
    return n, pmax


def _coverage(q, k, heads, scale, kv_div=1):
    """_lazy_rescales over every (query batch, head, row): rescale counts and largest P, flattened."""
    ns, ps = [], []
    for _, s in _scores64(q, k, heads, kv_div):
        n, p = _lazy_rescales(s, scale)
        ns.append(n.flatten())
        ps.append(p.flatten())
    return torch.cat(ns), torch.cat(ps)


def _spread_log2(q, k, heads, scale, kv_div=1):
    """Per row: (max - min) of the scores in log2 units, i.e. how many binades the row's P spans."""
    return torch.cat([((s.amax(-1) - s.amin(-1)) * scale * LOG2E).flatten() for _, s in _scores64(q, k, heads, kv_div)])


def _assert_coverage(data, n, pmax, G):
    """What each generator promises about the lazy rescale of a 128-key-block sweep over G blocks."""
    kind, x = DATA[data]
    if data == "ramp1":
        assert (n > 0).any(), f"{data}: no row rescales O"
    elif kind == "ramp":
        assert (n > 0).double().mean().item() >= 0.9, f"{data}: fewer than 90 % of the rows rescale O"
    elif kind == "sharp":
        assert (n > 0).double().mean().item() >= 0.75, f"{data}: fewer than 75 % of the rows rescale O"
    elif kind == "stair" and x > THR:
        assert (n == G - 1).all(), f"{data}: not every row rescales at every block"
    elif kind == "stair" and x > 0:
        assert (n == (G - 1) // 2).all(), f"{data}: not every row rescales at every second block"
        assert pmax.min().item() > 2 ** 7 and pmax.max().item() < 2 ** 8, f"{data}: P between rescales not in (2^7, 2^8)"
    elif kind == "stair":
        assert (n == 0).all(), f"{data}: a row rescales"
    elif kind == "tail":
        assert (n == 1).all(), f"{data}: not every row rescales exactly once (at the ragged last block)"


def _cov_str(n, pmax):
    n = n.double()
    return (f"rescales per row mean {n.mean().item():.2f} max {int(n.max().item())}, rows with >= 1: "
            f"{100 * (n > 0).double().mean().item():.1f} %, max P 2^{math.log2(pmax.max().item()):.2f}")


# ----------------------------------------------------------------------------------------------------- checks
def _viol(out, ref):
    return ((out.double() - ref).abs() > NS_ATOL + NS_RTOL * ref.abs()).double().mean().item()


def _check(out, ref, what, ns_max, extra=""):
    """test_kernels_gpu.py::_close's two bounds against the float64 reference: max|err| <= 3e-3 max|ref| + 1e-3, and
    at most ns_max of the outputs outside rtol 1e-3 / atol 1e-4."""
    assert out.shape == ref.shape, f"{what}: shape {out.shape} vs {ref.shape}"
    assert torch.isfinite(out).all(), f"{what}: non-finite output"
    err = (out.double() - ref).abs().max().item()
    bound = 3e-3 * ref.abs().max().item() + 1e-3
    viol = _viol(out, ref)
    print(f"{what}: max err {err:.3e} (bound {bound:.3e}); outside rtol 1e-3/atol 1e-4: {100 * viol:.4f} % "
          f"(allowed {100 * ns_max:.4f} %){'; ' + extra if extra else ''}")
    assert err <= bound, f"{what}: max err {err:.4e} > bound {bound:.4e}"
    assert viol <= ns_max, f"{what}: {100 * viol:.4f} % outside rtol 1e-3 / atol 1e-4 (allowed {100 * ns_max:.4f} %)"


def _guarded(rows, width):
    """Output buffer with 64 spare columns and 16 spare rows, filled with the sentinel."""
    return torch.full((rows + 16, width + 64), SENTINEL, dtype=torch.float16, device=DEV)


def _unguard(buf, rows, width, off, what):
    """The [rows, width] output at column `off`; asserts that nothing else in the buffer changed."""
    outside = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    outside[:rows, off:off + width] = False
    assert (buf[outside] == SENTINEL).all(), f"{what}: wrote outside the output slice"
    return buf[:rows, off:off + width]


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


# ----------------------------------------------------------------------------------------------------- CPU: the data
def _cpu_cov(data, Lq=64, Lk=1280, heads=2, B=2):
    q, k, _ = _gen(data, B, Lq, B, Lk, heads, seed=3, device="cpu")
    return _coverage(q, k, heads, SCALE)


def test_staircase_rescales_at_every_block():
    n, pmax = _cpu_cov("stair8.5")
    assert (n == 9).all(), n.unique()
    assert pmax.max().item() < 2 ** 9


def test_staircase_7_5_rescales_every_second_block_with_p_above_2_7():
    n, pmax = _cpu_cov("stair7.5")
    assert (n == 4).all(), n.unique()
    assert pmax.min().item() > 2 ** 7 and pmax.max().item() < 2 ** 8


def test_ramp_rescales_most_rows():
    for data in ("ramp1", "ramp4", "ramp12", "sharp"):
        n, pmax = _cpu_cov(data, Lq=256)
        _assert_coverage(data, n, pmax, 10)


def test_descending_never_rescales_and_underflows():
    q, k, _ = _gen("descending", 2, 64, 2, 1280, 2, seed=3, device="cpu")
    n, _ = _coverage(q, k, 2, SCALE)
    assert (n == 0).all()
    # the last blocks' P relative to the block-0 maximum lie below the fp16 normal range (2^-14) or round to 0
    assert (_spread_log2(q, k, 2, SCALE) > 24).all()


def test_tail_rescales_once_at_the_ragged_block():
    q, k, _ = _gen("tail", 2, 64, 2, 128 * 6 + 5, 2, seed=3, device="cpu")
    n, _ = _coverage(q, k, 2, SCALE)
    assert (n == 1).all()


def test_unit_spread_data_never_rescales():
    """The distribution of test_kernels_gpu.py's attention tests: the lazy rescale is not reached there."""
    g = torch.Generator().manual_seed(0)
    q, k = (torch.randn(1, 640, 128, generator=g).half() for _ in range(2))
    n, _ = _coverage(q, k, 2, SCALE)
    assert (n == 0).all()


def test_emulation_and_reference_agree():
    """The float64 reference adds two segments' softmax results, the emulated kernel arithmetic stays within the
    literal tolerance of it on soft data, and the eager and lazy emulations agree where the maximum never moves."""
    q, k, v = _gen("ramp1", 2, 96, 1, 300, 2, seed=5, device="cpu")
    _, k2, v2 = _gen("sharp", 2, 96, 2, 40, 2, seed=6, device="cpu")
    ref = _attn_ref64(q, [k, k2], [v, v2], 2, SCALE, [2, 1])
    sdpa = lambda kk, vv: F.scaled_dot_product_attention(*(t.double().reshape(2, -1, 2, 64).transpose(1, 2)
                                                           for t in (q, kk, vv))).transpose(1, 2).reshape(2, 96, 128)
    assert torch.allclose(ref, sdpa(k.expand(2, -1, -1), v.expand(2, -1, -1)) + sdpa(k2, v2), atol=1e-12)
    emu = _attn_emulated(q, [k, k2], [v, v2], 2, SCALE, [2, 1])
    assert _viol(emu, ref) < 0.01
    q, k, v = _gen("descending", 2, 96, 2, 640, 2, seed=7, device="cpu")
    assert torch.equal(_attn_emulated(q, k, v, 2, SCALE, thr=0.0), _attn_emulated(q, k, v, 2, SCALE))


# ----------------------------------------------------------------------------------------------------- tc_attn3_kernel
def _run_attn3(ops, data, B, Lq, Lk, heads, *, kv_div=1, layout="separate", out_off=0, seed=0):
    """One tc_attention call on `data` with K/V in the given layout, checked against the float64 reference."""
    C = heads * 64
    q, k, v = _gen(data, B, Lq, B // kv_div, Lk, heads, seed=seed)
    n, pmax = _coverage(q, k, heads, SCALE, kv_div)
    _assert_coverage(data, n, pmax, -(-Lk // BLOCK))
    buf = _guarded(B * Lq, C)
    if layout == "fused_qkv":             # engine.py:344: q / k / v are column slices of one [tokens][3C] projection
        qkv = torch.cat([q, k, v], -1)
        ops.attention(qkv, [dict(k=qkv, v=qkv, ldk=3 * C, ldv=3 * C, Lk=Lk, k_offset=C, v_offset=2 * C)], buf,
                      q_batches=B, Lq=Lq, heads=heads, scale=SCALE, ldq=3 * C, ldo=C + 64, out_offset=out_off)
    elif layout == "fused_kv":            # vae_engine.py:169: one [Lk][2C] tensor, v at column C
        kv = torch.cat([k, v], -1)
        ops.attention(q, [dict(k=kv, v=kv, ldk=2 * C, ldv=2 * C, Lk=Lk, kv_div=kv_div, v_offset=C)], buf,
                      q_batches=B, Lq=Lq, heads=heads, scale=SCALE, ldq=C, ldo=C + 64, out_offset=out_off)
    else:
        ops.attention(q, [dict(k=k, v=v, ldk=C, ldv=C, Lk=Lk, kv_div=kv_div)], buf, q_batches=B, Lq=Lq, heads=heads,
                      scale=SCALE, ldq=C, ldo=C + 64, out_offset=out_off)
    what = f"attn3 {data} B={B} Lq={Lq} Lk={Lk} h={heads} {layout}"
    out = _unguard(buf, B * Lq, C, out_off, what).reshape(B, Lq, C)
    ref = _attn_ref64(q, k, v, heads, SCALE, kv_div)
    _check(out, ref, what, _flash_ns(data, q, k, v, heads, SCALE, kv_div, ref), _cov_str(n, pmax))


# Ramp, sharp and tail rows put most of their weight on a few keys, so the fp16 rounding of P (up to 2^-11 relative) is
# not averaged away as at unit spread: the float64 emulation of the kernel arithmetic (_attn_emulated) itself has
# 0.36 % (ramp4), 0.17 % (ramp12), 0.12 % (sharp) and 0.18 % (tail) of the outputs outside rtol 1e-3 / atol 1e-4 at
# the shapes of test_attn3_online_softmax, above the 0.1 % of unit-spread data; tc_attn3_kernel measured 0.36 / 0.14 /
# 0.12 / 0.12 % there (B200, 1000 W limit).  (The eager rule of tc_attn_kernel: 0.10 % ramp4, 0.05 % sharp emulated.
# There the P of the row maximum is exactly 1; the lazy rule's 2^d, 0 <= d <= 8, is rounded to fp16 like every other
# P, which about doubles the fraction on near-argmax rows.)  These cases are held to 1.5x the emulation's fraction +
# 0.2 %; the staircases and descending rows (0 % emulated, 0 % measured) keep the flash-style limit.
EMULATED = {"ramp4", "ramp12", "sharp", "tail"}


def _flash_ns(data, q, k, v, heads, scale, kv_div, ref, thr=THR):
    if data not in EMULATED:
        return FLASH_NS
    return 1.5 * _viol(_attn_emulated(q, k, v, heads, scale, kv_div, thr=thr), ref) + 0.002


@pytest.mark.gpu
@pytest.mark.parametrize("single", ["0", "1"])
@pytest.mark.parametrize("data", list(DATA))
def test_attn3_online_softmax(ops, monkeypatch, data, single):
    """Every distribution through both CTA modes of tc_attn3_kernel (TC_ATTN_SINGLE is read on every call)."""
    monkeypatch.setenv("TC_ATTN_SINGLE", single)
    Lq, Lk = (300, 128 * 8 + 5) if data == "tail" else (1280, 1280)
    _run_attn3(ops, data, 2, Lq, Lk, 2, out_off=64 * (single == "1"), seed=11)


@pytest.mark.gpu
@pytest.mark.parametrize("single", ["0", "1"])
@pytest.mark.parametrize("data", ["ramp4", "stair8.5"])
def test_attn3_full_machine(ops, monkeypatch, data, single):
    """60 x 5 (batch, head) pairs at L = 2560, two per SM: thousands of CTAs rescaling O at the same time."""
    monkeypatch.setenv("TC_ATTN_SINGLE", single)
    _run_attn3(ops, data, 60, 2560, 2560, 5, seed=12)


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "stair8.5", "tail"])
def test_attn3_dual_reference_fusion_layout(ops, monkeypatch, data):
    """The VAE dual-reference fusion in the default dispatch (Lk > 4096: two query tiles per CTA sharing K/V): every
    query batch reads K/V batch 0 of one fused [Lk][2C] tensor (ldk = 2C, v at column C)."""
    monkeypatch.delenv("TC_ATTN_SINGLE", raising=False)
    Lk = 8192 + 5 if data == "tail" else 8192
    _run_attn3(ops, data, 3, 1024, Lk, 2, kv_div=3, layout="fused_kv", out_off=64, seed=13)


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "stair7.5"])
def test_attn3_fused_qkv_layout(ops, monkeypatch, data):
    """The spatial self attention's layout: q / k / v column slices of one [tokens][3C] tensor (ldq = ldk = 3C)."""
    monkeypatch.delenv("TC_ATTN_SINGLE", raising=False)
    _run_attn3(ops, data, 2, 1280, 1280, 2, layout="fused_qkv", seed=14)


# ----------------------------------------------------------------------------------------------------- tc_attn_kernel
def _two_seg(data, N, T, Lq, heads, Lk0, Lk1, seed):
    q, k0, v0 = _gen(data, N, Lq, -(-N // T), Lk0, heads, seed=seed)
    _, k1, v1 = _gen(data, N, Lq, N, Lk1, heads, seed=seed + 1)
    return q, [k0, k1], [v0, v1], [T, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "sharp"])
@pytest.mark.parametrize("Lk0,Lk1", [(77, 64), (300, 200), (81, 16)])
def test_attn_two_segments_long(ops, data, Lk0, Lk1):
    """Two K/V segments with more than 96 keys (ceil16(Lk0) + ceil16(Lk1) > 96) go to tc_attn_kernel: one online
    softmax per segment, the normalised results added.  (81, 16) is one key past the resident-K/V kernel's limit."""
    N, T, Lq, heads = 6, 3, 300, 2
    C = heads * 64
    q, ks, vs, divs = _two_seg(data, N, T, Lq, heads, Lk0, Lk1, seed=21)
    spread = torch.cat([_spread_log2(q, kk, heads, SCALE, d) for kk, d in zip(ks, divs)])
    assert spread.median().item() > 8, "scores not spread"
    buf = _guarded(N * Lq, C)
    ops.attention(q, [dict(k=ks[0], v=vs[0], ldk=C, ldv=C, Lk=Lk0, kv_div=T), dict(k=ks[1], v=vs[1], ldk=C, ldv=C, Lk=Lk1)],
                  buf, q_batches=N, Lq=Lq, heads=heads, scale=SCALE, ldq=C, ldo=C + 64)
    what = f"attn v2 two segments {data} {Lk0}+{Lk1}"
    out = _unguard(buf, N * Lq, C, 0, what).reshape(N, Lq, C)
    ref = _attn_ref64(q, ks, vs, heads, SCALE, divs)
    _check(out, ref, what, _flash_ns(data, q, ks, vs, heads, SCALE, divs, ref, thr=0.0),
           f"median score spread 2^{spread.median().item():.1f}")


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "sharp"])
def test_attn_v2_single_segment(ops, monkeypatch, data):
    """TC_ATTN_IMPL=v2 keeps single-segment problems on tc_attn_kernel (eager rescale of O in registers)."""
    monkeypatch.setenv("TC_ATTN_IMPL", "v2")
    B, L, heads = 2, 1280, 2
    C = heads * 64
    q, k, v = _gen(data, B, L, B, L, heads, seed=22)
    n, pmax = _coverage(q, k, heads, SCALE)
    _assert_coverage(data, n, pmax, L // BLOCK)
    buf = _guarded(B * L, C)
    ops.attention(q, [dict(k=k, v=v, ldk=C, ldv=C, Lk=L)], buf, q_batches=B, Lq=L, heads=heads, scale=SCALE, ldq=C,
                  ldo=C + 64, out_offset=64)
    what = f"attn v2 single segment {data}"
    out = _unguard(buf, B * L, C, 64, what).reshape(B, L, C)
    ref = _attn_ref64(q, k, v, heads, SCALE)
    _check(out, ref, what, _flash_ns(data, q, k, v, heads, SCALE, 1, ref, thr=0.0), _cov_str(n, pmax))


# ----------------------------------------------------------------------------------------------------- tc_attn_xs_kernel
@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "sharp"])
@pytest.mark.parametrize("N,T,Lq,Lk0,Lk1,fused", [
    (8, 4, 320, 77, 16, True),      # the UNet's text + image cross attention, K/V as in engine.py:355-357
    (6, 3, 333, 80, 16, False),     # exactly 96 keys (the dispatch boundary), ragged Lq
    (7, 3, 200, 1, 16, True),       # one text key; 7 query batches over kv_div = 3
    (7, 3, 333, 96, 0, False),      # one segment of 96 keys: the dispatch sends single segments to tc_attn3_kernel
])
def test_attn_xs_cross_attention(ops, data, N, T, Lq, Lk0, Lk1, fused):
    """Short K/V cross attention (tc_attn_xs_kernel): two independent softmaxes, P normalised then split into fp16
    hi + lo; the text segment is shared by T query batches."""
    heads = 2
    C = heads * 64
    if Lk1:
        q, ks, vs, divs = _two_seg(data, N, T, Lq, heads, Lk0, Lk1, seed=31)
    else:
        q, k0, v0 = _gen(data, N, Lq, -(-N // T), Lk0, heads, seed=31)
        ks, vs, divs = [k0], [v0], [T]
    spread = torch.cat([_spread_log2(q, kk, heads, SCALE, d) for kk, d in zip(ks, divs) if kk.shape[1] > 1])
    assert spread.median().item() > 8, "scores not spread"
    segs = []
    for kk, vv, d in zip(ks, vs, divs):
        if fused:
            kv = torch.cat([kk, vv], -1)
            segs.append(dict(k=kv, v=kv, ldk=2 * C, ldv=2 * C, Lk=kk.shape[1], kv_div=d, v_offset=C))
        else:
            segs.append(dict(k=kk, v=vv, ldk=C, ldv=C, Lk=kk.shape[1], kv_div=d))
    buf = _guarded(N * Lq, C)
    ops.attention(q, segs, buf, q_batches=N, Lq=Lq, heads=heads, scale=SCALE, ldq=C, ldo=C + 64, out_offset=64)
    what = f"attn xs {data} N={N} Lq={Lq} {Lk0}+{Lk1}{' fused kv' if fused else ''}"
    out = _unguard(buf, N * Lq, C, 64, what).reshape(N, Lq, C)
    ref = _attn_ref64(q, ks, vs, heads, SCALE, divs)
    ns = XS_NS if Lk1 else _flash_ns(data, q, ks, vs, heads, SCALE, divs, ref)
    _check(out, ref, what, ns, f"median score spread 2^{spread.median().item():.1f}")


# ----------------------------------------------------------------------------------------------------- temporal attention
@pytest.mark.gpu
@pytest.mark.parametrize("data", ["ramp4", "sharp"])
@pytest.mark.parametrize("T", [16, 20])
def test_temporal_attention_spread(ops, data, T):
    """Temporal self attention over T frames per (batch, pixel, head): T <= 16 on the mma.sync kernel, T = 20 on
    temporal_attn_kernel<32>; q / k / v are column slices of one [B][T][P][3C] tensor."""
    B, P, heads = 2, 40, 2
    C = heads * 64
    q, k, v = _gen(data, B * P, T, B * P, T, heads, seed=41)          # (b p) t c
    spread = _spread_log2(q, k, heads, SCALE)
    assert spread.median().item() > 8, "scores not spread"
    qkv = torch.cat([q, k, v], -1).reshape(B, P, T, 3 * C).permute(0, 2, 1, 3).contiguous()
    buf = _guarded(B * T * P, C)
    ops.temporal_attention(qkv, qkv, qkv, buf, ld=3 * C, ldo=C + 64, B=B, T=T, P=P, heads=heads, scale=SCALE,
                           k_offset=C, v_offset=2 * C)
    what = f"temporal attention {data} T={T}"
    out = _unguard(buf, B * T * P, C, 0, what).reshape(B, T, P, C)
    ref = _attn_ref64(q, k, v, heads, SCALE).reshape(B, P, T, C).permute(0, 2, 1, 3)
    _check(out, ref, what, TEMPORAL_NS, f"median score spread 2^{spread.median().item():.1f}")


# ----------------------------------------------------------------------------------------------------- tc_attn_wide_kernel
@pytest.mark.gpu
@pytest.mark.parametrize("data", ["stair7.5", "stair8.5", "descending"])
@pytest.mark.parametrize("D", [512, 128])
def test_attn_wide_lazy_rescale(ops, data, D):
    """The VAE mid-block attention (one head of D channels, q / k / v slices of one [L][3D] tensor) has the same lazy
    rule (tc_attn_wide.cu:38,276): staircases rescale at every (second) block, descending never."""
    N, L = 2, 1280
    scale = D ** -0.5
    q, k, v = _gen(data, N, L, N, L, 1, D=D, scale=scale, seed=51)
    n, pmax = _coverage(q, k, 1, scale)
    _assert_coverage(data, n, pmax, L // BLOCK)
    qkv = torch.cat([q, k, v], -1)
    buf = _guarded(N * L, D)
    ops.attention_wide(qkv, buf, batches=N, L=L, D=D, scale=scale, ld=3 * D, ldo=D + 64, q_offset=0, k_offset=D,
                       v_offset=2 * D, out_offset=64)
    what = f"wide attention {data} D={D}"
    out = _unguard(buf, N * L, D, 64, what).reshape(N, L, D)
    ref = _attn_ref64(q, k, v, 1, scale)
    _check(out, ref, what, FLASH_NS, _cov_str(n, pmax))


# ----------------------------------------------------------------------------------------------------- dispatch
@pytest.mark.gpu
def test_attention_dispatch_reaches_each_kernel(ops, monkeypatch):
    """The shapes above reach the kernels they are meant for (a dispatch change would move coverage silently)."""
    from torch.profiler import ProfilerActivity, profile
    ours = ("tc_attn3_kernel", "tc_attn_kernel", "tc_attn_xs_kernel", "temporal_attn_mma_kernel",
            "temporal_attn_kernel", "tc_attn_wide_kernel")
    heads, C, Lq = 2, 128, 200
    q = torch.zeros(1, Lq, C, dtype=torch.float16, device=DEV)
    out = torch.zeros_like(q)
    kv = lambda Lk: dict(k=torch.zeros(1, Lk, C, dtype=torch.float16, device=DEV),
                         v=torch.zeros(1, Lk, C, dtype=torch.float16, device=DEV), ldk=C, ldv=C, Lk=Lk)
    attn = lambda *Lks: (lambda: ops.attention(q, [kv(n) for n in Lks], out, q_batches=1, Lq=Lq, heads=heads,
                                               scale=SCALE, ldq=C, ldo=C))
    qkv = torch.zeros(20 * 8, 3 * C, dtype=torch.float16, device=DEV)
    temporal = lambda T: (lambda: ops.temporal_attention(qkv, qkv, qkv, out, ld=3 * C, ldo=C, B=1, T=T, P=1, heads=heads,
                                                         scale=SCALE, k_offset=C, v_offset=2 * C))
    cases = [("tc_attn3_kernel", None, attn(96)), ("tc_attn3_kernel", None, attn(8192)),
             ("tc_attn_xs_kernel", None, attn(80, 16)), ("tc_attn_xs_kernel", None, attn(1, 16)),
             ("tc_attn_kernel", None, attn(81, 16)), ("tc_attn_kernel", None, attn(77, 64)),
             ("tc_attn_kernel", "v2", attn(1280)),
             ("temporal_attn_mma_kernel", None, temporal(16)), ("temporal_attn_kernel", None, temporal(20)),
             ("tc_attn_wide_kernel", None, lambda: ops.attention_wide(qkv, out, batches=1, L=64, D=128, scale=0.1,
                                                                      ld=3 * C, ldo=C, k_offset=C, v_offset=2 * C))]
    for expect, impl, fn in cases:
        if impl:
            monkeypatch.setenv("TC_ATTN_IMPL", impl)
        else:
            monkeypatch.delenv("TC_ATTN_IMPL", raising=False)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = {k for e in prof.key_averages() for k in ours if re.search(rf"\b{k}\b", e.key)}
        assert names == {expect}, f"expected {expect}, launched {names or 'none of the attention kernels'}"
