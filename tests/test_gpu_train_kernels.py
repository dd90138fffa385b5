"""The non-GEMM kernels of the training path (csrc/train_kernels.cu), one at a time, against float64 references on
the CPU, through the pllb_debug_train_* / pllb_debug_s2s_attn hooks (include/pllb.h).

The MLM, RescoreBert and CorrectBart trainers share these kernels; their parity tests can only bound the per-tensor
error of whole-model gradients (bf16 GEMM operands), which a kernel wrong on a few rows, at one stride or under
dropout slips under.  Here every input is exactly representable in bf16 and the reference is computed in float64
from exactly those values, so a kernel's only error is its fp32 arithmetic, and it is bounded row by row:
* fp32 outputs: the largest error of a row over the largest reference magnitude of that row;
* bf16 outputs: within half a bf16 ulp of the reference plus the family's fp32 bound times the row's magnitude;
* every output buffer is pre-filled with a sentinel (a NaN bit pattern for fp32, 0xFFFF for bf16) and one extra
  row or element past its end; what the contract does not write must still hold it.
Dropout is restated bit for bit (drop_factor in train_kernels.cu), so the masks of the forward pass and their reuse
in the backward pass are checked exactly, at p in {0, 0.1, 0.5}.

Each bound is about 4x the worst value measured on a B200 (DESIGN.md §4, profiles/train_kernels_gpu_tests.log).
The tests without the gpu mark show that plausible bugs move the float64 reference by more than these bounds."""
import ctypes
import math

import numpy as np
import pytest
import torch

from asr_rescoring_b200 import _lib

# ------------------------------------------------------------------------------------------------ bounds
# (measured worst on one B200 in the comment of each)
# attention fp32 outputs (dq, dk, dv, D): per row, the largest error over the largest magnitude sum of that row (the sum
# of |terms| the output adds up, attn_ref); also the fp32 slack of the bf16 ctx over the row's largest |ctx|.
# Measured: dv 1.7e-6, ctx 6.1e-7, dk 3.8e-7, D 3.3e-7, dq 1.9e-7
ATT_REL = 7e-6
ATT_LSE = 1e-5       # attention log-sum-exp, absolute (nats); measured 2.3e-6
LN_REL = 1e-6        # LayerNorm forward / backward, per row; measured 2.5e-7
# LayerNorm forward on rows of mean 1e3 and standard deviation 1: fp32 cannot hold their mean closer than 3e-5 (half
# its spacing at 1000), so xhat is off by that much over the standard deviation; measured 4.3e-5
LN_CANCEL_REL = 1.7e-4
CE_REL = 4e-6        # cross entropy: per-row loss over max(1, |loss|) (measured 9.5e-7); fp32 slack of dlogits (2.6e-7)
EMB_REL = 8e-7       # embedding gradients (dword, dpos, dtype), per row; measured 2.0e-7
COLSUM_REL = 8e-7    # column sums: |error| / sum of |terms| of the column; measured 1.9e-7
GELU_REL = 5e-7      # GELU forward / backward: |error| / (|reference| + 1); measured 1.2e-7

DEV = "cuda"
NAN32 = 0x7FC0DEAD   # fp32 sentinel: a quiet NaN with a payload
SEED = 0x243F6A8885A308D3


def gpu_test(f):
    return pytest.mark.usefixtures("require_gpu")(pytest.mark.gpu(f))


# ------------------------------------------------------------------------------------------------ dropout
def drop_params(p):
    """thresh and 1 / (1 - p) as the trainers compute them (train_api.cu: drop_of)."""
    if p <= 0:
        return 0, 1.0
    thresh = int(min(4294967295.0, float(np.float32(p)) * 4294967296.0))
    return thresh, float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def drop_factor(seed, site, idx, p):
    """float64 factor (0 or 1 / (1 - p)) of the elements idx (uint64) of dropout site `site`: splitmix64 of
    seed + site * 0x9E3779B97F4A7C15 + idx * 0xD1B54A32D192ED03 with uint64 wrap-around, kept iff bits 63..32 >= thresh."""
    thresh, inv = drop_params(p)
    idx = np.asarray(idx, np.uint64)
    if thresh == 0:
        return np.ones(idx.shape)
    with np.errstate(over="ignore"):
        x = np.uint64((seed + site * 0x9E3779B97F4A7C15) % 2 ** 64) + idx * np.uint64(0xD1B54A32D192ED03)
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return np.where((x >> np.uint64(32)) >= np.uint64(thresh), inv, 0.0)


# ------------------------------------------------------------------------------------------------ helpers
def bf16r(x):
    """float64 tensor of the bf16 values nearest x (round to nearest even)."""
    return torch.as_tensor(np.asarray(x, np.float32)).bfloat16().double()


def f32_buf(n, fill=None):
    """DEVICE fp32 buffer of n + 1 elements: `fill` (float64 tensor of n values) or the sentinel, then a sentinel."""
    t = torch.full((n + 1,), NAN32, dtype=torch.int32, device=DEV).view(torch.float32)
    if fill is not None:
        t[:n] = fill.reshape(-1).float().to(DEV)
    return t


def bf16_buf(n, fill=None):
    t = torch.full((n + 1,), -1, dtype=torch.int16, device=DEV)
    if fill is not None:
        t.view(torch.bfloat16)[:n] = fill.reshape(-1).bfloat16().to(DEV)
    return t


def untouched(t, lo, hi=None):
    """the sentinel still in elements [lo, hi) of a buffer made by f32_buf / bf16_buf."""
    s = t.view(torch.int32) if t.dtype == torch.float32 else t
    v = s[lo:hi]
    return bool((v == (NAN32 if t.dtype == torch.float32 else -1)).all())


def host(t, n=None, shape=None):
    """float64 CPU copy of the first n elements (bf16 buffers are int16 raw bits)."""
    v = t.view(torch.bfloat16) if t.dtype == torch.int16 else t
    v = v[:n].double().cpu()
    return v.reshape(shape) if shape is not None else v


def ptr(t, off=0):
    return None if t is None else ctypes.c_void_p(t.data_ptr() + off * t.element_size())


def seed_buf():
    return torch.tensor([SEED], dtype=torch.int64, device=DEV)


def call(name, *args, rc=0):
    lib = _lib.load()
    got = getattr(lib, name)(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    if rc == 0:
        _lib.check(got)
    return got


def row_rel(got, ref):
    """per row: max |got - ref| / max |ref| (0 / 0 = 0)."""
    got = np.asarray(got, np.float64).reshape(len(ref), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    num, den = np.abs(got - ref).max(1), np.abs(ref).max(1)
    return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.where(num > 0, np.inf, 0.0))


def half_ulp_bf16(ref):
    a = np.abs(ref)
    e = np.floor(np.log2(np.where(a > 0, a, 1.0)))
    return np.where(a > 0, 2.0 ** (e - 8), 0.0)


def bf16_row_excess(got, ref):
    """per row: max over the row of (|got - ref| - half a bf16 ulp of ref) / max |ref|; <= 0 when every element is
    within half an ulp."""
    got = np.asarray(got, np.float64).reshape(len(ref), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    ex = (np.abs(got - ref) - half_ulp_bf16(ref)).max(1)
    den = np.abs(ref).max(1)
    return np.where(den > 0, ex / np.where(den > 0, den, 1.0), np.where(ex > 0, np.inf, 0.0))


def row_rel_mag(got, ref, mag):
    """per row: max |got - ref| / max mag, mag the magnitude sum of every element (0 / 0 = 0)."""
    got, ref, mag = (np.asarray(t, np.float64).reshape(len(ref), -1) for t in (got, ref, mag))
    num, den = np.abs(got - ref).max(1), mag.max(1)
    return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.where(num > 0, np.inf, 0.0))


def worst(x):
    return float(np.max(x)) if np.size(x) else 0.0


# ------------------------------------------------------------------------------------------------ attention
def attn_ref(q, k, v, visible, M, dctx):
    """float64 attention of q [B, NH, Tq, 64] over k, v [B, NH, Tk, 64]: visible bool [B, 1|NH, Tq, Tk], dropout factors
    M [B, NH, Tq, Tk] on the probabilities, upstream gradient dctx [B, NH, Tq, 64].
    Returns ctx, lse, dq, dk, dv, D (= sum_j P dP = dctx . ctx), and the magnitude sums of dq, dk, dv and D: the same
    sums over |terms|, the scale of their fp32 rounding error (an exact gradient can be 0, e.g. dk of a key that is the
    only one its queries see)."""
    ql, kl, vl = (t.clone().requires_grad_(True) for t in (q, k, v))
    s = (ql @ kl.transpose(-1, -2) * 0.125).masked_fill(~visible, -math.inf)
    lse = torch.logsumexp(s, -1)
    P = torch.exp(s - lse[..., None])
    ctx = (P * M) @ vl
    ctx.backward(dctx)
    P, ctx = P.detach(), ctx.detach()
    adP = (dctx.abs() @ v.abs().transpose(-1, -2)) * M                # |dP|, dP = (dctx . v) * mask
    aD = (P * adP).sum(-1)
    adS = P * (adP + aD[..., None])                                    # |dS|, dS = P (dP - D)
    mag = ((adS @ k.abs()) * 0.125, (adS.transpose(-1, -2) @ q.abs()) * 0.125, (P * M).transpose(-1, -2) @ dctx.abs(), aD)
    return ctx, lse.detach(), ql.grad, kl.grad, vl.grad, (dctx * ctx).sum(-1), mag


def heads(x, B, T, NH):
    """[B*T, NH*64] -> [B, NH, T, 64]"""
    return x.reshape(B, T, NH, 64).permute(0, 2, 1, 3)


def rows_of(x):
    """[B, NH, T, 64] -> [B*T, NH*64]"""
    B, NH, T, _ = x.shape
    return x.permute(0, 2, 1, 3).reshape(B * T, NH * 64)


def attn_masks(B, NH, Tq, Tk, n_valid, causal, seed, site, p):
    i = torch.arange(Tq)[:, None]
    j = torch.arange(Tk)[None, :]
    if causal:
        visible = (j <= i)[None, None].expand(B, 1, Tq, Tk)
    else:
        visible = (j[None] < torch.as_tensor(n_valid)[:, None, None])[:, None]
    M = torch.from_numpy(drop_factor(seed, site, np.arange(B * NH * Tq * Tk, dtype=np.uint64), p).reshape(B, NH, Tq, Tk))
    return visible, M


def ref_rows(r, NH):
    """attn_ref's results in the kernels' row layout: ctx, lse, dq, dk, dv, D and the magnitudes of dq, dk, dv, D."""
    ctx, lse, dq, dk, dv, D, (mq, mk, mv, mD) = r
    per_head = lambda x: x.permute(0, 2, 1).reshape(-1, NH)                     # noqa: E731
    return (rows_of(ctx), per_head(lse), rows_of(dq), rows_of(dk), rows_of(dv), per_head(D),
            (rows_of(mq), rows_of(mk), rows_of(mv), per_head(mD)))


def check_attn_outputs(tag, ref, got, key_rows_masked):
    """ref (from ref_rows) / got: ctx, lse, dq, dk, dv, D in row form; key_rows_masked: bool [B*Tk] (dk = dv = 0
    exactly)."""
    ctx_r, lse_r, dq_r, dk_r, dv_r, D_r, (mq, mk, mv, mD) = ref
    ctx_g, lse_g, dq_g, dk_g, dv_g, D_g = got
    m = {"ctx": worst(bf16_row_excess(ctx_g, ctx_r)), "lse": float((lse_g - lse_r).abs().max()),
         "dq": worst(row_rel_mag(dq_g, dq_r, mq)), "D": worst(row_rel_mag(D_g, D_r, mD))}
    live = ~key_rows_masked
    m["dk"] = worst(row_rel_mag(dk_g[live], dk_r[live], mk[live]))
    m["dv"] = worst(row_rel_mag(dv_g[live], dv_r[live], mv[live]))
    print(f"[{tag}] " + " ".join(f"{k} {v:.2e}" for k, v in m.items()))
    assert m["ctx"] <= ATT_REL and m["lse"] <= ATT_LSE, m
    assert m["dq"] <= ATT_REL and m["dk"] <= ATT_REL and m["dv"] <= ATT_REL and m["D"] <= ATT_REL, m
    assert bool((dk_g[key_rows_masked] == 0).all()) and bool((dv_g[key_rows_masked] == 0).all())


ATTN_T = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512]
ATTN_NH = [4, 8, 12, 16]        # the trainers take hidden 256 .. 1024, so 4 .. 16 heads of 64
PS = [0.0, 0.1, 0.5]


def ragged(T, B, rng):
    """n_valid of B sequences: T, 1, then random lengths in [1, T]."""
    return np.array(([T, 1] + list(rng.integers(1, T + 1, B)))[:B], np.int32)


@gpu_test
@pytest.mark.parametrize("T", ATTN_T)
def test_padded_self_attention(T):
    """attn_fwd_train + attn_bwd_q / attn_bwd_kv (MLM and RescoreBert encoders): B zero-padded sequences, queries past
    n_valid (pad rows) attend to the n_valid real keys, pad keys get dk = dv = 0."""
    rng = np.random.default_rng(T)
    NH = ATTN_NH[ATTN_T.index(T) % 4]
    H, B = NH * 64, 3
    n_valid = ragged(T, B, rng)
    qkv = bf16r(rng.normal(0, 1.5, (B * T, 3 * H)))
    dctx = bf16r(rng.normal(0, 1, (B * T, H)))
    d_qkv, d_dctx, d_nv, seed = bf16_buf(qkv.numel(), qkv), f32_buf(dctx.numel(), dctx), torch.from_numpy(n_valid).to(DEV), seed_buf()
    q, k, v = (heads(qkv[:, c * H:(c + 1) * H], B, T, NH) for c in range(3))
    for p in PS:
        site = 2 + 8 * int(p * 10)
        visible, M = attn_masks(B, NH, T, T, n_valid, False, SEED, site, p)
        ref = ref_rows(attn_ref(q, k, v, visible, M, heads(dctx, B, T, NH)), NH)
        ctx_b, lse_b, dqkv_b, D_b = bf16_buf(B * T * H), f32_buf(B * T * NH), f32_buf(B * T * 3 * H), f32_buf(B * T * NH)
        call("pllb_debug_train_attn", ptr(d_qkv), ptr(d_nv), B, T, H, ptr(d_dctx), ptr(seed), p, site, ptr(ctx_b), ptr(lse_b),
             ptr(dqkv_b), ptr(D_b))
        for buf, n in ((ctx_b, B * T * H), (lse_b, B * T * NH), (dqkv_b, B * T * 3 * H), (D_b, B * T * NH)):
            assert untouched(buf, n) and not untouched(buf, 0, n), "a write past the end, or a hole"
        g = host(dqkv_b, B * T * 3 * H, (B * T, 3 * H))
        masked_keys = torch.as_tensor(np.concatenate([np.arange(T) >= n for n in n_valid]))
        check_attn_outputs(f"self T={T} NH={NH} p={p}", ref,
                           (host(ctx_b, B * T * H, (B * T, H)), host(lse_b, B * T * NH, (B * T, NH)), g[:, :H], g[:, H:2 * H],
                            g[:, 2 * H:], host(D_b, B * T * NH, (B * T, NH))), masked_keys)


@gpu_test
@pytest.mark.parametrize("T", ATTN_T)
def test_causal_attention(T):
    """attn_*_s2s<causal> (the decoder's self-attention) in the trainer's layout: q | k | v in one [B*T, 3H] buffer
    (ldq = ldkv = 3H), dq | dk | dv into one [B*T, 3H] buffer."""
    rng = np.random.default_rng(100 + T)
    NH = ATTN_NH[(ATTN_T.index(T) + 1) % 4]
    H, B = NH * 64, 2
    qkv = bf16r(rng.normal(0, 1.5, (B * T, 3 * H)))
    dctx = bf16r(rng.normal(0, 1, (B * T, H)))
    d_qkv, d_dctx, seed = bf16_buf(qkv.numel(), qkv), f32_buf(dctx.numel(), dctx), seed_buf()
    q, k, v = (heads(qkv[:, c * H:(c + 1) * H], B, T, NH) for c in range(3))
    for p in PS:
        site = 2 + 8 * int(p * 10)
        visible, M = attn_masks(B, NH, T, T, None, True, SEED, site, p)
        ref = ref_rows(attn_ref(q, k, v, visible, M, heads(dctx, B, T, NH)), NH)
        ctx_b, lse_b, dqkv_b, D_b = bf16_buf(B * T * H), f32_buf(B * T * NH), f32_buf(B * T * 3 * H), f32_buf(B * T * NH)
        call("pllb_debug_s2s_attn", ptr(d_qkv), ptr(d_qkv, H), ptr(d_qkv, 2 * H), 3 * H, 3 * H, None, B, T, T, NH, 1,
             ptr(d_dctx), ptr(seed), p, site, ptr(ctx_b), ptr(lse_b), ptr(dqkv_b), 3 * H, ptr(dqkv_b, H), ptr(dqkv_b, 2 * H),
             3 * H, ptr(D_b))
        for buf, n in ((ctx_b, B * T * H), (lse_b, B * T * NH), (dqkv_b, B * T * 3 * H), (D_b, B * T * NH)):
            assert untouched(buf, n) and not untouched(buf, 0, n)
        g = host(dqkv_b, B * T * 3 * H, (B * T, 3 * H))
        check_attn_outputs(f"causal T={T} NH={NH} p={p}", ref,
                           (host(ctx_b, B * T * H, (B * T, H)), host(lse_b, B * T * NH, (B * T, NH)), g[:, :H], g[:, H:2 * H],
                            g[:, 2 * H:], host(D_b, B * T * NH, (B * T, NH))), torch.zeros(B * T, dtype=torch.bool))


CROSS = [(33, 129), (129, 1), (512, 65), (1, 512), (65, 33), (257, 512)]


@gpu_test
@pytest.mark.parametrize("Tq,Tk", CROSS)
def test_cross_attention_in_the_stacked_kv_layout(Tq, Tk):
    """attn_*_s2s<cross> (decoder over encoder rows) in the trainer's layout: the K|V of all NL = 3 decoder layers in
    one [B*Tk, 2H*NL] buffer, layer l at columns 2H*l (k) and 2H*l + H (v), dK|dV likewise.  Layer 1 is run: the
    columns of layers 0 and 2 of the gradient buffer keep their sentinel."""
    rng = np.random.default_rng(1000 * Tq + Tk)
    NH = ATTN_NH[CROSS.index((Tq, Tk)) % 4]
    H, B, NL, l = NH * 64, 3, 3, 1
    KV = 2 * H * NL
    n_valid = ragged(Tk, B, rng)
    qb = bf16r(rng.normal(0, 1.5, (B * Tq, H)))
    kv = bf16r(rng.normal(0, 1.5, (B * Tk, KV)))
    dctx = bf16r(rng.normal(0, 1, (B * Tq, H)))
    d_q, d_kv, d_dctx = bf16_buf(qb.numel(), qb), bf16_buf(kv.numel(), kv), f32_buf(dctx.numel(), dctx)
    d_nv, seed = torch.from_numpy(n_valid).to(DEV), seed_buf()
    q = heads(qb, B, Tq, NH)
    k, v = heads(kv[:, 2 * H * l:2 * H * l + H], B, Tk, NH), heads(kv[:, 2 * H * l + H:2 * H * (l + 1)], B, Tk, NH)
    for p in PS:
        site = 5 + 8 * int(p * 10)
        visible, M = attn_masks(B, NH, Tq, Tk, n_valid, False, SEED, site, p)
        ref = ref_rows(attn_ref(q, k, v, visible, M, heads(dctx, B, Tq, NH)), NH)
        ctx_b, lse_b, dq_b, dkv_b, D_b = (bf16_buf(B * Tq * H), f32_buf(B * Tq * NH), f32_buf(B * Tq * H), f32_buf(B * Tk * KV),
                                          f32_buf(B * Tq * NH))
        call("pllb_debug_s2s_attn", ptr(d_q), ptr(d_kv, 2 * H * l), ptr(d_kv, 2 * H * l + H), H, KV, ptr(d_nv), B, Tq, Tk, NH, 0,
             ptr(d_dctx), ptr(seed), p, site, ptr(ctx_b), ptr(lse_b), ptr(dq_b), H, ptr(dkv_b, 2 * H * l),
             ptr(dkv_b, 2 * H * l + H), KV, ptr(D_b))
        for buf, n in ((ctx_b, B * Tq * H), (lse_b, B * Tq * NH), (dq_b, B * Tq * H), (D_b, B * Tq * NH)):
            assert untouched(buf, n) and not untouched(buf, 0, n)
        raw = dkv_b[:B * Tk * KV].view(torch.int32).reshape(B * Tk, KV).cpu()
        own = torch.zeros(KV, dtype=torch.bool)
        own[2 * H * l:2 * H * (l + 1)] = True
        assert bool((raw[:, ~own] == NAN32).all()), "a write into another layer's columns"
        assert bool((raw[:, own] != NAN32).all()) and untouched(dkv_b, B * Tk * KV)
        g = host(dkv_b, B * Tk * KV, (B * Tk, KV))
        masked_keys = torch.as_tensor(np.concatenate([np.arange(Tk) >= n for n in n_valid]))
        check_attn_outputs(f"cross Tq={Tq} Tk={Tk} NH={NH} p={p}", ref,
                           (host(ctx_b, B * Tq * H, (B * Tq, H)), host(lse_b, B * Tq * NH, (B * Tq, NH)),
                            host(dq_b, B * Tq * H, (B * Tq, H)), g[:, 2 * H * l:2 * H * l + H], g[:, 2 * H * l + H:2 * H * (l + 1)],
                            host(D_b, B * Tq * NH, (B * Tq, NH))), masked_keys)


# ------------------------------------------------------------------------------------------------ LayerNorm
def ln_ref(z, g, b, eps, biased=True):
    """float64 LayerNorm of z [R, H]: xhat, rstd, out = xhat * g + b."""
    mean = z.mean(1, keepdim=True)
    var = ((z - mean) ** 2).sum(1, keepdim=True) / (z.shape[1] if biased else z.shape[1] - 1)
    rstd = 1.0 / torch.sqrt(var + eps)
    xhat = (z - mean) * rstd
    return xhat, rstd[:, 0], xhat * g + b


LN_H = [256, 512, 768, 1024]
LN_R = [1, 3, 5, 4097]
LN_CASES = [(H, R) for H in LN_H for R in LN_R]


def ln_inputs(H, R, rng):
    g = bf16r(rng.normal(1, 0.3, H))
    b = bf16r(rng.normal(0, 0.3, H))
    return g, b


@gpu_test
@pytest.mark.parametrize("H,R", LN_CASES)
def test_layernorm_forward(H, R):
    """ln_fwd (LN(dropout(y) + res)), ln_fwd<EMBED> (BERT embeddings, dropout after the LayerNorm) and bart_embed
    (word * scale + pos): xhat, rstd, the fp32 and bf16 outputs, at eps 1e-12 and 1e-5.  The plain form has rows of mean
    1e3 and standard deviation 1 (the first and the last row)."""
    k = LN_CASES.index((H, R))
    rng = np.random.default_rng(k)
    eps = (1e-12, 1e-5)[k % 2]
    p = PS[k % 3]
    g, b = ln_inputs(H, R, rng)
    d_g, d_b, seed = f32_buf(H, g), f32_buf(H, b), seed_buf()
    site = 3 + 8 * k
    F = torch.from_numpy(drop_factor(SEED, site, np.arange(R * H, dtype=np.uint64), p).reshape(R, H))
    # ---- plain: z = dropout(y) + res
    y = bf16r(rng.normal(0, 2, (R, H)))
    res = bf16r(rng.normal(0, 1, (R, H)))
    cancel = torch.zeros(R, dtype=torch.bool)
    cancel[0] = cancel[-1] = R > 1
    res[cancel] = torch.from_numpy((1000 + rng.normal(0, 1, (int(cancel.sum()), H))).astype(np.float32).astype(np.float64))
    y[cancel] = 0
    z = y * F + res
    forms = {"plain": (z, dict(form=0, y=f32_buf(R * H, y), res=f32_buf(R * H, res)))}
    # ---- embeddings: ids over T positions, a word table with repeated rows
    T, vocab, scale = min(R, 37), 50, 1.7
    ids = rng.integers(0, vocab, R).astype(np.int32)
    word, pos, typ = (bf16r(rng.normal(0, 1, s)) for s in ((vocab, H), (T, H), (2, H)))
    rpos = torch.as_tensor(np.arange(R) % T)
    forms["embed"] = (word[ids] + pos[rpos] + typ[0], dict(form=1))
    forms["bart"] = (word[ids] * float(np.float32(scale)) + pos[rpos], dict(form=2))
    d_ids, d_word, d_pos, d_typ = torch.from_numpy(ids).to(DEV), f32_buf(vocab * H, word), f32_buf(T * H, pos), f32_buf(2 * H, typ)
    for name, (zz, a) in forms.items():
        xhat, rstd, out = ln_ref(zz, g, b, eps)
        if name != "plain":
            out = out * F                                           # dropout after the LayerNorm
        o32, o16, xh, rs = f32_buf(R * H), bf16_buf(R * H), f32_buf(R * H), f32_buf(R)
        call("pllb_debug_train_ln_fwd", a["form"], ptr(a.get("y")), ptr(a.get("res")), ptr(d_ids), T, ptr(d_word), vocab,
             ptr(d_pos), ptr(d_typ), scale, ptr(d_g), ptr(d_b), eps, R, H, ptr(seed), p, site, ptr(o32), ptr(o16), ptr(xh),
             ptr(rs))
        for buf, n in ((o32, R * H), (o16, R * H), (xh, R * H), (rs, R)):
            assert untouched(buf, n) and not untouched(buf, 0, n)
        got = dict(xhat=host(xh, R * H, (R, H)), out32=host(o32, R * H, (R, H)))
        errs = {kk: row_rel(got[kk], ref) for kk, ref in (("xhat", xhat), ("out32", out))}
        errs["rstd"] = np.abs(host(rs, R).numpy() / rstd.numpy() - 1)
        errs["out16"] = bf16_row_excess(host(o16, R * H, (R, H)), out)
        c = cancel.numpy() if name == "plain" else np.zeros(R, bool)
        m = {kk: worst(e[~c]) for kk, e in errs.items()}
        mc = {kk: worst(e[c]) for kk, e in errs.items()}
        print(f"[ln fwd {name} H={H} R={R} eps={eps} p={p}] " + " ".join(f"{kk} {v:.2e}" for kk, v in m.items())
              + ("  mean-1e3 rows: " + " ".join(f"{kk} {v:.2e}" for kk, v in mc.items()) if c.any() else ""))
        assert all(v <= LN_REL for v in m.values()), m
        assert all(v <= LN_CANCEL_REL for v in mc.values()), mc


@gpu_test
@pytest.mark.parametrize("H,R", LN_CASES)
def test_layernorm_backward(H, R):
    """ln_bwd in the three ways the trainers call it: no residual gradient with the output-side mask (dz_drop); a
    separate residual gradient with the input-side mask; and in place, add == dz with the output-side mask into dz_drop
    (train_api.cu's residual chain)."""
    k = LN_CASES.index((H, R))
    rng = np.random.default_rng(50 + k)
    eps, p = (1e-12, 1e-5)[k % 2], PS[(k + 1) % 3]
    g, _ = ln_inputs(H, R, rng)
    z = torch.from_numpy(rng.normal(0.3, 1.7, (R, H)))
    xhat, rstd, _ = ln_ref(z, g, 0, eps)
    xhat32, rstd32 = xhat.float().double(), rstd.float().double()
    d_g, d_xh, d_rs, seed = f32_buf(H, g), f32_buf(R * H, xhat32), f32_buf(R, rstd32), seed_buf()
    dy = bf16r(rng.normal(0, 1, (R, H)))
    add = bf16r(rng.normal(0, 1, (R, H)))
    s_in, s_out = 4 + 8 * k, 3 + 8 * k
    f_in = drop_factor(SEED, s_in, np.arange(R * H, dtype=np.uint64), p).reshape(R, H)
    f_out = drop_factor(SEED, s_out, np.arange(R * H, dtype=np.uint64), p).reshape(R, H)

    def dz_ref(t):
        zz = z.clone().requires_grad_(True)
        x, _, _ = ln_ref(zz, g, 0, eps)
        (x * g).backward(t)
        return zz.grad

    for mode in ("out_mask", "in_mask", "aliased"):
        d_dy = f32_buf(R * H, dy)
        d_dz, d_dzd = f32_buf(R * H, add if mode == "aliased" else None), f32_buf(R * H)
        if mode == "out_mask":
            t32 = dy.numpy().astype(np.float32)
            args = (None, -1, s_out, ptr(d_dzd))
        elif mode == "in_mask":
            d_add = f32_buf(R * H, add)
            t32 = (dy.numpy().astype(np.float32) + add.numpy().astype(np.float32)) * f_in.astype(np.float32)
            args = (ptr(d_add), s_in, -1, None)
        else:                   # the trainers' residual chain: add == dz, with the output-side mask into dz_drop
            t32 = dy.numpy().astype(np.float32) + add.numpy().astype(np.float32)
            args = (ptr(d_dz), -1, s_out, ptr(d_dzd))
        call("pllb_debug_train_ln_bwd", ptr(d_dy), args[0], ptr(d_g), ptr(d_xh), ptr(d_rs), R, H, ptr(seed), p, args[1],
             args[2], ptr(d_dz), args[3])
        ref = dz_ref(torch.from_numpy(t32.astype(np.float64)))
        got_dy = host(d_dy, R * H, (R, H)).numpy()
        assert np.array_equal(got_dy.astype(np.float32), t32), "dy must hold (dy + add) * mask, in fp32"
        e = row_rel(host(d_dz, R * H, (R, H)), ref)
        m = {"dz": worst(e)}
        if mode in ("out_mask", "aliased"):
            m["dz_drop"] = worst(row_rel(host(d_dzd, R * H, (R, H)), ref * f_out))
            assert untouched(d_dzd, R * H) and not untouched(d_dzd, 0, R * H)
        else:
            assert untouched(d_dzd, 0)
        assert untouched(d_dz, R * H) and untouched(d_dy, R * H)
        print(f"[ln bwd {mode} H={H} R={R} p={p}] " + " ".join(f"{kk} {v:.2e}" for kk, v in m.items()))
        assert all(v <= LN_REL for v in m.values()), m


# ------------------------------------------------------------------------------------------------ cross entropy
def ce_ref(x, labels, V):
    """per-row loss and softmax - onehot over the first V columns (labels -100: 0 and a zero row)."""
    x = x[:, :V]
    lp = torch.log_softmax(x, 1)
    lab = torch.as_tensor(labels, dtype=torch.long)
    keep = lab >= 0
    loss = torch.zeros(len(x), dtype=torch.float64)
    loss[keep] = -lp[keep, lab[keep]]
    d = torch.exp(lp)
    d[keep, lab[keep]] -= 1
    d[~keep] = 0
    return loss, d


CE_CASES = [(300, 4096), (8000, 4096), (21128, 1024)]


@gpu_test
@pytest.mark.parametrize("ignore", [False, True])
@pytest.mark.parametrize("V,R", CE_CASES)
def test_cross_entropy(V, R, ignore):
    """ce_kernel + loss_mean_kernel (MLM) and ce_ignore_kernel + loss_mean_valid_kernel (CorrectBart), Vp = V rounded up
    to 256 with 1e30 in the pad columns (never read).  Labels 0 and V - 1, row scales from 0.1 to 20, a row with one
    dominant logit of +80 elsewhere and one at its label; dlogits columns >= V exactly 0."""
    rng = np.random.default_rng(V + R + ignore)
    Vp = (V + 255) // 256 * 256
    x = rng.normal(0, 1, (R, Vp)) * np.geomspace(0.1, 20, R)[:, None]
    labels = rng.integers(0, V, R).astype(np.int32)
    if ignore:
        labels[rng.random(R) < 0.35] = -100
        labels[4] = -100
    labels[0], labels[1] = 0, V - 1                   # after the -100 rows, so both edges are always labelled
    labels[2:4] = rng.integers(0, V, 2)
    x[2, (labels[2] + 7) % V] = 80.0
    x[3, labels[3]] = 80.0
    x = bf16r(x)
    x[:, V:] = 1e30
    d_x = f32_buf(R * Vp, x)
    batches = [labels]
    if ignore:
        one = np.full(R, -100, np.int32)
        one[R // 2] = V - 1
        batches.append(one)
    for lab in batches:
        loss, dl = ce_ref(x, lab, V)
        d_lab = torch.from_numpy(lab).to(DEV)
        lr, dlog, out = f32_buf(R), bf16_buf(R * Vp), f32_buf(2)
        call("pllb_debug_train_ce", ptr(d_x), ptr(d_lab), R, V, Vp, int(ignore), ptr(lr), ptr(dlog), ptr(out))
        got_l = host(lr, R)
        got_d = host(dlog, R * Vp, (R, Vp))
        assert untouched(lr, R) and untouched(dlog, R * Vp) and not untouched(dlog, 0, R * Vp)
        assert bool((got_d[:, V:] == 0).all()), "dlogits columns >= V must be 0"
        e_loss = (got_l - loss).abs() / loss.abs().clamp_min(1.0)
        e_d = bf16_row_excess(got_d[:, :V], dl)
        lab_rows = lab >= 0
        n = int(lab_rows.sum())
        mean_ref = float(got_l.numpy()[lab_rows].astype(np.float64).sum() / n)       # the mean of the fp32 row losses
        got_out = host(out, 2)
        print(f"[ce V={V} R={R} ignore={ignore} N={n}] loss {worst(e_loss.numpy()):.2e} dlogits {worst(e_d):.2e} "
              f"mean {abs(float(got_out[0]) - mean_ref) / mean_ref:.2e}")
        assert worst(e_loss.numpy()) <= CE_REL and worst(e_d) <= CE_REL
        assert abs(float(got_out[0]) - mean_ref) <= 2 ** -23 * abs(mean_ref)
        if ignore:
            assert bool((got_l[~torch.as_tensor(lab_rows)] == 0).all())
            assert bool((got_d[~torch.as_tensor(lab_rows)] == 0).all())
            assert np.float32(float(got_out[1])) == np.float32(1.0) / np.float32(n)
            assert untouched(out, 2)
        else:
            assert untouched(out, 1)


# ------------------------------------------------------------------------------------------------ embedding backward
@gpu_test
@pytest.mark.parametrize("form", ["bert", "bart"])
@pytest.mark.parametrize("H", LN_H)
def test_embedding_backward(H, form):
    """pos_grad + colsum + word_grad (BERT form) and the BART form with scale != 1: ids repeated across distant rows, the
    pad id present (skipped for the word rows, counted for positions and type), dword pre-loaded (the kernel adds),
    position rows >= T exactly 0, and in the BART form dz scaled in place."""
    rng = np.random.default_rng(H + (form == "bart"))
    B, T, pos_rows, vocab, pad = 3, 129, 160, 40, 0
    R = B * T
    ids = rng.integers(0, vocab, R).astype(np.int32)
    ids[rng.random(R) < 0.1] = pad
    ids[0], ids[R - 1] = 7, 7                     # the same id in the first and the last row
    dz = bf16r(rng.normal(0, 1, (R, H)))
    dword0 = bf16r(rng.normal(0, 1, (vocab, H)))
    scale = 1.7 if form == "bart" else 1.0
    dz_s = torch.from_numpy((dz.numpy().astype(np.float32) * np.float32(scale)).astype(np.float64))
    keep = ids != pad
    dword = dword0.clone()
    dword.index_add_(0, torch.as_tensor(ids[keep], dtype=torch.long), dz_s[torch.as_tensor(keep)])
    dpos = torch.zeros(pos_rows, H, dtype=torch.float64)
    dpos[:T] = dz.reshape(B, T, H).sum(0)
    for scratch in ((False, True) if form == "bert" else (False,)):
        d_dz, d_ids = f32_buf(R * H, dz), torch.from_numpy(ids).to(DEV)
        d_w, d_p, d_t = f32_buf(vocab * H, dword0), f32_buf(pos_rows * H), f32_buf(H)
        d_s = f32_buf(128 * H) if scratch else None
        call("pllb_debug_train_embed_bwd", int(form == "bart"), ptr(d_dz), ptr(d_ids), B, T, H, pos_rows, pad, scale, ptr(d_w),
             vocab, ptr(d_p), ptr(d_t) if form == "bert" else None, ptr(d_s))
        gw, gp = host(d_w, vocab * H, (vocab, H)), host(d_p, pos_rows * H, (pos_rows, H))
        assert untouched(d_w, vocab * H) and untouched(d_p, pos_rows * H)
        assert bool((gp[T:] == 0).all()), "position rows >= T must be 0"
        unused = np.setdiff1d(np.arange(vocab), ids[keep])
        assert bool((gw[unused] == dword0[unused]).all()), "rows no id maps to (the pad row among them) must stay as they were"
        m = {"dword": worst(row_rel(gw, dword)), "dpos": worst(row_rel(gp[:T], dpos[:T]))}
        if form == "bert":
            m["dtype"] = worst(row_rel(host(d_t, H)[None], dz.sum(0)[None]))
            assert untouched(d_t, H)
            assert bool((host(d_dz, R * H, (R, H)) == dz).all()), "the BERT form leaves dz as it is"
        else:
            assert np.array_equal(host(d_dz, R * H, (R, H)).numpy().astype(np.float32), dz_s.numpy().astype(np.float32))
        print(f"[embed bwd {form} H={H} scratch={scratch}] " + " ".join(f"{kk} {v:.2e}" for kk, v in m.items()))
        assert all(v <= EMB_REL for v in m.values()), m


# ------------------------------------------------------------------------------------------------ colsum
COLSUM = [(1, 21248), (63, 1), (64, 768), (65, 21248), (4095, 33), (16391, 31), (16391, 768), (4095, 1), (64, 1)]


@gpu_test
@pytest.mark.parametrize("R,C", COLSUM)
def test_column_sums(R, C):
    """colsum (+ colsum_final when the rows are split into S > 1 slices): bf16 and fp32 input, with and without xhat
    (the LayerNorm parameter gradients), with and without scratch (S = 1 or up to 64 slices)."""
    rng = np.random.default_rng(R * 7 + C)
    dy = bf16r(rng.normal(0.5, 1, (R, C)))
    xh = bf16r(rng.normal(0, 1, (R, C)))
    ref_sum, ref_dot = dy.sum(0), (dy * xh).sum(0)
    den_sum, den_dot = dy.abs().sum(0), (dy * xh).abs().sum(0)
    d_f32, d_b16, d_xh = f32_buf(R * C, dy), bf16_buf(R * C, dy), f32_buf(R * C, xh)
    for bf in (False, True):
        for with_xhat in (False, True):
            for scratch in (False, True):
                o_s, o_d = f32_buf(C), f32_buf(C)
                s = f32_buf(128 * C) if scratch else None
                call("pllb_debug_train_colsum", ptr(d_b16 if bf else d_f32), int(bf), ptr(d_xh) if with_xhat else None, R, C,
                     ptr(o_s), ptr(o_d) if with_xhat else None, ptr(s))
                e = (host(o_s, C) - ref_sum).abs() / den_sum.clamp_min(1e-30)
                m = {"sum": float(e.max())}
                assert untouched(o_s, C) and not untouched(o_s, 0, C)
                if with_xhat:
                    m["dot"] = float(((host(o_d, C) - ref_dot).abs() / den_dot.clamp_min(1e-30)).max())
                    assert untouched(o_d, C) and not untouched(o_d, 0, C)
                else:
                    assert untouched(o_d, 0)
                print(f"[colsum R={R} C={C} bf16={bf} xhat={with_xhat} scratch={scratch}] "
                      + " ".join(f"{kk} {v:.2e}" for kk, v in m.items()))
                assert all(v <= COLSUM_REL for v in m.values()), m


# ------------------------------------------------------------------------------------------------ cast_transpose
CT = [(1, 1, 64), (33, 47, 64), (100, 250, 128), (1000, 33, 1024), (64, 64, 64), (257, 768, 320)]


@gpu_test
@pytest.mark.parametrize("R,C,Rp", CT)
def test_cast_transpose_is_bit_exact(R, C, Rp):
    """cast_transpose: round to nearest even as torch's .bfloat16() (ties included), dstT [C, Rp] zero in columns >= R;
    dst16 only, dstT only, both; fp32 and bf16 sources.  This is also the witness for a transpose without the zero
    fill: dstT starts as the 0xFFFF sentinel, so a column >= R left unwritten fails the bit-exact comparison with +0
    (the shapes (1, 1, 64), (33, 47, 64), (100, 250, 128) and (257, 768, 320) have Rp > R)."""
    rng = np.random.default_rng(R + C + Rp)
    src = rng.normal(0, 3, (R, C)).astype(np.float32)
    bits = src.view(np.uint32)
    bits[::3] = (bits[::3] & 0xFFFF0000) | 0x8000          # exact ties between two bf16 values
    src_t = torch.from_numpy(src)
    exp16 = src_t.bfloat16().view(torch.int16)
    expT = torch.zeros(C, Rp, dtype=torch.int16)
    expT[:, :R] = exp16.t()
    d32 = torch.from_numpy(src.reshape(-1)).to(DEV)
    d16 = exp16.reshape(-1).to(DEV)
    for src_bf16 in (False, True):
        for want16, wantT in ((True, False), (False, True), (True, True)):
            o16 = bf16_buf(R * C) if want16 else None
            oT = bf16_buf(C * Rp) if wantT else None
            call("pllb_debug_train_cast_transpose", ptr(d16 if src_bf16 else d32), int(src_bf16), R, C, Rp, ptr(o16), ptr(oT))
            if want16:
                assert torch.equal(o16[:R * C].cpu().reshape(R, C), exp16) and untouched(o16, R * C)
            if wantT:
                assert torch.equal(oT[:C * Rp].cpu().reshape(C, Rp), expT) and untouched(oT, C * Rp)


# ------------------------------------------------------------------------------------------------ GELU
def gelu_ref(x):
    x = torch.as_tensor(x, dtype=torch.float64)
    c = 0.5 * (1 + torch.erf(x / math.sqrt(2)))
    return x * c, c + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


@gpu_test
def test_gelu_forward_and_backward():
    """gelu_fwd (bf16 and fp32 outputs) and gelu_bwd (dg *= GELU'(f)) against the float64 erf form, on a grid with
    +-0, +-1e-3, +-3, +-10, +-30 and random values."""
    rng = np.random.default_rng(3)
    special = np.array([0.0, -0.0, 1e-3, -1e-3, 1, -1, 3, -3, 10, -10, 30, -30], np.float32)
    f = np.concatenate([special, np.linspace(-12, 12, 50001, dtype=np.float32), rng.normal(0, 3, 50000).astype(np.float32)])
    f = bf16r(f).numpy()
    n = len(f)
    fwd, grad = gelu_ref(f)
    dg0 = bf16r(rng.normal(0, 1, n))
    d_f = f32_buf(n, torch.from_numpy(f))
    o16, o32, dg = bf16_buf(n), f32_buf(n), f32_buf(n, dg0)
    call("pllb_debug_train_gelu", ptr(d_f), n, ptr(o16), ptr(o32), ptr(dg))
    assert untouched(o16, n) and untouched(o32, n) and untouched(dg, n)
    g32, g16, gdg = host(o32, n), host(o16, n), host(dg, n)
    e32 = ((g32 - fwd).abs() / (fwd.abs() + 1)).numpy()
    e16 = ((g16 - fwd).abs() - torch.from_numpy(half_ulp_bf16(fwd.numpy()))).numpy() / (np.abs(fwd.numpy()) + 1)
    edg = ((gdg - dg0 * grad).abs() / ((dg0 * grad).abs() + dg0.abs() + 1e-300)).numpy()
    print(f"[gelu] fwd32 {e32.max():.2e} fwd16 {e16.max():.2e} bwd {edg.max():.2e}")
    assert e32.max() <= GELU_REL and e16.max() <= GELU_REL and edg.max() <= GELU_REL
    assert np.signbit(g32[1].item()) == np.signbit(np.float32(-0.0) * 0.5)       # -0 stays a zero
    assert float(g32[0]) == 0 and float(g32[1]) == 0


# ------------------------------------------------------------------------------------------------ long-K GEMMs
GEMM_C = 48.0        # |error| <= GEMM_C * 2^-23 * (|A| @ |W|^T); measured 11.8 (K = 16384), 6.8 (K = 4096)


@gpu_test
@pytest.mark.parametrize("K", [4096, 16384])
def test_weight_gradient_gemm_shapes(K):
    """The tcgen05 GEMM at the shapes of the weight-gradient GEMMs (dW [N_out, K_in] = dY^T . X over the padded rows K):
    M in {768, 3072, 21248} (hidden, intermediate, padded vocabulary), N in {768, 1024}, K = 4096 and 16384 rows.  Each
    element against float64 (computed on the device), bounded by fp32 accumulation over K terms."""
    from asr_rescoring_b200 import engine
    g = torch.Generator(device=DEV).manual_seed(K)
    for M in (768, 3072, 21248):
        for N in (768, 1024):
            A = torch.randn(M, K, device=DEV, generator=g).bfloat16()
            W = torch.randn(N, K, device=DEV, generator=g).bfloat16()
            bias = torch.zeros(N, device=DEV)
            out = engine.debug_gemm(A, W, bias, 2).double()
            ref = A.double() @ W.double().t()
            mag = A.double().abs() @ W.double().abs().t()
            c = float(((out - ref).abs() / (2.0 ** -23 * mag)).max())
            print(f"[gemm M={M} N={N} K={K}] max |error| / (2^-23 |A||W|^T) = {c:.3f}")
            assert c <= GEMM_C, (M, N, K, c)
            del A, W, out, ref, mag
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ rejections
@gpu_test
def test_hooks_reject_bad_arguments():
    """Each hook refuses bad scalars, null pointers and out-of-range device indices with PLLB_ERR_INVALID and launches
    nothing (the output keeps its sentinel)."""
    B, T, H, NH = 2, 8, 256, 4
    qkv, dctx = bf16_buf(B * T * 3 * H, bf16r(np.zeros((B * T, 3 * H)))), f32_buf(B * T * H, torch.zeros(B * T * H))
    nv_ok = torch.tensor([T, 1], dtype=torch.int32, device=DEV)
    seed = seed_buf()

    def attn(nv=nv_ok, B_=B, T_=T, H_=H, p=0.1, seed_=seed, qkv_=qkv, qoff=0, doff=0):
        ctx, lse, dqkv, D = bf16_buf(B * T * H), f32_buf(B * T * NH), f32_buf(B * T * 3 * H), f32_buf(B * T * NH)
        rc = call("pllb_debug_train_attn", ptr(qkv_, qoff), ptr(nv), B_, T_, H_, ptr(dctx), ptr(seed_), p, 2, ptr(ctx),
                  ptr(lse), ptr(dqkv, doff), ptr(D), rc=None)
        return rc, untouched(ctx, 0, B * T * H)
    assert attn() == (0, False)
    for kw in (dict(nv=torch.tensor([0, 1], dtype=torch.int32, device=DEV)), dict(nv=torch.tensor([T + 1, 1], dtype=torch.int32, device=DEV)),
               dict(H_=320), dict(H_=128), dict(T_=0), dict(T_=513), dict(B_=0), dict(p=1.0), dict(p=-0.1), dict(seed_=None),
               dict(qkv_=None), dict(nv=None), dict(qoff=4), dict(doff=1)):      # misaligned: qkv by 8 bytes, dqkv by 4
        assert attn(**kw) == (1, True), kw

    def s2s(causal=1, Tq=T, Tk=T, ldq=3 * H, ldkv=3 * H, lddq=3 * H, NH_=NH, nv=None, p=0.0, koff=0, dkoff=0):
        ctx, lse, d, D = bf16_buf(B * T * H), f32_buf(B * T * NH), f32_buf(B * T * 3 * H), f32_buf(B * T * NH)
        rc = call("pllb_debug_s2s_attn", ptr(qkv), ptr(qkv, H + koff), ptr(qkv, 2 * H), ldq, ldkv, ptr(nv), B, Tq, Tk, NH_,
                  causal, ptr(dctx), ptr(seed), p, 2, ptr(ctx), ptr(lse), ptr(d), lddq, ptr(d, H + dkoff), ptr(d, 2 * H), 3 * H,
                  ptr(D), rc=None)
        return rc, untouched(ctx, 0, B * T * H)
    assert s2s() == (0, False) and s2s(causal=0, nv=nv_ok) == (0, False)
    for kw in (dict(Tq=4), dict(ldkv=3 * H + 4), dict(ldq=3 * H + 2), dict(lddq=H - 2), dict(NH_=5), dict(causal=0),
               dict(koff=2), dict(dkoff=1),
               dict(causal=0, nv=torch.tensor([T + 1, 1], dtype=torch.int32, device=DEV)), dict(Tk=600, Tq=600), dict(p=1.5)):
        assert s2s(**kw) == (1, True), kw

    R = 8
    g, x = f32_buf(H, torch.ones(H)), f32_buf(R * H, torch.zeros(R * H))
    ids_bad = torch.tensor([0] * (R - 1) + [50], dtype=torch.int32, device=DEV)

    def ln(form=0, H_=H, R_=R, ids=None, eps=1e-5, T_=4):
        o = f32_buf(R * H)
        rc = call("pllb_debug_train_ln_fwd", form, ptr(x), None, ptr(ids), T_, ptr(x), 50, ptr(x), ptr(x), 1.0, ptr(g), ptr(g),
                  eps, R_, H_, None, 0.0, 0, ptr(o), None, None, None, rc=None)
        return rc, untouched(o, 0, R * H)
    assert ln() == (0, False)
    for kw in (dict(form=3), dict(H_=384), dict(R_=0), dict(eps=0.0), dict(form=1, ids=ids_bad), dict(form=1, ids=None),
               dict(form=1, ids=torch.zeros(R, dtype=torch.int32, device=DEV), T_=513)):
        assert ln(**kw) == (1, True), kw
    dz = f32_buf(R * H)
    assert call("pllb_debug_train_ln_bwd", ptr(x), None, ptr(g), ptr(x), ptr(g), R, 200, None, 0.0, -1, -1, ptr(dz), None, rc=None) == 1
    assert call("pllb_debug_train_ln_bwd", ptr(x), None, ptr(g), ptr(x), ptr(g), R, H, None, 0.5, -1, 3, ptr(dz), None, rc=None) == 1
    assert untouched(dz, 0, R * H)

    V, Vp = 300, 512
    logits = f32_buf(R * Vp, torch.zeros(R * Vp))

    def ce(lab, ignore=0, V_=V, Vp_=Vp):
        lr, out, d_lab = f32_buf(R), f32_buf(2), torch.tensor(lab, dtype=torch.int32, device=DEV)
        rc = call("pllb_debug_train_ce", ptr(logits), ptr(d_lab), R, V_, Vp_, ignore, ptr(lr), None, ptr(out), rc=None)
        return rc, untouched(lr, 0, R)
    assert ce([0] * R) == (0, False) and ce([-100] * (R - 1) + [3], 1) == (0, False)
    for args in (([0] * (R - 1) + [V],), ([0] * (R - 1) + [-100],), ([-100] * R, 1), ([-1] + [0] * (R - 1), 1), ([0] * R, 0, V, V - 1)):
        assert ce(*args) == (1, True), args

    def emb(ids, form=0, pos_rows=T, H_=H):
        dpos, dword, dtype0 = f32_buf(pos_rows * H), f32_buf(50 * H), f32_buf(H)
        rc = call("pllb_debug_train_embed_bwd", form, ptr(x), ptr(ids), 1, T, H_, pos_rows, 0, 1.0, ptr(dword), 50,
                  ptr(dpos), ptr(dtype0), None, rc=None)
        return rc, untouched(dpos, 0, max(pos_rows, 1) * H)
    ok_ids = torch.zeros(T, dtype=torch.int32, device=DEV)
    assert emb(ok_ids) == (0, False)
    for kw in (dict(ids=ids_bad), dict(ids=ok_ids, form=2), dict(ids=ok_ids, pos_rows=T - 1), dict(ids=ok_ids, H_=96)):
        assert emb(**kw) == (1, True), kw

    o = f32_buf(H)
    assert call("pllb_debug_train_colsum", ptr(x), 0, None, 0, H, ptr(o), None, None, rc=None) == 1
    assert call("pllb_debug_train_colsum", ptr(x), 0, None, R, H, ptr(o), ptr(o), None, rc=None) == 1     # out_dot needs xhat
    assert untouched(o, 0, H)
    t16 = bf16_buf(R * H)
    assert call("pllb_debug_train_cast_transpose", ptr(x), 0, R, H, R - 1, None, ptr(t16), rc=None) == 1
    assert call("pllb_debug_train_cast_transpose", ptr(x), 0, R, H, R, None, None, rc=None) == 1
    assert call("pllb_debug_train_gelu", ptr(x), 0, ptr(t16), None, None, rc=None) == 1
    assert call("pllb_debug_train_gelu", None, R, ptr(t16), None, None, rc=None) == 1
    assert untouched(t16, 0, R * H)


# ------------------------------------------------------------------------------------------------ witnesses (CPU)
# Each plausible bug moves the float64 reference by more than its family's bound, in the metric the GPU test of that
# family applies, on most of the rows it affects, so the GPU tests above would see it.  A transpose without the zero
# fill needs no witness here: test_cast_transpose_is_bit_exact sees it directly (its docstring says how).
def _attn_case(B, T, NH, n_valid, seed=0):
    rng = np.random.default_rng(seed)
    q, k, v, dctx = (torch.from_numpy(rng.normal(0, 1.5, (B, NH, T, 64))) for _ in range(4))
    return q, k, v, dctx


def seen(good, bad, NH):
    """The per-row metrics check_attn_outputs applies, with the float64 results of a buggy kernel (`bad`, its ctx rounded
    to bf16 as the kernel stores it) in place of the device's: how far each row is past its bound."""
    g, b = ref_rows(good, NH), ref_rows(bad, NH)
    mq, mk, mv, mD = g[6]
    return {"ctx": bf16_row_excess(bf16r(b[0].numpy()), g[0]) / ATT_REL,
            "lse": (b[1] - g[1]).abs().amax(1).numpy() / ATT_LSE,
            "dq": row_rel_mag(b[2], g[2], mq) / ATT_REL, "dk": row_rel_mag(b[3], g[3], mk) / ATT_REL,
            "dv": row_rel_mag(b[4], g[4], mv) / ATT_REL, "D": row_rel_mag(b[5], g[5], mD) / ATT_REL}


def test_witness_keys_capped_at_32():
    B, T, NH = 2, 65, 4
    n_valid = np.array([T, 40])
    q, k, v, dctx = _attn_case(B, T, NH, n_valid)
    vis, M = attn_masks(B, NH, T, T, n_valid, False, SEED, 2, 0.0)
    capped = vis & (torch.arange(T) < 32)
    e = seen(attn_ref(q, k, v, vis, M, dctx), attn_ref(q, k, v, capped, M, dctx), NH)
    keys_below_32 = np.tile(np.arange(T) < 32, B)          # keys >= 32 lose their gradient altogether
    for name, x in e.items():
        rows = keys_below_32 if name in ("dk", "dv") else slice(None)
        assert (x[rows] > 1).mean() > 0.9, (name, np.median(x[rows]))


def test_witness_causal_limit_i_instead_of_i_plus_1():
    B, T, NH = 1, 40, 4
    q, k, v, dctx = _attn_case(B, T, NH, None, 1)
    vis, M = attn_masks(B, NH, T, T, None, True, SEED, 2, 0.0)
    short = vis & ~torch.eye(T, dtype=torch.bool)
    short[..., 0, 0] = True           # row 0 would see no key at all; keep it so the softmax stays defined
    e = seen(attn_ref(q, k, v, vis, M, dctx), attn_ref(q, k, v, short, M, dctx), NH)
    for name in ("ctx", "lse", "dq", "D"):
        assert (e[name][1:] > 1).mean() > 0.9, (name, np.median(e[name][1:]))


def test_witness_cross_dropout_index_with_tq_for_tk():
    B, Tq, Tk, NH, p = 2, 33, 65, 4, 0.1
    rng = np.random.default_rng(2)
    q = torch.from_numpy(rng.normal(0, 1.5, (B, NH, Tq, 64)))
    k, v = (torch.from_numpy(rng.normal(0, 1.5, (B, NH, Tk, 64))) for _ in range(2))
    dctx = torch.from_numpy(rng.normal(0, 1, (B, NH, Tq, 64)))
    n_valid = np.array([Tk, 50])
    vis, M = attn_masks(B, NH, Tq, Tk, n_valid, False, SEED, 5, p)
    bh, i, j = np.meshgrid(np.arange(B * NH), np.arange(Tq), np.arange(Tk), indexing="ij")
    wrong = ((bh * Tq + i) * Tq + j).astype(np.uint64)
    Mw = torch.from_numpy(drop_factor(SEED, 5, wrong.reshape(-1), p).reshape(B, NH, Tq, Tk))
    e = seen(attn_ref(q, k, v, vis, M, dctx), attn_ref(q, k, v, vis, Mw, dctx), NH)
    live_keys = np.concatenate([np.arange(Tk) < n for n in n_valid])      # masked keys: dk = dv = 0 exactly either way
    for name in ("ctx", "dq", "dk", "dv"):                # the log-sum-exp does not see the dropout mask
        x = e[name][live_keys] if name in ("dk", "dv") else e[name]
        assert (x > 1).mean() > 0.9, (name, np.median(x))


def test_witness_layernorm_variance_over_h_minus_1():
    rng = np.random.default_rng(4)
    for H in LN_H:
        z = torch.from_numpy(rng.normal(0, 1, (5, H)))
        a, b = ln_ref(z, 1.0, 0.0, 1e-12)[0], ln_ref(z, 1.0, 0.0, 1e-12, biased=False)[0]
        assert row_rel(b.numpy(), a.numpy()).min() > 10 * LN_REL, H


def test_witness_softmax_over_pad_columns():
    B, T, NH = 2, 33, 4
    n_valid = np.array([20, 1])
    q, k, v, dctx = _attn_case(B, T, NH, n_valid, 5)
    vis, M = attn_masks(B, NH, T, T, n_valid, False, SEED, 2, 0.0)
    e = seen(attn_ref(q, k, v, vis, M, dctx), attn_ref(q, k, v, torch.ones_like(vis), M, dctx), NH)
    for name in ("ctx", "lse", "dq", "D"):
        assert (e[name] > 1).mean() > 0.9, (name, np.median(e[name]))


def test_witness_word_gradient_with_the_pad_id():
    rng = np.random.default_rng(6)
    ids = rng.integers(0, 10, 200)
    ids[::7] = 0
    dz = torch.from_numpy(rng.normal(0, 1, (200, 256)))
    dword0 = torch.from_numpy(rng.normal(0, 1, (10, 256)))
    good, bad = dword0.clone(), dword0.clone()
    good.index_add_(0, torch.as_tensor(ids[ids != 0]), dz[torch.as_tensor(ids != 0)])
    bad.index_add_(0, torch.as_tensor(ids), dz)
    assert row_rel(bad[:1].numpy(), good[:1].numpy()).min() > 1000 * EMB_REL


def test_dropout_restatement_keeps_the_rate():
    """The numpy restatement of drop_factor keeps a fraction 1 - p of the elements (a check of the restatement, not of
    the kernels, which the tests above compare with it exactly)."""
    for p in (0.1, 0.5):
        f = drop_factor(SEED, 3, np.arange(200000, dtype=np.uint64), p)
        assert abs((f == 0).mean() - p) < 0.005
        assert set(np.unique(f)) == {0.0, drop_params(p)[1]}
