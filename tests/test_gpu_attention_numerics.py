"""Attention numerics: the tcgen05 kernels against a float64 reference, element by element, with first-order error bounds.

test_gpu_attention.py compares with the fp32 CPU oracle under global norms on unit-scale random inputs.  Those inputs never make
the lazy rescale of O fire with a non-zero O (scores spread ~1.4 log2 units, the threshold is 8), and a global norm cannot see a
single leaked or dropped key.  Here every output element, lse entry and gradient element is held to its own bound (see
``_fwd_ref`` and ``_bwd_ref``), on input regimes built to reach the code those tests cannot:

  diffuse   unit-scale random q, k, v: the control.
  qknorm<w> q / k rows of RMS w (what the QKV epilogue's RMSNorm with weight w produces) around a shared direction: sharp rows
            with a few dominant keys, not one-hot ones.
  late_max  every query row meets a larger score in every later key tile -- rises of ~7.9 and ~8.1 log2 units, on both sides of
            the kernels' RESCALE_THRESHOLD = 8, and larger ones -- up to the last, partial tile, so O is rescaled while non-zero
            and P gets close to 2^8.
  uniform   q = 0: the output is the mean of V over the visible keys; a key too many or too few shows directly.
  poison    keys the kernel must not see (past kv_len, the next image's rows after a partial last tile, the packed layout's pad
            rows, |i - j| = w + 1 for a window) score ~30 nats above every visible key and carry large V: any leak dominates.
            In the backward pass the rows that must be ignored also carry large dO and a wrong, finite lse / delta.

Layouts: dense (flash), prefix key lengths (zero_invalid_rows), sliding window, and packed NaFlex rows (pack_plan / pack_rows /
attention_packed / vtk_attention_bwd_packed_bf16); head_dim 64 (persistent kernel) and 128 (one-shot two-tile kernel).
The last test reruns the d = 64 forward on persistent grids of 2, 3 and 37 SMs ("reserve_sms"), where every CTA walks many work
items, and requires bit-identical output and lse."""
import math
import os
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
F64 = torch.float64
U = 2.0 ** -8                # unit roundoff of bf16 (8 significant bits, round to nearest)
E32 = 2.0 ** -24             # unit roundoff of fp32
LOG2E = 1.0 / math.log(2.0)
LN2 = math.log(2.0)
# Calibrated on a B200 (1000 W power limit): the largest error / (first-order bound with c = 1) over every case of this file was
# 0.90 for the forward output (late_max, d = 64, N = 1000), 0.05 for lse (whose bound sums worst-case fp32 terms), and 0.93 / 0.34
# / 0.32 for dv / dk / dq.  c = 1.5 leaves room for the worst case of the rounding the bounds describe, not for a second source of
# error: a kernel that skips the O rescale or lets one masked key through exceeds them by orders of magnitude.
C_FWD = 1.5
C_LSE = 1.5
C_BWD = 1.5
HEADS = 2
NS = [1, 127, 128, 129, 255, 257, 1000, 4096]
WINDOWS = [0, 1, 127, 128, 129, None]      # None: a window >= N (every key visible)
REGIMES = ["diffuse", "qknorm1", "qknorm2", "qknorm3", "late_max", "uniform", "poison"]
DEV = "cuda"                 # where the float64 reference runs
SENT = -12288.0              # sentinel of output / lse / gradient buffers (exact in bf16 and fp32)
POISON_V = 1024.0            # |V| of rows the kernel must not read
# late_max: rises of the per-tile max in log2 units at the nominal row amplitude; each row's amplitude is jittered by +-3 %, so the
# 7.9 / 8.1 rises land on both sides of the threshold for different rows, and a 3.0 rise fires only once the stale max falls behind
LATE_RISES = [7.9, 8.1, 12.0, 3.0, 7.9, 8.1, 5.0, 20.0]


@pytest.fixture(scope="module")
def L():
    from vitok_b200 import _lib
    _lib.load()
    return _lib


# ------------------------------------------------------------------------------------------------------------------------------
# input regimes: q, k, v as [B, N, heads, d] float32 holding bf16 values; rows >= lens[b] are rows image b must not attend to
# ------------------------------------------------------------------------------------------------------------------------------
def _bf(x):
    return x.to(BF).float()


def _unit(x):
    return torch.nn.functional.normalize(x, dim=-1)


def _gen(regime, lens, N, d, seed):
    g = torch.Generator().manual_seed(seed)
    B, H = len(lens), HEADS

    def randn(*s):
        return torch.randn(*s, generator=g)

    shape = (B, N, H, d)
    inv = torch.arange(N)[None, :] >= torch.tensor(lens)[:, None]        # [B, N] rows past each image's valid tokens
    v = randn(*shape)
    if regime == "diffuse":
        return _bf(randn(*shape)), _bf(randn(*shape)), _bf(v)
    if regime.startswith("qknorm"):
        w = float(regime[6:])
        u = _unit(randn(H, d))

        def rows():
            return w * math.sqrt(d) * _unit(u + _unit(randn(*shape)))
        q, k = rows(), rows()
        k[inv] = 4.0 * k[inv]
    elif regime == "late_max":
        sc = LOG2E / math.sqrt(d)
        u = _unit(randn(H, d))

        def perp(x):                                   # the part of x orthogonal to u
            return x - (x * u).sum(-1, keepdim=True) * u
        amp = 2.0 * math.sqrt(d) * (1.0 + 0.03 * (2.0 * torch.rand(B, N, H, 1, generator=g) - 1.0))
        q = amp * u + perp(randn(*shape))              # background scores ~ N(0, 1.44^2) log2 units
        k = perp(randn(*shape))
        level = 6.0                                    # the spike of tile 0 sits above its background
        for b, n in enumerate(lens):
            for t in range((n + 127) // 128):
                if t > 0:
                    level += LATE_RISES[(t - 1) % len(LATE_RISES)]
                width = min(128, n - 128 * t)
                j = 128 * t + (37 * t + 11) % width
                k[b, j] = (level / (sc * 2.0 * math.sqrt(d))) * u
            level = 6.0
        k[inv] = 4.0 * randn(int(inv.sum()), H, d)
    elif regime == "uniform":
        q, k = torch.zeros(shape), randn(*shape)
    elif regime == "poison":
        # image b's queries point along e[b + 1]; its keys carry e[b] and e[b + 2], the query directions of its neighbours, so that
        # the next image's rows score high for image b (a forward leak past a partial tile) and image b's keys score high for the
        # next image's queries (a backward leak of MODE 0's query rows); its own rows past kv_len carry e[b + 1]
        assert B + 2 <= d // 2
        A, P = 2.0 * math.sqrt(d), 18.0                # A * P / sqrt(d) = 36 nats
        q, k = torch.zeros(shape), torch.zeros(shape)          # visible scores: noise in the upper half, ~N(0, 2) nats
        q[..., d // 2:] = randn(B, N, H, d - d // 2) * math.sqrt(2.0)
        k[..., d // 2:] = randn(B, N, H, d - d // 2) * math.sqrt(2.0)
        e = torch.eye(d)
        for b in range(B):
            q[b] += A * e[b + 1]
            k[b, ~inv[b]] += P * (e[b] + e[b + 2])
            k[b, inv[b]] += P * e[b + 1]
    else:
        raise ValueError(regime)
    if regime != "diffuse":
        v[inv] = POISON_V * torch.sign(randn(int(inv.sum()), H, d))
    return _bf(q), _bf(k), _bf(v)


def _gen_window_poison(B, N, d, w, seed):
    """Scores that depend on the offset i - j only and peak at |i - j| = w + 1, >= 30 nats above every offset inside the window:
    q_i = (cos(f i), sin(f i)), k_j = a (cos(f j), sin(f j)) over d/2 random frequencies f gives q_i . k_j = sum_f a_f cos(f (i - j)),
    and a_f = s cos(f (w + 1)) puts the maximum at the two offsets just outside the window."""
    g = torch.Generator().manual_seed(seed)
    F = d // 2
    f = (0.05 + (math.pi - 0.1) * torch.rand(F, generator=g, dtype=F64))
    a = torch.cos(f * (w + 1))
    off = torch.arange(0, w + 1, dtype=F64)
    inside = (a[None, :] * torch.cos(f[None, :] * off[:, None])).sum(1).max().item()
    gap = (a * a).sum().item() - inside
    assert gap > 0.1 * F, gap
    s = 30.0 * math.sqrt(d) / gap
    pos = torch.arange(N, dtype=F64)[:, None] * f[None, :]
    q = torch.cat([torch.cos(pos), torch.sin(pos)], 1)
    k = torch.cat([torch.cos(pos), torch.sin(pos)], 1) * torch.cat([a, a]) * s
    q = q[None, :, None, :].expand(B, N, HEADS, d).float()
    k = k[None, :, None, :].expand(B, N, HEADS, d).float()
    return _bf(q), _bf(k), _bf(torch.randn(B, N, HEADS, d, generator=g))


def _inputs(regime, lens, N, d, seed, window=None):
    if regime == "poison" and window is not None and window < N:
        return _gen_window_poison(len(lens), N, d, window, seed)
    return _gen(regime, lens, N, d, seed)


def _qkv(q, k, v):
    B, N, H, d = q.shape
    return torch.cat([t.reshape(B * N, H * d) for t in (q, k, v)], 1).to(BF).cuda()


# ------------------------------------------------------------------------------------------------------------------------------
# float64 reference and bounds
# ------------------------------------------------------------------------------------------------------------------------------
def _scores2(q, k, w, q0=0):
    """[H, m, n] scores q k^T / sqrt(d) in log2 units for query rows q0 .. q0+m-1 against keys 0 .. n-1, -inf outside the window."""
    s = torch.matmul(q, k.transpose(-1, -2)) * (LOG2E / math.sqrt(q.shape[-1]))
    if w is not None:
        i = torch.arange(q0, q0 + q.shape[-2], device=q.device)[:, None]
        j = torch.arange(k.shape[-2], device=q.device)[None, :]
        s = s.masked_fill((i - j).abs() > w, float("-inf"))
    return s


def _fwd_ref(q, k, v, w=None, chunk=1024):
    """Reference of one image: q [m, H, d] (query rows 0..m-1), k / v [n, H, d] the keys it may see (n >= 1), window w or None.

    Returns o, b_o, lse2, tau with o [m, H, d] = softmax(q k^T / sqrt(d)) v and lse2 [m, H] = log2 sum_j 2^(s_ij), s in log2 units,
    all in float64 on the bf16 input values, and the first-order bounds of the kernels' errors:

    The kernels compute s in fp32 on the tensor core, p_ij = ex2.approx(s_ij - m_i) against a running (lazy) max, l_i = sum p_ij
    in fp32 from the unrounded p, O_i = sum bf16(p_ij) v_j in fp32, and o_i = bf16(O_i / l_i).  Let tau_i bound the error, in log2
    units, of every exponent s_ij - m_i (and of lse):
        tau_i = sc d 2^-24 |q_i| max_j|k_j|        fp32 dot product of length d (|sum a_k b_k| error <= d eps sum|a_k b_k|)
              + log2(e) (2^-22 + n 2^-24)          ex2.approx's relative error; fp32 sum of n terms in l
              + 2^-23 (max_j|s_ij| + |lse_i|)      the FFMA s * sc - m and the final m + log2(l)
    so every p carries a relative error e_i = ln(2) tau_i before it is rounded to bf16 (relative error u = 2^-8).  To first order
        o_i - o_ref_i = sum_j (P~_ij - p_ij) / l_i v_j - o_ref_i (l_i - l_ref_i) / l_ref_i + rounding of o
    and the terms are bounded by (u + e_i) sum_j p_ij |v_j|, e_i |o_ref_i| and u |o_ref_i|:
        |o - o_ref| <= c_fwd ((u + e_i) sum_j p_ij |v_j| + (u + e_i) |o_ref_i|) + 2^-24 max|v|
    (sum_j p |v| is one more float64 product, with |V|).  The lazy max changes nothing here: p <= 2^8 is rounded to bf16 with the
    same relative error, and the rescale of O by alpha = 2^(m_old - m_new) is one more fp32 rounding.  The lse bound is c_lse tau_i.
    A kernel that skips the O rescale or leaks one key misses this bound by orders of magnitude (it is ~u of the output scale)."""
    H, d = q.shape[1], q.shape[2]
    sc = LOG2E / math.sqrt(d)
    qh, kh, vh = (t.to(device=DEV, dtype=F64).transpose(0, 1) for t in (q, k, v))      # [H, rows, d]
    kmax = kh.norm(dim=-1).amax(-1)                                                        # [H]
    n = kh.shape[1]
    o, pav, lse, tau = [], [], [], []
    for c0 in range(0, qh.shape[1], chunk):
        qc = qh[:, c0:c0 + chunk]
        s = _scores2(qc, kh, w, c0)
        ls = torch.logsumexp(s * LN2, -1) * LOG2E                                          # [H, m]
        p = torch.exp2(s - ls[..., None])
        o.append(p @ vh)
        pav.append(p @ vh.abs())
        lse.append(ls)
        smax = s.masked_fill(torch.isinf(s), 0.0).abs().amax(-1)
        tau.append(sc * d * E32 * qc.norm(dim=-1) * kmax[:, None] + LOG2E * (2.0 ** -22 + n * E32) + 2 * E32 * (smax + ls.abs()))
    o, pav, lse, tau = (torch.cat(t, 1) for t in (o, pav, lse, tau))
    e = LN2 * tau[..., None]
    b_o = (U + e) * (pav + o.abs()) + E32 * vh.abs().max()
    return o.transpose(0, 1), b_o.transpose(0, 1), lse.transpose(0, 1), tau.transpose(0, 1)


def _bwd_ref(q, k, v, do, b_o, tau, w=None, chunk=1024):
    """Gradients of one image (q [m, H, d] query rows, k / v [n, H, d] visible keys, do [m, H, d]) and their first-order bounds.

    The kernels form P = ex2(s * sc - lse) with the forward kernel's lse and delta_i = sum_d dO_i O_i over the forward kernel's bf16
    O (as the training step does), then dS = P (dP - delta) / sqrt(d) with dP = dO V^T in fp32, and accumulate in fp32
    dV = bf16(P)^T dO, dK = bf16(dS)^T Q, dQ = bf16(dS) K.  Replacing every rounded quantity by u times its magnitude:
      P     relative error u (bf16) + e_i = ln(2) tau_i (the exponent: S in fp32, lse of the forward, ex2.approx)
      delta |delta - delta_ref| <= D_i = sum_d |dO_i| b_o_i + d 2^-24 (|dO_i| . |O_i| + |dO_i| max_j|v_j|)
            (the forward output's own bound; fp32 sums of delta and dP)
      dS    |dS~ - dS| <= (u + e_i) |dS_ij| + P_ij D_i / sqrt(d)          (p unrounded in dS; dS rounded to bf16)
      grad  + u |grad| (the bf16 store)
    so that
      |dV_j - ref| <= P^T ((u + e) |dO|) + u |dV_j|
      |dQ_i - ref| <= (u + e_i) (|dS| |K|)_i + D_i (P |K|)_i / sqrt(d) + u |dQ_i|
      |dK_j - ref| <= (|dS|^T ((u + e) |Q|))_j + (P^T (D |Q|))_j / sqrt(d) + u |dK_j|
    and each gradient is held to c_bwd times its bound, plus 2^-24 of its largest magnitude."""
    H, d = q.shape[1], q.shape[2]
    scale = 1.0 / math.sqrt(d)
    qh, kh, vh, dh = (t.to(device=DEV, dtype=F64).transpose(0, 1) for t in (q, k, v, do))
    bo = b_o.transpose(0, 1)
    ee = U + LN2 * tau.transpose(0, 1)                                                     # [H, m]
    vmax = vh.norm(dim=-1).amax(-1)
    dq, bdq = [], []
    dk = torch.zeros_like(kh); dv = torch.zeros_like(kh); bdk = torch.zeros_like(kh); bdv = torch.zeros_like(kh)
    for c0 in range(0, qh.shape[1], chunk):
        qc, dc, ec = qh[:, c0:c0 + chunk], dh[:, c0:c0 + chunk], ee[:, c0:c0 + chunk]
        s = _scores2(qc, kh, w, c0)
        p = torch.exp2(s - (torch.logsumexp(s * LN2, -1) * LOG2E)[..., None])
        o = p @ vh
        delta = (dc * o).sum(-1)
        D = (dc.abs() * bo[:, c0:c0 + chunk]).sum(-1) + d * E32 * ((dc.abs() * o.abs()).sum(-1) + dc.norm(dim=-1) * vmax[:, None])
        dp = dc @ vh.transpose(-1, -2)
        ds = p * (dp - delta[..., None]) * scale
        dq.append(ds @ kh)
        bdq.append(ec[..., None] * (ds.abs() @ kh.abs()) + D[..., None] * (p @ kh.abs()) * scale)
        dv += p.transpose(-1, -2) @ dc
        dk += ds.transpose(-1, -2) @ qc
        bdv += p.transpose(-1, -2) @ (ec[..., None] * dc.abs())
        bdk += ds.abs().transpose(-1, -2) @ (ec[..., None] * qc.abs()) + p.transpose(-1, -2) @ (D[..., None] * qc.abs()) * scale
    dq, bdq = torch.cat(dq, 1), torch.cat(bdq, 1)
    out = []
    for g_, b_ in ((dq, bdq), (dk, bdk), (dv, bdv)):
        out += [g_.transpose(0, 1), (b_ + U * g_.abs()).transpose(0, 1)]
    return out


class Worst:
    """Largest error / bound seen by a test per checked quantity (the last word of the tag: out, lse, dq, dk, dv), for the log."""

    def __init__(self, name):
        self.name, self.worst = name, {}

    def check(self, tag, got, ref, bound, c):
        """got, ref, bound: same shape (got any float dtype).  Asserts |got - ref| <= c * bound everywhere."""
        got = got.to(F64)
        assert bool(torch.isfinite(got).all()), f"{self.name} {tag}: non-finite values"
        err = (got - ref.to(F64)).abs()
        ratio = err / bound.clamp_min(1e-300)
        i = int(ratio.argmax())
        r = float(ratio.flatten()[i])
        kind = tag.split()[-1]
        if r >= self.worst.get(kind, (-1.0, ""))[0]:
            self.worst[kind] = (r, tag)
        assert r <= c, (f"{self.name} {tag}: error {float(err.flatten()[i]):.4e} = {r:.3g} x its bound {float(bound.flatten()[i]):.4e} "
                        f"(allowed {c}) at flat index {i}: got {float(got.flatten()[i]):.6g}, ref {float(ref.flatten()[i]):.6g}")
        return r

    def report(self):
        print(f"[numerics] {self.name}: worst error/bound " + ", ".join(f"{k} {r:.3f} ({t})" for k, (r, t) in self.worst.items()))


def _check_fwd(wst, tag, out_rows, lse_rows, q, k, v, w=None):
    """out_rows [m, H*d] bf16, lse_rows [m, H] of one image whose query rows are q (m rows) and visible keys k / v."""
    o, b_o, lse, tau = _fwd_ref(q, k, v, w)
    m, H, d = q.shape
    wst.check(f"{tag} out", out_rows.view(m, H, d), o, b_o, C_FWD)
    wst.check(f"{tag} lse", lse_rows, lse, tau, C_LSE)
    return b_o, tau


def _lens(N):
    """A prefix / packed batch: a full image, an empty one, a one-token one and two partial ones."""
    return [N, 0, 1, (N + 1) // 2, max(N - 3, 1)]


def _mask(lens, N):
    m = torch.zeros(len(lens), N, dtype=torch.bool)
    for b, n in enumerate(lens):
        m[b, :n] = True
    return m


def _seed(*parts):
    return zlib.crc32(repr(parts).encode()) & 0x7FFFFFFF


# ------------------------------------------------------------------------------------------------------------------------------
# forward
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_forward_dense(L, d, regime):
    """No mask, two images: every query row sees its image's N keys; after a partial last tile the next image's rows follow."""
    wst = Worst(f"fwd dense d={d} {regime}")
    for N in NS:
        B = 2
        q, k, v = _inputs(regime, [N] * B, N, d, seed=_seed("dense", d, regime, N))
        lse = torch.full((B * N, HEADS), SENT, device="cuda")
        out = L.attention(_qkv(q, k, v), B, N, HEADS, d, None, lse=lse)
        for b in range(B):
            _check_fwd(wst, f"N={N} img {b}", out[b * N:(b + 1) * N], lse[b * N:(b + 1) * N], q[b], k[b], v[b])
    wst.report()


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_forward_prefix(L, d, regime):
    """Prefix key lengths (images of N, 0, 1 and partial valid tokens); query rows past kv_len are exactly 0 with lse = +inf."""
    wst = Worst(f"fwd prefix d={d} {regime}")
    for N in NS:
        lens = _lens(N)
        B = len(lens)
        q, k, v = _inputs(regime, lens, N, d, seed=_seed("prefix", d, regime, N))
        lse = torch.full((B * N, HEADS), SENT, device="cuda")
        out = L.attention(_qkv(q, k, v), B, N, HEADS, d, _mask(lens, N).cuda(), lse=lse)
        for b, n in enumerate(lens):
            r0 = b * N
            if n:
                _check_fwd(wst, f"N={N} img {b} (kv_len {n})", out[r0:r0 + n], lse[r0:r0 + n], q[b, :n], k[b, :n], v[b, :n])
            assert bool((out[r0 + n:r0 + N] == 0).all()), (N, b, "rows past kv_len must be 0")
            assert bool((lse[r0 + n:r0 + N] == float("inf")).all()), (N, b, "rows past kv_len must have lse +inf")
    wst.report()


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_forward_window(L, d, regime):
    """Sliding window |i - j| <= w for w in 0, 1, 127, 128, 129 and >= N."""
    wst = Worst(f"fwd window d={d} {regime}")
    for N in NS:
        for w in WINDOWS:
            w = N + 7 if w is None else w
            B = 1
            q, k, v = _inputs(regime, [N] * B, N, d, seed=_seed("window", d, regime, N, w), window=w)
            lse = torch.full((B * N, HEADS), SENT, device="cuda")
            out = L.attention(_qkv(q, k, v), B, N, HEADS, d, None, window=w, lse=lse)
            _check_fwd(wst, f"N={N} w={w}", out, lse, q[0], k[0], v[0], w)
    wst.report()


def _packed_inputs(L, regime, lens, N, d, seed, qrows):
    """The padded batch, its pack plan and the packed qkv, whose pad rows (which no kernel may read) are poisoned."""
    q, k, v = _inputs(regime, lens, N, d, seed)
    B = len(lens)
    plan = L.pack_plan(_mask(lens, N).cuda(), 16, qrows)
    pk = L.pack_rows(_qkv(q, k, v).view(B, N, -1), plan)
    cu, nv = plan["cu"].cpu().tolist(), plan["n_valid"].cpu().tolist()
    assert nv == list(lens)
    if regime != "diffuse":
        D = HEADS * d
        g = torch.Generator().manual_seed(seed + 1)
        for b in range(B):
            r0, r1 = cu[b] + nv[b], cu[b + 1]
            if r1 > r0:
                pk[r0:r1, :2 * D] = (8.0 * torch.randn(r1 - r0, 2 * D, generator=g)).to(BF).cuda()
                pk[r0:r1, 2 * D:] = POISON_V * torch.sign(torch.randn(r1 - r0, D, generator=g)).to(BF).cuda()
    return q, k, v, plan, pk, cu, nv


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_forward_packed(L, d, regime):
    """Packed NaFlex rows (qrows 128 for d = 64, 256 for d = 128), with an empty image: valid rows against the reference, the
    images' pad rows exactly 0 with lse +inf, rows past the last image untouched."""
    wst = Worst(f"fwd packed d={d} {regime}")
    for N in NS:
        lens = _lens(N)
        B, D = len(lens), HEADS * d
        q, k, v, plan, pk, cu, nv = _packed_inputs(L, regime, lens, N, d, _seed("packed", d, regime, N), 128 if d == 64 else 256)
        out = torch.full((pk.shape[0], D), SENT, dtype=BF, device="cuda")
        lse = torch.full((pk.shape[0], HEADS), SENT, device="cuda")
        L.attention_packed(pk, plan, B, N, HEADS, d, lse=lse, out=out)
        for b, n in enumerate(nv):
            if n:
                _check_fwd(wst, f"N={N} img {b} ({n} tokens)", out[cu[b]:cu[b] + n], lse[cu[b]:cu[b] + n], q[b, :n], k[b, :n], v[b, :n])
            assert bool((out[cu[b] + n:cu[b + 1]] == 0).all()) and bool((lse[cu[b] + n:cu[b + 1]] == float("inf")).all()), (N, b)
        assert bool((out[cu[B]:] == SENT).all()) and bool((lse[cu[B]:] == SENT).all()), N
    wst.report()


# ------------------------------------------------------------------------------------------------------------------------------
# backward
# ------------------------------------------------------------------------------------------------------------------------------
def _delta(L, out, do, rows, d):
    delta = torch.zeros(out.shape[0], HEADS, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_attn_delta(out.data_ptr(), out.stride(0), do.data_ptr(), do.stride(0), delta.data_ptr(), rows, HEADS, d,
                                    L.stream_ptr()))
    return delta


def _check_grads(wst, tag, dqkv_rows, q, k, v, do, b_o, tau, w=None):
    """dqkv_rows [n, 3*H*d] of one image whose query rows are q / do and whose visible keys are k / v (same n rows)."""
    n, H, d = q.shape
    g = dqkv_rows.view(n, 3, H, d)
    dq, bdq, dk, bdk, dv, bdv = _bwd_ref(q, k, v, do, b_o, tau, w)
    for i, (nm, ref, bd) in enumerate((("dq", dq, bdq), ("dk", dk, bdk), ("dv", dv, bdv))):
        wst.check(f"{tag} {nm}", g[:, i], ref, bd + E32 * ref.abs().max(), C_BWD)


def _grad_do(lens, N, d, seed, poison):
    """dO: unit-scale where it counts, large (POISON_V / 8) in rows that must not contribute when ``poison``."""
    g = torch.Generator().manual_seed(seed)
    do = torch.randn(len(lens), N, HEADS, d, generator=g)
    if poison:
        inv = torch.arange(N)[None, :] >= torch.tensor(lens)[:, None]
        do[inv] = (POISON_V / 8) * torch.sign(do[inv])
    return _bf(do)


def _bwd_padded(L, qkv, do, lse, delta, kl, B, N, d, zero_invalid, w):
    D = HEADS * d
    dqkv = torch.full((B * N, 3 * D), SENT, dtype=BF, device="cuda")
    b0, g0 = qkv.data_ptr(), dqkv.data_ptr()
    L.check(L.load().vtk_attention_bwd_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, do.data_ptr(), D, lse.data_ptr(), delta.data_ptr(),
                                            g0, g0 + 2 * D, g0 + 4 * D, 3 * D, L.ptr(kl), B, N, HEADS, d, zero_invalid, w, L.stream_ptr()))
    return dqkv


BWD_CASES = ([("dense", N, None) for N in NS] + [("prefix", N, None) for N in NS] +
             [("window", N, w) for N in [127, 129, 1000, 4096] for w in WINDOWS])


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_backward_padded(L, d, regime):
    """vtk_attention_bwd_bf16 with lse and delta from the forward kernel: dense, prefix key lengths (poisoned dO / lse / delta in
    the rows past kv_len, whose dq and whose keys' dk / dv must be exactly 0) and sliding windows."""
    wst = Worst(f"bwd padded d={d} {regime}")
    D = HEADS * d
    for layout, N, w in BWD_CASES:
        w = (N + 7 if w is None else w) if layout == "window" else None
        lens = _lens(N) if layout == "prefix" else [N] * (1 if layout == "window" else 2)
        B = len(lens)
        seed = _seed("bwd", layout, d, regime, N, w)
        q, k, v = _inputs(regime, lens, N, d, seed, window=w)
        qkv = _qkv(q, k, v)
        do = _grad_do(lens, N, d, seed + 1, regime != "diffuse")
        do_flat = do.reshape(B * N, D).to(BF).cuda()
        mask = _mask(lens, N).cuda() if layout == "prefix" else None
        lse = torch.empty(B * N, HEADS, device="cuda")
        out = L.attention(qkv, B, N, HEADS, d, mask, window=-1 if w is None else w, lse=lse)
        delta = _delta(L, out, do_flat, B * N, d)
        kl = None
        if mask is not None:
            kl = L.kv_len(mask)
            live = mask.reshape(B * N, 1)
            lse = torch.where(live, lse, torch.zeros_like(lse))            # rows past kv_len: a finite, wrong lse and delta
            delta = torch.where(live, delta, torch.full_like(delta, 0.75 * POISON_V))
        dqkv = _bwd_padded(L, qkv, do_flat, lse, delta, kl, B, N, d, 1 if mask is not None else 0, -1 if w is None else w)
        for b, n in enumerate(lens):
            r0 = b * N
            if n:
                b_o, tau = _fwd_ref(q[b, :n], k[b, :n], v[b, :n], w)[1::2]
                _check_grads(wst, f"{layout} N={N} w={w} img {b} (kv_len {n})", dqkv[r0:r0 + n], q[b, :n], k[b, :n], v[b, :n],
                             do[b, :n], b_o, tau, w)
            assert bool((dqkv[r0 + n:r0 + N] == 0).all()), (layout, N, b, "dq of rows / dk, dv of keys past kv_len must be 0")
    wst.report()


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("d", [64, 128])
def test_backward_packed(L, d, regime):
    """vtk_attention_bwd_packed_bf16 (plan qrows 128; the d = 128 forward runs on a qrows 256 plan of the same mask) with the
    forward kernel's lse and delta; the images' pad rows carry large dO, lse 0 and a large delta and get exactly 0 gradients, rows
    past the last image are untouched, and the next image's rows after a partial tile (in the poison regime: queries that score
    ~36 nats on this image's keys) contribute nothing."""
    wst = Worst(f"bwd packed d={d} {regime}")
    D = HEADS * d
    for N in NS:
        lens = _lens(N)
        B = len(lens)
        seed = _seed("bwd packed", d, regime, N)
        q, k, v, plan, pk, cu, nv = _packed_inputs(L, regime, lens, N, d, seed, 128)
        plan_f = plan if d == 64 else L.pack_plan(_mask(lens, N).cuda(), 16, 256)
        do = _grad_do(lens, N, d, seed + 2, False)
        do_pk = L.pack_rows(do.reshape(B, N, D).to(BF).cuda(), plan)
        rows = pk.shape[0]
        out = torch.zeros(rows, D, dtype=BF, device="cuda")
        lse = torch.zeros(rows, HEADS, device="cuda")
        L.attention_packed(pk, plan_f, B, N, HEADS, d, lse=lse, out=out)
        delta = _delta(L, out, do_pk, cu[B], d)
        if regime != "diffuse":
            valid = torch.zeros(rows, 1, dtype=torch.bool, device="cuda")
            for b in range(B):
                valid[cu[b]:cu[b] + nv[b]] = True
            do_pk = torch.where(valid, do_pk, torch.full_like(do_pk, POISON_V / 8))
            lse = torch.where(valid, lse, torch.zeros_like(lse))
            delta = torch.where(valid, delta, torch.full_like(delta, 0.75 * POISON_V))
        dqkv = torch.full((rows, 3 * D), SENT, dtype=BF, device="cuda")
        b0, g0 = pk.data_ptr(), dqkv.data_ptr()
        L.check(L.load().vtk_attention_bwd_packed_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, do_pk.data_ptr(), D, lse.data_ptr(),
                                                       delta.data_ptr(), g0, g0 + 2 * D, g0 + 4 * D, 3 * D, plan["n_valid"].data_ptr(),
                                                       plan["cu"].data_ptr(), plan["cuq"].data_ptr(), plan["grp_img"].data_ptr(),
                                                       plan["grp_order"].data_ptr(), B, HEADS, d, rows, plan["grp_img"].numel(),
                                                       L.stream_ptr()))
        for b, n in enumerate(nv):
            if n:
                b_o, tau = _fwd_ref(q[b, :n], k[b, :n], v[b, :n])[1::2]
                _check_grads(wst, f"N={N} img {b} ({n} tokens)", dqkv[cu[b]:cu[b] + n], q[b, :n], k[b, :n], v[b, :n], do[b, :n], b_o, tau)
            assert bool((dqkv[cu[b] + n:cu[b + 1]] == 0).all()), (N, b, "pad rows must get 0 gradients")
        assert bool((dqkv[cu[B]:] == SENT).all()), (N, "rows past the last image must stay untouched")
    wst.report()


# ------------------------------------------------------------------------------------------------------------------------------
# persistent grid
# ------------------------------------------------------------------------------------------------------------------------------
def test_persistent_grid_invariance(L):
    """The d = 64 forward is a persistent kernel whose grid is min(work items, 2 x usable SMs).  With "reserve_sms" leaving 2, 3 and
    37 SMs usable, every CTA walks many items back to back: Q refills, K/V ring phases across items with different tile counts,
    inactive items, the deferred TMA store of O and (packed) the boustrophedon dealing that skips indices past the total.  Output and
    lse must be bit-identical to the default grid, on late-max inputs (O rescaled while non-zero) and with every layout."""
    d = 64
    sms = L.load().vtk_sm_count()
    assert sms > 37
    cases = []
    for N in (1000, 1024):                                  # direct stores / TMA stores of O
        q, k, v = _gen("late_max", [N] * 3, N, d, seed=_seed("grid dense", N))
        cases.append((f"dense N={N}", lambda qkv=_qkv(q, k, v), N=N: L.attention(qkv, 3, N, HEADS, d, None, lse=_lse(3 * N))))
    lens = [1024, 0, 1, 600, 129, 1000]
    q, k, v = _gen("late_max", lens, 1024, d, seed=_seed("grid prefix"))
    cases.append(("prefix", lambda qkv=_qkv(q, k, v): L.attention(qkv, len(lens), 1024, HEADS, d, _mask(lens, 1024).cuda(),
                                                                  lse=_lse(len(lens) * 1024))))
    q, k, v = _gen("late_max", [1000] * 2, 1000, d, seed=_seed("grid window"))
    cases.append(("window 129", lambda qkv=_qkv(q, k, v): L.attention(qkv, 2, 1000, HEADS, d, None, window=129, lse=_lse(2000))))
    q, k, v, plan, pk, cu, nv = _packed_inputs(L, "late_max", lens, 1024, d, _seed("grid packed"), 128)

    def packed(pk=pk, plan=plan):
        lse = _lse(pk.shape[0])
        out = torch.full((pk.shape[0], HEADS * d), SENT, dtype=BF, device="cuda")
        return L.attention_packed(pk, plan, len(lens), 1024, HEADS, d, lse=lse, out=out)
    cases.append(("packed", packed))

    def run(fn):
        _lse.last = None
        out = fn()
        return out.clone(), _lse.last.clone()
    default = int(os.environ.get("VTK_RESERVE_SMS", "0"))
    base = {name: run(fn) for name, fn in cases}
    try:
        for usable in (2, 3, 37):
            L.set_flag("reserve_sms", sms - usable)
            for name, fn in cases:
                out, lse = run(fn)
                assert torch.equal(out, base[name][0]), f"{name}: output differs on a grid of {2 * usable} CTAs"
                assert torch.equal(lse, base[name][1]), f"{name}: lse differs on a grid of {2 * usable} CTAs"
    finally:
        L.set_flag("reserve_sms", default)
    print(f"[numerics] persistent grid: {len(cases)} layouts bit-identical on grids of 4, 6 and 74 CTAs and the default")


def _lse(rows):
    _lse.last = torch.full((rows, HEADS), SENT, device="cuda")
    return _lse.last
