"""Shared builders for the parity tests: seeded synthetic inputs in the reference's geometry, the oracle's
answer for them, and the tolerance rule of SURVEY.md section 8(d)."""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import mma_oracle as O

MEDIA_ID, ASST_ID, PAD_ID = 32012, 32001, 32000


def make_prompt(B, L, N, n_img, q_frac=0.85, seed=0, pad_right=0, first_img=8):
    """lang_x / attention_mask with n_img <image> placeholders at evenly spaced offsets (first at `first_img`),
    one <|assistant|> token at q_frac of the text, optional right padding (SFT collate)."""
    g = np.random.default_rng(seed)
    lang = g.integers(3, 31000, size=(B, L)).astype(np.int64)
    am = np.ones((B, L), dtype=np.int64)
    for b in range(B):
        n_valid = L - (pad_right if b % 2 == 1 else 0)
        if n_img:
            step = max(1, (int(n_valid * q_frac) - first_img) // n_img)
            for k in range(n_img):
                lang[b, first_img + k * step] = MEDIA_ID
        qpos = int(n_valid * q_frac)
        while lang[b, qpos] == MEDIA_ID:
            qpos += 1
        lang[b, qpos] = ASST_ID
        lang[b, n_valid:] = PAD_ID
        am[b, n_valid:] = 0
    return lang, am


def qkv_inputs(B, T, H=32, D=96, seed=0, device="cpu", std=1.0):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B, T, H, D, generator=g) * std).to(torch.bfloat16)
    k = (torch.randn(B, T, H, D, generator=g) * std).to(torch.bfloat16)
    v = (torch.randn(B, T, H, D, generator=g) * std).to(torch.bfloat16)
    return q.to(device), k.to(device), v.to(device)


def oracle_attention(q, k, v, S, scaling, cos=None, sin=None, dtype=torch.float32, row_block=None):
    """q,k,v (B,T,H,D) bf16 (pre-RoPE if cos given: both q and k are rotated, mirroring Phi3Attention).
    Returns (B,T,H,D) in `dtype` arithmetic."""
    qf, kf, vf = (x.cpu().to(dtype).transpose(1, 2) for x in (q, k, v))
    if cos is not None:
        c = torch.cat([cos, cos], -1).cpu().to(dtype); s = torch.cat([sin, sin], -1).cpu().to(dtype)
        if c.shape[0] == 1:
            c = c.expand(qf.shape[0], -1, -1); s = s.expand(qf.shape[0], -1, -1)
        qf = O.apply_rope(qf, c, s); kf = O.apply_rope(kf, c, s)
    T = qf.shape[2]
    if S is not None:
        m4 = torch.from_numpy(O.expand_segments_to_4d(S, t_out=T))
    else:
        m4 = torch.tril(torch.ones(T, T, dtype=torch.int64))[None, None]
    add = O.invert_4d_mask(m4, dtype).to(dtype) if dtype != torch.float32 else O.invert_4d_mask(m4, dtype)
    return O.eager_attention(qf, kf, vf, add, scaling, row_block=row_block)


def live_rows(S, B, T):
    """(B,T) bool: rows with at least one visible key (fully masked rows are don't-care, see DESIGN.md)."""
    if S is None:
        return torch.ones(B, T, dtype=torch.bool)
    return torch.from_numpy(~O.fully_masked_rows(S))[:, :T]


def err_stats(x, ref, rows=None):
    x = x.detach().float().cpu(); ref = ref.detach().float().cpu()
    if rows is not None:
        x = x[rows]; ref = ref[rows]
    d = (x - ref).abs()
    return float(d.max()), float(d.pow(2).mean().sqrt()), float(ref.pow(2).mean().sqrt())


def within_tolerance(kernel, bf16_ref, fp32_ref, rows=None, floor=1e-3):
    """kernel error vs fp32 oracle <= 2 x error of the reference-style bf16 eager path + floor * RMS(ref)."""
    ek, _, rms = err_stats(kernel, fp32_ref, rows)
    eb, _, _ = err_stats(bf16_ref, fp32_ref, rows)
    return ek <= 2.0 * eb + floor * max(rms, 1.0), ek, eb, rms


# ------------------------------------------------------------------------------------------------------------------
# Rounding-point references for the decoder-layer kernels (test_gpu_layer_numerics.py).  Values are carried in fp64;
# a kernel's fp32 or bf16 rounding is applied explicitly where the kernel rounds.
U32 = 2.0 ** -24              # unit roundoff of fp32 (half an ulp, relative)
BF16_MAX = (2.0 - 2.0 ** -7) * 2.0 ** 127


def f32(x):
    """Round fp64 values to fp32 (IEEE round-to-nearest-even) and back to fp64."""
    return x.to(torch.float32).to(torch.float64)


def pow2(k):
    """2.0 ** k as fp64 for integer tensors k in [-1022, 1023], built from the exponent bits (torch.ldexp multiplies by
    pow(2, k), which is not exact for fp64 on every device)."""
    return ((k.to(torch.int64) + 1023) << 52).view(torch.float64)


def bf16_rne(x):
    """Round fp64 values to bf16, round-to-nearest-even, in ONE rounding from fp64; returned as fp64 (exactly
    representable in bf16, so a later .to(torch.bfloat16) is exact).  Done on the integer significand: bf16 keeps 8
    significant bits down to the normal limit 2^-126 and a fixed quantum of 2^-133 below it (subnormals); values from
    the midpoint between the largest finite bf16 and 2^128 upward round to inf.  (torch's own fp64 -> bf16 cast goes
    through fp32, a double rounding, which is why this is written out.)"""
    x = x.to(torch.float64)
    bits = x.view(torch.int64)
    neg = bits < 0
    biased = (bits >> 52) & 0x7FF
    sig = (bits & ((1 << 52) - 1)) | (1 << 52)                     # 1.m as an integer, value = sig * 2^(e - 52)
    e = biased - 1023
    drop = 45 + torch.clamp(-126 - e, min=0)                       # significand bits below the bf16 quantum
    drop = torch.clamp(drop, max=54)                               # >= 54: below half the smallest quantum -> 0
    half = torch.ones_like(drop) << (drop - 1)
    odd = (sig >> drop) & 1
    q = (sig + half - 1 + odd) >> drop                             # round half to even on the integer
    mag = q.to(torch.float64) * pow2(torch.clamp(e - 52 + drop, min=-133))      # q < 2^9: exact
    mag = torch.where(mag > BF16_MAX, torch.full_like(mag, math.inf), mag)
    mag = torch.where(biased == 0, torch.zeros_like(mag), mag)     # fp64 zeros and subnormals (< 2^-1022)
    out = torch.where(neg, -mag, mag)
    return torch.where(torch.isfinite(x), out, x)                  # inf and NaN pass through


def bf16_step(v, up):
    """The bf16 neighbour of bf16-representable fp64 values v, towards +inf (up) or -inf; +-0 step to +-2^-133."""
    b = v.to(torch.bfloat16).view(torch.int16).to(torch.int32) & 0xFFFF
    away = (b >> 15 == 0) == up                                    # moving away from zero in the magnitude
    zero = (b & 0x7FFF) == 0
    mag = torch.where(zero, torch.ones_like(b), torch.where(away, (b & 0x7FFF) + 1, (b & 0x7FFF) - 1))
    sign = torch.where(zero, torch.full_like(b, 0 if up else 0x8000), b & 0x8000)
    out = (sign | mag).to(torch.int16).view(torch.bfloat16).to(torch.float64)
    return torch.where(torch.isfinite(v), out, v)


def ulp32(x):
    """fp32 ulp of fp64 values (2^-149 in the subnormal range)."""
    _, ex = torch.frexp(x.abs().to(torch.float64))
    return pow2(torch.clamp(ex - 24, min=-149))


def ulp_bf16(x):
    """bf16 ulp of fp64 values (2^-133 in the subnormal range)."""
    _, ex = torch.frexp(x.abs().to(torch.float64))
    return pow2(torch.clamp(ex - 8, min=-133))


def bf16_branches(v64, eps_rel, eps_abs=0.0):
    """(ref, alt, band) of a bf16 rounding point.  v64 is the exact (fp64) value the kernel rounds; the kernel's fp32
    value before the rounding lies within eps_rel * |v64| + eps_abs of it.  ref = bf16_rne(v64).  Where the nearest
    rounding midpoint of v64 lies within that distance (band), the kernel may round to alt, the bf16 neighbour of ref
    across that midpoint, instead.  Two branches describe the rounding only while the distance stays below half a bf16
    ulp (at most one midpoint within reach), which is asserted."""
    v64 = v64.to(torch.float64)
    ref = bf16_rne(v64)
    up, dn = bf16_step(ref, True), bf16_step(ref, False)
    mid_up, mid_dn = (ref + up) / 2, (ref + dn) / 2                 # exact in fp64 (9 significant bits)
    d_up, d_dn = (v64 - mid_up).abs(), (v64 - mid_dn).abs()
    alt = torch.where(d_up <= d_dn, up, dn)
    tol = eps_rel * v64.abs() + eps_abs
    fin = torch.isfinite(v64)
    tol_t = torch.broadcast_to(torch.as_tensor(tol, dtype=torch.float64, device=v64.device), v64.shape)
    assert bool((tol_t[fin] < torch.minimum(up - ref, ref - dn)[fin] / 2).all()), \
        "rounding band wider than half a bf16 ulp: more than two outcomes"
    band = fin & (torch.minimum(d_up, d_dn) <= tol) & (tol > 0)     # an exact value rounds exactly
    return ref, alt, band


def accept_branches(got, ref, alt, band, what=""):
    """Every element of got (a bf16 tensor) must equal ref, or alt where band holds (values compared as numbers, so
    -0 == +0; NaN only matches NaN).  Returns the mask of accepted flips (got == alt != ref)."""
    g = got.to(torch.float64).to(ref.device)
    same = (g == ref) | (torch.isnan(g) & torch.isnan(ref))
    flip = band & ~same & (g == alt)
    bad = ~same & ~flip
    if bool(bad.any()):
        idx = bad.nonzero()[:6].tolist()
        ex = [(i, float(g[tuple(i)]), float(ref[tuple(i)]), float(alt[tuple(i)]), bool(band[tuple(i)])) for i in idx]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements are neither the rounding of the "
                             f"reference nor an accepted neighbour (index, got, ref, alt, in band): {ex}")
    return flip


def accept_bf16(got, v64, eps_rel, eps_abs=0.0, what=""):
    """Tie-aware comparison of a kernel's bf16 output with the fp64 value v64 it rounds.  The kernel's fp32 value lies in
    [v64 - tol, v64 + tol], tol = eps_rel |v64| + eps_abs, and round-to-nearest-even is monotone, so its bf16 lies in
    [bf16_rne(v64 - tol), bf16_rne(v64 + tol)]: bit-exact to bf16_rne(v64) where no rounding midpoint is within tol,
    either neighbour where one is, and every value of the interval where a cancellation makes tol span several bf16
    ulps (eps_abs of a rotation).  Returns the mask of accepted flips (got != bf16_rne(v64))."""
    v64 = v64.to(torch.float64)
    tol = eps_rel * v64.abs() + eps_abs
    ref, lo, hi = bf16_rne(v64), bf16_rne(v64 - tol), bf16_rne(v64 + tol)
    g = got.to(torch.float64).to(v64.device)
    same = (g == ref) | (torch.isnan(g) & torch.isnan(ref))
    flip = ~same & torch.isfinite(v64) & (g >= lo) & (g <= hi)
    bad = ~same & ~flip
    if bool(bad.any()):
        idx = bad.nonzero()[:6].tolist()
        ex = [(i, float(g[tuple(i)]), float(ref[tuple(i)]), float(lo[tuple(i)]), float(hi[tuple(i)])) for i in idx]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements lie outside the bf16 rounding of "
                             f"[v - tol, v + tol] (index, got, ref, lowest, highest accepted): {ex}")
    return flip


def flip_bound(v64, eps_rel, eps_abs=0.0):
    """Upper bound for the number of accepted flips: an element can only flip inside the band, whose width
    2 (eps_rel |v| + eps_abs) is at most 2^9 (eps_rel + eps_abs / |v|) of the bf16 ulp of v (ulp >= 2^-8 |v|).  For
    values spread over many ulps the expected count is the sum of those fractions; the bound is twice that plus 8."""
    v = v64.to(torch.float64).abs()
    e = eps_rel + eps_abs / torch.clamp(v, min=2.0 ** -133)
    frac = torch.clamp(2.0 ** 9 * e, max=1.0)
    if not torch.is_tensor(frac) or frac.dim() == 0:
        frac = torch.full_like(v, float(frac))
    return int(2 * float(frac[torch.isfinite(v)].sum()) + 8)


def sum_eps(depth):
    """Relative error bound of an fp32 sum of non-negative terms in which every term passes through at most `depth`
    roundings (additions, or the rounding of an FMA that adds it): depth * 2^-24, to first order."""
    return depth * U32


# ------------------------------------------------------------------------------------------------------------------
# Visibility census (test_gpu_attention_census.py): with K = 0 every score is 0, so every visible key weighs exactly 1
# and a one-hot V window (forward, decode) or a one-hot dO probe (backward) turns an output element into "does this
# (row, key) pair attend": 1/n_i or bf16(P) where it does, exactly 0 where it does not.  The references below are plain
# torch expressions of the oracle's predicate; they run on the device their tensors live on and never read the
# kernels' metadata tensors.
CENSUS_W = 32 * 96          # keys (forward, decode) or rows (backward) one launch maps: H * D output columns


class MaskRef:
    """The visibility predicate of expand_segments_to_4d in key coordinates, for B samples of Tk keys:
    allowed(i, j) = i < len & j < len & ((j <= i & valid[j]) | (row_lo[i] <= j < row_hi[i] & mutual[j])).
    seq_len (B,), row_lo / row_hi (B, Tk) int64; valid / mutual (B, Tk) bool."""

    def __init__(self, seq_len, valid, mutual, row_lo, row_hi):
        self.seq_len, self.valid, self.mutual = seq_len.to(torch.int64), valid.bool(), mutual.bool()
        self.row_lo, self.row_hi = row_lo.to(torch.int64), row_hi.to(torch.int64)

    @property
    def B(self):
        return self.valid.shape[0]

    @property
    def Tk(self):
        return self.valid.shape[1]

    def to(self, device):
        return MaskRef(*(x.to(device) for x in (self.seq_len, self.valid, self.mutual, self.row_lo, self.row_hi)))

    @staticmethod
    def from_segments(S, T=None, text_only=False):
        """The oracle's Segments (segments_ref) cut or zero-padded to T keys; text_only: image rows see later text keys
        only (expand_segments_to_4d's text_only)."""
        T = S.seg.shape[1] if T is None else T
        m = min(T, S.seg.shape[1])

        def cut(a, fill, dtype):
            out = torch.full((a.shape[0], T), fill, dtype=dtype)
            out[:, :m] = torch.from_numpy(np.ascontiguousarray(a[:, :m])).to(dtype)
            return out
        valid = cut(S.valid, 0, torch.bool)
        mutual = valid & (cut(S.seg, -1, torch.int64) == 0) if text_only else valid
        return MaskRef(torch.from_numpy(S.seq_len.astype(np.int64)), valid, mutual, cut(S.row_lo, 0, torch.int64),
                       cut(S.row_hi, 0, torch.int64))

    @staticmethod
    def causal(B, T, seq_len=None):
        """No metadata: every key up to the row (seq_len None = T for every sample)."""
        sl = torch.full((B,), T, dtype=torch.int64) if seq_len is None else torch.as_tensor(seq_len, dtype=torch.int64)
        ones = torch.ones(B, T, dtype=torch.bool)
        zero = torch.zeros(B, T, dtype=torch.int64)
        return MaskRef(sl, ones, ones, zero, zero)


def allowed_slab(R, rows, cols):
    """(B, r1 - r0, c1 - c0) bool: allowed(i, j) for rows i in range(*rows), keys j in range(*cols), key coordinates.
    Rows and keys at or beyond Tk see / are seen by nothing."""
    (r0, r1), (c0, c1) = rows, cols
    dev = R.valid.device
    i = torch.arange(r0, r1, device=dev)[None, :, None]
    j = torch.arange(c0, c1, device=dev)[None, None, :]
    ic, jc = i.clamp(max=R.Tk - 1)[0, :, 0], j.clamp(max=R.Tk - 1)[0, 0]
    n = torch.minimum(R.seq_len, torch.tensor(R.Tk, device=dev))[:, None, None]
    valid, mutual = R.valid[:, jc][:, None, :], R.mutual[:, jc][:, None, :]
    lo, hi = R.row_lo[:, ic][:, :, None], R.row_hi[:, ic][:, :, None]
    ok = ((j <= i) & valid) | ((j >= lo) & (j < hi) & mutual)
    return ok & (i < n) & (j < n)


def visible_counts(R):
    """(B, Tk) int64: number of keys each row sees (row sums of allowed), from prefix sums, not from allowed_slab."""
    dev = R.valid.device
    i = torch.arange(R.Tk, device=dev)[None]
    n = torch.minimum(R.seq_len, torch.tensor(R.Tk, device=dev))[:, None]
    z = torch.zeros(R.B, 1, dtype=torch.int64, device=dev)
    cv = torch.cat([z, (R.valid & (i < n)).to(torch.int64).cumsum(1)], 1)       # cv[k] = valid keys among [0, k)
    cm = torch.cat([z, (R.mutual & (i < n)).to(torch.int64).cumsum(1)], 1)
    causal = cv.gather(1, (i + 1).clamp(max=R.Tk).expand(R.B, -1))
    lo = torch.maximum(R.row_lo, i + 1).clamp(min=0).minimum(n)                  # keys after the row: not counted twice
    hi = R.row_hi.clamp(min=0).minimum(n)
    ext = torch.where(hi > lo, cm.gather(1, hi) - cm.gather(1, lo.minimum(hi)), torch.zeros_like(hi))
    return torch.where(i < n, causal + ext, torch.zeros_like(causal))


def decode_visible(kv_len, kv_start, valid, n_keys):
    """(B, n_keys) bool: the keys a decode query attends, kv_start[b] <= j < kv_len[b] and valid[b, j] (kv_start /
    valid None: 0 / every key)."""
    kv_len = torch.as_tensor(kv_len, dtype=torch.int64)
    j = torch.arange(n_keys, device=kv_len.device)[None]
    vis = j < kv_len[:, None]
    if kv_start is not None:
        vis &= j >= torch.as_tensor(kv_start, dtype=torch.int64, device=kv_len.device)[:, None]
    if valid is not None:
        vis &= valid[:, :n_keys].to(kv_len.device).bool()
    return vis


def recip_bf16(n):
    """bf16(fp32(1 / n)) as fp64 for integer counts n >= 1 (0 where n == 0): what a kernel writes for a visible key
    when every visible key weighs exactly 1 (fp32 IEEE division, one bf16 rounding)."""
    nf = n.to(torch.float32)
    r = torch.where(n > 0, 1.0 / nf.clamp(min=1), torch.zeros_like(nf))
    return r.to(torch.bfloat16).to(torch.float64)


def census_diff(got, want, rows, keys):
    """Pairs where the kernel's map (got != 0) and the reference map `want` disagree: (K, 5) float64 rows
    (b, row, key, got, want), sorted.  got / want are (B, len(rows), len(keys)); rows / keys the key-coordinate indices
    of those axes."""
    bad = (got != 0) != want
    idx = bad.nonzero()
    if idx.numel() == 0:
        return torch.zeros(0, 5, dtype=torch.float64)
    b, r, k = idx.unbind(1)                                           # nonzero() is in (b, row, key) order
    return torch.stack([b.double(), rows.to(idx.device)[r].double(), keys.to(idx.device)[k].double(),
                        got[b, r, k].double(), want[b, r, k].double()], 1).cpu()


def census_message(diff, what):
    b, r, k, g, w = diff[0].tolist()
    return (f"{what}: {diff.shape[0]} (row, key) pairs attended wrongly; first (b, row, key, got, want) = "
            f"({int(b)}, {int(r)}, {int(k)}, {g:.6g}, {bool(w)})")
