"""Shared bodies of the sampling-noise checks (CPU executor and B200): the production entries that draw in-kernel noise
(phk_sample_tokens with u == NULL, phk_head_sample[_rng], phk_sample_tail_rows) against the float64 reference of
tests/noise_ref.py.

Decisions.  `with_table` with the transform of the library under test (read through phk_noise_probe) separates "the
counters and the reduction are right" from "the transform is accurate": the kernel's pick must equal it on every row
whose two best reference scores differ by more than delta, the float32 rounding bound of the kernel's score
fma(l, fl(1/T), g) (plus, for the head, the fp32 accumulation bound dim * 2^-23 * sum|e w| of the bf16 operands, from
which the float64 logits are exact).  At most 0.1 % of the rows (at least one) may fall inside delta, and there the
pick must be one of the candidates.  The float64 `ideal` sampler is the bar for the transform: rows whose ideal gap
exceeds delta + 2 * GUMBEL_TOL must get its decision too.

Confidence.  1 - score = softmax(l)[pred] must match float64 within
    p * (CONF_REL + 2 * eps_l + CONF_PER_LOGIT * max|l|) + 2^-23,
CONF_REL covering the approximate exponentials (ex2.approx / __expf: 2 ulp each, about 2^-22) and the fp32 running sum,
eps_l the bound on the kernel's logit error, CONF_PER_LOGIT the rounding of the exponent argument l * log2(e)."""
import numpy as np
import torch

from phenaki_pytorch_b200 import _lib as L
from tests import noise_ref as R

GUMBEL_TOL = 1e-4                 # |device transform - gumbel64| over every input (tests/test_gpu_sampling_noise.py)
CONF_REL, CONF_PER_LOGIT = 2e-5, 2.0 ** -23
U24 = 2.0 ** -24


def _u32(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).to(dev)


def probe(lib, dev, *, bits=None, seed=0, offset=0, n=None, sync=lambda: None):
    """(bits, gumbel) through phk_noise_probe: the generator's words (bits None) or the transform of given words."""
    n = len(bits) if bits is not None else n
    bits_in = None if bits is None else _u32(bits, dev)
    out = torch.empty(n, dtype=torch.int32, device=dev)
    g = torch.empty(n, dtype=torch.float32, device=dev)
    L.check(lib.phk_noise_probe(L.ptr(bits_in), seed & (2 ** 64 - 1), offset & (2 ** 64 - 1), n, L.ptr(out), L.ptr(g),
                                L.stream_ptr()), "phk_noise_probe")
    sync()
    return out.cpu().numpy().view(np.uint32), g.cpu().numpy()


def device_table(lib, dev, sync=lambda: None):
    """The library's gumbel of every k (2^23 float32 values), i.e. of the words k << 9."""
    return probe(lib, dev, bits=np.arange(R.K_COUNT, dtype=np.uint32) << 9, sync=sync)[1]


def check_decisions(pred, l64, T, bits, table, eps_l, what):
    """pred [rows]; l64 float64 [rows, V] (exact logits); eps_l [rows, V] bound on the kernel's logit error."""
    rows = l64.shape[0]
    Te = max(float(T), 1e-10)
    g_tab = np.asarray(table, dtype=np.float64)[bits >> 9]
    s_tab = R.scores(l64, T, g_tab)
    inv_t = 1.0 / Te
    elem = eps_l * inv_t + np.abs(l64) * inv_t * U24 + (np.abs(s_tab) + eps_l * inv_t) * U24
    delta = 2.0 * elem.max(axis=1) * (1 + 1e-3)
    ref = s_tab.argmax(axis=1)
    gap = R.top2_gap(s_tab)
    amb = gap <= delta
    assert int(amb.sum()) <= max(1, rows // 1000), f"{what}: {int(amb.sum())} of {rows} rows inside delta"
    bad = np.nonzero((pred != ref) & ~amb)[0]
    assert len(bad) == 0, (f"{what}: rows {bad[:8].tolist()} pick {pred[bad[:8]].tolist()} instead of "
                           f"{ref[bad[:8]].tolist()} (gaps {gap[bad[:8]].tolist()}, delta {delta[bad[:8]].tolist()})")
    for r in np.nonzero(amb)[0]:
        assert s_tab[r, pred[r]] >= s_tab[r].max() - delta[r], f"{what}: row {r}: not a candidate"
    s_id = R.scores(l64, T, R.gumbel64(bits))
    clear = R.top2_gap(s_id) > delta + 2 * GUMBEL_TOL
    bad = np.nonzero((pred != s_id.argmax(axis=1)) & clear)[0]
    assert len(bad) == 0, f"{what}: rows {bad[:8].tolist()} differ from the float64 gumbel reference"


def check_confidence(score, pred, l64, eps_l, what):
    p64 = R.softmax64(l64)[np.arange(len(pred)), pred]
    p = 1.0 - score.astype(np.float64)
    tol = p64 * (CONF_REL + 2 * eps_l.max(axis=1) + CONF_PER_LOGIT * np.abs(l64).max(axis=1)) + 2.0 ** -23
    err = np.abs(p - p64)
    assert bool((err <= tol).all()), f"{what}: confidence off by {err.max():.3g} (tol {tol[err.argmax()]:.3g})"


# ---------------------------------------------------------------------------------------------------------------------
# phk_sample_tokens(u = NULL)
# ---------------------------------------------------------------------------------------------------------------------
def run_sample_tokens(lib, dev, table, *, rows, V, T, cfg=False, ld_extra=0, seg=None, null_out=None, seed=7,
                      offset=1000, data_seed=0, sync=lambda: None, cond=None):
    """One phk_sample_tokens(u=NULL) call on seeded logits, checked against the reference.
    ld_extra: row pitch V + ld_extra.  seg: (n, prime) -> the token rows read logits[:, prime:] of (rows / n, prime + n)
    rows.  null_out: one of "mask", "pred", "score" passed as NULL."""
    g = torch.Generator().manual_seed(data_seed)
    ld = V + ld_extra
    if seg:
        n, prime = seg
        b = rows // n
        lrows = np.array([(r // n) * (prime + n) + prime + r % n for r in range(rows)])
        total = b * (prime + n)
    else:
        lrows, total = np.arange(rows), rows
    if cond is None:
        cond = torch.randn((total, ld), generator=g) * 2 + 1
    null = torch.randn((total, ld), generator=g) if cfg else None
    scale = 3.0 if cfg else 1.0
    mask = (torch.rand(rows, generator=g) < 0.7).to(torch.uint8)
    ids0 = torch.randint(0, V, (rows,), generator=g)
    c64 = cond.double().numpy()[lrows, :V]
    if cfg:
        n64 = null.double().numpy()[lrows, :V]
        l64 = n64 + (c64 - n64) * scale
        eps_l = U24 * (2 * scale * np.abs(c64 - n64) + np.abs(l64)) * (1 + 1e-6)
    else:
        l64, eps_l = c64, np.zeros_like(c64)
    ids = ids0.clone().to(dev)
    pred = torch.full((rows,), -1, dtype=torch.int64, device=dev)
    score = torch.full((rows,), float("nan"), device=dev)
    d_cond, d_null = cond.to(dev), (null.to(dev) if cfg else None)
    d_mask = None if null_out == "mask" else mask.to(dev)
    seg_len, seg_stride, seg_off = (seg[0], seg[0] + seg[1], seg[1]) if seg else (0, 0, 0)
    L.check(lib.phk_sample_tokens(L.ptr(d_cond), L.ptr(d_null), ld, None, seed, offset, scale, T, L.ptr(d_mask), L.ptr(ids),
                                  None if null_out == "pred" else L.ptr(pred),
                                  None if null_out == "score" else L.ptr(score), rows, V, seg_len, seg_stride, seg_off,
                                  L.stream_ptr()), "phk_sample_tokens")
    sync()
    ids, pred, score = ids.cpu().numpy(), pred.cpu().numpy(), score.cpu().numpy()
    m = np.ones(rows, bool) if null_out == "mask" else mask.numpy().astype(bool)
    what = f"sample_tokens V={V} T={T} cfg={cfg} ld=V+{ld_extra} seg={seg} null={null_out}"
    got = ids if null_out == "pred" else pred
    sel = m if null_out == "pred" else np.ones(rows, bool)
    bits = R.row_bits(seed, offset, np.arange(rows), V)
    if T == 0:
        # pure argmax of the fp32 logits (|l| >= 0.1): exact ties go to the lowest index, as torch.argmax
        assert np.array_equal(got[sel], cond.numpy()[lrows, :V].argmax(axis=1)[sel]), f"{what}: argmax"
    else:
        check_decisions(got[sel], l64[sel], T, bits[sel], table, eps_l[sel], what)
    if null_out != "pred":
        assert np.array_equal(ids[m], pred[m]), f"{what}: ids = pred where masked"
    assert np.array_equal(ids[~m], ids0.numpy()[~m]), f"{what}: unmasked ids changed"
    if null_out != "score":
        assert bool((score[~m] == -1e4).all()), f"{what}: unmasked score"
        check_confidence(score[m], got[m], l64[m], eps_l[m], what)


def tie_logits(rows, V, seed):
    """Logits for the T = 0 check: |l| >= 0.1 around the maximum, and in every other row an exact tie of two maximal
    entries that the kernel must resolve towards the lower index.  The tied value is a power of two, so l * 1e10 is a
    float32 number and fma(l, 1e10, g) rounds back to it for every gumbel g."""
    g = torch.Generator().manual_seed(seed)
    cond = (torch.randn((rows, V), generator=g) + 1.0).clamp(max=7.0)
    for r in range(0, rows, 2):
        i = int(torch.randint(0, V, (1,), generator=g))
        cond[r, i] = cond[r, (i + 1 + r) % V] = 8.0
    return cond


# ---------------------------------------------------------------------------------------------------------------------
# phk_head_sample[_rng]: emb bf16 [emb_rows, ld_emb], W bf16 [V, dim] -> exact float64 logits from those operands
# ---------------------------------------------------------------------------------------------------------------------
def head_operands(n_tokens, V, dim, *, emb_rows=None, ld_emb=None, bias=True, w_zero=False, data_seed=0, w_scale=0.05):
    """emb ~ N(0, 1), bias ~ N(0, 1), W ~ N(0, w_scale^2 / dim), all bf16-exact.  The small product term keeps the
    worst-case accumulation bound (dim * 2^-23 * sum|e w|) far below the score gaps, so that at most 0.1 % of the rows
    are ambiguous even at dim 512, V 65536; the bias and the noise spread the scores."""
    g = torch.Generator().manual_seed(data_seed)
    emb_rows, ld_emb = emb_rows or n_tokens, ld_emb or dim
    emb = torch.randn((emb_rows, ld_emb), generator=g).bfloat16()
    W = torch.zeros((V, dim)).bfloat16() if w_zero else (torch.randn((V, dim), generator=g) * (w_scale / dim ** 0.5)).bfloat16()
    b = torch.randn((V,), generator=g) if bias else None
    return emb, W, b


def head_reference(emb, W, bias, n_tokens, dim):
    e = emb[:n_tokens, :dim].double()
    w = W.double()
    l64 = (e @ w.t()).numpy()
    acc_bound = dim * 2.0 ** -23 * (e.abs() @ w.abs().t()).numpy()
    if bias is not None:
        l64 = l64 + bias.double().numpy()[None, :]
    eps_l = acc_bound + U24 * (np.abs(l64) + acc_bound)   # accumulation, then the fp32 bias add
    return l64, eps_l


def run_head(lib, dev, emb, W, bias, *, n_tokens, V, dim, T, seed, offset, rng_state=None, mask=None, sync=lambda: None):
    d_emb, d_W = emb.to(dev), W.to(dev)
    d_b = bias.to(dev) if bias is not None else None
    ids = torch.full((n_tokens,), -1, dtype=torch.int64, device=dev)
    pred = torch.full((n_tokens,), -1, dtype=torch.int64, device=dev)
    score = torch.full((n_tokens,), float("nan"), device=dev)
    nb = lib.phk_head_sample_scratch_bytes(n_tokens)
    scratch = torch.empty(int(nb), dtype=torch.uint8, device=dev)
    d_mask = mask.to(dev) if mask is not None else None
    L.check(lib.phk_head_sample_rng(L.ptr(d_emb), emb.shape[1], emb.shape[0], L.ptr(d_W), W.shape[1], L.ptr(d_b), n_tokens,
                                    V, dim, T, seed, offset, L.ptr(rng_state), L.ptr(d_mask), L.ptr(ids), L.ptr(pred),
                                    L.ptr(score), L.ptr(scratch), nb, L.stream_ptr()), "phk_head_sample_rng")
    sync()
    return ids.cpu().numpy(), pred.cpu().numpy(), score.cpu().numpy()


def check_head(lib, dev, table, *, n_tokens, V, dim, T, emb_rows=None, ld_emb=None, bias=True, w_zero=False, seed=11,
               offset=5, data_seed=0, sync=lambda: None):
    emb, W, b = head_operands(n_tokens, V, dim, emb_rows=emb_rows, ld_emb=ld_emb, bias=bias, w_zero=w_zero,
                              data_seed=data_seed)
    _, pred, score = run_head(lib, dev, emb, W, b, n_tokens=n_tokens, V=V, dim=dim, T=T, seed=seed, offset=offset, sync=sync)
    l64, eps_l = head_reference(emb, W, b, n_tokens, dim)
    what = f"head n={n_tokens} V={V} dim={dim} T={T} bias={bias} w_zero={w_zero}"
    bits = R.row_bits(seed, offset, np.arange(n_tokens), V)
    check_decisions(pred, l64, T, bits, table, eps_l, what)
    check_confidence(score, pred, l64, eps_l, what)


# ---------------------------------------------------------------------------------------------------------------------
# phk_sample_tail_rows at T > 0: gamma = 0 and cond_scale = 1 make every gathered embedding exactly beta (bf16 values),
# so the float64 logits W beta + bias are exact; the rows outside the sampled tokens (the prime prefix) hold NaN, which
# would reach the decisions of any row gathered from there.
# ---------------------------------------------------------------------------------------------------------------------
def check_tail_noise(lib, dev, table, *, b, n, k, V, dim, prime, T=0.9, seed=3, offset=2 ** 32 - 40, data_seed=0,
                     sync=lambda: None):
    g = torch.Generator().manual_seed(data_seed)
    stride = prime + n
    xc = torch.randn((b * stride, dim), generator=g)
    xn = torch.randn((b * stride, dim), generator=g)
    for i in range(b):
        xc[i * stride:i * stride + prime] = float("nan")
        xn[i * stride:i * stride + prime] = float("nan")
    gamma = torch.zeros(dim)
    beta = torch.randn((dim,), generator=g).bfloat16().float()
    W = (torch.randn((V, dim), generator=g) * (0.05 / dim ** 0.5)).bfloat16()   # small: see head_operands
    bias = torch.randn((V,), generator=g)
    mask = torch.zeros((b, n), dtype=torch.uint8)
    for i in range(b):
        mask[i, torch.randperm(n, generator=g)[:k]] = 1
    ids0 = torch.randint(0, V, (b, n), generator=g)
    d = [t.to(dev) for t in (xc, xn, gamma, beta, W, bias, mask)]
    ids = ids0.clone().to(dev)
    pred = torch.empty((b, n), dtype=torch.int64, device=dev)
    score = torch.empty((b, n), device=dev)
    nb = lib.phk_sample_tail_scratch_bytes(b, k, dim)
    scratch = torch.empty(int(nb), dtype=torch.uint8, device=dev)
    L.check(lib.phk_sample_tail_rows(L.ptr(d[0]), L.ptr(d[1]), L.ptr(d[2]), L.ptr(d[3]), 1.0, L.ptr(d[4]), dim, L.ptr(d[5]),
                                     b, n, k, V, dim, T, seed, offset, None, L.ptr(d[6]), L.ptr(ids), L.ptr(pred),
                                     L.ptr(score), stride, prime, L.ptr(scratch), nb, L.stream_ptr()), "phk_sample_tail_rows")
    sync()
    ids, pred, score = ids.cpu().numpy(), pred.cpu().numpy(), score.cpu().numpy()
    e = beta.double()[None, :]
    w = W.double()
    l_row = (e @ w.t()).numpy()[0] + bias.double().numpy()
    acc = dim * 2.0 ** -23 * (e.abs() @ w.abs().t()).numpy()[0]
    m = mask.numpy().astype(bool)
    pos = [np.nonzero(m[i])[0] for i in range(b)]                 # compact row i * k + j <- j-th masked position
    crow = np.concatenate([i * k + np.arange(k) for i in range(b)])
    flat = np.concatenate([i * n + pos[i] for i in range(b)])
    l64 = np.broadcast_to(l_row, (b * k, V))
    eps_l = np.broadcast_to(acc + U24 * (np.abs(l_row) + acc), (b * k, V))
    bits = R.row_bits(seed, offset, crow, V)
    what = f"sample_tail b={b} n={n} k={k} V={V} prime={prime} T={T}"
    check_decisions(ids.reshape(-1)[flat], l64, T, bits, table, eps_l, what)
    assert np.array_equal(pred.reshape(-1)[flat], ids.reshape(-1)[flat]), what
    check_confidence(score.reshape(-1)[flat], ids.reshape(-1)[flat], l64, eps_l, what)
    assert np.array_equal(ids[~m], ids0.numpy()[~m]) and np.array_equal(pred[~m], ids0.numpy()[~m]), f"{what}: untouched"
    assert bool((score[~m] == -1e4).all()), f"{what}: unmasked score"


# ---------------------------------------------------------------------------------------------------------------------
# distribution: chi-square of the sampled histogram against softmax(l / T)
# ---------------------------------------------------------------------------------------------------------------------
def chi2_pvalue(counts, probs):
    """Pearson chi-square p-value; categories expected below 5 draws are pooled into one."""
    from scipy import stats
    n = counts.sum()
    exp = probs * n
    small = exp < 5
    c = np.append(counts[~small], counts[small].sum())
    e = np.append(exp[~small], exp[small].sum())
    if e[-1] == 0:
        c, e = c[:-1], e[:-1]
    return float(stats.chisquare(c, e).pvalue)


def chi2_logits(T):
    """V = 16 logit vectors for the distribution checks; the last one has a token ~10 below the best in l / T units,
    so the tail of the gumbel draws (large g for that token) is exercised."""
    g = torch.Generator().manual_seed(42)
    a = (torch.randn(16, generator=g) * 1.5).double().numpy()
    flat = np.zeros(16)
    deficit = (torch.randn(16, generator=g) * 0.3).double().numpy()
    deficit[5] = deficit.max() - 10.0 * T
    return {"randn": a, "flat": flat, "deficit": deficit}


def find_near_one(seed0, offset, rows, V, k_min=R.K_COUNT - 2):
    """(seed, row, v) of the first seed >= seed0 whose noise at (offset, rows x V) has a word with k >= k_min."""
    for seed in range(seed0, seed0 + 2000):
        bits = R.row_bits(seed, offset, np.arange(rows), V)
        hit = np.argwhere((bits >> 9) >= k_min)
        if len(hit):
            return seed, int(hit[0][0]), int(hit[0][1])
    raise AssertionError("no near-1 draw found")
