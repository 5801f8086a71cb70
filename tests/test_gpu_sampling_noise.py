"""GPU: the in-kernel sampling noise of the B200 kernels (Philox4x32-7 words, the gumbel transform on the fast-math
unit) and the production entries that draw it -- phk_sample_tokens(u=NULL), the fused tcgen05 head phk_head_sample /
phk_head_sample_rng (also replayed from a CUDA graph with phk_rng_advance), phk_sample_tail_rows -- against the float64
reference of tests/noise_ref.py.  Tolerances and the decision rule are stated in tests/noise_cases.py."""
import numpy as np
import pytest
import torch

from phenaki_pytorch_b200 import _lib as L
from tests import noise_cases as N
from tests import noise_ref as R

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def sync():
    torch.cuda.synchronize()


@pytest.fixture(scope="module")
def table():
    return N.device_table(L.lib(), DEV, sync=sync)


# ---- (a) the words -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [12345, 2 ** 32 + 77, 2 ** 63 + 0x1234_5678_9ABC])
@pytest.mark.parametrize("offset", [0, 2 ** 32 - 5, 3 * 680_000_000 + 12])
def test_device_noise_words_equal_the_definition(seed, offset):
    n = 4 * 1000 + 3
    bits, _ = N.probe(L.lib(), DEV, seed=seed, offset=offset, n=n, sync=sync)
    assert np.array_equal(bits, R.stream_bits(seed, offset, n))


# ---- (b) the transform, over every input ---------------------------------------------------------------------------
def test_device_gumbel_transform_over_all_inputs(table):
    """All 2^23 uniforms: finite, non-decreasing in k (1e-5 allowed for the approximate logarithm), and within
    N.GUMBEL_TOL of -log(-log u) in float64 (range [-2.8115, 16.6355])."""
    g64 = R.gumbel64_table()
    assert bool(np.isfinite(table).all()), f"non-finite at k = {np.nonzero(~np.isfinite(table))[0][:8].tolist()}"
    d = np.diff(table.astype(np.float64))
    assert d.min() >= -1e-5, f"decreases by {-d.min():.3g} at k = {int(d.argmin())}"
    err = np.abs(table.astype(np.float64) - g64)
    k = int(err.argmax())
    print(f"max |g_dev - gumbel64| = {err[k]:.3g} at k = {k}")
    assert err[k] <= N.GUMBEL_TOL, f"|g_dev - gumbel64| = {err[k]:.3g} at k = {k} (device {table[k]}, float64 {g64[k]})"


# ---- (c) the production entries ------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [1, 3, 5, 128, 130, 4099, 65536])
@pytest.mark.parametrize("T", [0.05, 0.9, 2.0])
@pytest.mark.parametrize("cfg", [False, True])
def test_sample_tokens_noise_decisions(table, V, T, cfg):
    rows = 48 if V >= 4096 else 300
    N.run_sample_tokens(L.lib(), DEV, table, rows=rows, V=V, T=T, cfg=cfg, seed=2 ** 63 + 5, offset=2 ** 32 - 7 * V,
                        data_seed=V, sync=sync)


@pytest.mark.parametrize("V,ld_extra,seg,null_out", [
    (4099, 1, None, None), (130, 1, None, None), (1000, 4, None, None), (517, 0, (37, 11), None),
    (1024, 0, None, "mask"), (130, 0, None, "pred"), (4099, 4, None, "score"),
])
def test_sample_tokens_noise_layouts(table, V, ld_extra, seg, null_out):
    N.run_sample_tokens(L.lib(), DEV, table, rows=148, V=V, T=0.9, cfg=True, ld_extra=ld_extra, seg=seg, null_out=null_out,
                        seed=99, offset=6_800_000_000, data_seed=V + ld_extra, sync=sync)


@pytest.mark.parametrize("V", [3, 130, 65536])
def test_sample_tokens_temperature_zero_takes_the_first_maximum(table, V):
    rows = 64
    N.run_sample_tokens(L.lib(), DEV, table, rows=rows, V=V, T=0.0, cond=N.tie_logits(rows, V, V), sync=sync)


@pytest.mark.parametrize("n_tokens,V,dim,bias,emb_rows,ld_emb", [
    (300, 100, 64, True, None, None),         # V < 128, V % 4 == 0
    (200, 1000, 128, False, None, None),      # V % 32 != 0, no bias
    (130, 4099, 512, True, None, None),       # V % 4 != 0: the bias scalar path; n_tokens % 128 != 0
    (600, 65536, 512, True, None, None),      # 5 token tiles: uneven vocabulary splits (512 tiles as 28 x 18 + 8)
    (19000, 66, 64, True, None, None),        # 149 token tiles: one vocabulary split
    (250, 3000, 128, True, 300, 136),         # emb_rows > n_tokens, ld_emb > dim
])
@pytest.mark.parametrize("T", [0.05, 0.9])
def test_head_noise_decisions(table, n_tokens, V, dim, bias, emb_rows, ld_emb, T):
    N.check_head(L.lib(), DEV, table, n_tokens=n_tokens, V=V, dim=dim, T=T, bias=bias, emb_rows=emb_rows, ld_emb=ld_emb,
                 seed=2 ** 40 + n_tokens, offset=2 ** 32 - 3 * V, data_seed=V, sync=sync)


def test_head_with_zero_weights_is_the_epilogue_alone(table):
    """W = 0: the logits are the bias exactly, so the epilogue (noise, argmax, softmax) is checked free of GEMM error."""
    N.check_head(L.lib(), DEV, table, n_tokens=700, V=5003, dim=64, T=0.9, w_zero=True, sync=sync)


def test_head_temperature_zero_ties_across_vocabulary_splits():
    """T = 0, W = 0, the maximal bias at v = 5 and v = V - 7 (different vocabulary splits of the 1-tile call): the lower
    index must win every row, which the merge of the partials (head_finalize_kernel) decides."""
    n_tokens, V, dim = 100, 8192, 64
    emb, W, b = N.head_operands(n_tokens, V, dim, w_zero=True)
    b = b.clamp(max=3.0)
    b[5] = b[V - 7] = 4.0          # a power of two: fma(4, 1e10, g) rounds to 4e10 for every g, so the tie is exact
    _, pred, _ = N.run_head(L.lib(), DEV, emb, W, b, n_tokens=n_tokens, V=V, dim=dim, T=0.0, seed=1, offset=0, sync=sync)
    assert bool((pred == 5).all()), f"picks {np.unique(pred).tolist()}"


def test_head_rng_key_in_device_memory_equals_by_value():
    n_tokens, V, dim = 300, 1000, 128
    emb, W, b = N.head_operands(n_tokens, V, dim, data_seed=3)
    seed, offset = 2 ** 63 + 99, 2 ** 32 - 1000
    by_value = N.run_head(L.lib(), DEV, emb, W, b, n_tokens=n_tokens, V=V, dim=dim, T=0.9, seed=seed, offset=offset, sync=sync)
    state = torch.tensor([seed - 2 ** 64, offset], dtype=torch.int64, device=DEV)
    in_mem = N.run_head(L.lib(), DEV, emb, W, b, n_tokens=n_tokens, V=V, dim=dim, T=0.9, seed=0, offset=0, rng_state=state,
                        sync=sync)
    for x, y in zip(by_value, in_mem):
        assert np.array_equal(x, y)


def test_head_rng_graph_replays_advance_the_key(table):
    """phk_head_sample_rng + phk_rng_advance(stride) captured in one CUDA graph: replay i draws at offset + i * stride."""
    lib = L.lib()
    n_tokens, V, dim, T = 256, 3000, 128, 0.9
    emb, W, b = N.head_operands(n_tokens, V, dim, data_seed=4)
    seed, offset, stride = 2 ** 33 + 7, 2 ** 32 - 200_000, n_tokens * ((V + 3) // 4) + 4
    d_emb, d_W, d_b = emb.to(DEV), W.to(DEV), b.to(DEV)
    state = torch.tensor([seed, offset], dtype=torch.int64, device=DEV)
    pred = torch.empty(n_tokens, dtype=torch.int64, device=DEV)
    score = torch.empty(n_tokens, device=DEV)
    nb = lib.phk_head_sample_scratch_bytes(n_tokens)
    scratch = torch.empty(int(nb), dtype=torch.uint8, device=DEV)

    def step():
        L.check(lib.phk_head_sample_rng(L.ptr(d_emb), dim, n_tokens, L.ptr(d_W), dim, L.ptr(d_b), n_tokens, V, dim, T, 0, 0,
                                        L.ptr(state), None, None, L.ptr(pred), L.ptr(score), L.ptr(scratch), nb,
                                        L.stream_ptr()), "phk_head_sample_rng")
        L.check(lib.phk_rng_advance(L.ptr(state), stride, L.stream_ptr()), "phk_rng_advance")

    step()                                   # once eagerly: one-time kernel configuration happens outside the capture
    sync()
    state.copy_(torch.tensor([seed, offset], dtype=torch.int64))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    state.copy_(torch.tensor([seed, offset], dtype=torch.int64))
    sync()
    l64, eps_l = N.head_reference(emb, W, b, n_tokens, dim)
    for i in range(3):
        graph.replay()
        sync()
        bits = R.row_bits(seed, offset + i * stride, np.arange(n_tokens), V)
        N.check_decisions(pred.cpu().numpy(), l64, T, bits, table, eps_l, f"graph replay {i}")
    assert int(state[1].cpu()) == offset + 3 * stride


@pytest.mark.parametrize("b,n,k,V,dim,prime", [(3, 120, 50, 4099, 256, 24), (2, 576, 288, 65536, 512, 64)])
def test_sample_tail_counts_noise_by_compact_row(table, b, n, k, V, dim, prime):
    N.check_tail_noise(L.lib(), DEV, table, b=b, n=n, k=k, V=V, dim=dim, prime=prime, sync=sync)


def test_near_one_draw_never_lifts_a_hopeless_token(table):
    """A draw with k >= 2^23 - 2 (u within 2.5e-7 of 1) on a token whose l / T is 40 below the row's best: the float64
    reference can never pick it (gumbels span [-2.81, 16.64]), so neither may phk_sample_tokens nor phk_head_sample."""
    rows, V, T, offset = 64, 4096, 0.9, 2 ** 32 - 1000
    seed, row, v = N.find_near_one(1, offset, rows, V)
    logits = torch.randn(V, generator=torch.Generator().manual_seed(8))     # every row: the same logits (the head's bias)
    logits[v] = float(logits.max()) - 40.0 * T
    l64 = np.broadcast_to(logits.double().numpy(), (rows, V))
    bits = R.row_bits(seed, offset, np.arange(rows), V)
    ideal = R.ideal(l64, T, bits)
    assert ideal[row] != v
    pred = torch.empty(rows, dtype=torch.int64, device=DEV)
    cond = logits.to(DEV).expand(rows, V).contiguous()
    L.check(L.lib().phk_sample_tokens(L.ptr(cond), None, V, None, seed, offset, 1.0, T, None, None, L.ptr(pred), None, rows,
                                      V, 0, 0, 0, L.stream_ptr()), "phk_sample_tokens")
    sync()
    got = pred.cpu().numpy()
    assert got[row] == ideal[row], f"phk_sample_tokens picks {got[row]} (device g {table[bits[row, v] >> 9]})"
    assert not (got == v).any()
    emb, W, _ = N.head_operands(rows, V, 64, w_zero=True)
    _, hp, _ = N.run_head(L.lib(), DEV, emb, W, logits, n_tokens=rows, V=V, dim=64, T=T, seed=seed, offset=offset, sync=sync)
    assert hp[row] == ideal[row], f"phk_head_sample picks {hp[row]}"
    assert not (hp == v).any()


# ---- (d) the distribution through the kernels ----------------------------------------------------------------------
@pytest.mark.parametrize("entry", ["sample_tokens", "head"])
@pytest.mark.parametrize("T", [0.3, 1.0, 2.0])
def test_kernel_draws_follow_softmax_of_logits_over_temperature(entry, T):
    """2^20 rows of the same V = 16 logits through the kernel: the histogram of picks passes the chi-square against
    softmax(l / T) (p > 1e-6), as the float64 definition does in tests/test_sampling_noise_cpu.py."""
    rows, V = 2 ** 20, 16
    lib = L.lib()
    for name, l in N.chi2_logits(T).items():
        lt = torch.from_numpy(l).float()
        if entry == "sample_tokens":
            pred = torch.empty(rows, dtype=torch.int64, device=DEV)
            L.check(lib.phk_sample_tokens(L.ptr(lt.to(DEV).expand(rows, V).contiguous()), None, V, None, 2024, 2 ** 32 - 3,
                                          1.0, T, None, None, L.ptr(pred), None, rows, V, 0, 0, 0, L.stream_ptr()),
                    "phk_sample_tokens")
            sync()
            pick = pred.cpu().numpy()
        else:
            emb = torch.zeros((rows, 64), dtype=torch.bfloat16)
            W = torch.zeros((V, 64), dtype=torch.bfloat16)
            _, pick, _ = N.run_head(lib, DEV, emb, W, lt, n_tokens=rows, V=V, dim=64, T=T, seed=2024, offset=2 ** 32 - 3,
                                    sync=sync)
        counts = np.bincount(pick, minlength=V)
        assert counts.sum() == rows
        p = N.chi2_pvalue(counts, R.softmax64(lt.double().numpy() / T))
        assert p > 1e-6, f"{entry} {name}: chi-square p = {p:.3g}"
