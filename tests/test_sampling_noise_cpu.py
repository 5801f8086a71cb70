"""CPU: the definition of the in-kernel sampling noise (tests/noise_ref.py) against Random123's known answers and the
distribution it must sample, and the CPU executor (tests/cuda_emu) running the shipped noise code and the production
entries phk_sample_tokens(u=NULL) / phk_sample_tail_rows at T > 0 against that definition.  The same entry checks run
on the B200 in tests/test_gpu_sampling_noise.py."""
import numpy as np
import pytest
import torch

from phenaki_pytorch_b200 import _lib as L
from tests import emu_runtime
from tests import noise_cases as N
from tests import noise_ref as R

CPU = torch.device("cpu")


# Random123 kat_vectors: (rounds, counter, key, output)
KAT = [
    (10, [0] * 4, [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    (10, [0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    (10, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
    (7, [0] * 4, [0, 0], [0x5F6FB709, 0x0D893F64, 0x4F121F81, 0x4F730A48]),
    (7, [0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x5207DDC2, 0x45165E59, 0x4D8EE751, 0x8C52F662]),
    (7, [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0x4DFCCABA, 0x190A87F0, 0xC47362BA, 0xB6B5242A]),
]


@pytest.mark.parametrize("rounds,ctr,key,want", KAT)
def test_philox_reference_reproduces_the_known_answers(rounds, ctr, key, want):
    got = R.philox4x32(np.array([ctr], dtype=np.uint64), key, rounds)[0]
    assert [int(x) for x in got] == want


def test_counter_layout_carries_into_the_high_word():
    """Rows that straddle 2^32: the counter is one 64-bit number, so the word of (offset, row, v) equals the word of the
    single counter offset + row * ceil(V/4) + v // 4 -- and (c lo, c hi) = (0, 1) is not (0, 0)."""
    V, rows, offset = 10, 6, 2 ** 32 - 5
    bits = R.row_bits(17, offset, np.arange(rows), V)
    per = (V + 3) // 4
    for r in range(rows):
        for v in range(V):
            c = offset + r * per + v // 4
            word = R.philox4x32(np.array([[c & 0xFFFFFFFF, c >> 32, 0, 0]], dtype=np.uint64), (17, 0))[0][v % 4]
            assert bits[r, v] == word
    low = R.counter_bits(17, np.array([0], dtype=np.uint64))[0]
    high = R.counter_bits(17, np.array([2 ** 32], dtype=np.uint64))[0]
    assert not np.array_equal(low, high)
    assert np.array_equal(R.stream_bits(17, offset, 4 * per * rows).reshape(rows, per * 4)[:, :V], bits)


def test_uniform_and_gumbel_reference_edges():
    assert R.uniform(np.array([0], np.uint32))[0] == 2.0 ** -24
    assert R.uniform(np.array([0xFFFFFFFF], np.uint32))[0] == 1 - 2.0 ** -24
    g = R.gumbel64_table()
    assert np.all(np.diff(g) > 0)
    assert abs(g[0] - (-2.8115409)) < 1e-6 and abs(g[-1] - 16.6355323) < 1e-6


@pytest.mark.parametrize("T", [0.3, 1.0, 2.0])
def test_ideal_sampler_draws_softmax_of_logits_over_temperature(T):
    """The definition itself (7 rounds, 24-bit uniforms, -log(-log u)): 2^20 argmax draws per logit vector follow
    softmax(l / T) (Pearson chi-square, p > 1e-6; fixed seeds, so the outcome is deterministic)."""
    n, V = 2 ** 20, 16
    bits = R.stream_bits(2024, 7 * 2 ** 22, n * V).reshape(n, V)   # rows of 4 counters each, as phk_sample_tokens
    g = R.gumbel64(bits)
    for name, l in N.chi2_logits(T).items():
        pick = np.argmax(l[None, :] / T + g, axis=1)
        counts = np.bincount(pick, minlength=V)
        p = N.chi2_pvalue(counts, R.softmax64(l / T))
        assert p > 1e-6, f"{name}: chi-square p = {p:.3g}"


# ---------------------------------------------------------------------------------------------------------------------
# CPU executor
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    return emu_runtime.build_emu()


@pytest.fixture(autouse=True)
def _cpu(lib, monkeypatch):
    monkeypatch.setattr(L, "stream_ptr", lambda: None)
    monkeypatch.setattr(L, "lib", lambda: lib)


@pytest.fixture(scope="module")
def table(lib):
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(L, "stream_ptr", lambda: None)
        return N.device_table(lib, CPU)


@pytest.mark.parametrize("seed,offset", [(5, 0), (2 ** 40 + 3, 2 ** 32 - 5), (2 ** 63 + 12345, 6_800_000_123)])
def test_executor_noise_words_equal_the_definition(lib, seed, offset):
    n = 4 * 37 + 3
    bits, g = N.probe(lib, CPU, seed=seed, offset=offset, n=n)
    assert np.array_equal(bits, R.stream_bits(seed, offset, n))
    assert np.all(np.isfinite(g))


def test_executor_transform_is_the_probe_table(lib, table):
    """bits_in mode returns the transform of the given words: the same values as the k table."""
    bits = R.stream_bits(9, 0, 1000)
    out, g = N.probe(lib, CPU, bits=bits)
    assert np.array_equal(out, bits) and np.array_equal(g, table[bits >> 9])


@pytest.mark.parametrize("V,T,cfg,ld_extra,seg,null_out", [
    (1, 0.9, False, 0, None, None),
    (5, 0.9, True, 1, None, None),
    (130, 2.0, False, 0, None, "score"),
    (128, 0.05, True, 4, (5, 3), None),
    (259, 0.9, False, 1, None, "pred"),
    (64, 0.9, True, 0, None, "mask"),
])
def test_executor_sample_tokens_noise_decisions(lib, table, V, T, cfg, ld_extra, seg, null_out):
    N.run_sample_tokens(lib, CPU, table, rows=20, V=V, T=T, cfg=cfg, ld_extra=ld_extra, seg=seg, null_out=null_out,
                        seed=2 ** 33 + 1, offset=2 ** 32 - 9)


def test_executor_sample_tokens_temperature_zero_ties(lib, table):
    N.run_sample_tokens(lib, CPU, table, rows=12, V=9, T=0.0, cond=N.tie_logits(12, 9, 4))


def test_executor_sample_tail_counts_noise_by_compact_row(lib, table):
    N.check_tail_noise(lib, CPU, table, b=2, n=24, k=9, V=70, dim=128, prime=5)
