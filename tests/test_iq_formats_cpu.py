"""Integer IQ input formats, host side: the dequantisation table of include/habdec_b200.h (HBD_IQ_*) as api.dequantise
states it, and the quantise helper the GPU tests and tools/bench_iq_formats.py make integer data with."""
import numpy as np
import pytest

from habdec_b200 import api


def _formula(codes, fmt):
    v = codes.astype(np.float64)
    return {api.IQ_CS16: v / 32768.0, api.IQ_CS8: v / 128.0, api.IQ_CU8: (v - 128.0) / 128.0}[fmt]


@pytest.mark.parametrize("fmt,dtype", [(api.IQ_CS16, np.int16), (api.IQ_CS8, np.int8), (api.IQ_CU8, np.uint8)])
def test_dequantise_every_code_exactly(fmt, dtype):
    """Every code of the format, as I and as Q, equals the defining formula evaluated in float64 -- exactly, so the value
    is representable in float32 and an integer push can be bit for bit the cf32 push of these values."""
    info = np.iinfo(dtype)
    codes = np.arange(info.min, info.max + 1, dtype=np.int64).astype(dtype)
    iq = np.stack([codes, codes[::-1]], axis=-1).reshape(-1)           # I = code, Q = reversed codes
    got = api.dequantise(iq, fmt)
    assert got.dtype == np.complex64 and got.shape == (len(codes),)
    want = _formula(codes, fmt)
    assert np.array_equal(got.real.astype(np.float64), want)
    assert np.array_equal(got.imag.astype(np.float64), want[::-1])
    assert np.array_equal(want.astype(np.float32).astype(np.float64), want)
    assert api.IQ_BYTES[fmt] == 2 * np.dtype(dtype).itemsize


def test_cu8_is_cs8_of_flipped_sign_bit():
    codes = np.arange(256, dtype=np.uint8)
    iq = np.stack([codes, codes], axis=-1).reshape(-1)
    assert np.array_equal(api.dequantise(iq, api.IQ_CU8), api.dequantise((iq ^ 0x80).view(np.int8), api.IQ_CS8))


@pytest.mark.parametrize("fmt", [api.IQ_CS16, api.IQ_CS8, api.IQ_CU8])
def test_quantise_round_trip(fmt):
    rng = np.random.default_rng(3)
    x = (0.4 * (rng.standard_normal((3, 1000)) + 1j * rng.standard_normal((3, 1000)))).astype(np.complex64)
    q = api.quantise(x, fmt, scale=1.0)
    assert q.shape == (3, 2000) and q.dtype == {api.IQ_CS16: np.int16, api.IQ_CS8: np.int8, api.IQ_CU8: np.uint8}[fmt]
    y = api.dequantise(q, fmt)
    assert y.shape == x.shape
    lsb = {api.IQ_CS16: 1 / 32768, api.IQ_CS8: 1 / 128, api.IQ_CU8: 1 / 128}[fmt]
    inside = (np.abs(x.real) < 0.99) & (np.abs(x.imag) < 0.99)
    assert np.all(np.abs(y.real - x.real)[inside] <= lsb / 2 + 1e-7)
    assert np.all(np.abs(y.imag - x.imag)[inside] <= lsb / 2 + 1e-7)
    assert np.array_equal(api.quantise(y, fmt), q)                        # dequantised values are fixed points
    big = api.dequantise(api.quantise(np.array([4 + 4j, -4 - 4j], np.complex64), fmt), fmt)   # clipped, not wrapped
    assert big[0].real > 0.98 and big[1].real == -1.0


def test_quantise_torch_matches_numpy():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(5)
    x = (0.3 * (rng.standard_normal((2, 777)) + 1j * rng.standard_normal((2, 777)))).astype(np.complex64)
    for fmt in (api.IQ_CS16, api.IQ_CS8, api.IQ_CU8):
        assert np.array_equal(api.quantise(torch.from_numpy(x), fmt, 0.8).numpy(), api.quantise(x, fmt, 0.8))


def test_dequantise_rejects_a_mismatched_dtype():
    with pytest.raises(ValueError):
        api.dequantise(np.zeros(4, np.int8), api.IQ_CS16)
