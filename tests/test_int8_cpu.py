"""CPU-only checks of the int8 shard format: argument validation of the new C entry points (it happens before any CUDA
call) and the numeric contract of the CPU oracle the GPU tests compare against."""
import numpy as np
import pytest
import torch

from tests.int8_oracle import dequantize, quantize_rows, scores


def _lib():
    from sgpt_b200 import _lib

    return _lib, _lib.lib()


def test_quantize_entry_point_validates_arguments():
    _l, lib = _lib()
    for D in (0, 8, 24, 65536 + 16):
        assert lib.sgpt_quantize_rows_i8(None, 0, 4, D, None, None, None, None) == 1, D
    assert b"multiple of 16" in lib.sgpt_last_error()
    assert lib.sgpt_quantize_rows_i8(None, 0, 4, 64, None, None, None, None) == 1  # null buffers
    assert b"null" in lib.sgpt_last_error()
    assert lib.sgpt_quantize_rows_i8(None, 1, 0, 64, None, None, None, None) == 0  # nothing to do


@pytest.mark.parametrize("entry", ["sgpt_search_ex", "sgpt_search_packed_ex", "sgpt_search_gather_ex"])
def test_search_ex_entry_points_validate_before_any_cuda_call(entry):
    _l, lib = _lib()
    fn = getattr(lib, entry)

    def call(elem, D):  # null outputs (and, for the gather form, a null context)
        if entry == "sgpt_search_ex":
            return fn(None, None, None, None, 4, 1000, D, 10, 0, None, None, None, 0, elem, None)
        if entry == "sgpt_search_packed_ex":
            return fn(None, None, None, None, 4, 1000, D, 10, 0, None, None, 0, elem, None)
        return fn(None, None, None, None, None, 4, 1000, D, 10, 0, None, None, None, None, 0, elem, None)

    assert call(2, 64) == 1 and b"unknown element type" in lib.sgpt_last_error()
    assert call(-1, 64) == 1
    for D in (8, 72, 65536 + 16):  # int8 rows: D % 16 == 0 and D <= 65536
        assert call(_l.ELEM_I8, D) == 1 and b"multiple of 16" in lib.sgpt_last_error(), D
    assert call(_l.ELEM_I8, 64) == 1  # null outputs (or, for the gather form, a null context)
    assert b"null" in lib.sgpt_last_error()
    assert call(_l.ELEM_BF16, 72) == 1 and b"null" in lib.sgpt_last_error()  # bf16 keeps D % 8


def test_bf16_entry_points_keep_their_checks():
    _l, lib = _lib()
    assert lib.sgpt_search(None, None, None, None, 4, 1000, 64, 10, 0, None, None, None, 0, None) == 1
    assert b"null output" in lib.sgpt_last_error()
    assert lib.sgpt_search_packed(None, None, None, None, 4, 1000, 64, 10, 0, None, None, 0, None) == 1


def test_shard_rejects_bad_int8_shapes_without_a_gpu():
    from sgpt_b200 import CorpusShard

    with pytest.raises(ValueError, match="multiple of 16"):
        CorpusShard(24, 10, device="cpu", dtype="int8")
    with pytest.raises(ValueError, match="dtype"):
        CorpusShard(64, 10, device="cpu", dtype="fp8")


def test_oracle_quantizer_rules():
    x = np.array([[0.0] * 16,
                  [127.0, -127.0, 63.5, -63.5, 0.5, -0.5, 1.5, 2.5] + [0.0] * 8,  # s = 1: halves round to even
                  [1.0, -2.0, 3.0] + [0.25] * 13], dtype=np.float32)
    c, s, inv = quantize_rows(x)
    assert s[0] == 0 and np.all(c[0] == 0) and inv[0] == np.float32(1e12)
    assert s[1] == np.float32(1.0)
    assert c[1, :8].tolist() == [127, -127, 64, -64, 0, 0, 2, 2]
    assert np.abs(c).max() <= 127 and c.dtype == np.int8
    assert np.float32(3.0) / np.float32(127.0) == s[2]
    n2 = int((c[2].astype(np.int64) ** 2).sum())
    assert inv[2] == np.float32(1.0) / np.sqrt(np.float32(n2))
    # bf16 input is widened exactly
    xb = torch.randn(5, 64, generator=torch.Generator().manual_seed(1)).to(torch.bfloat16)
    cb, sb, ib = quantize_rows(xb)
    cf, sf, if_ = quantize_rows(xb.float().numpy())
    assert np.array_equal(cb, cf) and np.array_equal(sb, sf) and np.array_equal(ib, if_)


@pytest.mark.parametrize("fn", ["cos_sim", "dot"])
def test_oracle_scores_equal_fp64_scores_of_the_dequantized_rows(fn):
    """The fp32 score of the integer formula equals cos_sim / dot_score of the dequantized rows s * c (evaluated in fp64)
    within fp32 rounding: one int->float conversion and two multiplications, each <= 2^-24 relative."""
    g = torch.Generator().manual_seed(7)
    qx, dx = torch.randn(9, 768, generator=g), torch.randn(300, 768, generator=g) * 3.0
    dx[5] = 0.0  # zero row: score 0 either way
    qq, dq = quantize_rows(qx), quantize_rows(dx)
    got = scores(qq, dq, fn).double()
    a, b = torch.from_numpy(dequantize(qq)), torch.from_numpy(dequantize(dq))
    if fn == "cos_sim":
        want = (a / a.norm(dim=1, keepdim=True).clamp_min(1e-12)) @ (b / b.norm(dim=1, keepdim=True).clamp_min(1e-12)).T
    else:
        want = a @ b.T
    # 3 roundings of 2^-24 on each score, plus (cos_sim) the 3 roundings of each side's 1/||c||: float(n2), sqrt, divide
    tol = 16 * 2.0 ** -24 * want.abs() + 1e-30
    assert torch.all((got - want).abs() <= tol), ((got - want).abs() / want.abs().clamp_min(1e-30)).max().item()
    assert torch.all(got[:, 5] == 0)
