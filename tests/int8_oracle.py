"""CPU oracle of the int8 shard format (include/sgpt_b200.h sgpt_quantize_rows_i8 and the int8 search scores).

Every step is IEEE fp32 with round-to-nearest-even, exactly as the kernels compute it, so the GPU results must match
bit for bit: per row s = max|x| / 127, c = clamp(rint(x / s), -127, 127) (s == 0 -> c = 0), inv = 1 / max(sqrt((float)
sum c^2), 1e-12); scores cos_sim = ((float)acc * inv_q) * inv_d and dot = ((float)acc * s_q) * s_d with acc = sum cq cd,
exact.
"""
import numpy as np
import torch


def quantize_rows(x):
    """fp32 / bf16 rows [n, D] (torch or numpy) -> (codes int8 [n, D], scale fp32 [n], inv_norm fp32 [n]) as numpy."""
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().float().numpy()  # bf16 -> fp32 is exact
    x = np.ascontiguousarray(x, dtype=np.float32)
    a = np.abs(x).max(axis=1) if x.shape[1] else np.zeros(x.shape[0], np.float32)
    s = (a / np.float32(127.0)).astype(np.float32)
    ok = s > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        q = x / np.where(ok, s, np.float32(1.0))[:, None]
    c = np.clip(np.rint(q), -127, 127)
    c[~ok] = 0
    c = c.astype(np.int8)
    n2 = (c.astype(np.int64) ** 2).sum(axis=1)
    assert n2.max(initial=0) < 2 ** 31
    inv = (np.float32(1.0) / np.maximum(np.sqrt(n2.astype(np.float32)), np.float32(1e-12))).astype(np.float32)
    return c, s, inv


def exact_acc(cq, cd):
    """sum_j cq_j cd_j for every (query, doc) pair, exact: |products| <= 127^2 and |sums| <= 127^2 x 65536 < 2^53, so a
    float64 matrix product is exact in any summation order."""
    return torch.from_numpy(cq.astype(np.float64)) @ torch.from_numpy(cd.astype(np.float64)).T


def scores(q_quant, d_quant, score_function):
    """fp32 score matrix [nq, n] of quantized queries against quantized documents (the outputs of quantize_rows)."""
    (cq, sq, iq), (cd, sd, idd) = q_quant, d_quant
    acc = exact_acc(cq, cd).numpy().astype(np.float32)  # exact integer -> fp32, round to nearest even
    if score_function == "cos_sim":
        fq, fd = iq, idd
    elif score_function == "dot":
        fq, fd = sq, sd
    else:
        raise ValueError(score_function)
    return torch.from_numpy((acc * fq[:, None]).astype(np.float32) * fd[None, :])


def dequantize(quant):
    c, s, _ = quant
    return c.astype(np.float64) * s.astype(np.float64)[:, None]


def topk(full, k):
    """Sorted top-k of a dense score matrix: (scores, indices), ties by ascending index."""
    k = min(k, full.shape[1])
    order = torch.argsort(-full.double(), dim=1, stable=True)[:, :k]
    return torch.gather(full, 1, order), order


def assert_same_topk(s_dev, i_dev, full, k, id_base=0):
    """GPU result == oracle: scores bit-identical, ids identical with ties at the cut compared as sets."""
    want_s, want_i = topk(full, k)
    kk = want_s.shape[1]
    s, i = s_dev[:, :kk].cpu(), i_dev[:, :kk].cpu() - id_base
    assert torch.equal(s, want_s), (s - want_s).abs().max().item()
    for qi in range(s.shape[0]):
        cut = want_s[qi, -1].item()
        above_w = {int(j) for j, v in zip(want_i[qi], want_s[qi]) if v.item() > cut}
        above_g = {int(j) for j, v in zip(i[qi], s[qi]) if v.item() > cut}
        assert above_w == above_g, qi
        at_cut = set(torch.nonzero(full[qi] == cut).flatten().tolist())
        assert {int(j) for j, v in zip(i[qi], s[qi]) if v.item() == cut} <= at_cut, qi
        assert len(set(i[qi].tolist())) == kk, qi
