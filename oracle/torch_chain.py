"""The reference's eviction op chain restated with stock PyTorch ops (runs on CPU or GPU).

*** TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE. *** Used by tests (-m gpu: same-device comparison against
the CUDA kernels) and by bench.py as the "reference op chain on this GPU" baseline. The reference is not a dependency
of this repository, so the chain is restated here op for op; tests/test_torch_chain_vs_reference.py (and the
`*_bit_identical_to_reference` tests) check it bit-for-bit against the outputs the reference classes recorded in tests/golden.

Follows pyramidkv/pyramidkv_utils.py: budget :205-220; scoring :253-263 (== :317-327); pooling :264-269;
top-k :270; gather + concat :271-282; H2O :544-575; StreamingLLM :607-619; repeat_kv :108-117; L2Norm :406-431.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def repeat_kv(x: torch.Tensor, n_rep: int) -> torch.Tensor:
    """[b, Hkv, S, D] -> [b, Hkv*n_rep, S, D] materialised copy (pyramidkv_utils.py:108-117)."""
    if n_rep == 1:
        return x
    b, h, s, d = x.shape
    return x[:, :, None].expand(b, h, n_rep, s, d).reshape(b, h * n_rep, s, d)


def layer_budget(method, B, W, L, layer_idx, S, beta=20):
    if S < B:
        return 0, S
    if method != "pyramidkv":
        return 1, B - W
    lo = (B - W) // beta
    hi = (B - W) * 2 - lo
    if hi >= S - W:
        hi = S - W
        lo = (B - W) * 2 - hi
    step = (hi - lo) // (L - 1)
    return (1, B - W) if S < (B - W) * 2 else (1, hi - layer_idx * step)


def _window_mask(W, dtype, device):
    m = torch.full((W, W), torch.finfo(dtype).min, device=device)       # fp32, like the reference (:254)
    ar = torch.arange(W, device=device)
    m.masked_fill_(ar < (ar + 1).view(W, 1), 0)
    return m[None, None]


def scores(method, K, Q, W, kernel_size, pooling):
    """-> [b, H, S-W] tensor fed to topk."""
    D = Q.shape[-1]
    Qs = Q if method == "h2o" else Q[..., -W:, :]
    a = torch.matmul(Qs, K.transpose(2, 3)) / math.sqrt(D)
    a[:, :, -W:, -W:] += _window_mask(W, a.dtype, a.device)
    a = F.softmax(a, dim=-1, dtype=torch.float32).to(Q.dtype)
    if method == "h2o":
        return a[:, :, :, :-W].sum(dim=-2)
    s = a[:, :, -W:, :-W].sum(dim=-2)
    if pooling == "avgpool":
        return F.avg_pool1d(s, kernel_size=kernel_size, padding=kernel_size // 2, stride=1)
    if pooling == "maxpool":
        return F.max_pool1d(s, kernel_size=kernel_size, padding=kernel_size // 2, stride=1)
    raise ValueError("Pooling method not supported")


def select(scores_, k, tie_rule="torch"):
    """topk(k).indices. tie_rule="torch": the reference's call (tie order = whatever this torch build does on this
    device). tie_rule="lowest_index": the contract of the CUDA path — (value desc, index asc) via a stable sort."""
    if tie_rule == "torch":
        return scores_.topk(k, dim=-1).indices
    return torch.sort(scores_.float(), dim=-1, descending=True, stable=True).indices[..., :k]


def update_kv(method, K, Q, V, W, B, kernel_size=5, pooling="avgpool", num_layers=32, layer_idx=0, beta=20,
              return_indices=False, tie_rule="torch"):
    """K, Q, V: [b, H, S, D] with K/V already repeat_kv-expanded (as the reference's callers pass them)."""
    assert K.shape[-2] == Q.shape[-2]
    b, H, S, D = Q.shape
    mode, k = layer_budget(method, B, W, num_layers, layer_idx, S, beta)
    if mode == 0:
        return (K, V, None) if return_indices else (K, V)
    if method == "streamingllm":
        idx = torch.tensor(range(B - W), dtype=torch.int64).to(K.device)[None, None].repeat(b, H, 1)
    else:
        idx = select(scores(method, K, Q, W, kernel_size, pooling), k, tie_rule)
    gi = idx.unsqueeze(-1).expand(-1, -1, -1, D)
    Kc = torch.cat([K[:, :, :-W, :].gather(2, gi), K[:, :, -W:, :]], dim=2)
    Vc = torch.cat([V[:, :, :-W, :].gather(2, gi), V[:, :, -W:, :]], dim=2)
    return (Kc, Vc, idx) if return_indices else (Kc, Vc)


def l2norm_update_kv(K, V, B, skip=False, return_indices=False, tie_rule="torch"):
    """L2NormCluster.update_kv (pyramidkv_utils.py:406-431): keep the B tokens of smallest key norm, in argsort order; no
    window. `skip` = `self.layer_idx in self.skip_layers` (:416). tie_rule as in select()."""
    S, D = K.shape[-2], K.shape[-1]
    if S < B or skip:
        return (K, V, None) if return_indices else (K, V)
    norms = torch.norm(K, p=2, dim=-1)
    order = norms.argsort(dim=-1) if tie_rule == "torch" else torch.sort(norms.float(), dim=-1, stable=True).indices
    gi = order.unsqueeze(-1).expand(-1, -1, -1, D)
    Kc, Vc = K.gather(2, gi)[:, :, :B, :], V.gather(2, gi)[:, :, :B, :]
    return (Kc, Vc, order[..., :B]) if return_indices else (Kc, Vc)


# ---- AdaKV / HeadKV: ragged per-head budgets (pyramidkv_utils.py:622-878) ----
def adakv_scores(K, Q, W, kernel_size, pooling):
    """`calcul_attn_sore` (pyramidkv_utils.py:647-672, == :781-806): like the SnapKV scores, but the window rows are
    averaged (`.mean(dim=-2)`) instead of summed. -> [b, H, S-W]."""
    D = Q.shape[-1]
    a = torch.matmul(Q[..., -W:, :], K.transpose(2, 3)) / math.sqrt(D)
    a[:, :, -W:, -W:] += _window_mask(W, a.dtype, a.device)
    a = F.softmax(a, dim=-1, dtype=torch.float32).to(Q.dtype)
    s = a[:, :, -W:, :-W].mean(dim=-2)
    if pooling == "avgpool":
        return F.avg_pool1d(s, kernel_size=kernel_size, padding=kernel_size // 2, stride=1)
    if pooling == "maxpool":
        return F.max_pool1d(s, kernel_size=kernel_size, padding=kernel_size // 2, stride=1)
    raise ValueError("Pooling method not supported")


def adakv_capacities(score, base_capacity, floor_ratio, normalize, tie_rule="torch"):
    """Per-head budgets of AdaKVCluster.update_kv (pyramidkv_utils.py:702-717): the heads share num_heads * base_capacity
    slots in proportion to how many of the globally largest (optionally normalised) scores they own, mixed with a floor.
    score [1, H, n] -> (capacities int32 [H], sorted indices [1, H, n]). tie_rule "torch": the reference's calls;
    "lowest_index": stable sort per head + stable flat selection (lower head / better rank first) — the CUDA path's rule."""
    bsz, H, n = score.shape
    if tie_rule == "torch":
        srt, idx = score.sort(dim=-1, descending=True)
    else:
        srt, idx = torch.sort(score.float(), dim=-1, descending=True, stable=True)
        srt = srt.to(score.dtype)
    adaptive = srt
    if normalize:
        ratio = srt[..., :base_capacity].sum(dim=-1, keepdim=True) / srt.sum(dim=-1, keepdim=True)
        adaptive = adaptive * ratio
    flat = adaptive.reshape(bsz, n * H)
    if tie_rule == "torch":
        top = torch.topk(flat, k=H * base_capacity, dim=-1).indices
    else:
        top = torch.sort(flat.float(), dim=-1, descending=True, stable=True).indices[:, : H * base_capacity]
    heads = top // n
    cap = torch.zeros((bsz, H), device=score.device, dtype=heads.dtype)
    cap.scatter_add_(-1, heads, torch.ones_like(heads, dtype=cap.dtype))
    floor_capacity = int(base_capacity * floor_ratio)
    cap = torch.round(cap * (1 - floor_ratio) + floor_capacity).int()
    return cap[0], idx


def ragged_gather(K, V, sorted_idx, capacities, W):
    """The per-head loop of AdaKV / HeadKV update_kv (pyramidkv_utils.py:731-757, :852-878): head h keeps its capacities[h]
    best tokens (in sorted order) followed by the last W tokens; the heads are concatenated into ONE flat [sum_h len_h, D]
    tensor. Returns (k_flat, v_flat, head_lens list)."""
    D = K.shape[-1]
    ks, vs, lens = [], [], []
    for h in range(K.shape[1]):
        ci = sorted_idx[:, h:h + 1, : int(capacities[h])]
        gi = ci.reshape(1, 1, -1, 1).expand(-1, -1, -1, D)
        ks.append(torch.cat([K[:, h:h + 1].gather(2, gi), K[:, h:h + 1, -W:, :]], dim=2).reshape(-1, D))
        vs.append(torch.cat([V[:, h:h + 1].gather(2, gi), V[:, h:h + 1, -W:, :]], dim=2).reshape(-1, D))
        lens.append(int(ci.shape[-1]) + W)
    return torch.cat(ks, dim=0), torch.cat(vs, dim=0), lens


def adakv_update_kv(K, Q, V, W, B, kernel_size=7, pooling="maxpool", floor_ratio=0.2, normalize=True, tie_rule="torch"):
    """AdaKVCluster.update_kv (pyramidkv_utils.py:674-757). K, Q, V [1, H, S, D] (K/V repeat_kv-expanded).
    Returns (k_flat [sum len, D], v_flat, head_lens)."""
    base = B - W
    score = adakv_scores(K, Q, W, kernel_size, pooling)
    S, D = Q.shape[-2], Q.shape[-1]
    if base > score.size(-1):                                   # not compressed (:698-701)
        return K.reshape(-1, D), V.reshape(-1, D), [S] * Q.shape[1]
    cap, idx = adakv_capacities(score, base, floor_ratio, normalize, tie_rule)
    return ragged_gather(K, V, idx, cap, W)


def headkv_update_kv(K, Q, V, W, B, head_capacity, kernel_size=7, pooling="maxpool", tie_rule="torch"):
    """HeadKVCluster.update_kv (pyramidkv_utils.py:808-878): the same ragged gather with the budgets given per head
    (`head_capacity[layer_idx]`, from the runner's head-score file)."""
    base = B - W
    score = adakv_scores(K, Q, W, kernel_size, pooling)
    S, D = Q.shape[-2], Q.shape[-1]
    if base > score.size(-1):
        return K.reshape(-1, D), V.reshape(-1, D), [S] * Q.shape[1]
    if tie_rule == "torch":
        idx = score.sort(dim=-1, descending=True).indices
    else:
        idx = torch.sort(score.float(), dim=-1, descending=True, stable=True).indices
    return ragged_gather(K, V, idx, head_capacity, W)


def update_flatten_view(cache, state, head_lens, cu_lens):
    """The reference's native `update_flatten_view` (csrc/csrc/cuda_api.cu:11-53) restated with torch ops: the flat ragged
    cache [sum_h len_h, D] gets one row of `state` [H, D] appended behind every head's rows. head_lens [H] int32,
    cu_lens[h] = rows before head h (the reference passes cu_klen with H + 1 entries)."""
    out = []
    for h in range(state.shape[0]):
        b, n = int(cu_lens[h]), int(head_lens[h])
        out += [cache[b:b + n], state[h:h + 1]]
    return torch.cat(out, dim=0)


def eager_decode_attn(q, Kc, Vc):
    """llama_model.py:174-183 with q_len == 1 and no mask. q [b,H,1,D]; Kc,Vc [b,H,T,D]."""
    a = torch.matmul(q, Kc.transpose(2, 3)) / math.sqrt(q.shape[-1])
    a = F.softmax(a, dim=-1, dtype=torch.float32).to(q.dtype)
    return torch.matmul(a, Vc)
