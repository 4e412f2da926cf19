"""CPU: the L2Norm policy (SURVEY.md §8 f4; pyramidkv_utils.py:394-431) — oracle vs the golden vectors the unmodified
reference produced (tests/golden/make_golden_l2norm.py), budget/skip logic of the host mirror, and the plugin flow
through the test backend. The reference's `argsort` is not stable: the ORDER inside a class of equal norms (bf16 norms of
a 1K-token head take < 100 distinct values) is implementation-defined there, so the pins are: norms bit-exact, the
selected set strictly below the boundary norm identical, the kept rows' norm SEQUENCE identical, gather = byte copies."""
import os

import numpy as np
import pytest
import torch

from golden_util import GOLDEN_DIR, DTYPES, from_u16, make_inputs, sha256_of
from oracle_backend import OracleBackend

CASES = ["l2norm_s1024_b128_bf16", "l2norm_s777_b96_fp16", "l2norm_mha_d64_s640_b640_bf16", "l2norm_8b_s4096_b512_bf16"]


def _load(name):
    import json
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    m = json.loads(bytes(z["meta"]).decode())
    dt = DTYPES[m["dtype"]]
    q, k, v = make_inputs(m["seed"], m["Hq"], m["Hkv"], m["S"], m["D"], dt, m["scale"])
    assert (sha256_of(q), sha256_of(k), sha256_of(v)) == (m["sha_q"], m["sha_k"], m["sha_v"])
    return z, m, dt, q, k, v


@pytest.mark.parametrize("name", CASES)
def test_oracle_norms_and_selection_vs_reference(oracle, name):
    z, m, dt, q, k, v = _load(name)
    ref_norms = from_u16(z["norms"], dt)                      # [Hkv, S] as torch.norm produced them
    mine = oracle.key_norms(k)
    bad = int((mine.view(torch.int16) != ref_norms.view(torch.int16)).sum())
    assert bad <= (0 if m["dtype"] == "bf16" else max(1, mine.numel() // 5000)), f"{bad} norms differ from torch.norm"
    if bad:                                                   # fp16: a handful of values sit on a rounding boundary of the fp32 sum
        d = (mine.float() - ref_norms.float()).abs() / ref_norms.float()
        assert float(d.max()) <= 2.0 ** -10
    B, G = m["B"], m["Hq"] // m["Hkv"]
    ref_idx = torch.from_numpy(z["idx"])                      # [Hq, B] reference argsort order (unstable among equals)
    # selection on the REFERENCE's norms (stage injection), so a boundary-norm difference cannot blur the comparison
    keys = (ref_norms.view(torch.int16) ^ torch.tensor(-32768, dtype=torch.int16)).view(dt).repeat_interleave(G, dim=0).contiguous()
    idx = oracle.topk(keys, B, oracle.TIE_LOWEST_INDEX)
    nr = ref_norms.repeat_interleave(G, dim=0).float()
    assert torch.equal(torch.gather(nr, 1, idx), torch.gather(nr, 1, ref_idx)), "kept rows' norm sequence differs"
    for h in range(m["Hq"]):
        boundary = float(nr[h, ref_idx[h, -1]])
        below_ref = set(ref_idx[h][nr[h, ref_idx[h]] < boundary].tolist())
        below_mine = set(idx[h][nr[h, idx[h]] < boundary].tolist())
        assert below_ref == below_mine
        ties = idx[h][nr[h, idx[h]] == boundary]
        assert torch.equal(ties, torch.sort(ties).values)                        # lowest indices of the boundary class, ascending
        all_ties = torch.nonzero(nr[h] == boundary).flatten()
        assert torch.equal(ties, all_ties[: ties.numel()])
    # gather semantics: the reference's outputs are byte copies of the rows its own order names, no window rows
    assert sha256_of(oracle.gather(k, ref_idx, 0, m["Hq"])) == m["sha_k_out"]
    assert sha256_of(oracle.gather(v, ref_idx, 0, m["Hq"])) == m["sha_v_out"]


@pytest.mark.parametrize("name", CASES[:3])
def test_oracle_evict_l2norm_end_to_end(oracle, name):
    z, m, dt, q, k, v = _load(name)
    r = oracle.evict("l2norm", q, k, v, 0, m["B"])
    G = m["Hq"] // m["Hkv"]
    norms = oracle.key_norms(k)
    assert torch.equal(r.pooled.view(torch.int16), (norms.view(torch.int16) ^ torch.tensor(-32768, dtype=torch.int16)).repeat_interleave(G, dim=0))
    st = torch.sort(norms.float().repeat_interleave(G, dim=0), dim=-1, stable=True).indices[:, : m["B"]]
    assert torch.equal(r.idx, st)                                                  # == stable ascending argsort, truncated
    assert r.k_cache.shape == (m["Hq"], m["B"], m["D"])
    assert torch.equal(r.k_cache, oracle.gather(k, r.idx, 0, m["Hq"])) and torch.equal(r.v_cache, oracle.gather(v, r.idx, 0, m["Hq"]))
    with pytest.raises(ValueError):
        oracle.evict("l2norm", q, k, v, 8, m["B"])                               # L2Norm keeps no window


def test_torch_chain_l2norm_matches_oracle_under_stable_rule(oracle):
    from oracle import torch_chain as tc
    q, k, v = make_inputs(77, 8, 2, 500, 128, torch.bfloat16)
    K, V = tc.repeat_kv(k[None], 4), tc.repeat_kv(v[None], 4)
    Kc, Vc, idx = tc.l2norm_update_kv(K, V, 100, return_indices=True, tie_rule="lowest_index")
    r = oracle.evict("l2norm", q, k, v, 0, 100)
    assert torch.equal(idx[0], r.idx) and torch.equal(Kc[0], r.k_cache) and torch.equal(Vc[0], r.v_cache)
    assert tc.l2norm_update_kv(K, V, 600)[0] is K and tc.l2norm_update_kv(K, V, 100, skip=True)[0] is K


def test_torch_chain_l2norm_bit_identical_to_reference():
    """The torch restatement returns the K/V bytes the reference's L2NormCluster (skip_layers=[0, 1]) returned on every golden
    case, including the reference's own order inside classes of equal norms (sha256 recorded by make_golden_l2norm.py)."""
    from oracle import torch_chain as tc
    for name in CASES + ["l2norm_skip_layer_s300_b64_bf16", "l2norm_pass_s50_b64_bf16"]:
        z, m, dt, q, k, v = _load(name)
        G = m["Hq"] // m["Hkv"]
        mk, mv, order = tc.l2norm_update_kv(tc.repeat_kv(k[None], G), tc.repeat_kv(v[None], G), m["B"], skip=m["layer"] in (0, 1),
                                            return_indices=True)
        assert (order is not None) == m["evicted"] and mk.shape[2] == m["k_rows"], name
        if order is not None:
            assert torch.equal(order[0], torch.from_numpy(z["idx"])), name
        assert sha256_of(mk[0]) == m["sha_k_out"] and sha256_of(mv[0]) == m["sha_v_out"], name


def test_host_mirror_budget_skip_and_defaults(libpkv, oracle):
    from pyramidkv_b200 import kv_cluster as kc, ops
    assert ops.layer_budget("l2norm", 128, 0, 2, 0, 1000) == (1, 128) == oracle.layer_budget("l2norm", 128, 0, 2, 0, 1000)
    assert ops.layer_budget("l2norm", 128, 0, 2, 0, 100) == (0, 100)
    assert ops.layer_budget("l2norm", 128, 0, 2, 0, 128) == (1, 128)
    with pytest.raises(ValueError):
        ops.layer_budget("l2norm", 128, 8, 2, 0, 1000)
    c = kc.L2NormCluster(max_capacity_prompt=64, layer_idx=1, skip_layers=[0, 1], backend=OracleBackend())
    assert c.budget(500) == (0, 500)
    c = kc.L2NormCluster(max_capacity_prompt=64, layer_idx=2, skip_layers=[0, 1], backend=OracleBackend())
    assert c.budget(500) == (1, 64) and c.window_size == 0

    class Cfg:
        pass

    class Mod:
        config, layer_idx = Cfg(), 3
    m = Mod()
    kc.init_l2norm(m)                                         # pyramidkv_utils.py:954-968
    assert (m.config.max_capacity_prompt, m.config.layer_idx, m.config.skip_layers) == (4096, 0, [0, 1])
    assert isinstance(m.kv_cluster, kc.L2NormCluster) and m.kv_cluster.layer_idx == 3
    # reference-shaped update_kv on repeated tensors for a skipped layer returns the same objects
    q, k, v = make_inputs(5, 4, 4, 90, 64, torch.bfloat16)
    c = kc.L2NormCluster(max_capacity_prompt=32, layer_idx=0, skip_layers=[0, 1], backend=OracleBackend())
    ko, vo = c.update_kv(k[None], q[None], v[None], None, 1)
    assert ko.data_ptr() == k.data_ptr() and vo.data_ptr() == v.data_ptr()


def test_l2norm_through_the_plugin_flow(oracle):
    """replace_llama('l2norm') + generate on a tiny model through the test backend: skipped layers keep every row, the others keep
    max_capacity_prompt rows (+ decoded tokens); the static loop yields the same tokens."""
    from pyramidkv_b200 import generate as G, runner
    runner.patch("l2norm")
    try:
        model = runner.build_model("tiny-llama", torch.device("cpu"), torch.bfloat16, "eager")
        for layer in model.model.layers:
            layer.self_attn.config.max_capacity_prompt = 40
            layer.self_attn.config.skip_layers = [0, 1]
            layer.self_attn._pkv_backend = OracleBackend()
        ids = runner.synthetic_prompt(model.config.vocab_size, 120, 9, torch.device("cpu"))
        with torch.no_grad():
            out = model.generate(ids, attention_mask=torch.ones_like(ids), max_new_tokens=5, min_new_tokens=5, num_beams=1, do_sample=False,
                                 pad_token_id=0, return_dict_in_generate=True)
        rows = [int(l.keys.shape[-2]) for l in out.past_key_values.layers]
        assert rows == [124, 124, 44, 44]
        seq = G.greedy_generate(model, ids, 5)
        assert seq.tolist() == out.sequences.tolist()
    finally:
        from pyramidkv.monkeypatch import restore
        restore()
