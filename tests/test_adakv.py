"""CPU: AdaKV / HeadKV ragged budgets (SURVEY.md §8 f4; pyramidkv_utils.py:622-878) — oracle vs golden vectors of the
unmodified reference (tests/golden/make_golden_adakv.py) and the torch restatement vs the oracle under the stable tie rule.
Tie allocation at the global threshold (torch.topk on the flattened scores) and the order inside classes of equal scores
(unstable sort) are implementation-defined in the reference; pinned are: scores, the normalised scores the flat top-k sees,
counts above the threshold, and capacities wherever ties leave no freedom."""
import json
import os

import numpy as np
import pytest
import torch

from golden_util import DTYPES, GOLDEN_DIR, from_u16, make_inputs, sha256_of

ADAKV = ["adakv_s1024_b128_w32_bf16_norm", "adakv_s1024_b128_w32_bf16_raw", "adakv_s777_b96_w8_bf16_avg_flat",
         "adakv_mha_d64_s640_b80_w16_fp16", "adakv_8b_s2048_b256_w8_bf16"]


def _load(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    m = json.loads(bytes(z["meta"]).decode())
    dt = DTYPES[m["dtype"]]
    q, k, v = make_inputs(m["seed"], m["Hq"], m["Hkv"], m["S"], m["D"], dt, m["scale"])
    assert (sha256_of(q), sha256_of(k), sha256_of(v)) == (m["sha_q"], m["sha_k"], m["sha_v"])
    return z, m, dt, q, k, v


def _mismatch(a, b):
    return int((a.view(torch.int16) != b.view(torch.int16)).sum())


@pytest.mark.parametrize("name", ADAKV + ["headkv_s1024_b128_w32_bf16"])
def test_scores_close_to_reference(oracle, name):
    z, m, dt, q, k, v = _load(name)
    ref = from_u16(z["score"], dt)
    mine = oracle.adakv_scores(q, k, m["W"], m["kernel"], m["pooling"])
    bad = _mismatch(mine, ref)
    assert bad <= max(4, int(2e-3 * ref.numel())), f"{bad}/{ref.numel()} mean-pooled scores differ (softmax / GEMM rounding class)"
    d = (mine.view(torch.int16).int() - ref.view(torch.int16).int()).abs().max()
    assert int(d) <= 4


@pytest.mark.parametrize("name", ADAKV)
def test_capacities_by_stage_injection(oracle, name):
    """reference scores in -> normalised scores bit-identical (as multisets per head), counts above the threshold identical,
    capacities identical wherever the threshold class leaves no choice, always inside the interval the ties allow."""
    z, m, dt, q, k, v = _load(name)
    score = from_u16(z["score"], dt)
    base = m["B"] - m["W"]
    caps, gt, eq, thr, scaled = oracle.adakv_capacities(score, base, m["floor"], m["normalize"], details=True)
    ref_flat = from_u16(z["flat"], dt)                                      # [Hq, n] sorted descending per head
    assert torch.equal(torch.sort(scaled.float(), dim=-1, descending=True).values, ref_flat.float()), "normalised scores differ"
    counts = torch.from_numpy(z["counts"])                                  # slots per head in the reference's flat top-k
    K = m["Hq"] * base
    assert int(counts.sum()) == K
    t = torch.sort(ref_flat.float().flatten(), descending=True).values[K - 1]
    assert float(t) == float(thr.float())
    ref_gt = (ref_flat.float() > t).sum(-1)
    assert torch.equal(ref_gt, gt) and torch.all(counts >= gt) and torch.all(counts <= gt + eq)
    need = K - int(gt.sum())
    omf, fc = np.float32(1 - m["floor"]), int(base * m["floor"])
    rnd = lambda c: int(torch.round(torch.tensor(float(np.float32(c) * omf + np.float32(fc)))).item())
    ref_caps = torch.from_numpy(z["head_lens"]).long() - m["W"]
    assert [rnd(int(c)) for c in counts] == ref_caps.tolist()               # the rounding step itself (:715)
    # the oracle's rule: lower heads take the tied slots first
    exp, left = [], need
    for h in range(m["Hq"]):
        take = min(left, int(eq[h])); left -= take
        exp.append(rnd(int(gt[h]) + take))
    assert caps.tolist() == exp
    free = int(eq.sum()) - need                                             # tied candidates that do not get a slot
    if free == 0:
        assert caps.tolist() == ref_caps.tolist()
    for h in range(m["Hq"]):
        assert rnd(int(gt[h])) <= int(ref_caps[h]) <= rnd(int(gt[h] + eq[h]))


@pytest.mark.parametrize("name", ADAKV + ["headkv_s1024_b128_w32_bf16"])
def test_ragged_gather_semantics(oracle, name):
    """Rows of head h = its capacity[h] best tokens in (score desc, index asc) order, then the last W tokens; with the
    reference's own capacities the kept rows carry exactly the reference's score multiset (order inside ties is free)."""
    z, m, dt, q, k, v = _load(name)
    score = from_u16(z["score"], dt)
    W, Hq, G = m["W"], m["Hq"], m["Hq"] // m["Hkv"]
    caps = (torch.from_numpy(z["head_lens"]).long() - W).tolist()
    ks, vs, ids = oracle.ragged_evict(k, v, score, caps, W)
    assert sum(x.shape[0] for x in ks) == m["rows"]
    for h in range(Hq):
        c = caps[h]
        assert ks[h].shape == (c + W, m["D"])
        st = torch.sort(score[h].float(), descending=True, stable=True).indices[:c]
        assert torch.equal(ids[h], st)
        assert torch.equal(ks[h][:c], k[h // G][st]) and torch.equal(vs[h][:c], v[h // G][st])
        assert torch.equal(ks[h][c:], k[h // G][-W:]) and torch.equal(vs[h][c:], v[h // G][-W:])


def test_torch_chain_stable_rule_equals_oracle(oracle):
    from oracle import torch_chain as tc
    q, k, v = make_inputs(91, 8, 2, 900, 128, torch.bfloat16)
    K, V, Q = tc.repeat_kv(k[None], 4), tc.repeat_kv(v[None], 4), q[None]
    W, B = 32, 160
    score = tc.adakv_scores(K, Q, W, 7, "maxpool")
    for normalize in (True, False):
        cap, idx = tc.adakv_capacities(score, B - W, 0.2, normalize, tie_rule="lowest_index")
        assert cap.tolist() == oracle.adakv_capacities(score[0], B - W, 0.2, normalize).tolist()
        kf, vf, lens = tc.ragged_gather(K, V, idx, cap, W)
        ks, vs, _ = oracle.ragged_evict(k, v, score[0], cap.tolist(), W)
        assert torch.equal(kf, torch.cat(ks)) and torch.equal(vf, torch.cat(vs)) and lens == [int(c) + W for c in cap]


def test_torch_chain_bit_identical_to_reference():
    """The torch restatement reproduces what the reference's AdaKVCluster / HeadKVCluster returned on every golden case
    (recorded by tests/golden/make_golden_adakv.py): scores, flat K/V (sha256) and head lengths."""
    from oracle import torch_chain as tc
    for name in ADAKV + ["adakv_pass_s100_b256_w32_bf16", "headkv_s1024_b128_w32_bf16"]:
        z, m, dt, q, k, v = _load(name)
        G = m["Hq"] // m["Hkv"]
        K, V, Q = tc.repeat_kv(k[None], G), tc.repeat_kv(v[None], G), q[None]
        assert torch.equal(tc.adakv_scores(K, Q, m["W"], m["kernel"], m["pooling"])[0].view(torch.int16), from_u16(z["score"], dt).view(torch.int16)), name
        if m["kind"] == "adakv":
            mk, mv, lens = tc.adakv_update_kv(K, Q, V, m["W"], m["B"], m["kernel"], m["pooling"], m["floor"], m["normalize"])
        else:
            mk, mv, lens = tc.headkv_update_kv(K, Q, V, m["W"], m["B"], torch.tensor(m["head_capacity"]), m["kernel"], m["pooling"])
        assert sha256_of(mk) == m["sha_k_out"] and sha256_of(mv) == m["sha_v_out"], name
        assert lens == z["head_lens"].tolist() and mk.shape[0] == m["rows"], name


# ---------------- host mirror + plugin flow (test backend) ----------------
def _oracle_backend():
    from oracle_backend import OracleBackend
    return OracleBackend()


@pytest.mark.parametrize("name", ["adakv_s1024_b128_w32_bf16_norm", "adakv_s1024_b128_w32_bf16_raw", "adakv_8b_s2048_b256_w8_bf16"])
def test_cluster_update_kv_reference_shape_and_metadata(oracle, name):
    """AdaKVCluster.update_kv with the reference's signature: flat [sum len, D] outputs + the reference's metadata attributes,
    equal to the torch restatement under the stable tie rule (scores differ from torch's only in the softmax rounding class, so
    the comparison feeds the cluster's own scores)."""
    from oracle import torch_chain as tc
    from pyramidkv_b200 import kv_cluster as kc
    z, m, dt, q, k, v = _load(name)
    c = kc.AdaKVCluster(window_size=m["W"], kernel_size=m["kernel"], pooling=m["pooling"], max_capacity_prompt=m["B"], floor=m["floor"],
                        normalize=m["normalize"], layer_idx=0, num_hidden_layers=4, backend=_oracle_backend())
    kf, vf = c.update_kv(k[None], q[None], v[None])
    W, Hq, G = m["W"], m["Hq"], m["Hq"] // m["Hkv"]
    score = oracle.adakv_scores(q, k, W, m["kernel"], m["pooling"])
    caps = oracle.adakv_capacities(score, m["B"] - W, m["floor"], m["normalize"]).tolist()
    assert c.last_capacities == caps and c.head_lens.tolist() == [x + W for x in caps]
    assert c.klen_sum == sum(caps) + W * Hq == kf.shape[0] and c.max_seqlen_k == max(caps) + W
    assert c.cu_klen.tolist() == [0] + torch.cumsum(c.head_lens, 0).tolist() and c.cu_qlen.tolist() == list(range(Hq + 1))
    K, V = tc.repeat_kv(k[None], G), tc.repeat_kv(v[None], G)
    idx = torch.sort(score.float(), dim=-1, descending=True, stable=True).indices[None]
    rk, rv, lens = tc.ragged_gather(K, V, idx, caps, W)
    assert torch.equal(kf, rk) and torch.equal(vf, rv)
    # not compressed: everything is kept, metadata says q_len rows per head
    c2 = kc.AdaKVCluster(window_size=W, max_capacity_prompt=m["S"] + W + 1, floor=0.2, normalize=True, layer_idx=0, num_hidden_layers=4, backend=_oracle_backend())
    kf2, _ = c2.update_kv(k[None], q[None], v[None])
    assert kf2.shape[0] == Hq * m["S"] and c2.head_lens.tolist() == [m["S"]] * Hq


def test_headkv_cluster_and_init_errors(oracle):
    from pyramidkv_b200 import kv_cluster as kc
    z, m, dt, q, k, v = _load("headkv_s1024_b128_w32_bf16")
    hc = torch.tensor([m["head_capacity"]])
    c = kc.HeadKVCluster(window_size=m["W"], kernel_size=m["kernel"], pooling=m["pooling"], max_capacity_prompt=m["B"], layer_idx=0,
                         num_hidden_layers=4, head_capacity=hc, backend=_oracle_backend())
    kf, vf = c.update_kv(k[None], q[None], v[None])
    assert c.head_lens.tolist() == z["head_lens"].tolist() and kf.shape[0] == m["rows"]

    # a head budget above the n = S - W candidates keeps all n (the reference slices sorted_indices[..., :cap], :866-872)
    from oracle import torch_chain as tc
    q2, k2, v2 = make_inputs(17, 4, 4, 200, 128, torch.bfloat16)
    hc2 = torch.tensor([[300, 100, 50, 128]])
    c2 = kc.HeadKVCluster(window_size=8, kernel_size=7, pooling="maxpool", max_capacity_prompt=128, layer_idx=0, num_hidden_layers=4,
                          head_capacity=hc2, backend=_oracle_backend())
    kf2, vf2 = c2.update_kv(k2[None], q2[None], v2[None])
    _, _, lens = tc.headkv_update_kv(k2[None], q2[None], v2[None], 8, 128, hc2[0], 7, "maxpool")
    assert c2.head_lens.tolist() == lens == [200, 108, 58, 136] and kf2.shape[0] == sum(lens) == vf2.shape[0]
    assert set(map(tuple, kf2[:200].view(torch.int16).tolist())) == set(map(tuple, k2[0].view(torch.int16).tolist()))   # head 0 kept every row

    class Cfg:
        num_hidden_layers = 4

    class Mod:
        config, layer_idx = Cfg(), 0
    with pytest.raises(ValueError, match="Must have head_capacity"):       # pyramidkv_utils.py:1073
        kc.init_headkv(Mod())
    mod = Mod()
    mod.config.floor = 0.3
    kc.init_adakv(mod)                                                      # defaults :1035-1046
    cfg = mod.config
    assert (cfg.window_size, cfg.max_capacity_prompt, cfg.kernel_size, cfg.pooling, cfg.floor_ratio, cfg.normalize) == (32, 2048, 5, "maxpool", 0.2, True)
    first = mod.kv_cluster
    kc.init_adakv(mod)
    assert mod.kv_cluster is first and first.floor_ratio == 0.3             # built once (:1049), floor read from config.floor


@pytest.mark.parametrize("method", ["adakv", "headkv"])
def test_ragged_methods_through_the_plugin_flow(oracle, method):
    """replace_llama(method) + HF generate on a tiny model (test backend): per-head row counts grow by one per token, the static
    loop produces the same tokens, and the decode step equals attention over each head's own rows."""
    from oracle_backend import OracleBackend
    from pyramidkv_b200 import generate as G, runner
    from pyramidkv_b200.cache import PkvRaggedCacheLayer
    runner.patch(method)
    try:
        model = runner.build_model("tiny-llama", torch.device("cpu"), torch.bfloat16, "eager")
        L, Hq = model.config.num_hidden_layers, model.config.num_attention_heads
        cfg = model.config
        cfg.window_size, cfg.max_capacity_prompt, cfg.kernel_size, cfg.pooling, cfg.floor, cfg.normalize = 8, 40, 7, "maxpool", 0.2, True
        if method == "headkv":
            cfg.head_capacity = torch.tensor([[5 + 3 * ((l + h) % 7) for h in range(Hq)] for l in range(L)])
        for layer in model.model.layers:
            layer.self_attn._pkv_backend = OracleBackend()
        ids = runner.synthetic_prompt(cfg.vocab_size, 150, 21, torch.device("cpu"))
        new = 6
        with torch.no_grad():
            out = model.generate(ids, attention_mask=torch.ones_like(ids), max_new_tokens=new, min_new_tokens=new, num_beams=1,
                                 do_sample=False, pad_token_id=0, return_dict_in_generate=True)
        for l, layer in enumerate(out.past_key_values.layers):
            assert isinstance(layer, PkvRaggedCacheLayer) and layer.appended == new - 1
            caps = model.model.layers[l].self_attn.kv_cluster.last_capacities
            assert layer.head_rows_host == [c + 8 for c in caps]
            if method == "headkv":
                assert caps == cfg.head_capacity[l].tolist()
            else:
                assert abs(sum(caps) - Hq * 32) <= Hq                       # sum of budgets = H * base up to the per-head rounding
            kh, vh = layer.head_view(0)
            assert kh.shape[0] == caps[0] + 8 + new - 1
        seq = G.greedy_generate(model, ids, new)
        assert seq.tolist() == out.sequences.tolist()
        # short prompt: nothing is compressed, the layer is a plain (uniform) compacted cache
        short = runner.synthetic_prompt(cfg.vocab_size, 30, 22, torch.device("cpu"))
        with torch.no_grad():
            o2 = model.generate(short, attention_mask=torch.ones_like(short), max_new_tokens=2, min_new_tokens=2, num_beams=1,
                                do_sample=False, pad_token_id=0, return_dict_in_generate=True)
        assert not isinstance(o2.past_key_values.layers[0], PkvRaggedCacheLayer) and o2.past_key_values.layers[0].length == 31
    finally:
        from pyramidkv.monkeypatch import restore
        restore()
