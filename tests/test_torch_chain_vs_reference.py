"""CPU: the restated torch op chain (oracle/torch_chain.py) is bit-identical to the unmodified reference classes. The
reference's own outputs on every golden case are stored in tests/golden (tests/golden/make_golden.py): the selected
indices and the sha256 of the K/V that `update_kv` returned."""
import pytest
import torch

from golden_util import GoldenCase, golden_names, sha256_of


@pytest.mark.parametrize("name", golden_names())
def test_chain_equals_reference(name):
    from oracle import torch_chain as tc
    g = GoldenCase(name)
    m = g.meta
    G = m["Hq"] // m["Hkv"]
    K, V, Q = tc.repeat_kv(g.k[None], G), tc.repeat_kv(g.v[None], G), g.q[None]
    assert torch.equal(K[0], g.k.repeat_interleave(G, dim=0))
    ck, cv, idx = tc.update_kv(m["method"], K, Q, V, m["W"], m["B"], m["kernel"], m["pooling"], m["L"], m["layer"], return_indices=True)
    assert ck.shape[2] == m["k_rows"]
    if g.has("idx"):
        assert torch.equal(idx[0], g.t("idx"))
    assert sha256_of(ck[0]) == m["sha_k_out"] and sha256_of(cv[0]) == m["sha_v_out"]
