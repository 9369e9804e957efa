"""CPU: the oracle restatement against the UNMODIFIED reference.  The comparisons run against the
reference's own outputs stored under tests/golden (oracle/make_golden.py), so they run everywhere.
Only the key-by-key state_dict comparison (order, dtypes) is live and needs a reference checkout
(oracle/ref_shim.py, e.g. VQAE_REFERENCE_ROOT)."""
import numpy as np
import pytest
import torch

import helpers as H
import ref_shim
import vqae_oracle as O


def test_l4_not_l2():
    """The reference's metric is L4 (p = inputs.dim() = 4, vq.py:97,121-129), not Euclidean: the
    codes its EMAVectorQuantizer returned (quantizer.npz, bare case) are the L4 argmin."""
    g = H.golden("quantizer")
    x, embed = torch.from_numpy(g["bare_x"]), torch.from_numpy(g["bare_embed"])
    idx = torch.from_numpy(g["bare_idx"].astype(np.int64))
    flat = x.permute(0, 2, 3, 1).reshape(-1, 8)
    assert torch.equal(idx.reshape(-1), torch.cdist(flat, embed, 4).argmin(1))
    assert (idx.reshape(-1) != torch.cdist(flat, embed, 2).argmin(1)).float().mean() > 0.05
    _, o_idx, _, _ = O.ema_quantizer_forward(x, embed, 1.0)
    assert torch.equal(o_idx, idx)


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference checkout not available")
def test_state_dict_layout_matches_reference():
    import vqae_b200
    from vqae_b200.config import compose_vqae_conf
    model_mod = ref_shim.load_reference()[0]
    for n_down, n_params in ((3, 4934287), (4, 19750707)):      # SURVEY.md 8c cross-check
        conf = compose_vqae_conf(n_down=n_down)
        conf.pop("_target_"), conf.pop("_recursive_")
        r = model_mod.VQAE(**conf)
        m = vqae_b200.build_vqae(n_down=n_down)
        rs, ms = r.state_dict(), m.state_dict()
        assert list(rs.keys()) == list(ms.keys())
        assert all(rs[k].shape == ms[k].shape and rs[k].dtype == ms[k].dtype for k in rs)
        assert sum(p.numel() for p in m.parameters()) == n_params
        m.load_state_dict(rs)                                     # loads unchanged


@pytest.mark.parametrize("n_down, tag, n_params", [(3, "model_nd3_perturbed", 4934287),
                                                   (4, "model_nd4_perturbed_256", 19750707)])
def test_state_dict_size_matches_reference(n_down, tag, n_params):
    """The reference's parameter count (SURVEY.md 8c) and state_dict entry count (n_state, stored by
    oracle/make_golden.py from the reference's own state_dict).  Names and shapes of every entry the
    forward reads are pinned by test_oracle_equals_stored_reference: synthetic weights are seeded by
    key name, so weights made from this package's keys reproduce the reference's stored outputs only
    where name and shape agree."""
    import vqae_b200
    m = vqae_b200.build_vqae(n_down=n_down)
    assert sum(p.numel() for p in m.parameters()) == n_params
    assert len(m.state_dict()) == int(H.golden(tag)["n_state"])


def test_fixup_init_distribution_matches_reference():
    """Same Fixup initialisation rules (conv_block.py:218-237): conv3 = 0, conv1 std."""
    import vqae_b200
    m = vqae_b200.build_vqae(n_down=3)
    blk = m.encoder.pre_enc_layers[0][0]
    assert float(blk.branch_conv3.weight.abs().max()) == 0.0
    expected = np.sqrt(2 / 64) * 124 ** -0.5
    assert abs(float(blk.branch_conv1.weight.std()) - expected) / expected < 0.1


@pytest.mark.parametrize("tag", ["model_nd3_perturbed", "model_nd3_fixup", "model_nd4_perturbed_256"])
def test_oracle_equals_stored_reference(tag):
    """The oracle against the reference's own VQAE outputs for the same weights and input: codes
    exact, quantised latents (sampled as stored), reconstruction and loss to fp32 rounding."""
    _, sd, x = H.model_and_state(tag)
    g = H.golden(tag)
    with torch.no_grad():
        (o_enc,), (o_idx,), (o_loss,) = O.encoder_forward(x, sd)
        o_recon = O.decoder_forward((o_enc,), sd)
    assert np.array_equal(o_idx.numpy(), g["idx"].astype(np.int64))
    assert H.rel_err(o_enc[:, ::8, ::4, ::4], torch.from_numpy(g["enc_sub"])) < 1e-6
    assert H.rel_err(o_recon[:, :, ::8, ::8], torch.from_numpy(g["recon_sub"])) < 1e-5
    assert abs(o_loss.item() - float(g["loss"])) < 1e-7
