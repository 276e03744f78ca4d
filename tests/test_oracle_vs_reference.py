"""CPU: the oracle restatement against the unmodified reference, stage by stage with amplified inputs (end-to-end
parity alone is blind to e.g. a wrong GELU variant in corr_mlp, SURVEY Appendix A).  The reference's outputs on these
seeded inputs are pinned in tests/golden/reference_units.npz (oracle/make_golden.py); larger arrays keep every
THIN-th element."""
import pytest
import torch

from cases import O, load_golden
from oracle.make_golden import UNIT_TIME_LENGTHS, thin, unit_inputs


@pytest.fixture(scope="module")
def ref():
    sd, x = unit_inputs()
    return load_golden("reference_units"), sd, x


def test_updateformer_amplified(ref):
    want, sd, x = ref
    with torch.no_grad():
        got = thin(O.updateformer(sd, x["updateformer"]))
    assert float((got - want["updateformer"]).abs().max()) < 1e-4 * max(1.0, float(want["updateformer"].abs().max()))


def test_corr_volume_and_corr_mlp_amplified(ref):
    want, sd, x = ref
    with torch.no_grad():
        got = O.correlation_volume(x["corr_fmap"][0], x["corr_support"][0], x["corr_coords"])
        assert float((thin(got) - want["corr_volume"]).abs().max()) < 1e-4
        big = x["corr_mlp_in"]                                      # out of the regime where erf == tanh GELU
        assert torch.allclose(thin(O.mlp(sd, "corr_mlp", big, "none")), want["corr_mlp"], atol=1e-4)
        assert not torch.allclose(thin(O.mlp(sd, "corr_mlp", big, "tanh")), want["corr_mlp"], atol=1e-4)


def test_support_features(ref):
    want, sd, x = ref
    with torch.no_grad():
        got = O.support_features(x["sup_fmap"][0], x["sup_qf"][0], x["sup_qc"][0])
    assert float((thin(got) - want["support"]).abs().max()) < 1e-5


def test_posenc_and_time_embedding(ref):
    want, sd, x = ref
    assert torch.equal(O.posenc(x["posenc"]), want["posenc"])
    for t in UNIT_TIME_LENGTHS:
        assert torch.allclose(thin(O.time_embedding(sd, t)), want[f"time_embed{t}"], atol=0)


def test_encoder_and_pyramid(ref):
    want, sd, x = ref
    with torch.no_grad():
        assert float((thin(O.encoder(sd, x["encoder"])) - want["encoder"]).abs().max()) < 1e-4


def test_offline_forward_live(ref):
    want, sd, x = ref
    wc, wv = want["coords"], want["vis"]
    with torch.no_grad():
        gc, gv, gq = O.offline_forward(sd, x["video"], x["queries"], iters=3)
    assert float((gc - wc).abs().max()) < 1e-4 and float((gv - wv).abs().max()) < 1e-5
    assert float((wc[0, -1] - wc[0, 0]).abs().max()) > 0.5   # tracks move
