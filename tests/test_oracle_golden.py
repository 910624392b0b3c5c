"""CPU: the oracle restatement reproduces the golden vectors that the UNMODIFIED reference produced
(tests/golden/esvit_small.pt, written by oracle/make_golden.py): losses, centers and indices whole; outputs, gradients
and teacher weights by sum and norm and by a seeded sample of their elements."""
import pytest
import torch

from helpers import assert_matches_sample, assert_matches_stats, load_fixture
from oracle import losses as L
from oracle import step as ST
from oracle import swin as S


@pytest.fixture(scope="module")
def G():
    return load_fixture()


def _spec(G, dense):
    return S.SwinSpec(**dict(G["dense"]["meta"]["spec"], use_dense_prediction=dense))


def test_oracle_forward_matches_reference(G):
    D = G["dense"]
    spec = _spec(G, True)
    with torch.no_grad():
        s = S.multicrop_forward(D["crops"], D["state_dict"], spec)
        t = S.multicrop_forward(D["crops"][:2], D["state_dict"], spec)
    for a, k in zip(s[:3] + t[:3], ("s_cls", "s_region", "s_fea", "t_cls", "t_region", "t_fea")):
        assert_matches_sample(a, D["out_sample"][k], 2e-5, 1e-4, k)
        assert_matches_stats(a, D["out_stats"][k], 1e-5, k)
    assert s[3] == D["s_npatch"] and t[3] == D["t_npatch"]


def test_oracle_region_match_indices_bit_exact(G):
    """on the oracle's features (test_oracle_forward_matches_reference pins them to the reference's)"""
    D = G["dense"]
    B, ncrops = D["meta"]["batch"], D["meta"]["ncrops"]
    Tg, Tl = D["s_npatch"]
    split = [Tg * B] * 2 + [Tl * B] * (ncrops - 2)
    with torch.no_grad():
        s_fea = S.multicrop_forward(D["crops"], D["state_dict"], _spec(G, True))[2]
        t_fea = S.multicrop_forward(D["crops"][:2], D["state_dict"], _spec(G, True))[2]
    sf = torch.split(s_fea, split)
    tf = t_fea.chunk(2)
    for (iq, v), ref in D["indices"].items():
        T = Tg if v < 2 else Tl
        assert torch.equal(L.region_match(sf[v].view(B, T, -1), tf[iq].view(B, Tg, -1)), ref)


@pytest.mark.parametrize("dense", [True, False])
def test_oracle_training_steps_match_reference(G, dense):
    D = G["dense" if dense else "view"]
    sd = {k: v for k, v in G["dense"]["state_dict"].items() if dense or not k.startswith("head_dense")}
    crops = G["dense"]["crops"] if dense else G["dense"]["crops"][:2]
    orc = ST.OracleStep(sd, _spec(G, dense), D["meta"]["ncrops"], D["meta"]["out_dim"], **D["meta"]["hp"])
    losses = [orc.step(crops, epoch=0, keep_grads=(i == 0)) for i in range(D["meta"]["nsteps"])]
    for a, b in zip(losses, D["losses"]):
        assert abs(a - b) < 2e-5 * max(1.0, abs(b))
    for k, g in D["grads_step0_sample"].items():
        assert_matches_sample(orc.grads_step[k], g, 1e-7 + 1e-4 * float(g.abs().max()), 1e-3, k)
    for k, (ssum, nrm) in D["grads_step0_stats"].items():
        assert abs(float(orc.grads_step[k].double().norm()) - nrm) < 1e-3 * nrm + 1e-9, k
    assert torch.allclose(orc.center, D["center_after"], atol=1e-6)
    if dense:
        assert torch.allclose(orc.center_grid, D["center_grid_after"], atol=1e-6)
    for k, v in D["final_teacher_sample"].items():
        assert_matches_sample(orc.teacher[k], v, 1e-5, 0.0, k)
    for k, st in D["final_teacher_stats"].items():
        assert_matches_stats(orc.teacher[k], st, 1e-5, k)


def test_closed_forms():
    # rel-pos index & shift mask closed forms against the textbook construction
    ws = 7
    coords = torch.stack(torch.meshgrid(torch.arange(ws), torch.arange(ws), indexing="ij")).flatten(1)
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws - 1
    rel[:, :, 1] += ws - 1
    rel[:, :, 0] *= 2 * ws - 1
    assert torch.equal(rel.sum(-1), S.rel_pos_index(ws))
    m = S.shift_mask(6, 6, 7, 3)
    assert m.shape == (1, 49, 49) and float((m != 0).float().mean()) > 0.5


def test_oracle_w14_training_steps_match_reference():
    """ws = 14 geometry (Swin-S/B W14 configs: 2x2 shifted windows of 14, the single un-shifted 14x14 window of
    :206-209, heavily padded local-crop windows): losses, gradients, teacher EMA and centers of two training steps of the
    executed reference (tests/golden/esvit_small_w14.pt; weights and crops regenerated from their seeds)."""
    D = load_fixture("esvit_small_w14.pt")["dense"]
    M = D["meta"]
    spec = S.SwinSpec(**M["spec"])
    crops = D["crops"]
    with torch.no_grad():
        s = S.multicrop_forward(crops, D["state_dict"], spec)
    assert s[3] == D["s_npatch"]
    for a, k in zip(s[:3], ("s_cls", "s_region", "s_fea")):
        ssum, nrm = D["out_stats"][k]
        assert abs(float(a.double().norm()) - nrm) < 1e-4 * nrm, k
        assert abs(float(a.double().sum()) - ssum) < 1e-4 * nrm, k
        assert_matches_sample(a, D["out_sample"][k], 2e-5, 1e-4, k)
    orc = ST.OracleStep(D["state_dict"], spec, M["ncrops"], M["out_dim"], **M["hp"])
    losses = [orc.step(crops, epoch=0, keep_grads=(i == 0)) for i in range(M["nsteps"])]
    for a, b in zip(losses, D["losses"]):
        assert abs(a - b) < 2e-5 * max(1.0, abs(b))
    for k, g in D["grads_step0_sample"].items():
        assert_matches_sample(orc.grads_step[k], g, 1e-7 + 1e-4 * float(g.abs().max()), 1e-3, k)
    for k, (ssum, nrm) in D["grads_step0_stats"].items():
        assert abs(float(orc.grads_step[k].double().norm()) - nrm) < 1e-3 * nrm + 1e-9, k
    assert torch.allclose(orc.center, D["center_after"], atol=1e-6)
    for k, v in D["final_teacher_sample"].items():
        assert_matches_sample(orc.teacher[k], v, 1e-5, 0.0, k)
    for k, st in D["final_teacher_stats"].items():
        assert_matches_stats(orc.teacher[k], st, 1e-5, k)
