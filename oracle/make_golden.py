"""Generate tests/golden/*.pt by RUNNING THE UNMODIFIED REFERENCE in the build container.

TEST INFRASTRUCTURE.  Usage (only where /root/reference exists):

    python -m oracle.make_golden            # writes tests/golden/esvit_small.pt and esvit_small_w14.pt

The step loop below is main_esvit.py:541-590 driven through the reference's own
modules (SwinTransformer.forward, DINOHead, DINOLoss/DDINOLoss, utils.clip_gradients,
utils.cancel_gradients_last_layer, utils.get_params_groups, torch.optim.AdamW, the EMA
loop) on CPU fp32 (the fp32 branch of train_one_epoch, with the undefined `model` at
:571 read as `student`).  The oracle is asserted against every stored vector while the
file is written, so a committed fixture is also a record that the oracle matched.
"""
from __future__ import annotations

import os
import sys
import warnings

import torch

from . import losses as L
from . import reference_import as R
from . import step as ST
from . import swin as S

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

SMALL = dict(img_size=112, embed_dim=32, depths=(2, 2, 2), num_heads=(1, 2, 4), window_size=7)
# ws = 14 geometry (Swin-S/B W14 configs): 112^2 -> 28x28 tokens = 2x2 windows of 14 (+ shift 7), then ONE un-shifted 14x14
# window (:206-209), then 7x7; 48^2 local crops -> 12 / 6 / 3 tokens, i.e. heavily padded windows
SMALL_W14 = dict(img_size=112, embed_dim=32, depths=(2, 2, 2), num_heads=(1, 2, 4), window_size=14)
HEAD = dict(hidden_dim=128, bottleneck_dim=64)
K = 384
INIT_SEED = 0
HP = dict(lr=5e-4, weight_decay=0.04, clip_grad=3.0, freeze_last_layer=1, momentum_teacher=0.996,
          teacher_temp=0.04, student_temp=0.1, center_momentum=0.9)


def build(dense: bool, small=None):
    """The reference's own modules, initialised with the seeded weights of ST.synthetic_state_dict (the fixture stores
    the seed and the layout, not the weights)."""
    ns = R.load()
    spec = S.SwinSpec(use_dense_prediction=dense, **(small or SMALL))
    m = R.build_swin(spec, K)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m.head = ns.DINOHead(m.num_features, K, **HEAD)
        if dense:
            m.head_dense = ns.DINOHead(m.num_features, K, **HEAD)
    ref = m.state_dict()
    sd = ST.synthetic_state_dict([(k, tuple(v.shape)) for k, v in ref.items()], INIT_SEED)
    for k, v in ref.items():
        assert sd[k].dtype == v.dtype and (v.dtype.is_floating_point or torch.equal(sd[k], v)), k
    m.load_state_dict(sd)
    return ns, spec, m


def reference_steps(ns, m_student, m_teacher, loss_mod, crops, nsteps, dense):
    params_groups = ns.get_params_groups(m_student)
    opt = torch.optim.AdamW(params_groups)
    rec = []
    for it in range(nsteps):
        for i, pg in enumerate(opt.param_groups):
            pg["lr"] = HP["lr"]
            if i == 0:
                pg["weight_decay"] = HP["weight_decay"]
        teacher_output = m_teacher(crops[:2])
        student_output = m_student(crops)
        loss = loss_mod(student_output, teacher_output, 0, None)
        opt.zero_grad()
        loss.backward()
        grads = {n: p.grad.detach().clone() for n, p in m_student.named_parameters() if p.grad is not None}
        ns.clip_gradients(m_student, HP["clip_grad"])
        ns.cancel_gradients_last_layer(0, m_student, HP["freeze_last_layer"])
        opt.step()
        with torch.no_grad():
            mm = HP["momentum_teacher"]
            for param_q, param_k in zip(m_student.parameters(), m_teacher.parameters()):
                param_k.data.mul_(mm).add_((1 - mm) * param_q.detach().data)
        rec.append(dict(loss=float(loss), student_output=student_output, teacher_output=teacher_output,
                        grads=grads))
    return rec


FULL_GRADS = ("patch_embed.proj.weight", "patch_embed.norm.weight", "layers.0.blocks.1.attn.relative_position_bias_table",
              "layers.0.blocks.1.attn.qkv.weight", "layers.1.blocks.1.attn.qkv.bias", "layers.1.blocks.0.mlp.fc1.weight",
              "layers.1.downsample.reduction.weight", "layers.1.downsample.norm.bias", "layers.2.blocks.1.attn.proj.weight",
              "norm.weight", "head.mlp.4.weight", "head.last_layer.weight_v", "head_dense.mlp.0.weight",
              "head_dense.last_layer.weight_v")


def stats(d):
    return {k: (float(v.double().sum()), float(v.double().norm())) for k, v in d.items()}


def make(dense: bool, sd_init=None, small=None, compact: bool = False):
    """The fixture keeps the seeds and the layout of the inputs (crops and weights are regenerated from them), losses,
    centers, sums and norms of every gradient / parameter / output and a seeded sample of the elements of a few of them.
    compact: no teacher outputs or region-match indices."""
    small = small or SMALL
    R.ensure_process_group()
    ns, spec, student = build(dense, small=small)
    if sd_init is not None:  # the view-only fixture shares the dense fixture's backbone + `head` weights
        student.load_state_dict({k: v for k, v in sd_init.items() if not k.startswith("head_dense")})
    _, _, teacher = build(dense, small=small)
    teacher.load_state_dict(student.state_dict())
    for p in teacher.parameters():
        p.requires_grad = False
    sd0 = {k: v.detach().clone() for k, v in student.state_dict().items()}
    B, n_local = 2, 3
    ncrops = 2 + n_local if dense else 2
    crops = ST.synthetic_crops(B, n_local, seed=1234, global_size=112, local_size=48)
    if not dense:
        crops = crops[:2]
    Loss = ns.DDINOLoss if dense else ns.DINOLoss
    loss_mod = Loss(K, ncrops, 0.04, HP["teacher_temp"], 0, 10, HP["student_temp"], HP["center_momentum"])
    nsteps = 2
    rec = reference_steps(ns, student, teacher, loss_mod, crops, nsteps, dense)

    # ---- the oracle must reproduce all of it -------------------------------------------------
    orc = ST.OracleStep(sd0, spec, ncrops, K, **HP)
    o_losses = []
    for it in range(nsteps):
        o_losses.append(orc.step(crops, epoch=0, keep_grads=(it == 0)))
    for a, b in zip(o_losses, [r["loss"] for r in rec]):
        assert abs(a - b) < 2e-5 * max(1, abs(b)), (a, b)
    for k, g in rec[0]["grads"].items():
        og = orc.grads_step[k]
        assert torch.allclose(og, g, atol=1e-7 + 1e-4 * float(g.abs().max()), rtol=1e-3), k
    sd_s, sd_t = student.state_dict(), teacher.state_dict()
    for k in orc.names:
        # AdamW's first steps are ~lr*sign(g): ill-conditioned where g ~ 0, so the bulk must agree
        # tightly and the outliers are bounded by nsteps*lr.
        d = (orc.student[k].detach() - sd_s[k]).abs()
        assert float(d.max()) <= 2.2 * HP["lr"] and float((d < 2e-5).float().mean()) > 0.98, (k, float(d.max()))
        d = (orc.teacher[k] - sd_t[k]).abs()
        assert float(d.max()) < 1e-5, k
    assert torch.allclose(orc.center, loss_mod.center, atol=1e-6)

    r0 = rec[0]
    so, to = r0["student_output"], r0["teacher_output"]
    outputs = dict(s_cls=so[0], s_region=so[1], s_fea=so[2]) if dense else dict(s_out=so, t_out=to)
    if dense and not compact:
        outputs.update(t_cls=to[0], t_region=to[1], t_fea=to[2])
    outputs = {k: v.detach() for k, v in outputs.items()}
    out = dict(
        meta=dict(spec=dict(small, use_dense_prediction=dense), head=HEAD, out_dim=K, batch=B,
                  n_local=n_local if dense else 0, ncrops=ncrops, hp=HP, nsteps=nsteps,
                  crop_seed=1234, global_size=112, local_size=48,
                  init_seed=INIT_SEED, layout=[(k, tuple(v.shape)) for k, v in sd0.items()],
                  generator="oracle/make_golden.py (reference run on CPU fp32, torch %s)" % torch.__version__),
        losses=[r["loss"] for r in rec], center_after=loss_mod.center.clone(),
        final_student_stats=stats({k: sd_s[k] for k in orc.names}),
        final_teacher_stats=stats({k: sd_t[k] for k in orc.names}),
        final_teacher_sample={k: ST.sample_elements(sd_t[k]) for k in FULL_GRADS if k in sd_t},
        grads_step0_stats=stats(r0["grads"]),
        grads_step0_sample={k: ST.sample_elements(r0["grads"][k]) for k in FULL_GRADS if k in r0["grads"]},
        out_stats=stats(outputs), out_sample={k: ST.sample_elements(v) for k, v in outputs.items()},
    )
    if dense:
        out["s_npatch"] = list(so[3])
    if dense and not compact:
        out.update(t_npatch=list(to[3]), center_grid_after=loss_mod.center_grid.clone())
        # argmax indices of the first step, recomputed with the reference's own expression (main_esvit.py:735-736)
        Bn, N = B, to[3][0]
        split = [so[3][0]] * 2 + [so[3][1]] * (ncrops - 2)
        s_f = torch.split(so[2].detach(), [i * Bn for i in split], dim=0)
        t_f = to[2].detach().chunk(2)
        idx = {}
        for iq in range(2):
            for v in range(ncrops):
                if v == iq:
                    continue
                a = torch.nn.functional.normalize(s_f[v].view(Bn, split[v], -1), p=2, dim=-1)
                b = torch.nn.functional.normalize(t_f[iq].view(Bn, N, -1), p=2, dim=-1)
                idx[(iq, v)] = torch.matmul(a, b.permute(0, 2, 1)).max(dim=2)[1]
                assert torch.equal(idx[(iq, v)], orc.indices_step[(iq, v)])
        out["indices"] = idx
        assert torch.allclose(orc.center_grid, loss_mod.center_grid, atol=1e-6)
    return out


if __name__ == "__main__":
    if not R.available():
        sys.exit("reference tree not found; golden vectors can only be generated in the build container")
    dense = make(True)
    view = make(False, ST.synthetic_state_dict(dense["meta"]["layout"], INIT_SEED))
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "esvit_small.pt")
    torch.save(dict(dense=dense, view=view), path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB; losses", dense["losses"], view["losses"])
    w14 = make(True, small=SMALL_W14, compact=True)
    path = os.path.join(OUT, "esvit_small_w14.pt")
    torch.save(dict(dense=w14), path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB; losses", w14["losses"])
