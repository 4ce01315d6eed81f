"""GPU parity: K4 fused PPO loss, K7 optimiser step and PPO_Learner.update vs the torch-CPU oracle."""
import numpy as np
import pytest
import torch

from helpers import build_product_ppo_model, ppo_config
from oracle.learners import PPOLearnerOracle, ppo_clip_terms
from oracle.nets import SharedActorCriticOracle

pytestmark = pytest.mark.gpu


def _loss_inputs(rng, B, A, clip_heavy=False):
    logits = rng.normal(size=(B, A)).astype(np.float32) * 2
    value = rng.normal(size=B).astype(np.float32)
    act = rng.integers(0, A, size=B).astype(np.float32)
    ret = rng.normal(size=B).astype(np.float32)
    adv = rng.normal(size=B).astype(np.float32)
    adv[:3] = 0.0
    old = (rng.normal(size=B) * (1.0 if clip_heavy else 0.1) - np.log(A)).astype(np.float32)
    return logits, value, act, ret, adv, old


@pytest.mark.parametrize("B,A", [(8192, 4), (1000, 6), (257, 18), (64, 2), (33, 40)])
def test_ppo_loss_kernel_matches_torch_autograd(B, A):
    from xuance_b200 import _lib
    rng = np.random.default_rng(B + A)
    logits, value, act, ret, adv, old = _loss_inputs(rng, B, A, clip_heavy=(A == 6))
    clip, vf, ent = 0.2, 0.25, 0.01
    # oracle: torch autograd on CPU of ppo_learner.py:46-60
    lt = torch.tensor(logits, requires_grad=True)
    vt = torch.tensor(value, requires_grad=True)
    a_loss, c_loss, e_loss, ratio = ppo_clip_terms(lt, vt, torch.tensor(act), torch.tensor(ret), torch.tensor(adv),
                                                   torch.tensor(old), clip)
    loss = a_loss - ent * e_loss + vf * c_loss
    loss.backward()
    cr = ((ratio < 1 - clip).sum() + (ratio > 1 + clip).sum()) / ratio.shape[0]
    dev = "cuda:0"
    t_in = [torch.tensor(x, device=dev) for x in (logits, value, act, old, adv, ret)]   # keep alive across launches
    dl = torch.empty((B, A), device=dev)
    dv = torch.empty(B, device=dev)
    stats = torch.zeros(8, device=dev)
    scratch = _lib.scratch(torch.device(dev))
    for _ in range(2):   # twice: the ticket counter must re-arm
        _lib.call("xb_ppo_loss_fwd_bwd", *[_lib.ptr(t) for t in t_in], B, A, B, clip, vf, ent, 0, _lib.ptr(dl),
                  _lib.ptr(dv), _lib.ptr(stats), _lib.ptr(scratch))
    s = stats.cpu().numpy()
    np.testing.assert_allclose(s[0], a_loss.item(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(s[1], c_loss.item(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(s[2], e_loss.item(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(s[3], vt.mean().item(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(s[4], cr.item(), rtol=0, atol=1e-7)
    np.testing.assert_allclose(s[5], loss.item(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(dl.cpu().numpy(), lt.grad.numpy(), rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(dv.cpu().numpy(), vt.grad.numpy(), rtol=1e-5, atol=1e-10)


def test_fused_adam_matches_torch_adam_with_clip():
    from xuance_b200.torch.utils import FusedAdam
    torch.manual_seed(0)
    shapes = [(32, 4, 8, 8), (32,), (512, 6400), (7,), (3, 5)]
    cpu_params = [torch.nn.Parameter(torch.randn(s) * 0.1) for s in shapes]
    gpu_params = [torch.nn.Parameter(p.detach().clone().cuda()) for p in cpu_params]
    opt_c = torch.optim.Adam(cpu_params, 2.5e-4, eps=1e-5)
    opt_g = FusedAdam(gpu_params, 2.5e-4, eps=1e-5)
    sch_c = torch.optim.lr_scheduler.LinearLR(opt_c, 1.0, 0.5, total_iters=10)
    sch_g = torch.optim.lr_scheduler.LinearLR(opt_g, 1.0, 0.5, total_iters=10)
    for it in range(6):
        grads = [torch.randn(s) * (3.0 if it % 2 == 0 else 0.001) for s in shapes]
        opt_c.zero_grad(), opt_g.zero_grad()
        for p, q, g in zip(cpu_params, gpu_params, grads):
            p.grad = g.clone()
            q.grad.copy_(g)
        total = torch.nn.utils.clip_grad_norm_(cpu_params, 0.5)
        opt_c.step(), sch_c.step()
        opt_g.step(max_norm=0.5), sch_g.step()
        np.testing.assert_allclose(float(opt_g.grad_norm), float(total), rtol=3e-4)  # torch sums 3.3M squares in fp32; K7 in fp64
        assert opt_g.param_groups[0]["lr"] == opt_c.param_groups[0]["lr"]
        for p, q in zip(cpu_params, gpu_params):
            np.testing.assert_allclose(q.detach().cpu().numpy(), p.detach().numpy(), rtol=2e-5, atol=2e-7)
    sd = opt_g.state_dict()
    assert set(sd["state"][0].keys()) >= {"step", "exp_avg", "exp_avg_sq"}
    np.testing.assert_allclose(sd["state"][2]["exp_avg"].cpu().numpy(), opt_c.state_dict()["state"][2]["exp_avg"].numpy(),
                               rtol=1e-4, atol=1e-8)


@pytest.mark.parametrize("compute,tol", [("fp32", 2e-4)])
def test_ppo_learner_update_matches_oracle(compute, tol):
    """Three consecutive updates on identical inputs / initial weights: info terms, then parameters."""
    from xuance_b200.torch.learners import PPO_Learner
    from xuance_b200.common import BaseCallback
    torch.manual_seed(1)
    A, B = 6, 256
    oracle_model = SharedActorCriticOracle(A)
    model = build_product_ppo_model(A, "cuda:0")
    model.load_state_dict(oracle_model.state_dict())         # same parameter names as the reference
    model.representation.set_compute(compute)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = ppo_config("cuda:0", running_steps=256 * 128 * 10)
    learner = PPO_Learner(cfg, model, BaseCallback())
    orc = PPOLearnerOracle(oracle_model, end_factor_lr_decay=0.5, total_iters=learner.total_iters)
    rng = np.random.default_rng(5)
    for it in range(3):
        samples = {
            "obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8),
            "actions": rng.integers(0, A, size=B).astype(np.float32),
            "returns": rng.normal(size=B).astype(np.float32),
            "advantages": rng.normal(size=B).astype(np.float32),
            "aux_batch": {"old_logp": (rng.normal(size=B) * 0.05 - np.log(A)).astype(np.float32)},
            "values": rng.normal(size=B).astype(np.float32), "batch_size": B,
        }
        info_o = orc.update(**samples)
        dev_samples = dict(samples, obs=torch.from_numpy(samples["obs"]).cuda())
        info_p = learner.update(**dev_samples)
        for k in ("actor_loss", "critic_loss", "entropy", "predict_value"):
            np.testing.assert_allclose(info_p[k], info_o[k], rtol=tol, atol=1e-5, err_msg=k)
        assert info_p["learning_rate"] == info_o["learning_rate"]
        np.testing.assert_allclose(info_p["clip_ratio"], float(info_o["clip_ratio"]), atol=1.0 / B + 1e-7)
    so, sp = oracle_model.state_dict(), model.state_dict()
    for k in so:
        np.testing.assert_allclose(sp[k].cpu().numpy(), so[k].numpy(), rtol=1e-3, atol=1e-4, err_msg=k)  # Adam: |step| ~ lr


@pytest.mark.parametrize("kind", ["a2c", "pg"])
def test_a2c_pg_learners_match_oracle(kind):
    """Sibling learners on the same K4 kernel (loss_kind = 1): A2C and PG (SURVEY.md section 8f-3).  The fp32 encoder's
    convolutions run without cuDNN here: on B200 cuDNN's fp32 weight-gradient algorithm for conv2 is off by enough, on a
    few PG gradient elements near Adam's eps, to move those weights by ~lr after three steps."""
    with torch.backends.cudnn.flags(enabled=False, benchmark=False, deterministic=False, allow_tf32=False):
        _a2c_pg_learners_match_oracle(kind)


def _a2c_pg_learners_match_oracle(kind):
    from xuance_b200.torch.learners import A2C_Learner, PG_Learner
    from xuance_b200.common import BaseCallback
    torch.manual_seed(2)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    A, B = 5, 128
    oracle_model = SharedActorCriticOracle(A)
    model = build_product_ppo_model(A, "cuda:0")
    model.load_state_dict(oracle_model.state_dict())
    cfg = ppo_config("cuda:0", running_steps=256 * 128 * 10)
    learner = (A2C_Learner if kind == "a2c" else PG_Learner)(cfg, model, BaseCallback())
    orc = PPOLearnerOracle(oracle_model, end_factor_lr_decay=0.5, kind=kind,
                           total_iters=cfg.running_steps if kind == "a2c" else learner.total_iters)
    rng = np.random.default_rng(6)
    for it in range(3):
        samples = {"obs": rng.integers(0, 256, size=(B, 84, 84, 4), dtype=np.uint8),
                   "actions": rng.integers(0, A, size=B).astype(np.float32),
                   "returns": rng.normal(size=B).astype(np.float32), "advantages": rng.normal(size=B).astype(np.float32),
                   "aux_batch": {"old_logp": np.zeros(B, np.float32)}, "batch_size": B}
        io = orc.update(**samples)
        ip = learner.update(**dict(samples, obs=torch.from_numpy(samples["obs"]).cuda()))
        np.testing.assert_allclose(ip["actor-loss"], io["actor_loss"], rtol=2e-4, atol=1e-5)
        np.testing.assert_allclose(ip["entropy"], io["entropy"], rtol=2e-4)
        if kind == "a2c":
            np.testing.assert_allclose(ip["critic-loss"], io["critic_loss"], rtol=2e-4, atol=1e-5)
        assert ip["learning_rate"] == io["learning_rate"]
    so, sp = oracle_model.state_dict(), model.state_dict()
    for k in so:
        np.testing.assert_allclose(sp[k].cpu().numpy(), so[k].numpy(), rtol=1e-3, atol=1e-4, err_msg=k)
