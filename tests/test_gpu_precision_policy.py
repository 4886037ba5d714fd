"""GPU: evidence for the precision policy (VERDICT r1 next-round #5).  north_star: ">= 4x the reference's single-GPU
PyTorch renderer ... with matching PSNR / eikonal loss".

Protocol.  One 300-step training run of the reference's fp32 training step on this GPU (clip 0.99 + Adam(eps=1e-7),
deterministic strata, a learnable synthetic scene) is the baseline; its weights are snapshotted at steps 100 / 200 / 300.
The baseline runs the restatement oracle/neuconw_port.py (pinned to the unmodified reference by tests/test_oracle_golden.py),
and its curve is held against tests/golden/precision_curve.npz, the same run of the unmodified reference on a B200
(oracle/make_golden.py): first step within 1e-4, the first 25 steps within 1 %.  The same run (same initial weights,
same batches) is repeated in `bf16x3` (3 bf16 products per GEMM), `mixed` (3 products forward, plain-bf16 backward
GEMMs) and `bf16` (one product everywhere).

 (1) ON IDENTICAL, TRAINED WEIGHTS (each snapshot loaded into the CUDA path): total loss within 5e-4 relative, PSNR within
     0.01 dB, eikonal term within 1e-3 relative for bf16x3 / mixed (their forward passes are the same arithmetic; every
     rendered OUTPUT holds 1e-4 of its range, these are ratios of small differences of outputs), and the flat parameter gradient's
     cosine similarity with the baseline's autograd gradient >= 0.9999 (bf16x3) / >= 0.995 (mixed).  Deterministic.
 (2) TRAJECTORIES: training is chaotic - the runs agree to < 1 % for ~75 steps, then decorrelate (any perturbation of
     the order of fp32 rounding does that, the fp32 reference against itself included), so tail statistics are compared
     within a band that reflects this: mean PSNR of the last 100 steps within 1.0 dB of the unmodified reference's stored
     curve (observed spread over repeated runs of this test: bf16x3 -0.6 .. -0.2 dB, mixed 0.0 .. +0.4 dB); loss and eikonal
     tails are REPORTED (gpurun_out/precision_study.json -> profiles/), not asserted.
`bf16` is reported only."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle import neuconw_port as port
from oracle import synth

pytestmark = pytest.mark.gpu
STEPS, R, LR = 300, 1024, 5e-4
KW = dict(n_samples=32, n_importance=32, up_sample_steps=4, n_outside=4, n_vocab=64)


def _scene_batches(n_batches, seed=0):
    """learnable target: a shaded sphere (radius 0.5) in front of a direction-dependent sky, seen from a camera ring."""
    from nrw.raycache import synthetic_cache

    rays, _ = synthetic_cache(n_batches * R, n_images=32, n_vocab=64, seed=seed)
    o, d = rays[:, 0:3], rays[:, 3:6]
    b = (o * d).sum(-1)
    disc = b * b - ((o * o).sum(-1) - 0.25)
    hit = disc > 0
    t = -b - torch.sqrt(disc.clamp_min(0))
    n = (o + t[:, None] * d) / 0.5
    shade = 0.5 + 0.5 * n
    sky = torch.stack([0.3 + 0.2 * d[:, 1], 0.5 + 0.3 * d[:, 1], 0.8 + 0.1 * d[:, 0]], -1).clamp(0, 1)
    rgb = torch.where(hit[:, None], shade, sky).float()
    label = torch.where(hit, torch.zeros_like(t), torch.full_like(t, 2.0))            # sky label where the ray misses
    out = []
    for i in range(n_batches):
        sl = slice(i * R, (i + 1) * R)
        out.append({"rays": torch.cat([rays[sl, :8], rays[sl, 10:12]], 1).contiguous(), "rgbs": rgb[sl].contiguous(),
                    "ts": rays[sl, 8].long(), "label": label[sl].contiguous()})
    return out


def _make_nrw(mode):
    from nrw.train import TrainSystem

    sysm = TrainSystem(torch.device("cuda", 0), precision=mode, chunk_rows=65536, batch_size=R, canonical_lr=LR, canonical_bs=R, **KW)
    sysm.renderer.perturb = 0.0
    sysm.track_metrics = True
    return sysm


def _run_nrw(mode, batches):
    sysm = _make_nrw(mode)
    init = {k: v.detach().cpu().clone() for k, v in sysm.renderer.engine.named_params()}
    init["embedding_a.weight"] = sysm.embedding_a.weight.detach().cpu().clone()
    hist = []
    for i in range(STEPS):
        sysm.training_step(batches[i % len(batches)])
        hist.append(torch.stack([sysm.last_metrics[k].reshape(()) for k in ("loss", "psnr", "eikonal", "s_val")]))
    return torch.stack(hist).cpu(), init


def _ref_cfg():
    return synth.PathConfig(n_samples=KW["n_samples"], n_importance=KW["n_importance"], up_sample_steps=KW["up_sample_steps"],
                            n_outside=KW["n_outside"], n_vocab=KW["n_vocab"], perturb=0.0, cos_anneal_ratio=0.0, igr_weight=0.0001)


def _initial_weights():
    """the seeded initial weights of the CUDA path (TrainSystem seed), reference state_dict names"""
    sysm = _make_nrw("bf16x3")
    init = {k: v.detach().cpu().clone() for k, v in sysm.renderer.engine.named_params()}
    init["embedding_a.weight"] = sysm.embedding_a.weight.detach().cpu().clone()
    return init


class _PortRunner:
    """What oracle.ref_runner.RefRunner does with the reference's modules, on the restated step: render -> loss ->
    backward -> clip_grad_norm_(0.99) -> Adam(eps=1e-7)."""

    def __init__(self, cfg, init, device):
        self.cfg = cfg
        self.P = {k: v.to(device).clone() for k, v in init.items()}
        self.optimizer = torch.optim.Adam(list(self.P.values()), lr=LR, eps=1e-7, weight_decay=0)

    def train_step(self, batch):
        res, loss, self.grads = port.train_step(self.P, self.cfg, batch, perturb_overwrite=0)
        with torch.no_grad():
            mse = ((res["color"].detach() - batch["rgbs"]) ** 2).mean()
            self.last_metrics = {"loss": loss, "psnr": -10.0 * torch.log10(mse),
                                 "eikonal": res["gradient_error"].detach().mean(), "s_val": res["s_val"].detach().mean()}
        if self.optimizer is not None:
            for k, p in self.P.items():
                p.grad = self.grads[k]
            torch.nn.utils.clip_grad_norm_(list(self.P.values()), 0.99)
            self.optimizer.step()


def _run_reference(init, batches, probe):
    """-> (curve, snapshots {step: (state dict, metrics on `probe`, flat-gradient dict on `probe`)})"""
    cfg = _ref_cfg()
    r = _PortRunner(cfg, init, "cuda")
    hist, snaps = [], {}
    for i in range(STEPS):
        cfg.cos_anneal_ratio = min(1.0, i / 50000)                    # NeuconWSystem.get_cos_anneal_ratio
        r.train_step(batches[i % len(batches)])
        hist.append(torch.stack([r.last_metrics[k].reshape(()) for k in ("loss", "psnr", "eikonal", "s_val")]))
        if (i + 1) % 100 == 0:
            state = {k: v.detach().clone() for k, v in r.P.items()}
            opt, r.optimizer = r.optimizer, None                      # gradient only: no update on the probe batch
            cfg.cos_anneal_ratio = min(1.0, (i + 1) / 50000)
            r.train_step(probe)
            r.optimizer = opt
            grads = {k: g.detach().clone() for k, g in r.grads.items() if not k.startswith("embedding_a.")}
            snaps[i + 1] = (state, {k: float(v) for k, v in r.last_metrics.items()}, grads)
    return torch.stack(hist).cpu(), snaps


def _probe_nrw(mode, snaps, probe):
    """loss / PSNR / eikonal and the flat gradient of the CUDA path on the reference's snapshot weights."""
    sysm = _make_nrw(mode)
    out = {}
    for step, (state, ref_metrics, ref_grads) in snaps.items():
        sysm.neuconw.load_state_dict({k[len("neuconw."):]: v for k, v in state.items() if k.startswith("neuconw.")})
        sysm.nerf.load_state_dict({k[len("nerf."):]: v for k, v in state.items() if k.startswith("nerf.")})
        sysm.embedding_a.load_state_dict({"weight": state["embedding_a.weight"]})
        sysm.global_step = step
        _, flat, _ = sysm.compute_grads(probe)
        eng = sysm.renderer.engine
        dot = nn = rr = 0.0
        for k, _p in eng.named_params():
            shape, off, numel = eng.index[k]
            g_c, g_r = flat[off:off + numel].double(), ref_grads[k].reshape(-1).double()
            dot += float((g_c * g_r).sum()); nn += float((g_c * g_c).sum()); rr += float((g_r * g_r).sum())
        m = {k: float(v) for k, v in sysm.last_metrics.items()}
        out[step] = {"metrics": m, "reference_metrics": ref_metrics, "grad_cosine": dot / (nn ** 0.5 * rr ** 0.5 + 1e-30),
                     "grad_norm_ratio": (nn / (rr + 1e-30)) ** 0.5}
    return out


def test_precision_policy_training_curves():
    all_b = _scene_batches(17)
    batches = [{k: v.cuda() for k, v in b.items()} for b in all_b[:16]]
    probe = {k: v.cuda() for k, v in all_b[16].items()}              # held-out batch for the snapshot comparison
    curves, init = {}, None
    for mode in ("bf16x3", "mixed", "bf16"):
        curves[mode], init0 = _run_nrw(mode, batches)
        init = init or init0
    curves["fp32_port"], snaps = _run_reference(init, batches, probe)
    curves["fp32_reference"] = torch.from_numpy(np.load(os.path.join(GOLDEN, "precision_curve.npz"))["curve"])
    probes = {mode: _probe_nrw(mode, snaps, probe) for mode in ("bf16x3", "mixed", "bf16")}
    tail = {k: v[-100:].mean(0) for k, v in curves.items()}
    ref = tail["fp32_reference"]
    report = {"steps": STEPS, "rays": R, "lr": LR, "columns": ["loss", "psnr_db", "eikonal", "s_val"],
              "first_step": {k: [float(x) for x in v[0]] for k, v in curves.items()},
              "mean_of_last_100_steps": {k: [float(x) for x in v] for k, v in tail.items()},
              "every_25th_step": {k: [[float(x) for x in row] for row in v[::25]] for k, v in curves.items()},
              "on_reference_snapshot_weights": probes}
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump(report, open(os.path.join(ROOT, "gpurun_out", "precision_study.json"), "w"), indent=1)
    print(json.dumps({"tail": report["mean_of_last_100_steps"], "snapshots": probes}, indent=1))
    # same starting point, the restated baseline follows the unmodified reference until the trajectories decorrelate,
    # and the baseline actually trains
    for mode in ("bf16x3", "fp32_port"):
        assert abs(float(curves[mode][0, 0] - curves["fp32_reference"][0, 0])) < 1e-4 * abs(float(curves["fp32_reference"][0, 0])), mode
    early = (curves["fp32_port"][:25, 0] - curves["fp32_reference"][:25, 0]).abs() / curves["fp32_reference"][:25, 0].abs()
    assert float(early.max()) < 1e-2, float(early.max())
    assert float(curves["fp32_port"][-100:, 1].mean() - curves["fp32_port"][:5, 1].mean()) > 10.0
    # (1) identical trained weights: forward quantities and gradient direction
    for mode, cos_min in (("bf16x3", 0.9999), ("mixed", 0.995)):
        for step, pr in probes[mode].items():
            for k, tol_rel, tol_abs in (("loss", 5e-4, 0.0), ("psnr", 0.0, 0.01), ("eikonal", 1e-3, 1e-7)):
                a, b = pr["metrics"][k], pr["reference_metrics"][k]
                assert abs(a - b) <= tol_rel * abs(b) + tol_abs, (mode, step, k, a, b)
            assert pr["grad_cosine"] >= cos_min, (mode, step, pr["grad_cosine"])
            assert abs(pr["grad_norm_ratio"] - 1.0) < 0.02, (mode, step, pr["grad_norm_ratio"])
    # (2) trajectories: PSNR tail within the chaos band
    for mode in ("bf16x3", "mixed"):
        assert abs(float(tail[mode][1] - ref[1])) < 1.0, (mode, "psnr", float(tail[mode][1]), float(ref[1]))
