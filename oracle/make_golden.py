"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE.  Run:  python -m oracle.make_golden
Imports /root/reference through ``oracle.ref_import`` (third-party imports stubbed),
loads ``oracle.synth.make_params`` weights into the reference's own ``NeuconW`` /
``NeRF`` / ``nn.Embedding`` modules, drives ``NeuconWRenderer.render`` +
``NeuconWLoss`` + ``backward`` on ``oracle.synth.make_rays`` batches and stores the
stage-boundary tensors.  Large parameter gradients are stored as seeded random
projections (``grad_probe``) + norms so the fixtures stay small.
"""
import os
import sys
import tempfile
import types
import warnings

import numpy as np
import torch

from . import ref_import, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests",
                          "golden")

SDF_CONFIG = dict(d_in=3, d_out=513, d_hidden=512, n_layers=8, skip_in=(4,), multires=6, bias=0.5,
                  scale=1, geometric_init=True, weight_norm=True, inside_outside=False)
COLOR_CONFIG = dict(d_in=9, d_feature=512, mode="idr", d_out=3, d_hidden=256, n_layers=4,
                    head_channels=128, static_head_layers=2, weight_norm=True, multires_view=4)


def install_injected_hits(renderer, hits, device="cpu"):
    """Config C3 without Kaolin: replace ONLY the Kaolin-backed ``get_near_far`` symbol that
    ``rendering/renderer.py`` imported (tools/prepare_data/generate_voxel.py:311) by a function returning injected
    trace results, and hand the renderer two placeholder octree dicts.  The reference's own
    ``get_near_far_octree`` / ``get_near_far_sdf`` / ``sparse_sampler`` arithmetic (renderer.py:380-568) runs unmodified."""
    import rendering.renderer as rr  # type: ignore

    coarse_tag, fine_tag = object(), object()

    def fake_get_near_far(rays_o, rays_d, octree, *a, **k):
        if octree is fine_tag:
            return hits["surface"].to(rays_o.device).clone(), None
        assert octree is coarse_tag
        return hits["sfm_near"].to(rays_o.device).clone(), hits["sfm_far"].to(rays_o.device).clone()

    rr.get_near_far = fake_get_near_far
    od = lambda tag, extra: dict(octree=tag, scene_origin=torch.zeros(3), scale=1.0, level=1, spc_data=None, **extra)
    renderer.octree_data = od(coarse_tag, {})
    renderer.fine_octree_data = od(fine_tag, {"voxel_size": hits["fine_voxel_sfm"]})
    renderer.nerf_far_override = True
    renderer.voxel_size = hits["voxel_size"]


def build_reference(cfg: synth.PathConfig, P):
    """Construct the reference modules and load the synthetic parameters into them."""
    ref = ref_import.load()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        neuconw = ref.NeuconW(sdfNet_config=SDF_CONFIG, colorNet_config=COLOR_CONFIG,
                              SNet_config=dict(init_val=0.3), in_channels_a=cfg.n_a, encode_a=True)
        nerf = ref.NeRF(D=8, d_in=4, d_in_view=3, W=256, multires=10, multires_view=4, output_ch=4,
                        skips=[4], encode_appearance=True, in_channels_a=cfg.n_a,
                        in_channels_dir=27, use_viewdirs=True)
    emb = torch.nn.Embedding(cfg.n_vocab, cfg.n_a)
    neuconw.load_state_dict({k[len("neuconw."):]: v for k, v in P.items() if k.startswith("neuconw.")})
    nerf.load_state_dict({k[len("nerf."):]: v for k, v in P.items() if k.startswith("nerf.")})
    emb.load_state_dict({"weight": P["embedding_a.weight"]})
    scene = tempfile.mkdtemp(prefix="nrw_scene_")
    import yaml
    with open(os.path.join(scene, "config.yaml"), "w") as f:
        yaml.safe_dump(dict(origin=[float(x) for x in cfg.origin], radius=float(cfg.radius),
                            sfm2gt=np.eye(4).tolist(),
                            eval_bbx=[[-cfg.radius] * 3, [cfg.radius] * 3]), f)
    renderer = ref.NeuconWRenderer(
        nerf=nerf, neuconw=neuconw, embeddings={"a": emb}, n_samples=cfg.n_samples,
        s_val_base=cfg.s_val_base, n_importance=cfg.n_importance, n_outside=cfg.n_outside,
        up_sample_steps=cfg.up_sample_steps, perturb=cfg.perturb, origin=list(cfg.origin),
        radius=cfg.radius, render_bg=cfg.render_bg, mesh_mask_list=cfg.mesh_mask_list,
        floor_normal=False, floor_labels=["road"], depth_loss=cfg.depth_loss,
        spc_options=dict(voxel_size=0.1, recontruct_path=scene, min_track_length=0),
        sample_range=cfg.sample_range, boundary_samples=cfg.boundary_samples,
        nerf_far_override=False, trim_sphere=cfg.trim_sphere)
    config = types.SimpleNamespace(NEUCONW=types.SimpleNamespace(
        MESH_MASK_LIST=cfg.mesh_mask_list, DEPTH_LOSS=cfg.depth_loss, FLOOR_NORMAL=False))
    loss = ref.NeuconWLoss(coef=1.0, igr_weight=cfg.igr_weight, mask_weight=cfg.mask_weight,
                           depth_weight=cfg.depth_weight, floor_weight=0.01, config=config)
    return dict(neuconw=neuconw, nerf=nerf, emb=emb, renderer=renderer, loss=loss)


def reference_train_step(cfg, P, batch, perturb_overwrite=0, rand_seed=None, hits=None):
    """The reference's own forward/loss/backward (NeuconWSystem.forward semantics,
    lightning_modules/neuconw_system.py:159-176,337-360)."""
    m = build_reference(cfg, P)
    if hits is not None:
        install_injected_hits(m["renderer"], hits)
    if rand_seed is not None:
        torch.manual_seed(rand_seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = m["renderer"].render(batch["rays"], batch["ts"], batch["label"],
                                   perturb_overwrite=perturb_overwrite,
                                   background_rgb=torch.zeros([1, 3]),
                                   cos_anneal_ratio=cfg.cos_anneal_ratio)
        loss_d = m["loss"](res, batch["rgbs"])
        loss = sum(loss_d.values())
        loss.backward()
    grads = {}
    for prefix, mod in (("neuconw.", m["neuconw"]), ("nerf.", m["nerf"]), ("embedding_a.", m["emb"])):
        for k, p in mod.named_parameters():
            grads[prefix + k] = p.grad.detach().clone() if p.grad is not None else torch.zeros_like(p)
    return res, loss.detach(), grads, m


def grad_probe(grads, n_probe=4, seed=99):
    """Small digest of a gradient dict: per-parameter L2 norm + n_probe random projections."""
    out = {}
    for k in sorted(grads):
        g = grads[k].detach().double().reshape(-1)
        gen = torch.Generator().manual_seed(seed + (sum(map(ord, k)) % 100003))
        pr = torch.randn(n_probe, g.numel(), generator=gen, dtype=torch.float64)
        out[k] = torch.cat([g.norm().reshape(1), pr @ g]).numpy()
    return out


def sample_index(numel, key, n=256):
    """Seeded, sorted sample of up to n flat indices of a tensor with `numel` elements (depends on the name only)."""
    gen = torch.Generator().manual_seed(7 + (sum(map(ord, key)) % 100003))
    return torch.randperm(numel, generator=gen)[:n].sort().values


# tests/test_dataio_oracle.py: (n_items, world) of DataModule._get_local_split, (n, world) of utils.visualization.get_local_split
DATAIO_SPLITS = [(64, 8), (64, 3), (5, 4), (7, 1)]
DATAIO_RANGES = [(10, 4), (12, 4), (1, 3)]


def dataio_getitem_inputs():
    """500 ray-cache rows (rays[12] with image id / semantic label columns, rgbs[3]) and 97 drawn indices."""
    g = torch.Generator().manual_seed(0)
    n = 500
    all_rays = torch.randn(n, 12, generator=g)
    all_rays[:, 8] = torch.randint(0, 1500, (n,), generator=g).float()
    all_rays[:, 9] = torch.tensor([0.0, 2.0, 12.0, 20.0, 116.0, 127.0, 6.0])[torch.randint(0, 7, (n,), generator=g)]
    all_rgbs = torch.rand(n, 3, generator=g)
    idx = torch.randperm(n, generator=g)[:97]
    return all_rays, all_rgbs, idx


def make_dataio_golden():
    """The reference's data-path helpers on the inputs of tests/test_dataio_oracle.py -> tests/golden/dataio.npz."""
    ref_import.load()
    from datasets.data import DataModule  # type: ignore
    from datasets.mask_utils import get_label_id_mapping  # type: ignore
    from datasets.phototourism import PhototourismDataset  # type: ignore
    from utils.visualization import get_local_split  # type: ignore

    arrays = {}
    for n_items, world in DATAIO_SPLITS:
        items = [f"split_{i}" for i in range(n_items)]
        for rank in range(world):
            want = DataModule._get_local_split(None, items, world, rank)
            arrays[f"split.{n_items}_{world}_{rank}"] = np.array([int(s[len("split_"):]) for s in want], np.int64)
    all_rays, all_rgbs, idx = dataio_getitem_inputs()
    fake = types.SimpleNamespace(split="train", all_rays=all_rays, all_rgbs=all_rgbs, with_semantics=True)
    items = [PhototourismDataset.__getitem__(fake, int(i)) for i in idx]
    for k in items[0]:
        arrays["getitem." + k] = torch.stack([it[k] for it in items]).numpy()
    m = get_label_id_mapping()
    arrays["label.names"] = np.array(sorted(m))
    arrays["label.ids"] = np.array([m[k] for k in sorted(m)], np.int64)
    for n, world in DATAIO_RANGES:
        data = torch.arange(n * 3, dtype=torch.float32).reshape(n, 3) + 1
        for rank in range(world):
            arrays[f"local.{n}_{world}_{rank}"] = get_local_split(data, world, rank).numpy()
    return arrays


# tests/test_oracle_vs_reference.py: a config unlike the CASES below (s_val_base 2, cos_anneal 0.25, 6 outside samples)
PORT_CFG = dict(n_samples=12, n_importance=12, up_sample_steps=3, n_outside=6, s_val_base=2, cos_anneal_ratio=0.25)
PORT_RAYS, PORT_SEED = 24, 5


def make_port_golden():
    """One training step of the reference on the PORT_CFG batch (every output, the loss, a seeded sample of every parameter
    gradient with its max magnitude) and the reference modules' state_dict layout -> tests/golden/port_step.npz."""
    import json

    P = synth.make_params(seed=0)
    cfg = synth.PathConfig(**PORT_CFG, **synth.BRANDENBURG)
    batch = synth.make_rays(PORT_RAYS, cfg, seed=PORT_SEED)
    res, loss, grads, _ = reference_train_step(cfg, P, batch, perturb_overwrite=0)
    arrays = {f"out.{k}": v.detach().numpy() for k, v in res.items()}
    arrays["loss"] = loss.numpy()
    for k, g in grads.items():
        flat = g.reshape(-1)
        arrays["gs." + k] = flat[sample_index(flat.numel(), k)].numpy()
        arrays["gmax." + k] = flat.abs().max().numpy()
    m = build_reference(synth.PathConfig(), P)
    layout = {}
    for pre, mod in (("neuconw.", m["neuconw"]), ("nerf.", m["nerf"]), ("embedding_a.", m["emb"])):
        for k, v in mod.state_dict().items():
            layout[pre + k] = list(v.shape)
    arrays["state_dict_layout"] = np.array(json.dumps(layout, sort_keys=True))
    return arrays


# tests/test_gpu_fullsize_reference.py: the full C2 batch is stored for a seeded sample of its rays
FULL_RAYS, FULL_SEED, FULL_SAMPLE_RAYS, FULL_SAMPLE_GRAD = 8192, 17, 128, 32768
FULL_PER_RAY = ("color", "color_sphere", "color_bg", "cdf_fine", "gradients", "mask_error", "weights", "weights_sum", "weights_max",
                "inside_sphere", "depth")


def full_sample():
    """(ray indices, flat-gradient indices over the sorted neuconw. / nerf. parameter names) of the stored C2 sample."""
    gen = torch.Generator().manual_seed(2024)
    rays = torch.randperm(FULL_RAYS, generator=gen)[:FULL_SAMPLE_RAYS].sort().values
    total = sum(v.numel() for k, v in synth.make_params(seed=0).items() if not k.startswith("embedding_a."))
    return rays, torch.randperm(total, generator=gen)[:FULL_SAMPLE_GRAD].sort().values


def flat_grad(grads):
    return torch.cat([grads[k].double().reshape(-1) for k in sorted(grads)])


def make_fullsize_golden(device):
    """The reference's full training step on the whole C2 batch (8192 rays x 128 samples, fp32, TF32 off) on `device`:
    the per-ray outputs and z_vals of FULL_SAMPLE_RAYS rays, the loss, gradient_error, the squared norm of the neuconw +
    nerf gradient and FULL_SAMPLE_GRAD of its entries -> tests/golden/fullsize_c2.npz."""
    cfg = synth.PathConfig(**synth.BRANDENBURG)
    P = synth.make_params(seed=0)
    b = {k: v.to(device) for k, v in synth.make_rays(FULL_RAYS, cfg, seed=FULL_SEED).items()}
    torch.backends.cuda.matmul.allow_tf32 = False
    m = build_reference(cfg, P)
    for k in ("neuconw", "nerf", "emb"):
        m[k].to(device)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = m["renderer"].render(b["rays"], b["ts"], b["label"], perturb_overwrite=0,
                                   background_rgb=torch.zeros([1, 3], device=device), cos_anneal_ratio=cfg.cos_anneal_ratio)
        loss = sum(m["loss"](res, b["rgbs"]).values())
        loss.backward()
    o = ((b["rays"][:, 0:3] - m["renderer"].origin).float() / cfg.radius).float()       # render()'s own normalisation
    with torch.no_grad():
        _, z, _, _ = m["renderer"].sparse_sampler(o, b["rays"][:, 3:6], (b["rays"][:, 6:7] / cfg.radius).float(),
                                                  (b["rays"][:, 7:8] / cfg.radius).float(), 0)
    grads = {}
    for pre, mod in (("neuconw.", m["neuconw"]), ("nerf.", m["nerf"])):
        for k, p in mod.named_parameters():
            grads[pre + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).detach().cpu()
    rays, gidx = full_sample()
    g = flat_grad(grads)
    arrays = {f"out.{k}": res[k].detach().cpu()[rays].numpy() for k in FULL_PER_RAY}
    arrays.update(z_vals=z.cpu()[rays].numpy(), loss=loss.detach().cpu().numpy(),
                  gradient_error=res["gradient_error"].detach().cpu().numpy(),
                  grad_norm2=np.array(float((g * g).sum())), grad_sample=g[gidx].numpy())
    return arrays


def make_precision_golden(device):
    """The reference's 300-step fp32 training run of tests/test_gpu_precision_policy.py on `device` (same initial
    weights, batches and schedule): loss / PSNR / eikonal / s_val of every step -> tests/golden/precision_curve.npz."""
    sys.path.insert(0, os.path.dirname(GOLDEN_DIR))
    import test_gpu_precision_policy as tp  # type: ignore
    from . import ref_runner

    all_b = tp._scene_batches(17)
    batches = [{k: v.to(device) for k, v in b.items()} for b in all_b[:16]]
    init = tp._initial_weights()
    cfg = tp._ref_cfg()
    r = ref_runner.RefRunner(cfg, init, device=device, lr=tp.LR)
    hist = []
    for i in range(tp.STEPS):
        cfg.cos_anneal_ratio = min(1.0, i / 50000)                    # NeuconWSystem.get_cos_anneal_ratio
        r.train_step(batches[i % len(batches)], perturb_overwrite=0)
        hist.append(torch.stack([r.last_metrics[k].reshape(()) for k in ("loss", "psnr", "eikonal", "s_val")]))
    return {"curve": torch.stack(hist).cpu().numpy()}


CASES = {
    # name: (cfg, n_rays, perturb_overwrite, torch seed for perturb draws)
    "small_det": (synth.PathConfig(n_samples=16, n_importance=8, up_sample_steps=2, n_outside=4), 48, 0, None),
    "small_perturb": (synth.PathConfig(n_samples=16, n_importance=16, up_sample_steps=4, n_outside=4,
                                       perturb=1.0, **synth.BRANDENBURG), 48, -1, 123),
    "c1_slice": (synth.C1, 32, 0, None),
    # config C3: SfM-octree near/far override + surface-guided fine sampling + boundary samples with INJECTED octree
    # trace results (synth.make_injected_hits), perturbed strata, scene frame
    "fine_c3": (synth.PathConfig(n_samples=16, n_importance=16, up_sample_steps=4, n_outside=4, perturb=1.0,
                                 boundary_samples=10, sample_range=8.0, **synth.BRANDENBURG), 48, -1, 321),
}
FINE_CASES = {"fine_c3"}


def save(out_dir, name, arrays):
    path = os.path.join(out_dir, f"{name}.npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {os.path.getsize(path) / 1024:.1f} KiB")


def main():
    """python -m oracle.make_golden [--cases] [--cpu-extra] [--gpu OUT_DIR]: no flag regenerates the CASES files; the
    GPU files are written to OUT_DIR (then copied to tests/golden)."""
    if not ref_import.available():
        print("reference tree not available; cannot regenerate golden vectors", file=sys.stderr)
        sys.exit(1)
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    argv = sys.argv[1:] or ["--cases"]
    if "--cpu-extra" in argv:
        save(GOLDEN_DIR, "dataio", make_dataio_golden())
        save(GOLDEN_DIR, "port_step", make_port_golden())
    if "--gpu" in argv:
        out = argv[argv.index("--gpu") + 1]
        os.makedirs(out, exist_ok=True)
        save(out, "fullsize_c2", make_fullsize_golden(torch.device("cuda", 0)))
        save(out, "precision_curve", make_precision_golden(torch.device("cuda", 0)))
    if "--cases" not in argv:
        return
    P = synth.make_params(seed=0)
    for name, (cfg, n_rays, pov, rseed) in CASES.items():
        batch = synth.make_rays(n_rays, cfg, seed=11)
        hits = synth.make_injected_hits(batch, cfg) if name in FINE_CASES else None
        res, loss, grads, m = reference_train_step(cfg, P, batch, perturb_overwrite=pov, rand_seed=rseed, hits=hits)
        # re-run the sampler alone for z_vals (deterministic given the same torch seed)
        o = ((batch["rays"][:, 0:3] - torch.tensor(cfg.origin, dtype=torch.float64).float()) / cfg.radius).float()
        near, far = (batch["rays"][:, 6:7] / cfg.radius).float(), (batch["rays"][:, 7:8] / cfg.radius).float()
        if rseed is not None:
            torch.manual_seed(rseed)
        with torch.no_grad():
            _, z, z_out, sd = m["renderer"].sparse_sampler(
                o, batch["rays"][:, 3:6], near.clone(), far.clone(), cfg.perturb if pov < 0 else pov)
        arrays = {f"out.{k}": v.detach().numpy() for k, v in res.items()}
        arrays.update(z_vals=z.numpy(), z_vals_outside=z_out.numpy(), sample_dist=sd.numpy(),
                      loss=loss.numpy())
        for k, v in grad_probe(grads).items():
            arrays["gp." + k] = v
        for k in ("neuconw.deviation_network.variance", "neuconw.sdf_net.lin8.bias",
                  "neuconw.color_net.lin4.bias", "nerf.alpha_linear.weight", "nerf.rgb_linear.bias",
                  "neuconw.sdf_net.lin0.weight_g"):
            arrays["g." + k] = grads[k].numpy()
        path = os.path.join(GOLDEN_DIR, f"{name}.npz")
        np.savez_compressed(path, **arrays)
        print(f"wrote {path}: loss={float(loss):.6f} {os.path.getsize(path) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
