"""Generate golden vectors by running the *reference* SceneRF renderer (unmodified, imported from
/root/reference) on the deterministic synthetic inputs of scenerf_b200.synth.

Runs ONLY in the build container (needs /root/reference); the GPU box never executes this.
    python tests/golden/make_goldens.py            # rewrites tests/golden/*.npz

How the reference is made importable without touching it (SURVEY.md 8c / Appendix A):
  * `pytorch_lightning` is absent -> a 10-line stand-in module whose LightningModule is nn.Module;
  * `UNet2DSphere.build` would call torch.hub (network) -> replaced by a stub returning nn.Identity.
The two RNG draws of a chunk (utils.py:84 torch.rand_like, utils.py:208-211 torch.normal) are recorded by
wrapping the torch functions, so that every other implementation can be fed identical noise.

Stored per case: inputs that are not regenerable from synth (noise), stage-boundary tensors and the 12-key
output dict of render_rays_batch (scenerf.py:456-469).
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("SCENERF_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

from scenerf_b200 import synth  # noqa: E402


def _install_shims():
    pl = types.ModuleType("pytorch_lightning")

    class _LM(nn.Module):
        def save_hyperparameters(self, *a, **k):
            pass

        def log(self, *a, **k):
            pass

        @property
        def device(self):
            return next(self.parameters()).device

    pl.LightningModule = _LM
    sys.modules["pytorch_lightning"] = pl
    import scenerf.models.unet2d_sphere as U
    U.UNet2DSphere.build = classmethod(lambda cls, **kw: nn.Identity())


def build_reference_model(cfg: synth.SceneConfig, seed=11):
    _install_shims()
    if cfg.dataset == "kitti":
        from scenerf.models.scenerf import SceneRF
    else:
        from scenerf.models.scenerf_bf import SceneRF
    m = SceneRF(som_sigma=cfg.som_sigma, std=cfg.std, img_size=(cfg.img_W, cfg.img_H),
                max_sample_depth=cfg.max_sample_depth, n_gaussians=cfg.n_gaussians,
                n_pts_uni=cfg.n_pts_uni, n_pts_per_gaussian=cfg.n_pts_per_gaussian,
                add_fov_hor=cfg.add_fov_hor, add_fov_ver=cfg.add_fov_ver,
                sphere_H=cfg.sphere_H, sphere_W=cfg.sphere_W).eval()
    pm, pg = synth.make_model_params(cfg, seed)
    m.mlp.load_state_dict({k: torch.from_numpy(v) for k, v in pm.items()})
    m.mlp_gaussian.load_state_dict({k: torch.from_numpy(v) for k, v in pg.items()})
    return m


class _Recorder:
    """Records the reference's RNG draws and a few stage-boundary tensors."""

    def __init__(self, model):
        self.model = model
        self.rec = {}
        self._orig = {}

    def __enter__(self):
        import scenerf.models.utils as RU
        rec = self.rec
        o_rand_like, o_normal = torch.rand_like, torch.normal
        self._orig = dict(rand_like=o_rand_like, normal=o_normal)

        def rand_like(x, *a, **k):
            r = o_rand_like(x, *a, **k)
            rec.setdefault("noise_u", []).append(r.detach().clone())
            return r

        def normal(*a, **k):
            r = o_normal(*a, **k)
            rec.setdefault("noise_n", []).append(r.detach().clone())
            return r

        torch.rand_like, torch.normal = rand_like, normal
        sm = self.model.spherical_mapping
        o_from = sm.from_pixels
        self._orig["from_pixels"] = o_from

        def from_pixels(inv_K, pix_coords=None):
            out = o_from(inv_K=inv_K, pix_coords=pix_coords)
            rec.setdefault("sphere_coords", []).append(out[1].detach().clone())
            rec.setdefault("proj_pix", []).append(pix_coords.detach().clone())
            return out

        sm.from_pixels = from_pixels
        o_predict = self.model.predict
        self._orig["predict"] = o_predict

        def predict(*a, **k):
            rec.setdefault("predict_cam_pts", []).append(k["cam_pts"].detach().clone())
            rec.setdefault("predict_viewdir", []).append(k["viewdir"].detach().clone())
            out = o_predict(*a, **k)
            if isinstance(out, tuple):
                rec.setdefault("predict_density", []).append(out[0].detach().clone())
                rec.setdefault("predict_color", []).append(out[1].detach().clone())
            else:
                rec.setdefault("predict_offset", []).append(out.detach().clone())
            return out

        self.model.predict = predict
        return self

    def __exit__(self, *exc):
        torch.rand_like, torch.normal = self._orig["rand_like"], self._orig["normal"]
        self.model.spherical_mapping.from_pixels = self._orig["from_pixels"]
        self.model.predict = self._orig["predict"]


def run_render_case(cfg, pixels, pyr_seed, torch_seed=0, **model_kw):
    model = build_reference_model(cfg, **model_kw)
    x_rgb = {k: torch.from_numpy(v) for k, v in synth.make_pyramid(pyr_seed, cfg.sphere_W, cfg.sphere_H).items()}
    K = torch.from_numpy(cfg.K)
    T = torch.from_numpy(cfg.T)
    pix = torch.from_numpy(pixels)
    torch.manual_seed(torch_seed)
    with torch.no_grad(), _Recorder(model) as r:
        if cfg.dataset == "kitti":
            out = model.render_rays_batch(K, T, x_rgb, ray_batch_size=pix.shape[0], sampled_pixels=pix)
        else:
            out = model.render_rays_batch(K, T, x_rgb, sampled_pixels=pix, ray_batch_size=pix.shape[0])
    rec = r.rec
    R = pix.shape[0]
    g = {k: v.numpy() for k, v in out.items()}
    g["noise_u"] = rec["noise_u"][0].reshape(R, -1).numpy()
    g["noise_n"] = rec["noise_n"][0].reshape(R, -1).numpy()
    # predict call 0 = gaussian proposal (R,G,3) ; call 1 = main pass (R,S,3)
    g["gauss_pts"] = rec["predict_cam_pts"][0].numpy()
    g["gauss_offset"] = rec["predict_offset"][0].numpy()
    g["main_pts"] = rec["predict_cam_pts"][1].numpy()
    g["viewdir"] = rec["predict_viewdir"][1].numpy()
    g["main_color"] = rec["predict_color"][0].numpy()
    g["gauss_sphere"] = rec["sphere_coords"][0].numpy().astype(np.int32)
    g["main_sphere"] = rec["sphere_coords"][1].numpy().astype(np.int32)
    g["pixels"] = pixels
    return g


def run_predict_case(cfg, cam_pts, viewdir, pyr_seed, **model_kw):
    """Direct call of SceneRF.predict (scenerf.py:505-547) on crafted points (adversarial gather cases)."""
    model = build_reference_model(cfg, **model_kw)
    x_rgb = {k: torch.from_numpy(v) for k, v in synth.make_pyramid(pyr_seed, cfg.sphere_W, cfg.sphere_H).items()}
    K = torch.from_numpy(cfg.K)
    with torch.no_grad(), _Recorder(model) as r:
        kw = dict(mlp=model.mlp, cam_pts=torch.from_numpy(cam_pts), x_rgb=x_rgb, cam_K=K,
                  viewdir=torch.from_numpy(viewdir))
        if cfg.dataset == "kitti":
            kw["T_cam2velo"] = None
        density, color = model.predict(**kw)
        kw["mlp"] = model.mlp_gaussian
        offset = model.predict(output_type="offset", **kw)
    return dict(cam_pts=cam_pts, viewdir=viewdir, density=density.numpy(), color=color.numpy(),
                offset=offset.numpy(), sphere=r.rec["sphere_coords"][0].numpy().astype(np.int32),
                proj_pix=r.rec["proj_pix"][0].numpy())


def adversarial_points(cfg, n_cols=48, n_per=8, seed=5):
    """Points (in the infer-camera frame) whose sphere coordinates land where the reference's quirks bite
    (SURVEY 8a a7/a10): top-left (W//s,H//s) corners of scales 2..16 incl. the boundary row/column, points
    behind the camera (pixel sentinel (-1,-1)), points outside the sphere grid, and ordinary points."""
    v_min, v_max, h_min, h_max = cfg.angles()
    W, H = cfg.sphere_W, cfg.sphere_H
    targets = []
    for s in (1, 2, 4, 8, 16):
        wn, hn = W // s, H // s
        for sx in (0, 1, wn // 2, wn - 1, wn, wn + 1):
            for sy in (0, 1, hn // 2, hn - 1, hn, hn + 1):
                targets.append((sx, sy))
    targets = targets[: n_cols * n_per - 64] if len(targets) > n_cols * n_per - 64 else targets
    pts = []
    u = synth.hash_unit(seed, 4 * len(targets)).astype(np.float64)
    for i, (sx, sy) in enumerate(targets):
        # invert the angle mapping (spherical_mapping.py:95-115) at the pixel centre (+ small jitter)
        h = h_min + (sx + 0.3 * (u[4 * i] - 0.5)) / (W - 1) * (h_max - h_min)
        v = v_min + (sy + 0.3 * (u[4 * i + 1] - 0.5)) / (H - 1) * (v_max - v_min)
        hr, vr = np.deg2rad(180.0 - h), np.deg2rad(v)
        d = np.array([np.sin(vr) * np.cos(hr), -np.cos(vr), np.sin(vr) * np.sin(hr)])
        r = 2.0 + 30.0 * u[4 * i + 2]
        pts.append(d * r)
    pts = np.array(pts, dtype=np.float32)
    n_total = n_cols * n_per
    extra = n_total - pts.shape[0]
    e = synth.hash_uniform(seed + 1, 3 * extra).reshape(extra, 3)
    ex = np.stack([e[:, 0] * 30.0, e[:, 1] * 6.0, e[:, 2] * 40.0 + 10.0], axis=1).astype(np.float32)
    ex[: extra // 4, 2] = -np.abs(ex[: extra // 4, 2])          # behind the camera
    ex[extra // 4: extra // 2, 0] *= 8.0                         # far outside the horizontal FOV
    pts = np.concatenate([pts, ex], axis=0)
    cam_pts = pts.reshape(n_cols, n_per, 3)
    viewdir = (synth.hash_uniform(seed + 2, n_cols * 3).reshape(n_cols, 3) * np.float32(0.8)).astype(np.float32)
    return np.ascontiguousarray(cam_pts), np.ascontiguousarray(viewdir)


CASES = {}


def case(fn):
    CASES[fn.__name__] = fn
    return fn


@case
def kitti_mini():
    cfg = synth.config_A(name="kitti_mini", sphere_W=300, sphere_H=90, yaw_deg=10.0, tz=1.0)
    return run_render_case(cfg, synth.random_pixels(21, 96, cfg.img_W, cfg.img_H), pyr_seed=31)


@case
def kitti_s128():
    cfg = synth.config_B(name="kitti_s128", sphere_W=306, sphere_H=92)
    pix = synth.grid_pixels(cfg.img_W, cfg.img_H, stride=61)[:48]
    return run_render_case(cfg, np.ascontiguousarray(pix), pyr_seed=32)


@case
def bf_mini():
    cfg = synth.config_C(name="bf_mini", sphere_W=160, sphere_H=120, n_pts_uni=32)
    return run_render_case(cfg, synth.random_pixels(23, 64, cfg.img_W, cfg.img_H), pyr_seed=33)


@case
def bf_s96():
    """BASELINE.json config C geometry: BundleFusion, U=64, G=4, P=8 -> S = 96 samples (not a power of two)."""
    cfg = synth.config_C(name="bf_s96", sphere_W=160, sphere_H=120)
    pix = synth.grid_pixels(cfg.img_W, cfg.img_H, stride=67)[:40]
    return run_render_case(cfg, np.ascontiguousarray(pix), pyr_seed=38)


@case
def kitti_identity():
    """T = identity-ish (tz=0): all samples of a ray share one sphere pixel (SURVEY hard part 3c)."""
    cfg = synth.config_A(name="kitti_identity", sphere_W=300, sphere_H=90, yaw_deg=0.0, tz=0.0)
    return run_render_case(cfg, synth.random_pixels(24, 32, cfg.img_W, cfg.img_H), pyr_seed=34)


FULL_KEEP = ("depth", "color", "gaussian_means", "gaussian_stds", "weights_at_depth", "closest_pts_to_depths", "loss_kl",
             "alphas", "som_vars", "densities", "weights", "depth_volumes", "noise_u", "noise_n", "pixels", "main_sphere",
             "gauss_sphere")


def full_size_pixels(cfg, n=256):
    """n integer pixels of the x-major full-frame grid (render_colors.py:103-111), spread over the whole image."""
    grid = synth.grid_pixels(cfg.img_W, cfg.img_H)
    idx = (np.arange(n, dtype=np.int64) * (grid.shape[0] // n + 1) + 13) % grid.shape[0]
    return np.ascontiguousarray(grid[idx])


def run_full_case(cfg, pyr_seed):
    g = run_render_case(cfg, full_size_pixels(cfg), pyr_seed=pyr_seed)
    return {k: g[k] for k in FULL_KEEP}


@case
def full_B():
    """BASELINE.json configs[1] at FULL size: sphere grid 1226x370 (281 MB pyramid), S = 128; 256 rays of the frame."""
    return run_full_case(synth.config_B(name="full_B"), 41)


@case
def full_Bp():
    """config B' (SURVEY 8d): the reference-default 1500x452 sphere grid (420 MB pyramid), S = 128."""
    return run_full_case(synth.config_B(name="full_Bp", sphere_W=1500, sphere_H=452), 42)


@case
def full_C():
    """BASELINE.json configs[2] at FULL size: BundleFusion 640x480 sphere grid (190 MB pyramid), S = 96."""
    return run_full_case(synth.config_C(name="full_C"), 43)


@case
def predict_adversarial_kitti():
    cfg = synth.config_A(name="adv_kitti", sphere_W=300, sphere_H=90)
    pts, vd = adversarial_points(cfg)
    return run_predict_case(cfg, pts, vd, pyr_seed=35)


@case
def predict_adversarial_kitti_full():
    """Reference-default sphere grid 1500x452: W_t != W_n for scales 8/16 (fractional taps)."""
    cfg = synth.config_A(name="adv_kitti_full")
    pts, vd = adversarial_points(cfg, n_cols=40, n_per=8)
    return run_predict_case(cfg, pts, vd, pyr_seed=36)


@case
def predict_adversarial_bf():
    cfg = synth.config_C(name="adv_bf", sphere_W=160, sphere_H=120)
    pts, vd = adversarial_points(cfg)
    pts = pts * np.float32(0.2)
    return run_predict_case(cfg, pts, vd, pyr_seed=37)


def tsdf_inputs():
    """Synthetic depth sweep for the TSDF golden: 3 poses (sample_rel_poses style), small images, scaled intrinsics."""
    H, W = 48, 160
    K = np.array([[707.0912 * W / 1220.0, 0, 601.8873 * W / 1220.0], [0, 707.0912 * H / 370.0, 183.1104 * H / 370.0], [0, 0, 1]])
    T_velo2cam = np.array([[0.0, -1.0, 0.0, 0.0], [0.0, 0.0, -1.0, -0.08], [1.0, 0.0, 0.0, -0.27], [0, 0, 0, 1.0]])
    frames = []
    for i, (yaw, tz) in enumerate(((0.0, 0.0), (10.0, 1.5), (-10.0, 3.0))):
        depth = (4.0 + 6.0 * synth.hash_unit(50 + i, H * W).reshape(H, W) + np.linspace(0, 4, W)[None, :]).astype(np.float32)
        depth[synth.hash_unit(60 + i, H * W).reshape(H, W) < 0.05] = 0.0           # holes
        rgb = np.floor(synth.hash_unit(70 + i, H * W * 3).reshape(H, W, 3) * 256.0).astype(np.float64)
        rel = synth.yaw_translate(yaw, tz).astype(np.float64)
        frames.append((rgb, depth, np.linalg.inv(T_velo2cam) @ rel))
    vol_bnds = np.zeros((3, 2))
    vol_bnds[:, 0] = [0, -6.4, -2]
    vol_bnds[:, 1] = vol_bnds[:, 0] + [12.8, 12.8, 3.2]
    return K, frames, vol_bnds


@case
def tsdf_fusion():
    """The reference's TSDFVolume (CPU / numba path, fusion.py:219-324) on a 3-pose synthetic depth sweep."""
    sk = types.ModuleType("skimage")
    sk.measure = types.ModuleType("skimage.measure")
    sys.modules.setdefault("skimage", sk)
    sys.modules.setdefault("skimage.measure", sk.measure)
    import scenerf.data.utils.fusion as fusion
    K, frames, vol_bnds = tsdf_inputs()
    vol = fusion.TSDFVolume(vol_bnds.copy(), voxel_size=0.2, trunc_margin=10, use_gpu=False)
    out = {}
    for i, (rgb, depth, pose) in enumerate(frames):
        vol.integrate(rgb, depth, K, pose, obs_weight=1.)
        out["rgb%d" % i], out["depth%d" % i], out["pose%d" % i] = rgb.astype(np.float32), depth, pose
    tsdf, color = vol.get_volume()
    out.update(K=K, vol_bnds=vol_bnds, tsdf=tsdf.copy(), color=color.copy(), weight=vol._weight_vol_cpu.copy())
    return out


GRAD_KEYS = ("depth", "color", "gaussian_means", "gaussian_stds", "weights_at_depth", "closest_pts_to_depths", "loss_kl",
             "alphas", "densities", "weights", "depth_volumes")          # som_vars: see DESIGN.md (non-differentiable here)


def cotangent(key_idx, shape):
    n = int(np.prod(shape))
    return synth.hash_normalish(900 + key_idx, n).reshape(shape).astype(np.float32)


def grad_digest(name, G, out):
    """Big gradient tensors are stored as projections: G@u, G.T@v (fixed pseudo-random u, v) and the strided block
    G[::16, ::16]; small ones in full."""
    G = np.ascontiguousarray(G, dtype=np.float32)
    if G.ndim == 1 or G.size <= 65536:
        out["g:" + name] = G
        return
    u = synth.hash_normalish(700, G.shape[1]).astype(np.float64)
    v = synth.hash_normalish(701, G.shape[0]).astype(np.float64)
    out["gu:" + name] = (G.astype(np.float64) @ u).astype(np.float32)
    out["gv:" + name] = (G.astype(np.float64).T @ v).astype(np.float32)
    out["gs:" + name] = G[::16, ::16].copy()


def run_grad_case(cfg, pixels, pyr_seed):
    """Reference autograd through render_rays_batch: L = sum_k <out_k, C_k> with fixed cotangents C_k; gradients w.r.t.
    the 2 x 22 MLP parameter tensors, the 5 pyramid tensors and the raw MLP outputs."""
    model = build_reference_model(cfg)
    for p_ in model.parameters():
        p_.requires_grad_(True)
    x_rgb = {k: torch.from_numpy(v).requires_grad_(True) for k, v in synth.make_pyramid(pyr_seed, cfg.sphere_W, cfg.sphere_H).items()}
    raws = {}
    def keep(tag):
        def hook(m, i, o):
            o.retain_grad()
            raws[tag] = o
        return hook
    model.mlp.register_forward_hook(keep("main"))
    model.mlp_gaussian.register_forward_hook(keep("gauss"))
    K, T, pix = torch.from_numpy(cfg.K), torch.from_numpy(cfg.T), torch.from_numpy(pixels)
    torch.manual_seed(0)
    with _Recorder(model) as r:
        if cfg.dataset == "kitti":
            out = model.render_rays_batch(K, T, x_rgb, ray_batch_size=pix.shape[0], sampled_pixels=pix)
        else:
            out = model.render_rays_batch(K, T, x_rgb, sampled_pixels=pix, ray_batch_size=pix.shape[0])
    L = 0
    for i, k in enumerate(GRAD_KEYS):
        L = L + (out[k] * torch.from_numpy(cotangent(i, tuple(out[k].shape)))).sum()
    L.backward()
    R = pix.shape[0]
    g = {k: v.detach().numpy() for k, v in out.items()}
    g["noise_u"] = r.rec["noise_u"][0].reshape(R, -1).numpy()
    g["noise_n"] = r.rec["noise_n"][0].reshape(R, -1).numpy()
    g["pixels"] = pixels
    g["loss"] = np.float64(L.item())
    g["graw_main"] = raws["main"].grad.reshape(-1, 4).numpy()
    g["graw_gauss"] = raws["gauss"].grad.reshape(-1, 2).numpy()
    for tag, net in (("main", model.mlp), ("gauss", model.mlp_gaussian)):
        for name, p_ in net.named_parameters():
            grad_digest("%s.%s" % (tag, name), p_.grad.numpy(), g)
    for k, t in x_rgb.items():
        G = t.grad.numpy()
        g["gpyr_chsum:" + k] = G.sum(axis=(1, 2), dtype=np.float64).astype(np.float32)
        g["gpyr_pixsum:" + k] = G.sum(axis=0, dtype=np.float64).astype(np.float32)
        g["gpyr_head:" + k] = G[:4].copy()
        g["gpyr_abs:" + k] = np.float64(np.abs(G).sum(dtype=np.float64))
    return g


@case
def grad_kitti():
    cfg = synth.config_A(name="grad_kitti", sphere_W=300, sphere_H=90, yaw_deg=10.0, tz=1.0)
    return run_grad_case(cfg, synth.random_pixels(23, 48, cfg.img_W, cfg.img_H), pyr_seed=41)


@case
def grad_bf():
    cfg = synth.config_C(name="grad_bf", sphere_W=160, sphere_H=120, n_pts_uni=32)
    return run_grad_case(cfg, synth.random_pixels(24, 40, cfg.img_W, cfg.img_H), pyr_seed=42)


@case
def sphere_feature():
    """DecoderSphere.get_sphere_feature (unet2d_sphere.py:138-166): image-plane feature maps resampled onto the sphere grid
    through the pixel -> sphere-pixel table of SphericalMapping.from_pixels.  Duplicate sphere cells are resolved by
    index_put_ on ONE CPU thread, i.e. the last image pixel in row-major order wins."""
    _install_shims()
    from scenerf.models.unet2d_sphere import DecoderSphere
    from scenerf.models.spherical_mapping import SphericalMapping
    torch.set_num_threads(1)
    W, H, oW, oH = 122, 37, 150, 45
    K = synth.KITTI_K.copy()
    K[:2] /= 10.0
    cfg = synth.config_A(name="sf", sphere_W=oW, sphere_H=oH)
    v0, v1, h0, h1 = cfg.angles()
    sm = SphericalMapping(v_angle_max=v1, v_angle_min=v0, h_angle_max=h1, h_angle_min=h0, img_W=W, img_H=H, out_img_W=oW, out_img_H=oH)
    pix, pix_sphere, _ = sm.from_pixels(inv_K=torch.inverse(torch.from_numpy(K)))
    dec = DecoderSphere.__new__(DecoderSphere)
    torch.nn.Module.__init__(dec)
    dec.out_img_W, dec.out_img_H = oW, oH
    out = dict(pix=pix.numpy(), pix_sphere=pix_sphere.numpy(), K=K, dims=np.array([W, H, oW, oH]))
    for scale, C in ((1, 6), (2, 8), (4, 5)):
        h, w = -(-H // scale), -(-W // scale)
        x = torch.from_numpy(synth.hash_normalish(300 + scale, C * h * w).reshape(1, C, h, w).astype(np.float32))
        out["x_%d" % scale] = x.numpy()[0]
        out["feat_%d" % scale] = dec.get_sphere_feature(x, pix, pix_sphere, scale).numpy()[0]
    return out


DECODER_CASE = dict(num_features=128, bottleneck=48, W=128, H=64, oW=150, oH=46, seed=21)


def decoder_inputs(c=DECODER_CASE):
    """Deterministic encoder maps (the six `features[...]` DecoderSphere.forward reads, unet2d_sphere.py:168-175) + camera."""
    chans = {1: 3, 2: 32, 4: 48, 8: 80, 16: 224, 32: c["bottleneck"]}
    feats = {}
    for s, ch in chans.items():
        h, w = -(-c["H"] // s), -(-c["W"] // s)
        feats[s] = synth.hash_normalish(500 + s, ch * h * w).reshape(ch, h, w).astype(np.float32)
    K = synth.KITTI_K.copy()
    K[:2] /= 9.5
    return feats, K


@case
def decoder_sphere():
    """DecoderSphere.forward (unet2d_sphere.py:167-206) in eval mode on deterministic weights: conv2, six get_sphere_feature
    resamplings, five UpSampleBN stacks -> the five maps of the x_rgb pyramid."""
    _install_shims()
    from scenerf.models.unet2d_sphere import DecoderSphere
    from scenerf.models.spherical_mapping import SphericalMapping
    torch.set_num_threads(1)
    c = DECODER_CASE
    feats, K = decoder_inputs()
    cfg = synth.config_A(name="dec", sphere_W=c["oW"], sphere_H=c["oH"])
    v0, v1, h0, h1 = cfg.angles()
    sm = SphericalMapping(v_angle_max=v1, v_angle_min=v0, h_angle_max=h1, h_angle_min=h0, img_W=c["W"], img_H=c["H"],
                          out_img_W=c["oW"], out_img_H=c["oH"])
    pix, pix_sphere, _ = sm.from_pixels(inv_K=torch.inverse(torch.from_numpy(K)))
    dec = DecoderSphere(num_features=c["num_features"], bottleneck_features=c["bottleneck"], out_feature=16, out_img_W=c["oW"],
                        out_img_H=c["oH"]).eval()
    params = synth.make_decoder_params(c["num_features"], c["bottleneck"], c["seed"])
    missing, unexpected = dec.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=False)
    assert not unexpected and all(m.startswith("resize_") or m.endswith("num_batches_tracked") for m in missing), (missing, unexpected)
    features = [None] * 12
    for idx, s in ((0, 1), (4, 2), (5, 4), (6, 8), (8, 16), (11, 32)):
        features[idx] = torch.from_numpy(feats[s])[None]
    with torch.no_grad():
        out = dec(features, pix, pix_sphere)
    g = {k: v[0].numpy() for k, v in out.items()}
    g.update(pix=pix.numpy(), pix_sphere=pix_sphere.numpy(), K=K)
    return g


def sweep_setup():
    """Small-image stand-in of generate_novel_depths.py: 244x74 image (KITTI intrinsics / 5), stride-4 grid (61x19 rays),
    the 6 poses of sample_rel_poses(step=1.0, angle=10, max_distance=1.1)."""
    cfg = synth.config_A(name="sweep_kitti", sphere_W=300, sphere_H=90)
    cfg.img_W, cfg.img_H = 244, 74
    cfg.K = synth.KITTI_K.copy()
    cfg.K[:2] /= 5.0
    return cfg, 4, dict(step=1.0, angle=10, max_distance=1.1), 39


@case
def sweep_kitti():
    """generate_novel_depths.py:52,103-152 + depth2tsdf.py:87-103 run with the reference's own functions on a small image."""
    import torch.nn.functional as F
    _install_shims()
    from scenerf.models.utils import sample_rel_poses, sample_rel_poses_bf
    sk = types.ModuleType("skimage")
    sk.measure = types.ModuleType("skimage.measure")
    sys.modules.setdefault("skimage", sk)
    sys.modules.setdefault("skimage.measure", sk.measure)
    import scenerf.data.utils.fusion as fusion
    cfg, scale, pose_kw, pyr_seed = sweep_setup()
    out = {}
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        bf = sample_rel_poses_bf(angle=15, max_distance=0.7, step=0.2)
    out["bf_pose_keys"] = np.array([[float(s), float(a)] for s, a in bf.keys()], dtype=np.float64)
    out["bf_poses"] = np.stack([v.numpy() for v in bf.values()])
    full = sample_rel_poses(step=0.5, angle=10, max_distance=10.1)
    out["full_pose_keys"] = np.array([[float(s), float(a)] for s, a in full.keys()], dtype=np.float64)
    out["full_poses"] = np.stack([v.numpy() for v in full.values()])
    rel_poses = sample_rel_poses(**pose_kw)
    out["pose_keys"] = np.array([[float(s), float(a)] for s, a in rel_poses.keys()], dtype=np.float64)
    out["poses"] = np.stack([v.numpy() for v in rel_poses.values()])

    model = build_reference_model(cfg)
    x_rgb = {k: torch.from_numpy(v) for k, v in synth.make_pyramid(pyr_seed, cfg.sphere_W, cfg.sphere_H).items()}
    cam_K = torch.from_numpy(cfg.K)
    img_size = (cfg.img_W, cfg.img_H)
    T_velo2cam = np.array([[0.0, -1.0, 0.0, 0.0], [0.0, 0.0, -1.0, -0.08], [1.0, 0.0, 0.0, -0.27], [0, 0, 0, 1.0]])
    vol_bnds = np.zeros((3, 2))
    vol_bnds[:, 0] = [0, -6.4, -2]
    vol_bnds[:, 1] = vol_bnds[:, 0] + [12.8, 12.8, 3.2]
    vol = fusion.TSDFVolume(vol_bnds.copy(), voxel_size=0.2, use_gpu=False)
    torch.manual_seed(0)
    for i, ((step, angle), rel_pose) in enumerate(rel_poses.items()):
        # generate_novel_depths.py:103-147, verbatim sequence of torch calls
        xs = torch.arange(start=0, end=img_size[0], step=scale).type_as(cam_K)
        ys = torch.arange(start=0, end=img_size[1], step=scale).type_as(cam_K)
        grid_x, grid_y = torch.meshgrid(xs, ys)
        rendered_im_size = grid_x.shape
        sampled_pixels = torch.cat([grid_x.unsqueeze(-1), grid_y.unsqueeze(-1)], dim=2).reshape(-1, 2)
        with torch.no_grad(), _Recorder(model) as r:
            rd = model.render_rays_batch(cam_K, rel_pose.type_as(cam_K), x_rgb, ray_batch_size=5000,
                                         sampled_pixels=sampled_pixels)
        depth_rendered = rd["depth"].reshape(rendered_im_size[0], rendered_im_size[1])
        color_rendered = rd["color"].reshape(rendered_im_size[0], rendered_im_size[1], 3)
        depth_rendered = F.interpolate(depth_rendered.T.unsqueeze(0).unsqueeze(0), size=(img_size[1], img_size[0]), mode="bilinear")
        color_rendered = F.interpolate(color_rendered.permute(2, 1, 0).unsqueeze(0), size=(img_size[1], img_size[0]), mode="bilinear")
        color_np = color_rendered.clamp(0, 1).squeeze().permute(2, 1, 0).detach().cpu().numpy()
        color_np = np.transpose(color_np, (1, 0, 2))
        depth_np = depth_rendered.squeeze().detach().cpu().numpy()
        # plt.imsave (matplotlib ScalarMappable.to_rgba(bytes=True): (x*255).astype(uint8)); PNG is lossless;
        # depth2tsdf.py:19-26,98 reads it back as float32/255.0 and multiplies by 255.0
        u8 = (color_np * 255).astype(np.uint8)
        rgb = (np.array(u8, dtype=np.float32) / 255.0) * 255.0
        vol.integrate(rgb, depth_np, cfg.K, np.linalg.inv(T_velo2cam) @ rel_pose.numpy(), obs_weight=1.)
        R = sampled_pixels.shape[0]
        out["noise_u%d" % i] = r.rec["noise_u"][0].reshape(R, -1).numpy()
        out["noise_n%d" % i] = r.rec["noise_n"][0].reshape(R, -1).numpy()
        out["depth_rays%d" % i], out["color_rays%d" % i] = rd["depth"].numpy(), rd["color"].numpy()
        if i in (0, 4):           # full images only for two poses (fixture size)
            out["depth%d" % i], out["color%d" % i], out["rgb_tsdf%d" % i] = depth_np, color_np.astype(np.float16), u8
    tsdf, color = vol.get_volume()
    out.update(pixels=sampled_pixels.numpy(), K=cfg.K, T_velo2cam=T_velo2cam, vol_bnds=vol_bnds, tsdf=tsdf.copy(),
               tsdf_color=color.copy(), tsdf_weight=vol._weight_vol_cpu.copy())
    # a non-integer-ratio resampling case for the interpolation restatement (stride 3 grid of a 50x23 image)
    g = torch.from_numpy(synth.hash_normalish(77, 17 * 8).reshape(17, 8).astype(np.float32))
    out["interp_src"] = g.numpy()
    out["interp_dst"] = F.interpolate(g.T.unsqueeze(0).unsqueeze(0), size=(23, 50), mode="bilinear").squeeze().numpy()
    return out


@case
def angles_kat():
    """The only known-answer check in the reference: scripts/determine_angles.py <-> scenerf.py:84-87 and
    scenerf_bf.py:84-87.  We run the same functions on every pixel and store min/max."""
    _install_shims()
    from scenerf.models.spherical_mapping import SphericalMapping, pix_2_cam_pts
    out = {}
    for name, K, W, H in (("kitti", synth.KITTI_K, 1220, 370), ("bf", synth.BF_K, 640, 480)):
        invK = torch.inverse(torch.from_numpy(K))
        m = SphericalMapping(v_angle_max=0, v_angle_min=0, h_angle_max=0, h_angle_min=0, img_W=W, img_H=H,
                             out_img_W=0, out_img_H=0)
        mesh = np.meshgrid(range(W), range(H), indexing="xy")
        ids = torch.from_numpy(np.stack(mesh, 0).astype(np.float32))
        pix = torch.cat([ids[0].reshape(-1, 1), ids[1].reshape(-1, 1)], 1)
        cam = pix_2_cam_pts(pix, invK, torch.ones(pix.shape[0]))
        v, h, _ = m.cam_pts_2_angle(cam)
        out[name] = np.array([v.min(), v.max(), h.min(), h.max()], dtype=np.float32)
    return out


@case
def reference_sources():
    """sha256 of every reference file oracle/build_ref.py stages into oracle/_ref, so that a staged copy can be checked
    on a machine without the reference tree."""
    import hashlib
    from oracle import build_ref
    digests = []
    for rel in build_ref.FILES:
        with open(os.path.join(REF, rel), "rb") as f:
            digests.append(hashlib.sha256(f.read()).hexdigest())
    return {"files": np.array(build_ref.FILES), "sha256": np.array(digests)}


def main():
    only = sys.argv[1:]
    for name, fn in CASES.items():
        if only and name not in only:
            continue
        g = fn()
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **g)
        print("%-32s %8.1f KB  keys=%d" % (name, os.path.getsize(path) / 1024.0, len(g)))


if __name__ == "__main__":
    main()
