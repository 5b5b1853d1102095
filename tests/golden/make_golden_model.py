"""Generates tests/golden/reference_model.npz by running the reference's OWN scene/gaussian_model.py
(/root/reference/scene/gaussian_model.py: training_setup :176-211, update_learning_rate :213-223, densify_and_prune :452-469,
reset_opacity :258-261) and torch.optim.Adam on the CPU in this container.

The reference class cannot be imported as-is here: it imports `plyfile` and `simple_knn._C` (absent; neither is used by the
methods exercised) and hard-codes device="cuda" in torch.zeros / torch.ones calls.  This script
  * registers EMPTY stand-in modules for `plyfile` and `simple_knn._C`,
  * wraps torch.zeros so the device keyword is dropped,
and otherwise runs the reference code unmodified, loaded straight from its file (scene/__init__.py pulls in the dataset
readers, which are not needed).  /root/reference does not exist on the GPU box, hence the committed fixture.

    python tests/golden/make_golden_model.py
"""
import importlib.util
import os
import sys
import types
from argparse import ArgumentParser

import numpy as np
import torch

REF = "/root/reference"
sys.path.insert(0, REF)

_zeros = torch.zeros


def _cpu_zeros(*a, **k):
    k.pop("device", None)
    return _zeros(*a, **k)


torch.zeros = _cpu_zeros
ply = types.ModuleType("plyfile")
ply.PlyData = ply.PlyElement = object
sys.modules["plyfile"] = ply
knn = types.ModuleType("simple_knn")
knn_c = types.ModuleType("simple_knn._C")
knn_c.distCUDA2 = None
sys.modules["simple_knn"], sys.modules["simple_knn._C"] = knn, knn_c

spec = importlib.util.spec_from_file_location("ref_gaussian_model", os.path.join(REF, "scene", "gaussian_model.py"))
GM = importlib.util.module_from_spec(spec)
spec.loader.exec_module(GM)
from arguments import OptimizationParams  # noqa: E402

opt = OptimizationParams(ArgumentParser())
out = {}

g = torch.Generator().manual_seed(4321)
P0, EXTENT = 64, 4.0          # ten full snapshots of parameters and both Adam moments: the fixture stays under 1 MB
pc = GM.GaussianModel(3)
pc.active_sh_degree = 3
pc.spatial_lr_scale = EXTENT
nnP = torch.nn.Parameter
pc._xyz = nnP(torch.randn(P0, 3, generator=g))
pc._features_dc = nnP(torch.randn(P0, 1, 3, generator=g) * 0.5)
pc._features_rest = nnP(torch.randn(P0, 15, 3, generator=g) * 0.1)
# log-scales straddling percent_dense*extent = 0.04 (log = -3.2) and a few above 0.1*extent = 0.4 (log = -0.9)
pc._scaling = nnP(torch.randn(P0, 3, generator=g) * 1.0 - 3.6)
pc._rotation = nnP(torch.randn(P0, 4, generator=g))
# opacity logits: sigmoid < 0.005 needs logit < -5.3 -- make some
pc._opacity = nnP(torch.rand(P0, 1, generator=g) * 9.0 - 6.5)
pc.max_radii2D = torch.zeros(P0)
pc.pretrained_exposures = None                      # create_from_pcd :173-176 (per-image exposure; not on this path)
pc._exposure = nnP(torch.eye(3, 4)[None].repeat(1, 1, 1))
for k in ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity"):
    out["init" + k] = getattr(pc, k).detach().numpy().copy()
pc.training_setup(opt)

# A loss whose gradient w.r.t. the ACTIVATED tensors is w + u * act (state dependent, reproducible by the tests)
names = ("xyz", "features", "opacity", "scaling", "rotation")
shapes = {"xyz": (3,), "features": (16, 3), "opacity": (1,), "scaling": (3,), "rotation": (4,)}
MAXP = 4 * P0
W = {n: torch.randn(MAXP, *shapes[n], generator=g) * 1e-3 for n in names}
U = {n: torch.randn(MAXP, *shapes[n], generator=g) * 1e-3 for n in names}
for n in names:
    out["w_" + n], out["u_" + n] = W[n].numpy(), U[n].numpy()


def activated():
    return {"xyz": pc.get_xyz, "features": pc.get_features, "opacity": pc.get_opacity, "scaling": pc.get_scaling,
            "rotation": pc.get_rotation}


def snapshot(tag):
    for k in ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity"):
        out[f"{tag}{k}"] = getattr(pc, k).detach().numpy().copy()
    for grp in pc.optimizer.param_groups:
        st = pc.optimizer.state.get(grp["params"][0], None)
        if st is not None:
            out[f"{tag}_m_{grp['name']}"] = st["exp_avg"].numpy().copy()
            out[f"{tag}_v_{grp['name']}"] = st["exp_avg_sq"].numpy().copy()
    out[f"{tag}_lr_xyz"] = np.float64([grp["lr"] for grp in pc.optimizer.param_groups if grp["name"] == "xyz"][0])


def train_step(iteration):
    pc.update_learning_rate(iteration)
    act = activated()
    P = pc.get_xyz.shape[0]
    loss = sum((W[n][:P] * act[n]).sum() + 0.5 * (U[n][:P] * act[n] ** 2).sum() for n in names)
    loss.backward()
    pc.optimizer.step()
    pc.optimizer.zero_grad(set_to_none=True)


it = 0
for _ in range(3):
    it += 1
    train_step(it)
snapshot("s3")

# densification statistics (train.py:166-167 / gaussian_model.py:471-473 would have produced these)
P = pc.get_xyz.shape[0]
denom = torch.randint(0, 4, (P, 1), generator=g).float()
accum = torch.rand(P, 1, generator=g) * 0.0008 * denom            # mean grad in [0, 0.0008): ~75 % over the 0.0002 threshold
pc.xyz_gradient_accum, pc.denom = accum.clone(), denom.clone()
pc.max_radii2D = torch.rand(P, generator=g) * 40.0                 # some > 20: must NOT prune (postfix zeroes it first)
radii = torch.randint(0, 30, (P,), generator=g).int()
out.update(dens_accum=accum.numpy(), dens_denom=denom.numpy(), dens_max_radii2D=pc.max_radii2D.numpy().copy(),
           dens_radii=radii.numpy(), dens_extent=np.float32(EXTENT), dens_seed=np.int64(77))
torch.manual_seed(77)
# the reference draws torch.normal(mean=0, std=stds): record that this equals randn * std on this torch build
_s = torch.get_rng_state()
_chk = torch.normal(mean=torch.zeros(10, 3), std=torch.full((10, 3), 2.0))
torch.set_rng_state(_s)
assert torch.equal(_chk, torch.randn(10, 3) * 2.0)
torch.manual_seed(77)
pc.densify_and_prune(opt.densify_grad_threshold, 0.005, EXTENT, 20, radii)
snapshot("d")
out["d_P"] = np.int64(pc.get_xyz.shape[0])
out["d_max_radii2D"] = pc.max_radii2D.numpy().copy()
out["d_accum"], out["d_denom"] = pc.xyz_gradient_accum.numpy().copy(), pc.denom.numpy().copy()
print("densify: P", P, "->", pc.get_xyz.shape[0])

for _ in range(2):
    it += 1
    train_step(it)
snapshot("s5")

pc.reset_opacity()
it += 1
train_step(it)
snapshot("s6")

# the same densification without the size threshold (iteration <= opacity_reset_interval: max_screen_size None)
P = pc.get_xyz.shape[0]
denom2 = torch.randint(0, 3, (P, 1), generator=g).float()
accum2 = torch.rand(P, 1, generator=g) * 0.0006 * denom2
pc.xyz_gradient_accum, pc.denom = accum2.clone(), denom2.clone()
out.update(dens2_accum=accum2.numpy(), dens2_denom=denom2.numpy())
torch.manual_seed(78)
pc.densify_and_prune(opt.densify_grad_threshold, 0.005, EXTENT, None, torch.zeros(P).int())
snapshot("d2")
out["d2_P"] = np.int64(pc.get_xyz.shape[0])
print("densify 2: P", P, "->", pc.get_xyz.shape[0])

# ---- train.py order (train.py:139-190): loss.backward() FIRST, then densify_and_prune / reset_opacity replace parameters (a
# fresh nn.Parameter has .grad None), THEN optimizer.step(): torch.optim.Adam skips every replaced parameter -- no update, no
# moment decay, no increment of that parameter's own step counter (which drives its bias correction from then on).
def backward_only(iteration):
    pc.update_learning_rate(iteration)
    act = activated()
    P = pc.get_xyz.shape[0]
    loss = sum((W[n][:P] * act[n]).sum() + 0.5 * (U[n][:P] * act[n] ** 2).sum() for n in names)
    loss.backward()


def snapshot_steps(tag):
    for grp in pc.optimizer.param_groups:
        st = pc.optimizer.state.get(grp["params"][0], None)
        out[f"{tag}_step_{grp['name']}"] = np.float64(float(st["step"]) if st is not None and "step" in st else 0.0)


it += 1
backward_only(it)
P = pc.get_xyz.shape[0]
assert P <= MAXP
denom3 = torch.randint(0, 3, (P, 1), generator=g).float()
accum3 = torch.rand(P, 1, generator=g) * 0.0004 * denom3
pc.xyz_gradient_accum, pc.denom = accum3.clone(), denom3.clone()
out.update(dens3_accum=accum3.numpy(), dens3_denom=denom3.numpy())
torch.manual_seed(79)
pc.densify_and_prune(opt.densify_grad_threshold, 0.005, EXTENT, 20, torch.zeros(P).int())
pc.optimizer.step()                                   # every parameter was just replaced: a no-op
pc.optimizer.zero_grad(set_to_none=True)
snapshot("t1")
snapshot_steps("t1")
out["t1_P"] = np.int64(pc.get_xyz.shape[0])
print("densify 3 (train.py order): P", P, "->", pc.get_xyz.shape[0])
assert pc.get_xyz.shape[0] <= MAXP

it += 1
train_step(it)
snapshot("t2")
snapshot_steps("t2")

it += 1
backward_only(it)
pc.reset_opacity()                                    # only the opacity parameter is replaced
pc.optimizer.step()                                   # five groups step, opacity does not
pc.optimizer.zero_grad(set_to_none=True)
snapshot("t3")
snapshot_steps("t3")

it += 1
train_step(it)                                        # opacity's step counter now lags the others by two
snapshot("t4")
snapshot_steps("t4")

for k in ("position_lr_init", "position_lr_final", "position_lr_delay_mult", "position_lr_max_steps", "feature_lr", "opacity_lr",
          "scaling_lr", "rotation_lr", "percent_dense", "densify_grad_threshold"):
    out["opt_" + k] = np.float64(getattr(opt, k))

dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_model.npz")
np.savez_compressed(dst, **out)
print("wrote", dst, len(out), "arrays,", os.path.getsize(dst) // 1024, "KiB")
