import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tests import parity_utils as PU
import toda_b200.pcdet_plugin as P
g = PU.load_golden("backbone_res_stage2.npz")
nf = int(g["voxel_features"].shape[1])
twin, net = PU.build_pair("VoxelResBackBone8x", nf, g["grid_size"], seed=int(g["seed"]))
hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
vf = torch.from_numpy(g["voxel_features"]).cuda(); vc = torch.from_numpy(g["voxel_coords"]).float().cuda()
cot = torch.randn(tuple(g["bev_shape"]), generator=torch.Generator().manual_seed(int(g["seed"])))
r = PU.run_backbone(net, hc, vf, vc, 2, cot=cot, train=True)
ro = PU.run_backbone(twin, PU._oracle_hc, torch.from_numpy(g["voxel_features"]), torch.from_numpy(g["voxel_coords"]).float(), 2, cot=cot, train=True)
def rl2(a, b): return float(np.linalg.norm(a.astype(np.float64) - b.astype(np.float64)) / max(np.linalg.norm(b.astype(np.float64)), 1e-30))
print("dvf gpu vs golden", rl2(r["dvoxel_features"], g["train_dvoxel_features"]), "oracle-now vs golden", rl2(ro["dvoxel_features"], g["train_dvoxel_features"]))
for k in ["x_conv1", "x_conv2", "x_conv3", "x_conv4"]:
    print(k, r[k + "_features"].shape)
print("enc", r["enc_features"].shape)
names = [str(n) for n in g["grad_names"]]
for n in names[:12] + names[-6:]:
    print("%-40s gpu-vs-oracle %.2e   norm %.3e" % (n, rl2(r["grads"][n], ro["grads"][n]), np.linalg.norm(ro["grads"][n])))
# ---- which BN backward call produces a wrong dbeta?
from toda_b200 import ops
orig = ops._bn_backward_phases
log = []
def spy(da, y, a, gamma, mean, rstd, training, relu, has_res, want_bf16, gsums=None, want_db=False):
    out = yield from orig(da, y, a, gamma, mean, rstd, training, relu, has_res, want_bf16, gsums, want_db)
    dy, dyb, dres, dgamma, dbeta, _ = out
    g = da * (a > 0) if relu else da
    ref_db = g.double().sum(0)
    xhat = (y.double() - mean.double()) * rstd.double()
    ref_dg = (g.double() * xhat).sum(0)
    log.append((y.shape, has_res, float((dbeta.double() - ref_db).norm() / ref_db.norm()), float((dgamma.double() - ref_dg).norm() / ref_dg.norm()),
                bool(torch.isfinite(da).all()), float(da.abs().max())))
    return out
ops._bn_backward_phases = spy
twin, net = PU.build_pair("VoxelResBackBone8x", nf, g["grid_size"], seed=int(g["seed"]))
r = PU.run_backbone(net, hc, vf, vc, 2, cot=cot, train=True)
for l in log[:8]: print(l)
# ---- compare d(x_conv4) between oracle and GPU
das = []
def spy2(da, y, a, gamma, mean, rstd, training, relu, has_res, want_bf16, gsums=None, want_db=False):
    das.append((da.detach().cpu().numpy().copy(), a.detach().cpu().numpy().copy()))
    return (yield from orig(da, y, a, gamma, mean, rstd, training, relu, has_res, want_bf16, gsums, want_db))
ops._bn_backward_phases = spy2
twin, net = PU.build_pair("VoxelResBackBone8x", nf, g["grid_size"], seed=int(g["seed"]))
net.train(); twin.train()
bd_g = hc(net({"voxel_features": vf.clone().requires_grad_(True), "voxel_coords": vc, "batch_size": 2}))
(bd_g["spatial_features"] * cot.cuda()).sum().backward()
x4g = bd_g["multi_scale_3d_features"]["x_conv4"]
vfo = torch.from_numpy(g["voxel_features"]).clone().requires_grad_(True)
bd_o = PU._oracle_hc(twin({"voxel_features": vfo, "voxel_coords": torch.from_numpy(g["voxel_coords"]).float(), "batch_size": 2}))
x4o = bd_o["multi_scale_3d_features"]["x_conv4"]
x4o.features.retain_grad()
(bd_o["spatial_features"] * cot).sum().backward()
da_g, a_g = das[1]
og = PU.canonical_order(x4g.indices.cpu().numpy()); oo = PU.canonical_order(x4o.indices.numpy())
assert np.array_equal(x4g.indices.cpu().numpy()[og], x4o.indices.numpy()[oo])
d = np.abs(da_g[og] - x4o.features.grad.numpy()[oo])
fa = np.abs(a_g[og] - x4o.features.detach().numpy()[oo])
zc = x4o.indices.numpy()[oo][:, 1]
print("d x_conv4: max err", d.max(), "rows with err>1e-4:", int((d.max(1) > 1e-4).sum()), "their z:", np.unique(zc[d.max(1) > 1e-4], return_counts=True), "fwd max err", fa.max())
print("rows per z", np.unique(zc, return_counts=True))
ag, ao = a_g[og], x4o.features.detach().numpy()[oo]
flip = (ag > 0) != (ao > 0)
print("relu mask flips at x_conv4:", int(flip.sum()), "of", flip.size, " |a| there:", np.abs(ag[flip]), np.abs(ao[flip]), " da there:", da_g[og][flip])
