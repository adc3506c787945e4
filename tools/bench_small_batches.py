"""Developer check: chain-steps/s of cfg3-shaped models with few chains (cluster variant of the evaluation kernel)."""
import sys, os, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
from gladsgp_b200 import _lib
if os.environ.get('GGP_LIB'):
    _lib.LIB_PATH = os.environ['GGP_LIB']
from gladsgp_b200 import svd, model as gmodel
from sepia.SepiaData import SepiaData
from sepia.SepiaModel import SepiaModel
t, y, mu, sd = bench.build_problem(400, 36, standardized=False)
data = SepiaData(t_sim=t, y_sim=y, y_ind_sim=np.linspace(0, 1, y.shape[1]))
data.transform_xt(t_notrans=np.arange(8)); data.standardize_y(y_mean=mu, y_sd=sd)
np.random.seed(1)
U, S, Vh = svd.randomized_svd(data.sim_data.y_std, 25, k=0, q=1)
K = ((S[:10, None] * Vh[:10]) / np.sqrt(512)).astype(np.float32)
data.create_K_basis(K=K)
model = SepiaModel(data)
gmodel.override_lamWOs(model, gmodel.pc_precision(data.sim_data))
res = {}
for chains in (1, 4, 16):
    model.do_mcmc_chains(5, chains); torch.cuda.synchronize()
    t0 = time.perf_counter(); model.do_mcmc_chains(30, chains); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    res[chains] = chains * 30 / dt
print(json.dumps(res))
