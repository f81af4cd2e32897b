"""Three all-task steps of BASELINE config 4 (ii) (256 policies, beta = 30, B = 4096, GPI over 256 reward vectors) for ncu:
   ncu --set full --clock-control none --import-source on -k regex:'step_prep|fold_gpi|mlp_forward_tc|td_kernel|dgrad_tc|wgrad_tc|adam_step' \
       -s 14 -c 7 -o gpurun_out/r02_config4 python scripts/profile_config4.py"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from deep_successor_features_for_transfer_b200.workloads import build_tsf_agent, synthetic_transitions, ENVS

N = int(sys.argv[1]) if len(sys.argv) > 1 else 256
shp = ENVS['reacher']
dsf, ag = build_tsf_agent('reacher', N, [256, 256], ['relu', 'relu'], 100, 30, 'bf16', True, seed=1034)
gen = torch.Generator().manual_seed(1024)
res = [tuple(t.cuda() for t in synthetic_transitions(4096, shp['S'], shp['A'], shp['D'], gen)) for _ in range(3)]
for k in range(3):
    ag.update_successor_all(res[k], use_gpi=True)
torch.cuda.synchronize()
print('done')
