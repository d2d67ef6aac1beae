#!/usr/bin/env python
"""Timing of the SRF band-convolution mode (band_kernel_srf) on 100 k bench-distribution samples;
SPART_B200_LIB selects an alternative build of the library.  usage: python tools/srfbench.py [sensor]
(default Sentinel2A-MSI)"""
import sys, json, os
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / 'spart-python_b200')); sys.path.insert(0, str(ROOT))
import torch, bench, spart_b200
dev=torch.device('cuda',0); eng=spart_b200.default_engine(dev)
n=100000
sensor=sys.argv[1] if len(sys.argv) > 1 else 'Sentinel2A-MSI'
P=bench.synthetic_params_torch(n, 20261020, dev)
out=None
for _ in range(2): out=eng.forward_bands(P,sensor,uniform_geometry=True,band_mode='srf')
torch.cuda.synchronize()
e0,e1=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(5): out=eng.forward_bands(P,sensor,uniform_geometry=True,band_mode='srf')
e1.record(); torch.cuda.synchronize()
ms=e0.elapsed_time(e1)/5
print(json.dumps({'lib':os.environ.get('SPART_B200_LIB','default'),'sensor':sensor,'srf_ms_per_100k':ms,'Msims':n/ms/1e3,'checksum':float(out.sum())}))
