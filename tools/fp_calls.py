import contextlib, io, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import svnet_b200 as sv
from svnet_b200 import _native as nv, fused
from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict
with contextlib.redirect_stdout(io.StringIO()):
    net = sv.SV_DGCNN_CLS(make_args(k=20, binary=False), 15)
net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=1003))
net = net.cuda().eval()
x = synthetic_clouds(32, 1024, 1003).cuda()
fused.CONCURRENT_HALVES = False
with torch.no_grad():
    for _ in range(3): net(x)
    torch.cuda.synchronize()
    nv.PROFILE[0] = set(nv.EXPORTS); nv.ORDER.clear()
    net(x); torch.cuda.synchronize()
for name, e0, e1 in nv.ORDER:
    print("%-28s %8.1f us" % (name, 1e3 * e0.elapsed_time(e1)))
