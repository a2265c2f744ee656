"""Per-kernel timing of one bf16 training step at B=8192 (scratch tool)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from roomslam_b200 import RoomSLAM, synth, functional as F_
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
torch.manual_seed(0)
m = RoomSLAM(dropout=float(os.environ.get("RS_PROBE_DROPOUT", "0.0")), precision="bf16").cuda().train()
x, tgt = synth.make_sample(B, 500, 10, seed=0, device="cuda")
def step():
    m.zero_grad(); l = m.compute_loss(m(x), tgt)["total"]; l.backward(); return l
for _ in range(3): step()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(3): step()
e1.record(); torch.cuda.synchronize()
F_.enable_kernel_timing(True); step(); k = F_.collect_kernel_timing(); F_.enable_kernel_timing(False)
print("ms/step %.2f" % (e0.elapsed_time(e1) / 3), {n: round(v[0], 2) for n, v in k.items()})
# per-launch detail (layer order: forward L0, L1; backward L1, L0)
F_.enable_kernel_timing(True); step(); torch.cuda.synchronize()
for name, a, b, fl in F_._KT["events"]:
    print("   %-36s %7.3f ms" % (name, a.elapsed_time(b)))
F_.enable_kernel_timing(False)
