"""Device timeline of the conv kernels of ONE bf16 forward (globaltimer stamps of first CTA entry / last CTA exit per launch):
shows the gaps between kernels and the overlap of the attention branch.  usage (GPU box): python tools/timeline_forward.py [batch]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import healthivert_gan_b200 as hv
from healthivert_gan_b200 import _lib
from oracle import synth

n = int(sys.argv[1]) if len(sys.argv) > 1 else 16
g = hv.Generator({"input_dim": 1, "ngf": 16}, True); g.load_state_dict(synth.synthetic_generator_state_dict()); g = g.cuda().eval(); g.precision = "bf16"
x, mask, cam, ratio = (t.cuda() for t in synth.synthetic_slices(n, seed=1))
L = _lib.lib()
L.hv_debug_conv_timeline.argtypes = [ctypes.c_void_p]
order = ("C1 C2 C3 C4 C5 C6 C7 C8 C9 C10 C11 C12 C20 C13 C14 C19 C15 C16 C17 F1 PM2 PM3 PM4 PM5 PM6 PM9 PM10 "
         "F2 F3 F4 F5 F6 F7 F8 F9 F10 A11 A12 A19 A13 A14 A15 A16 A17")
if int(os.environ.get("HV_NO_TAIL_FUSE") or 0) == 0:   # conv16 + heads of each stage run as one fused launch (CTAIL / ATAIL)
    order = order.replace("C16 C17", "CTAIL").replace("A16 A17", "ATAIL")
if int(os.environ.get("HV_NO_STEM_FUSE") or 0) == 0:   # conv1 + conv2 of each stage (+ pmconv2) run as one fused launch (CSTEM / FSTEM)
    order = order.replace("C1 C2 ", "CSTEM ").replace("F1 PM2 ", "FSTEM ").replace(" F2 ", " ")
order = order.split()
with torch.no_grad():
    for _ in range(3):
        g(x, mask, cam, ratio)
    torch.cuda.synchronize()
    buf = torch.zeros(4 * 64, dtype=torch.int64, device="cuda")
    buf[0::4] = 1 << 62
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    L.hv_debug_conv_timeline(buf.data_ptr())
    g(x, mask, cam, ratio)           # first use of the instances that carry the diagnostics (lazy module load), not measured
    torch.cuda.synchronize()
    buf.zero_()
    buf[0::4] = 1 << 62
    L.hv_debug_conv_timeline(buf.data_ptr())
    e0.record()
    g(x, mask, cam, ratio)
    e1.record()
    torch.cuda.synchronize()
    L.hv_debug_conv_timeline(None)
b = buf.cpu().tolist()
rows = [(order[i], b[4 * i], b[4 * i + 1]) for i in range(len(order)) if b[4 * i + 1]]
t0 = min(r[1] for r in rows)
print(f"forward (events) {e0.elapsed_time(e1) * 1e3:.0f} us; first conv entry -> last conv exit {(max(r[2] for r in rows) - t0) / 1e3:.0f} us")
prev_end = {}
main = [r for r in rows if not r[0].startswith("PM")]
side = [r for r in rows if r[0].startswith("PM")]
for name, lst in (("main stream", main), ("attention branch", side)):
    print(name)
    pe = None
    busy = 0
    for nm, s, e in lst:
        gap = (s - pe) / 1e3 if pe else 0.0
        busy += (e - s) / 1e3
        print(f"  {nm:5s} start {(s - t0) / 1e3:8.1f}  dur {(e - s) / 1e3:6.1f}  gap before {gap:6.1f}")
        pe = e
    print(f"  sum of durations {busy:.0f} us")
