"""Development: dump the clock64 trace of CTA 0 of the streaming conv kernel (needs a -DTTG_TRACE build)."""
import sys, os, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tartangan_b200 import ops, _lib
from tartangan_b200._lib import call, ptr
n, h, w, cin, cout, k = [int(v) for v in sys.argv[1:7]]
bf = torch.bfloat16
x = ops.empty_nhwc(n, cin, h, w, bf, 'cuda'); x.normal_()
wt = torch.randn(cout, cin, k, k, device='cuda') * 0.05
wp = ops._packed(wt, 0, 'tc')
y = ops.empty_nhwc(n, cout, h, w, bf, 'cuda')
fn = lambda: call('ttg_conv2d_tc', ptr(x), ptr(wp), None, ptr(y), n, h, w, cin, cout, k, _lib.BF16)
if len(sys.argv) > 7 and sys.argv[7] == 'wgrad':
    gy = ops.empty_nhwc(n, cout, h, w, bf, 'cuda'); gy.normal_()
    gw = torch.empty(cout, cin, k, k, device='cuda')
    ws = torch.empty(_lib.lib.ttg_conv2d_wgrad_tc_workspace_bytes(cin, cout, k) // 4 + 4, device='cuda')
    fn = lambda: call('ttg_conv2d_wgrad_tc', ptr(x), ptr(gy), ptr(gw), n, h, w, cin, cout, k, ptr(ws))
dll = _lib.lib.load()
buf = (ctypes.c_longlong * (16 * 256 * 2))()
for _ in range(3): fn()
dll.ttg_trace_read(buf, 1)
fn()
dll.ttg_trace_read(buf, 1)
ev = []
for role in range(16):
    for i in range(256):
        t0, t1 = buf[(role * 256 + i) * 2], buf[(role * 256 + i) * 2 + 1]
        if t0:
            ev.append((role, i, t0, t1))
t00 = min(e[2] for e in ev)
names = {1: 'mma.wait_wfull', 2: 'mma.wait_afull', 3: 'mma.wait_accempty', 4: 'str.wait_wempty', 5: 'epi.wait_accfull', 6: 'epi.run', 7: 'mma.issue4', 8: 'mma.commit', 9: 'wg.wait_done', 10: 'wg.epilogue', 11: 'wg.iss_wait_full', 12: 'wg.iss_issue', 13: 'wg.tma_wait_empty'}
for e in sorted(ev, key=lambda e: e[2]):
    print(f'{names.get(e[0], e[0]):18s} idx {e[1]:4d}  t0 {e[2]-t00:8d}  dur {e[3]-e[2]:7d}')
