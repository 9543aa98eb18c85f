"""In-situ timeline of one generator forward (PDL overlap intact): per launch the time from the previous launch's last CTA end
to this launch's first CTA start (gap), and its own span; launch i is op i of the plan's forward (op 0, the input conversion, has no
stamps).  python tools/timeline.py [workload] ; CSR_OPTS as in bench.py."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))
from bench import WORKLOADS  # noqa: E402
from climsr_b200._lib import lib  # noqa: E402
from climsr_b200.models import ESRGANGenerator  # noqa: E402

if __name__ == "__main__":
    wl = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    for kv in filter(None, os.environ.get("CSR_OPTS", "").split(",")):
        k, v = kv.split("=")
        lib.csr_set_option(int(k), int(v))
    lib.csr_set_option(11, 0)                                   # direct launches (graphs would freeze the launch parameters)
    in_ch, nb, gc, tiles, h, w = WORKLOADS[wl]
    torch.manual_seed(0)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc).cuda().eval()
    x = torch.rand((tiles, in_ch, h, w), device="cuda") * 2 - 1
    mask = (torch.rand((tiles, 1, 4 * h, 4 * w), device="cuda") > 0.3).float()
    elev = torch.rand((tiles, 1, 4 * h, 4 * w), device="cuda") * mask
    cap = 512
    with torch.no_grad():
        for _ in range(3):
            net(x, elev, mask)
        tl = torch.zeros(2 * cap, dtype=torch.int64, device="cuda")
        tl[0::2] = -1                                           # ~0ull
        lib.csr_debug_set_timeline(tl.data_ptr(), cap)
        net(x, elev, mask)
        torch.cuda.synchronize()
        lib.csr_debug_set_timeline(None, 0)
    t = tl.cpu().view(cap, 2)
    rows = [(i, int(t[i, 0]), int(t[i, 1])) for i in range(cap) if int(t[i, 1]) != 0]
    t0 = rows[0][1]
    print(f"{wl}: {len(rows)} launches, {(rows[-1][2] - t0) / 1e3:.1f} us from first start to last end")
    prev_end = t0
    agg = {}
    for i, s, e in rows:
        gap, span = (s - prev_end) / 1e3, (e - s) / 1e3
        print(f"launch {i:4d}  start {(s - t0) / 1e3:9.1f} us  gap {gap:6.1f}  span {span:7.1f}")
        prev_end = e
