import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vittles_b200 import ops
dev = torch.device('cuda', 0)
N, D = 2000000, 1024
X = ops.synth_design(1, 0, N, D, dev)
theta = 0.3 * ops.synth_theta(1, D, dev)
y = (torch.rand(N, device=dev, dtype=torch.float64) < 0.5).double()
w = torch.ones(N, device=dev, dtype=torch.float64)
def timed(fn, reps=5):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): out = fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out
t0, st = timed(lambda: ops.glm_stats(X, theta, y, w))
t1, st2 = timed(lambda: ops.glm_stats(X, theta, y, w, want_colmax=True))
s = st[2]
t2, _ = timed(lambda: ops.syrk_weighted(X, s, precision='f64_ozaki'), reps=3)
t3, _ = timed(lambda: ops.syrk_weighted(X, s, precision='f64_ozaki', colmax=st2[4]), reps=3)
print('stats %.3f ms, stats+colmax %.3f ms, syrk %.3f ms, syrk with colmax given %.3f ms' % (t0, t1, t2, t3))
