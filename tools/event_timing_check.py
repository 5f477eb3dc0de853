import sys, os, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import pendulum_batch, make_controller
B = 65536
cfg, X0, Xref = pendulum_batch(B, "identical")
K = make_controller(cfg, X0, Xref, B, 0); K.solve(); K.output()
dev = torch.device("cuda", 0); L, h = K._L, K.handle
stream = torch.cuda.Stream(dev); torch.cuda.synchronize(dev); torch.cuda.set_stream(stream)   # handle 0 would mean the library's own stream
L.bmpc_set_stream(h, stream.cuda_stream)
Ad = torch.tensor(cfg["Ad"], device=dev); Bd = torch.tensor(cfg["Bd"], device=dev)
Xd = torch.tensor(X0, device=dev); Xn = torch.empty_like(Xd)
U = [torch.zeros(B, 1, dtype=torch.float64, device=dev) for _ in range(2)]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
for mode in (1, 2):
    for doflush in (1, 0):
        rows = []
        for t in range(30):
            L.bmpc_bind_output(h, U[t & 1].data_ptr())
            if doflush: flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); ea = torch.cuda.Event(enable_timing=True); eb = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            L.bmpc_update(h, Xd.data_ptr(), U[(t & 1) ^ 1].data_ptr(), None, 1, mode)
            ea.record(stream)
            L.bmpc_solve(h)
            eb.record(stream)
            L.bmpc_output(h, None, None, 1, 1)
            e1.record(stream)
            torch.matmul(Xd, Ad.T, out=Xn); Xn.addmm_(U[t & 1], Bd.T)
            st = K.stats(); torch.cuda.synchronize(); Xd, Xn = Xn, Xd
            if t >= 10: rows.append((e0.elapsed_time(e1), e0.elapsed_time(ea), ea.elapsed_time(eb), eb.elapsed_time(e1), st["ms_admm"], st["ms_polish"]))
        r = np.median(np.array(rows), axis=0)
        print(f"mode={mode} flush={doflush}: step {r[0]:.4f} update {r[1]:.4f} solve {r[2]:.4f} output {r[3]:.4f} | stats admm {r[4]:.4f} polish {r[5]:.4f}")
