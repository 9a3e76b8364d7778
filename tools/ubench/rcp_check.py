import os, sys, ctypes as C, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from pnp_solver_test_b200 import _lib
rng = np.random.default_rng(5)
a = np.concatenate([rng.uniform(0.5, 2.0, 2000000), 10.0 ** rng.uniform(-250, 250, 100000)])
x = torch.from_numpy(a).cuda()
for sign in (1,):
    o = [torch.empty_like(x) for _ in range(3)]
    _lib.check(_lib.lib.pnpb200_selftest_math(C.c_int64(sign * a.size), C.c_void_p(x.data_ptr()), C.c_void_p(o[0].data_ptr()), C.c_void_p(o[1].data_ptr()), C.c_void_p(o[2].data_ptr()), None), "st")
    torch.cuda.synchronize()
    rcp = o[0].cpu().numpy()
    err = np.abs(rcp * a.astype(np.longdouble) - 1) / 2.0**-52
    exact = (rcp == 1.0 / a).mean()
    print("sign", sign, "max err ulp", float(err.max()), "correctly rounded frac", exact)
