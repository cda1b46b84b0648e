import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-nmf_b200"), os.path.join(ROOT, "tests")]
import torch
from conftest import load_npz
from torchnmf_b200 import PLCA
Z = load_npz("reference_next.npz")
def case(name): return {k.split("/", 1)[1]: Z[k] for k in Z.files if k.startswith(name + "/")}
for name in ("plca_small", "plca_prior", "plca_frozenZ", "plca_tc"):
    c = case(name)
    for prec in ("f32", "f16", "f16_split"):
        t = lambda k: torch.from_numpy(c[k].copy())
        m = PLCA(W=t("W0"), H=t("H0"), Z=t("Z0"), trainable_Z=bool(int(c["trainable_Z"]))).cuda()
        m.fit(t("V").cuda(), float("-inf"), int(c["iters"]), False, float(c["W_alpha"]), float(c["H_alpha"]), float(c["Z_alpha"]), precision=prec)
        errs = []
        for nm in ("W", "H", "Z"):
            want = t(nm); got = getattr(m, nm).data.cpu()
            errs.append(float(((got - want).abs() / (1e-3 * want.abs() + 1e-5 * want.abs().max())).max()))
        print(name, prec, m.last_fit_precision, "W %.2f H %.2f Z %.2f x tol" % tuple(errs), flush=True)
