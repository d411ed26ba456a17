#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (rgl-epfl/large-steps-pytorch) on the CPU.
The tests only read the stored files; the reference is needed only to regenerate them:
    LARGESTEPS_REF=<checkout of rgl-epfl/large-steps-pytorch> python tests/golden/make_golden.py

How the reference is made to run here without a GPU / without cholespy (nothing is copied into the repo):
  * largesteps/geometry.py hard-codes device='cuda' (geometry.py:60,83,125).  Its source text is read
    from the checkout at run time, the literal "device='cuda'" is replaced by "device='cpu'" in memory,
    and the result is exec'd as module `largesteps.geometry`.
  * largesteps/solvers.py imports cholespy (solvers.py:3), which is not installable offline.  A stub module
    is registered in sys.modules so ConjugateGradientSolver / DifferentiableSolve / from_differential(method='CG')
    import and run unmodified.  The Cholesky path itself cannot run (parity unpinned at that boundary).
"""
import os
import sys
import types
import importlib.util
import warnings

import numpy as np
import torch

REF = os.environ.get("LARGESTEPS_REF", "")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "..", "large-steps-pytorch_b200"))
from largesteps_b200 import workloads  # noqa: E402  (mesh generators only)

warnings.filterwarnings("ignore")
torch.set_num_threads(4)


def load_reference():
    if not os.path.isfile(os.path.join(REF, "largesteps", "geometry.py")):
        sys.exit("set LARGESTEPS_REF to a checkout of rgl-epfl/large-steps-pytorch")
    chol = types.ModuleType("cholespy")
    chol.CholeskySolverF = object
    chol.MatrixType = types.SimpleNamespace(COO=0)
    sys.modules["cholespy"] = chol
    pkg = types.ModuleType("largesteps")
    pkg.__path__ = [os.path.join(REF, "largesteps")]
    sys.modules["largesteps"] = pkg
    src = open(os.path.join(REF, "largesteps", "geometry.py")).read().replace("device='cuda'", "device='cpu'")
    geo = types.ModuleType("largesteps.geometry")
    exec(compile(src, os.path.join(REF, "largesteps", "geometry.py"), "exec"), geo.__dict__)
    sys.modules["largesteps.geometry"] = geo
    mods = {"geometry": geo}
    for name in ("solvers", "parameterize", "optimize"):
        spec = importlib.util.spec_from_file_location(f"largesteps.{name}", os.path.join(REF, "largesteps", f"{name}.py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[f"largesteps.{name}"] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods


def coo(M):
    M = M.coalesce()
    return M.indices().numpy().astype(np.int64), M.values().numpy().astype(np.float32)


def main():
    ref = load_reference()
    geo, par, sol, opt = ref["geometry"], ref["parameterize"], ref["solvers"], ref["optimize"]
    out = {}

    # ---- meshes -------------------------------------------------------------------------------------
    tet_v = np.array([[0, 0, 0], [1, 1, 0], [1, 0, 1], [0, 1, 1]], dtype=np.float32)
    tet_f = np.array([[0, 1, 2], [0, 3, 1], [0, 2, 3], [1, 3, 2]], dtype=np.int64)
    quad_v = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0]], dtype=np.float32)
    quad_f = np.array([[0, 1, 2], [0, 2, 3]], dtype=np.int64)
    ico_v, ico_f = workloads.icosphere(2)                       # 162 V
    bun_v64, bun_f = workloads.load_obj(os.path.join(REF, "ext/botsch-kobbelt-remesher-libigl/data/bunny.obj"))
    bun_v = bun_v64.astype(np.float32)
    # mesh with an isolated vertex (index 4 unused) and a non-manifold edge (3 faces on edge 0-1)
    odd_v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [5, 5, 5], [0.3, -1, 0.2]], dtype=np.float32)
    odd_f = np.array([[0, 1, 2], [0, 1, 3], [1, 0, 5]], dtype=np.int64)
    meshes = {"tet": (tet_v, tet_f), "quad": (quad_v, quad_f), "ico2": (ico_v, ico_f),
              "bunny": (bun_v, bun_f), "odd": (odd_v, odd_f)}
    np.savez_compressed(os.path.join(HERE, "bunny_mesh.npz"), verts=bun_v, faces=bun_f.astype(np.int32))

    # ---- assembly: geometry.py compute_matrix / laplacians ------------------------------------------
    cases = [("uni_l10", dict(lambda_=10.0)), ("uni_a095", dict(lambda_=1.0, alpha=0.95)),
             ("cot_l19", dict(lambda_=19.0, cotan=True)), ("cot_a09", dict(lambda_=1.0, alpha=0.9, cotan=True))]
    for mname, (v, f) in meshes.items():
        out[f"{mname}.verts"] = v
        out[f"{mname}.faces"] = f
        tv, tf = torch.from_numpy(v), torch.from_numpy(f)
        for cname, kw in cases:
            idx, val = coo(geo.compute_matrix(tv, tf, **kw))
            out[f"{mname}.{cname}.idx"] = idx
            out[f"{mname}.{cname}.val"] = val
        idx, val = coo(geo.laplacian_uniform(tv, tf))
        out[f"{mname}.Luni.idx"], out[f"{mname}.Luni.val"] = idx, val
        idx, val = coo(geo.laplacian_cot(tv, tf))
        out[f"{mname}.Lcot.idx"], out[f"{mname}.Lcot.val"] = idx, val
    try:
        geo.compute_matrix(torch.from_numpy(tet_v), torch.from_numpy(tet_f), 1.0, alpha=1.0)
        out["alpha_error"] = np.array("none")
    except ValueError as e:
        out["alpha_error"] = np.array(str(e))
    np.savez_compressed(os.path.join(HERE, "assembly.npz"), **out)

    # ---- to_differential / reference CG / from_differential(method='CG') + autograd ------------------
    sv = {}
    for mname, kw in (("ico2", dict(lambda_=10.0)), ("bunny", dict(lambda_=19.0, cotan=True))):
        v, f = meshes[mname]
        M = geo.compute_matrix(torch.from_numpy(v), torch.from_numpy(f), **kw)
        rng = np.random.default_rng(0)
        vv = torch.from_numpy((v + rng.normal(0, 0.01, v.shape)).astype(np.float32))
        u = par.to_differential(M, vv)
        b = (u + torch.from_numpy(np.random.default_rng(1).normal(0, 0.01, v.shape).astype(np.float32)))
        g = torch.from_numpy((1e-4 * np.random.default_rng(2).normal(0, 1, v.shape)).astype(np.float32))
        sv[f"{mname}.v"], sv[f"{mname}.u"], sv[f"{mname}.b"], sv[f"{mname}.g"] = vv.numpy(), u.numpy(), b.numpy(), g.numpy()
        cg = sol.ConjugateGradientSolver(M)
        x1 = cg.solve(b.clone())                       # cold
        x2 = cg.solve((b * 1.01).clone())              # warm start from x1 (solvers.py:107-110)
        xb = cg.solve(g.clone(), backward=True)
        sv[f"{mname}.cg_x1"], sv[f"{mname}.cg_x2"], sv[f"{mname}.cg_xb"] = x1.numpy(), x2.numpy(), xb.numpy()
        # differentiable path, exactly as scripts/main.py:173,206 use it
        uu = b.clone().requires_grad_(True)
        vout = par.from_differential(M, uu, "CG")
        (vout * g).sum().backward()
        sv[f"{mname}.fd_v"], sv[f"{mname}.fd_grad"] = vout.detach().numpy(), uu.grad.numpy()
    try:
        par.from_differential(M, b, "nope")
        sv["method_error"] = np.array("none")
    except ValueError as e:
        sv["method_error"] = np.array(str(e))
    try:
        sol.ConjugateGradientSolver(M).solve(b[:, 0])
        sv["shape_error"] = np.array("none")
    except ValueError as e:
        sv["shape_error"] = np.array(str(e))
    np.savez_compressed(os.path.join(HERE, "solve.npz"), **sv)

    # ---- AdamUniform (optimize.py:17-41) --------------------------------------------------------------
    ad = {}
    rng = np.random.default_rng(3)
    p0 = rng.normal(0, 1, (500, 3)).astype(np.float32)
    p = torch.nn.Parameter(torch.from_numpy(p0.copy()))
    o = opt.AdamUniform([p], lr=0.05, betas=(0.9, 0.999))
    ad["p0"] = p0
    for s in range(4):
        gnp = (rng.normal(0, 1, (500, 3)) * (10.0 ** (-s))).astype(np.float32)
        p.grad = torch.from_numpy(gnp.copy())
        o.step()
        ad[f"g{s}"] = gnp
        ad[f"p{s + 1}"] = p.detach().numpy().copy()
    np.savez_compressed(os.path.join(HERE, "adam.npz"), **ad)
    for fn in ("assembly.npz", "solve.npz", "adam.npz", "bunny_mesh.npz"):
        print(fn, os.path.getsize(os.path.join(HERE, fn)), "bytes")


if __name__ == "__main__":
    main()
