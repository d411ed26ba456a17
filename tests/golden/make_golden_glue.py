#!/usr/bin/env python
"""Generate tests/golden/glue.npz by running the UNMODIFIED reference loop glue (scripts/geometry.py of
rgl-epfl/large-steps-pytorch: remove_duplicates, average_edge_length, compute_face_normals, compute_vertex_normals) and the
(bi)Laplacian regulariser of scripts/main.py:192-195 on the CPU, in float32 (what the reference runs) and in float64 (a tight
reference for the gradients).

    LARGESTEPS_REF=<checkout of rgl-epfl/large-steps-pytorch> python tests/golden/make_golden_glue.py
"""
import importlib.util
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import load_reference, REF, workloads  # noqa: E402

warnings.filterwarnings("ignore")
torch.set_num_threads(4)


def main():
    spec = importlib.util.spec_from_file_location("ref_scripts_geometry", os.path.join(REF, "scripts", "geometry.py"))
    sg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sg)
    geo = load_reference()["geometry"]
    out = {}
    d = np.load(os.path.join(HERE, "bunny_mesh.npz"))
    meshes = {"ico2": workloads.icosphere(2), "bunny": (d["verts"], d["faces"].astype(np.int64))}
    for name, (v, f) in meshes.items():
        V = len(v)
        rng = np.random.default_rng(11)
        # a mesh with seams: the first V/8 vertices exist twice, and a third of the faces that touch them use the copy
        ndup = V // 8
        v_src = np.concatenate([v, v[:ndup]], axis=0).astype(np.float32)
        f_src = f.copy()
        pick = rng.random(f_src.shape) < 0.33
        f_src = np.where(pick & (f_src < ndup), f_src + V, f_src)
        tv, tf = torch.from_numpy(v_src), torch.from_numpy(f_src)
        v_unique, f_unique, dup = sg.remove_duplicates(tv, tf)
        out[f"{name}.v_src"], out[f"{name}.f_src"] = v_src, f_src
        out[f"{name}.v_unique"], out[f"{name}.f_unique"], out[f"{name}.dup"] = v_unique.numpy(), f_unique.numpy(), dup.numpy()
        out[f"{name}.avg_edge"] = sg.average_edge_length(v_unique, f_unique).numpy()
        W1 = rng.normal(size=(len(v_src), 3)).astype(np.float32)
        W2 = rng.normal(size=(len(v_src), 3)).astype(np.float32)
        W3 = rng.normal(size=(3, len(f_src))).astype(np.float32)
        out[f"{name}.W1"], out[f"{name}.W2"], out[f"{name}.W3"] = W1, W2, W3
        L = geo.laplacian_uniform(v_unique, f_unique)
        for dt, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
            x = (v_unique.to(dt) + 0.01 * torch.from_numpy(rng.normal(size=tuple(v_unique.shape))).to(dt) * 0).clone().requires_grad_(True)
            v_opt = x[dup]
            fn = sg.compute_face_normals(x, f_unique)
            n_unique = sg.compute_vertex_normals(x, f_unique, fn)
            n_opt = n_unique[dup]
            loss = (v_opt * torch.from_numpy(W1).to(dt)).sum() + (n_opt * torch.from_numpy(W2).to(dt)).sum() \
                + (fn * torch.from_numpy(W3).to(dt)).sum()
            loss.backward()
            if tag == "f32":      # the float64 face normals are read by no test and would take the file past 1 MB
                out[f"{name}.{tag}.face_normals"] = fn.detach().numpy()
            out[f"{name}.{tag}.vertex_normals"] = n_unique.detach().numpy()
            out[f"{name}.{tag}.n_opt"] = n_opt.detach().numpy()
            out[f"{name}.{tag}.loss"] = loss.detach().numpy()
            out[f"{name}.{tag}.grad"] = x.grad.numpy().copy()
            # regulariser (scripts/main.py:192-195)
            Ld = L.to(dt)
            for bil, rn in ((True, "bilap"), (False, "lap")):
                y = v_unique.to(dt).clone().requires_grad_(True)
                reg = (Ld @ y).square().mean() if bil else (y * (Ld @ y)).mean()
                reg.backward()
                out[f"{name}.{tag}.{rn}"] = reg.detach().numpy()
                out[f"{name}.{tag}.{rn}_grad"] = y.grad.numpy().copy()
    np.savez_compressed(os.path.join(HERE, "glue.npz"), **out)
    print("glue.npz", os.path.getsize(os.path.join(HERE, "glue.npz")), "bytes;",
          {k: out[k].shape for k in out if k.startswith("ico2.") and "f32" not in k and "f64" not in k})


if __name__ == "__main__":
    main()
