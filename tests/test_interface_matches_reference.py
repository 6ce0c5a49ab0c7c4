"""Drop-in boundary: the host-side mirrors must accept exactly what the reference's callers pass (SURVEY.md 8b).
The reference's signatures and the MPI construction + call its MPIRenderer.render makes were recorded from the unmodified
reference (tests/golden/reference_signatures.json, tests/golden/reference_mpi_call.npz, oracle/make_golden_interface.py)."""
import inspect
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN


def _params(fn):
    """The rows oracle/make_golden_interface.py recorded: (name, kind, repr(default)) without self."""
    return [[n, p.kind.name, repr(p.default)] for n, p in inspect.signature(fn).parameters.items() if n != "self"]


def _reference_signatures():
    with open(os.path.join(GOLDEN, "reference_signatures.json")) as f:
        return json.load(f)


def _decode_kwargs(z, prefix):
    """Inverse of make_golden_interface.encode_kwargs: the keyword arguments in the order the reference passed them."""
    kw = {}
    for name in z[prefix + "order"]:
        name = str(name)
        if f"{prefix}none/{name}" in z.files:
            kw[name] = None
        elif f"{prefix}t/{name}" in z.files:
            kw[name] = torch.from_numpy(z[f"{prefix}t/{name}"])
        elif f"{prefix}a/{name}" in z.files:
            kw[name] = z[f"{prefix}a/{name}"]
        elif f"{prefix}s/{name}" in z.files:
            kw[name] = z[f"{prefix}s/{name}"].item()
        else:
            n = sum(1 for k in z.files if k.startswith(f"{prefix}l/{name}/"))
            assert n > 0, name
            kw[name] = [torch.from_numpy(z[f"{prefix}l/{name}/{i}"]) for i in range(n)]
    return kw


def test_mpi_signatures():
    ref = _reference_signatures()["MPI"]
    import ml_gmpi_b200 as g
    assert _params(g.MPI.forward) == ref["forward"]                  # keyword-only, same names, same defaults
    assert _params(g.MPI.check_shapes) == ref["check_shapes"]
    init_ref = ref["__init__"]
    init_ours = _params(g.MPI.__init__)
    assert init_ours[: len(init_ref)] == init_ref                    # ours adds the optional `validate` after align_corners


def test_renderer_signatures():
    ref = _reference_signatures()["MPIRenderer"]
    from ml_gmpi_b200.renderer import MPIRenderer
    for name in ("render", "sample_cam_poses", "set_cam", "compute_mpi_spatial_volume"):
        assert _params(getattr(MPIRenderer, name)) == ref[name], name
    ref_init = ref["__init__"]
    ours_init = _params(MPIRenderer.__init__)
    assert ours_init[: len(ref_init)] == ref_init                    # ours adds the optional `validate`


def test_reference_call_site_binds():
    """mpi_renderer.py:451-461 calls self.mpi(batch_rgba=..., ..., c2w_mat=..., sphere_c=...): must bind to our forward."""
    import ml_gmpi_b200 as g
    sig = inspect.signature(g.MPI.forward)
    sig.bind(None, batch_rgba=1, batch_dhw=2, batch_ray_dir=3, batch_eye_pos=4, batch_z_dir=5, separate_background=None,
             assert_not_out_of_last_plane=True, c2w_mat=6, sphere_c=7)


def test_unmodified_reference_renderer_drives_the_drop_in():
    """INTEGRATION.md's patch (`gmpi.core.mpi_renderer.MPI = ml_gmpi_b200.MPI`), replayed: the unmodified reference
    MPIRenderer constructs MPI (mpi_renderer.py:47) and, inside `render`, calls it with the tensors its own pose sampling and
    ray generation produced (mpi_renderer.py:418-461).  Both were recorded; replayed against our class, the construction must
    take the reference's keywords and the call must get through our check_shapes and stop exactly at the "CUDA devices only"
    check -- the recorded tensors live on the CPU and there is no CPU fallback by design."""
    import ml_gmpi_b200 as g
    z = np.load(os.path.join(GOLDEN, "reference_mpi_call.npz"))
    init_kw, call_kw = _decode_kwargs(z, "init/"), _decode_kwargs(z, "call/")
    assert list(call_kw) == ["batch_rgba", "batch_dhw", "batch_ray_dir", "batch_eye_pos", "batch_z_dir", "separate_background",
                             "assert_not_out_of_last_plane", "c2w_mat", "sphere_c"]
    mpi = g.MPI(**init_kw)
    assert mpi._align_corners is True
    assert call_kw["batch_rgba"].shape == (2, 4, 4, 16, 16) and len(call_kw["batch_ray_dir"]) == 2
    with pytest.raises(RuntimeError, match="CUDA devices only"):
        mpi(**call_kw)
    # a malformed MPI is rejected by OUR check_shapes with the reference's message before any device work
    with pytest.raises(AssertionError, match="Expected rgba to be of shape"):
        mpi(batch_rgba=torch.rand(2, 4, 3, 16, 16), batch_dhw=torch.rand(2, 4, 3), batch_ray_dir=[torch.rand(1, 3, 8, 8)] * 2,
            batch_eye_pos=[torch.rand(1, 3)] * 2, batch_z_dir=[torch.rand(1, 3)] * 2, separate_background=None)
