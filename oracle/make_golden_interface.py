"""Golden fixtures for the drop-in boundary, produced by the UNMODIFIED reference on CPU:

    GMPI_REFERENCE_ROOT=<ml-gmpi checkout> python oracle/make_golden_interface.py

writes
  tests/golden/reference_signatures.json  every parameter (name, kind, default) of MPI.__init__ / forward / check_shapes and
                                          of every function of MPIRenderer
  tests/golden/reference_mpi_call.npz     the keyword arguments MPIRenderer constructs MPI with (mpi_renderer.py:47) and
                                          calls it with inside `render` (mpi_renderer.py:451-461), recorded by a stand-in MPI

The stand-in only observes: the reference's pose sampling and ray generation run unchanged.  The tests replay the recorded
construction and call against ml_gmpi_b200.MPI, so they need neither the reference nor a GPU.

TEST INFRASTRUCTURE ONLY.
"""
import inspect
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def signature_rows(fn):
    """[(name, kind, repr(default))] without self: the form tests/test_interface_matches_reference.py compares."""
    return [[n, p.kind.name, repr(p.default)] for n, p in inspect.signature(fn).parameters.items() if n != "self"]


def encode_kwargs(prefix, kw, out):
    """Keyword arguments -> npz entries: `<prefix>order` (names in call order), `<prefix>t/<name>` tensors,
    `<prefix>a/<name>` numpy arrays, `<prefix>l/<name>/<i>` lists of tensors, `<prefix>none/<name>` None,
    `<prefix>s/<name>` Python scalars."""
    out[prefix + "order"] = np.array(list(kw))
    for k, v in kw.items():
        if v is None:
            out[f"{prefix}none/{k}"] = np.zeros(0)
        elif isinstance(v, torch.Tensor):
            out[f"{prefix}t/{k}"] = v.detach().cpu().numpy()
        elif isinstance(v, np.ndarray):
            out[f"{prefix}a/{k}"] = v
        elif isinstance(v, (list, tuple)):
            assert all(isinstance(x, torch.Tensor) for x in v), k
            for i, x in enumerate(v):
                out[f"{prefix}l/{k}/{i}"] = x.detach().cpu().numpy()
        else:
            assert isinstance(v, (bool, int, float)), (k, type(v))
            out[f"{prefix}s/{k}"] = np.array(v)


def main():
    ref_mpi, ref_r = ref_shim.import_reference()
    sigs = {"MPI": {name: signature_rows(getattr(ref_mpi.MPI, name)) for name in ("__init__", "forward", "check_shapes")},
            "MPIRenderer": {name: signature_rows(fn) for name, fn in inspect.getmembers(ref_r.MPIRenderer, inspect.isfunction)}}

    rec = {}

    class RecordingMPI:
        def __init__(self, *args, **kw):
            assert not args
            rec["init"] = kw

        def __call__(self, *args, **kw):
            assert not args
            rec["call"] = kw
            n = len(kw["batch_ray_dir"])
            h, w = kw["batch_ray_dir"][0].shape[-2:]
            return torch.zeros(n, 3, h, w), torch.zeros(n, 1, h, w)

    old = ref_r.MPI
    ref_r.MPI = RecordingMPI
    try:
        r = ref_r.MPIRenderer(n_mpi_planes=4, device=torch.device("cpu"), **ref_shim.FFHQ_KWARGS)
        torch.manual_seed(0)
        rgba = torch.rand(2, 4, 4, 16, 16)
        r.render(rgba, 16, 16, given_yaws=torch.zeros(2, 1), given_pitches=torch.zeros(2, 1))
    finally:
        ref_r.MPI = old

    arrays = {}
    encode_kwargs("init/", rec["init"], arrays)
    encode_kwargs("call/", rec["call"], arrays)
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "reference_signatures.json"), "w") as f:
        json.dump(sigs, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(OUT, "reference_mpi_call.npz"), **arrays)
    print("wrote reference_signatures.json", {k: len(v) for k, v in sigs.items()}, "and reference_mpi_call.npz",
          list(rec["init"]), list(rec["call"]))


if __name__ == "__main__":
    main()
