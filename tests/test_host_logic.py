"""CPU-only checks of the host layer: the C-ABI library loads and exports every declared symbol,
weights ingestion (weight-norm fold) against torch's own, reference-surface behaviour of the
Python mirror, voxel grid quirk, synthetic generator determinism.  No compute calls (no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_library_exports_every_declared_symbol():
    from dsp_slam_b200 import _lib
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "dspgn.h")).read()
    declared = set(re.findall(r"\b(dspgn_[a-z_0-9]+)\s*\(", hdr))
    bound = {n for n, _, _ in _lib.SYMBOLS}
    assert declared == bound, declared ^ bound
    for n in declared:
        assert hasattr(lib, n)
    assert lib.dspgn_version() >= 100
    assert C.sizeof(_lib.ObjectOut) == 4 * _lib.RESULT_FLOATS


def test_no_cpu_fallback_without_gpu(golden_dir):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from dsp_slam_b200._lib import DspgnError
    from dsp_slam_b200.decoder import DecoderWeights, DeviceDecoder
    w = DecoderWeights.from_npz(os.path.join(golden_dir, "decoder_cars.npz"))
    with pytest.raises(DspgnError):
        DeviceDecoder(w, 0)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "dsp_slam_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("oracle/", "").replace("the oracle", "") or f == "synth.py", f


def test_weight_fold_matches_torch(golden_dir, stages):
    from dsp_slam_b200.decoder import DecoderWeights
    w = DecoderWeights.from_npz(os.path.join(golden_dir, "decoder_cars.npz"))
    assert w.latent_in_layer == 4 and w.latent_size == 64 and len(w.W) == 9
    for k in range(9):
        np.testing.assert_allclose(w.W[k], stages[f"cars_W{k}"], rtol=0, atol=2e-7)


def test_weights_from_live_module(golden_dir, stages):
    """from_module on an nn.Module with torch weight_norm hooks (what get_decoder returns)."""
    import json
    import torch
    import torch.nn as nn
    from dsp_slam_b200.decoder import DecoderWeights
    d = np.load(os.path.join(golden_dir, "decoder_cars.npz"))

    class Dec(nn.Module):          # structural stand-in with the attributes from_module reads
        def __init__(self):
            super().__init__()
            self.latent_in = [4]; self.xyz_in_all = False; self.use_tanh = False
            self.latent_dropout = False; self.weight_norm = True; self.norm_layers = list(range(8))
            dims = [67, 256, 256, 256, 189, 256, 256, 256, 256, 1]
            ins = [67, 256, 256, 256, 256, 256, 256, 256, 256]
            for k in range(9):
                lin = nn.Linear(ins[k], dims[k + 1])
                setattr(self, f"lin{k}", nn.utils.weight_norm(lin) if k < 8 else lin)
    m = Dec()
    m.load_state_dict({k: torch.from_numpy(d[k]) for k in d.files if k != "spec_json"})
    w = DecoderWeights.from_module(m.eval())
    for k in range(9):
        np.testing.assert_allclose(w.W[k], stages[f"cars_W{k}"], rtol=0, atol=2e-7)


def test_decoder_variants_are_ingested(golden_dir):
    """LayerNorm / xyz_in_all / use_tanh / several latent_in layers (deep_sdf_decoder.py:41-63,87-102) no longer raise
    at construction (inside LocalMapping's constructor that would kill the process, src/LocalMapping.cc:38-40): they
    are recorded in the decoder spec and routed to the fp32 SIMT engine; structural nonsense still raises."""
    from dsp_slam_b200.decoder import DecoderWeights
    w = DecoderWeights.from_npz(os.path.join(golden_dir, "decoder_variant.npz"))
    assert w.cat_kind == [0, 2, 1, 2, 1, 2] and w.use_tanh and not w.is_plain
    assert [x is not None for x in w.ln] == [True] * 5 + [False]
    assert w.ln[0][0].shape == (125,) and w.latent_in_layer == -1
    plain = DecoderWeights.from_npz(os.path.join(golden_dir, "decoder_cars.npz"))
    assert plain.is_plain and plain.cat_kind == [0, 0, 0, 0, 1, 0, 0, 0, 0]
    d = np.load(os.path.join(golden_dir, "decoder_cars.npz"))
    sd = {k: d[k] for k in d.files if k != "spec_json"}
    with pytest.raises(ValueError):                            # xyz_in_all on weights that were not built for it
        DecoderWeights.from_state_dict(sd, 64, latent_in=(4,), xyz_in_all=True)


def test_result_container_semantics():
    from dsp_slam_b200.optimizer import ResultDict
    r = ResultDict(t_cam_obj=None, code=None, is_good=False, loss=0.0)
    assert r.is_good is False and r["loss"] == 0.0
    with pytest.raises(KeyError):
        r.missing_key


def test_config_keys_read_like_the_reference(cfg_kitti):
    """Optimizer.__init__ must raise KeyError for a missing hyper-parameter (ForceKeyErrorDict
    behaviour, reconstruct/utils.py:82-84) before touching the GPU."""
    import copy
    from dsp_slam_b200.optimizer import Optimizer
    bad = copy.deepcopy(cfg_kitti)
    del bad["optimizer"]["joint_optim"]["k3"]
    with pytest.raises(KeyError):
        Optimizer(object(), bad)


def test_voxel_grid_quirk_matches_reference(golden_dir):
    """create_voxel_grid's integer-tensor true division (reconstruct/utils.py:107-108) reproduced."""
    from dsp_slam_b200.optimizer import create_voxel_grid
    v = np.load(os.path.join(golden_dir, "voxel.npz"))
    np.testing.assert_allclose(create_voxel_grid(8), v["vox8"], rtol=0, atol=1e-6)


def test_synth_is_deterministic_and_fortran_ordered():
    from dsp_slam_b200 import synth
    a = synth.make_object(3, 100, 50, 10)
    b = synth.make_object(3, 100, 50, 10)
    for k in ("pts", "rays", "depth", "t_cam_obj_init"):
        np.testing.assert_array_equal(a[k], b[k])
        assert a[k].dtype == np.float32
    assert a["pts"].flags.f_contiguous and a["rays"].shape == (60, 3) and a["depth"].shape == (50,)


def test_c_abi_rejects_bad_arguments_before_touching_cuda():
    """Argument validation of the C ABI returns DSPGN_E_ARG (-1) without needing a GPU."""
    import ctypes as C
    from dsp_slam_b200 import _lib
    lib = _lib.load()
    FP = C.POINTER(C.c_float)
    h = C.c_void_p()
    # null pointers
    assert lib.dspgn_decoder_create(None, None, None, 0, C.byref(h)) == -1
    assert b"null" in lib.dspgn_last_error()
    # inconsistent decoder shapes
    spec = _lib.DecoderSpec()
    spec.latent_size = 64; spec.num_linear = 3; spec.latent_in_layer = -1
    for k, (i, o) in enumerate([(67, 256), (200, 256), (256, 1)]):      # layer 1 in_dim != layer 0 out_dim
        spec.in_dim[k], spec.out_dim[k] = i, o
    W = [np.zeros((o, i), np.float32) for i, o in [(67, 256), (200, 256), (256, 1)]]
    b = [np.zeros(o, np.float32) for o in (256, 256, 1)]
    Wp = (FP * 3)(*[w.ctypes.data_as(FP) for w in W]); bp = (FP * 3)(*[x.ctypes.data_as(FP) for x in b])
    assert lib.dspgn_decoder_create(C.byref(spec), Wp, bp, 0, C.byref(h)) == -1
    assert b"in_dim" in lib.dspgn_last_error()
    spec.in_dim[1] = 256
    spec.out_dim[2] = 2                                                    # last layer must have one output
    assert lib.dspgn_decoder_create(C.byref(spec), Wp, bp, 0, C.byref(h)) == -1
    spec.out_dim[2] = 1
    spec.latent_size = 65                                                  # > DSPGN_MAX_CODE
    assert lib.dspgn_decoder_create(C.byref(spec), Wp, bp, 0, C.byref(h)) == -1
    # solver / run entry points with null handles
    assert lib.dspgn_run_batch(None, 0) == -1
    assert lib.dspgn_upload_batch(None, 1, None) == -1
    assert lib.dspgn_results(None, None) == -1
    assert lib.dspgn_solver_engine(None) == -1
    D = np.zeros((128, 16), np.float32)
    assert lib.dspgn_tc_selftest(0, 17, 1, D.ctypes.data_as(FP), D.ctypes.data_as(FP), D.ctypes.data_as(FP)) == -1   # N % 16


def test_optimizer_rejects_wrong_shapes(golden_dir, cfg_kitti):
    """Misuse raises (ValueError) in the host layer; only per-object numerical failures are soft."""
    from dsp_slam_b200.optimizer import BatchSolver
    from dsp_slam_b200 import _lib
    bs = BatchSolver.__new__(BatchSolver)
    bs.cfg = _lib.Config(); bs.cfg.code_len = 64
    with pytest.raises(ValueError):
        bs._pack([dict(t_cam_obj=np.eye(3, dtype=np.float32), pts=np.zeros((5, 3), np.float32))])
    with pytest.raises(ValueError):
        bs._pack([dict(t_cam_obj=np.eye(4, dtype=np.float32), pts=np.zeros((5, 2), np.float32))])
    # a code shorter than code_len is zero-padded (optimizer.py:97-100 slices code[:code_len])
    arr, keep = bs._pack([dict(t_cam_obj=np.eye(4, dtype=np.float32), pts=np.zeros((5, 3), np.float32), code=np.ones(10, np.float32))])
    assert [arr[0].code[i] for i in (0, 9, 10, 63)] == [1.0, 1.0, 0.0, 0.0]
    # float64 / list inputs are converted, Fortran order is passed through without a copy
    P = np.asfortranarray(np.random.default_rng(0).standard_normal((7, 3)).astype(np.float32))
    arr, keep = bs._pack([dict(t_cam_obj=np.eye(4).tolist(), pts=P)])
    assert arr[0].n_pts == 7 and arr[0].pts_rs == 1 and arr[0].pts_cs == 7 and arr[0].t_rs == 4 and arr[0].t_cs == 1
    assert arr[0].pts[arr[0].pts_cs * 2 + 3] == P[3, 2]


def test_reference_surface_never_raises(cfg_kitti):
    """The three entry points C++ calls through pybind11 have no handler above them
    (src/LocalMapping_util.cc:109-110,179-196): whatever goes wrong inside must come back as the reference's
    soft failure.  Exercised here without a GPU by breaking the solver underneath."""
    from dsp_slam_b200.optimizer import Optimizer, MeshExtractor

    class Boom:
        cfg = None

        def __getattr__(self, k):
            raise RuntimeError("no GPU here")

    opt = Optimizer.__new__(Optimizer)
    opt.code_len = 64
    opt.solver = Boom()
    r = opt.reconstruct_object(np.eye(4, dtype=np.float32), np.zeros((5, 3), np.float32), np.zeros((3, 3), np.float32), np.zeros(2, np.float32))
    assert r.is_good is False and r.t_cam_obj is None and r.code is None and r.loss == 0.0
    r = opt.reconstruct_object("garbage", None, None, None)
    assert r.is_good is False
    T = np.eye(4, dtype=np.float32); T[0, 3] = 2.0
    out = opt.estimate_pose_cam_obj(T, 1.7, np.zeros((5, 3), np.float32), np.zeros(64, np.float32))
    np.testing.assert_array_equal(out, T)                       # failed optimisation: input pose kept
    assert opt.estimate_pose_cam_obj("garbage", 1.0, None, None).shape == (4, 4)
    mx = MeshExtractor.__new__(MeshExtractor)
    mx.code_len, mx.voxels_dim, mx.solver, mx.voxel_points = 64, 8, Boom(), np.zeros((512, 3), np.float32)
    m = mx.extract_mesh_from_code(np.zeros(64, np.float32))
    assert m.vertices.shape == (0, 3) and m.faces.shape == (0, 3) and m.faces.dtype == np.int32


class _StrictConfig(dict):
    """Stand-in for the config object DSP-SLAM's reconstruct.utils.get_configs returns: the JSON tree with
    attribute access at every level, where a missing key raises KeyError (read as an item or as an attribute)."""

    def __init__(self, tree):
        super().__init__((k, _StrictConfig(v) if isinstance(v, dict) else v) for k, v in tree.items())

    def __getattr__(self, key):
        return self[key]


def test_drop_in_shim_module_next_to_the_reference_package(golden_dir):
    """integration/reconstruct/optimizer.py is the one-file replacement of the reference's
    reconstruct/optimizer.py: imported the way src/LocalMapping.cc:38 does (`reconstruct.optimizer`), it must expose
    Optimizer / MeshExtractor and read the reference's whole configs/config_kitti.json (stored verbatim as
    tests/golden/config_kitti_reference.json) through a config object that behaves like get_configs' result."""
    import importlib.util
    import json
    shim = os.path.join(ROOT, "integration", "reconstruct", "optimizer.py")
    assert os.path.isfile(shim)
    spec = importlib.util.spec_from_file_location("reconstruct_optimizer_shim", shim)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    from dsp_slam_b200 import optimizer as ours
    assert mod.Optimizer is ours.Optimizer and mod.MeshExtractor is ours.MeshExtractor
    with open(os.path.join(golden_dir, "config_kitti_reference.json")) as f:
        tree = json.load(f)
    cfg = _StrictConfig(tree)
    assert cfg.optimizer.joint_optim.k4 == 1e7 and cfg.data_type == "KITTI"
    with pytest.raises(KeyError):
        cfg.optimizer.missing_key
    # constructor reads the keys exactly like reconstruct/optimizer.py:27-43 before touching the GPU ...
    with pytest.raises(Exception) as ei:
        mod.Optimizer(object(), cfg)
    assert "cannot build decoder weights" in str(ei.value) or "libdspgn" in str(ei.value) or "CUDA" in str(ei.value)
    # ... and a missing key is the reference's KeyError
    bad = _StrictConfig(tree)
    del bad["optimizer"]["joint_optim"]["k3"]
    with pytest.raises(KeyError):
        mod.Optimizer(object(), bad)


def test_native_packer_equals_python_packer():
    """csrc/fastpack.c (CPython extension) fills the DspgnObjectIn records for plain float32 numpy inputs; anything else
    falls back to the Python path.  Both must produce byte-identical records."""
    import ctypes as C
    from dsp_slam_b200 import optimizer as O, synth, _lib
    if O._fastpack_mod() is None:
        pytest.skip("_fastpack extension not built")
    bs = O.BatchSolver.__new__(O.BatchSolver)
    bs.cfg = _lib.Config(); bs.cfg.code_len = 64
    objs = synth.make_batch(5, 300, 120, 40, cls=["cars", "chairs", "cars", "chairs", "cars"], init_code_frac=0.5)
    ins = []
    for i, o in enumerate(objs):
        d = dict(t_cam_obj=o["t_cam_obj_init"], pts=o["pts"], rays=o["rays"], depth=o["depth"], code=o["code_init"], class_id=i & 1)
        ins.append(d)
    ins[1] = dict(ins[1], pts=np.ascontiguousarray(ins[1]["pts"]), scale=1.7)                 # C-ordered, with a scale
    ins[2] = dict(t_cam_obj=ins[2]["t_cam_obj"], pts=ins[2]["pts"])                            # no rays, no code
    ins[3] = dict(t_cam_obj=ins[3]["t_cam_obj"], pts=ins[3]["pts"], pixels=np.asfortranarray(np.random.default_rng(0).random((50, 2), np.float32)),
                  inv_k=np.eye(3, dtype=np.float32), depth=np.zeros(10, np.float32), t_cam_world=np.eye(4, dtype=np.float32))

    def records(use_native):
        O._fastpack = False if use_native else None
        arr, keep = bs._pack(ins)
        return [bytes(C.string_at(C.addressof(arr[i]), C.sizeof(_lib.ObjectIn))) for i in range(len(ins))], keep
    try:
        fast, keep_f = records(True)
        slow, keep_s = records(False)
    finally:
        O._fastpack = False
    assert len(keep_f) == 2 and keep_f[1] is ins               # the native path keeps the record array and the caller's list
    assert fast == slow
    # float64 / list inputs: the native path declines, the Python path converts
    mixed = [dict(t_cam_obj=np.eye(4).tolist(), pts=np.zeros((5, 3)))]
    arr, keep = bs._pack(mixed)
    assert arr[0].n_pts == 5 and isinstance(keep[0], tuple) and keep[0][1].dtype == np.float32    # converted copies are kept alive


def test_shipped_library_is_tcgen05_code_for_sm_100a_only():
    """The product path is hand-written tcgen05 / TMEM code for sm_100a (no mma.sync / wgmma recompiles, no second
    architecture): disassemble the built library (cuobjdump, no GPU needed) and look for the opcodes that prove it
    (B200_PROFILING.md: tcgen05.mma -> UTCHMMA, tcgen05.ld/st -> LDTM/STTM, cp.async.bulk -> UBLKCP) in every kernel
    that runs decoder tiles; profiles/sass_summary.txt is the same listing per kernel."""
    import re
    import shutil
    import subprocess
    from dsp_slam_b200 import _lib
    if shutil.which("cuobjdump") is None or not os.path.isfile(_lib.LIB_PATH):
        pytest.skip("cuobjdump or the built library is not available")
    out = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    assert set(re.findall(r"arch = (sm_\w+)", out)) == {"sm_100a"}
    per_kernel, kern = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            kern = m.group(1)
            per_kernel[kern] = set()
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and kern:
            per_kernel[kern].add(m.group(1))
    tiles = [k for k in per_kernel if any(n in k for n in ("k_gn_persistent", "k_decoder_tc"))]
    assert len(tiles) == 3, sorted(per_kernel)
    for k in tiles:
        ops = per_kernel[k]
        assert {"UTCHMMA", "LDTM", "STTM", "UTCBAR", "UBLKCP"} <= ops, (k, sorted(ops)[:40])
    everything = set().union(*per_kernel.values())
    assert not any(op.startswith(("HMMA", "HGMMA", "IMMA")) for op in everything)     # no legacy tensor-core paths anywhere


def test_ctypes_mirror_has_the_layout_of_the_c_header(tmp_path):
    """The hand-written ctypes structures of dsp_slam_b200/_lib.py against include/dspgn.h as the C compiler lays it
    out: a generated C program prints sizeof / offsetof of every field, gcc compiles it against the real header."""
    import shutil
    import subprocess
    from dsp_slam_b200 import _lib
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    pairs = [("DspgnDecoderSpec", _lib.DecoderSpec), ("DspgnConfig", _lib.Config), ("DspgnObjectIn", _lib.ObjectIn),
             ("DspgnObjectOut", _lib.ObjectOut), ("DspgnCounters", _lib.Counters), ("DspgnIpcHandle", _lib.IpcHandle)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dspgn.h"', 'int main(void) {']
    for cname, st in pairs:
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in st._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  printf("MAX_CODE %d MAX_LINEAR %d RESULT_FLOATS %d IPC %d\\n", DSPGN_MAX_CODE, DSPGN_MAX_LINEAR, '
              'DSPGN_RESULT_FLOATS, DSPGN_IPC_HANDLE_BYTES);', '  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([cc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.rsplit(" ", 1) for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True)
               .stdout.splitlines() if not line.startswith("MAX_CODE"))
    for cname, st in pairs:
        assert int(got[cname]) == C.sizeof(st), cname
        for fname, _ in st._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(st, fname).offset, (cname, fname)
    consts = subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines()[-1].split()
    assert [int(consts[i]) for i in (1, 3, 5, 7)] == [_lib.MAX_CODE, _lib.MAX_LINEAR, _lib.RESULT_FLOATS, _lib.IPC_HANDLE_BYTES]
