"""CPU: the drop-in boundary -- state_dict layout, registry, C-ABI symbol table, loud failure without CUDA."""
import ctypes
import os
import re

import pytest
import torch

import savsr_b200
from oracle.state_dict_fixture import make_state_dict, state_dict_spec
from savsr_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
YAML_KWARGS = dict(num_in_ch=3, num_feat=64, num_frame=7, slid_win=3, fusion_win=5, interval=0, w1_num_block=4, w2_num_block=2,
                   n_resgroups=4, n_resblocks=8, center_frame_idx=None)     # options/test/SAVSR/test_SAVSR_Vid4_asBI.yml:830-842


@pytest.fixture(scope="module")
def net():
    return savsr_b200.build_network(dict(type="SAVSR", **YAML_KWARGS))


def test_registry_and_constructor(net):
    assert "SAVSR" in savsr_b200.ARCH_REGISTRY
    assert type(net).__name__ == "SAVSR" and net.scale == (4, 4)
    with pytest.raises(KeyError):
        savsr_b200.ARCH_REGISTRY.get("NoSuchArch")
    with pytest.raises(NotImplementedError):
        savsr_b200.SAVSR(interval=1)


def test_state_dict_layout_matches_reference(net):
    spec = state_dict_spec()                 # pinned to the reference by scripts/make_golden.py (strict load + key order)
    sd = net.state_dict()
    assert list(sd) == [k for k, _, _ in spec] and len(sd) == 791
    for k, shape, _ in spec:
        assert tuple(sd[k].shape) == tuple(shape), k
    assert sum(p.numel() for p in net.parameters()) == 18890044
    net.load_state_dict(make_state_dict(1), strict=True)
    assert "SAVSR(" in str(net)


def test_set_scale_and_hw(net):
    net.set_scale((1.5, 4))
    assert net.scale == (1.5, 4)
    assert savsr_b200.get_HW(33, 35, (1.5, 1.5)) == (50, 52)      # python round: half to even
    assert savsr_b200.get_HW(144, 180, 4) == (576, 720)


def test_no_cpu_fallback(net):
    net.eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(torch.zeros(1, 7, 3, 8, 8))
    with pytest.raises(ValueError):
        net.plan_for(torch.zeros(1, 5, 3, 8, 8))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "savsr_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(savsr_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = _capi.load()                        # raises if the .so is missing or lacks a bound symbol
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/savsr_b200.h but not exported"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    assert lib.savsr_abi_version() == _capi.ABI_VERSION == 4


def test_struct_layouts_match_header():
    assert ctypes.sizeof(_capi.ConvGroup) == 104 and _capi.ConvGroup.weight.offset == 48 and _capi.ConvGroup.src_channels.offset == 96
    assert _capi.OsaParams.pool.offset == 16 + 16 * 8 and ctypes.sizeof(_capi.SatuWeights) == 96
    # training entry points (train_ops.cu / train_attn.cu carry the matching static_asserts on the C side)
    assert ctypes.sizeof(_capi.Axpby) == 20 and ctypes.sizeof(_capi.Nchw3) == 8
    assert ctypes.sizeof(_capi.GradPrep) == 72 and _capi.GradPrep.cscale.offset == 24 and _capi.GradPrep.dbias.offset == 64
    assert ctypes.sizeof(_capi.PackChunk) == 40 and ctypes.sizeof(_capi.WgradItem) == 48 and _capi.WgradItem.sample_stride.offset == 40
    assert ctypes.sizeof(_capi.MaskTrain) == 456 and _capi.MaskTrain.gamma.offset == 176 and _capi.MaskTrain.dmask.offset == 400
    assert ctypes.sizeof(_capi.OsaTrain) == 56 and _capi.OsaTrain.state.offset == 40 and ctypes.sizeof(_capi.OsaGrads) == 160


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU error path")
def test_context_creation_fails_loudly_without_gpu():
    with pytest.raises(_capi.SavsrError):
        _capi.Context(0)
    lib = _capi.load()
    assert lib.savsr_arena_bytes(2, 3, 10, 12) == 2 * 3 * 10 * 12 * 64 * 2
    assert lib.savsr_packed_weight_bytes(64, 192, 3) == 64 * 192 * 9 * 2
    assert lib.savsr_ctx_sm_count(None) == 0


# A pristine checkout of the reference, reduced to what the overlay has to get past: lbasicsr/__init__.py imports the generated
# version.py (absent before setup.py runs) and the archs; lbasicsr/archs/__init__.py imports every *_arch.py beside it by module name;
# the registry asserts that a name is registered once.  The reference's own savsr_arch.py must never be the one that loads.
REFERENCE_STAND_IN = {
    "lbasicsr/__init__.py": "from .archs import *  # noqa: F401,F403\nfrom .version import __gitsha__, __version__  # noqa: F401\n",
    "lbasicsr/utils/__init__.py": "",
    "lbasicsr/utils/registry.py": (
        "class Registry:\n"
        "    def __init__(self, name):\n"
        "        self._name, self._obj_map = name, {}\n"
        "    def _do_register(self, name, obj):\n"
        "        assert name not in self._obj_map, f\"An object named '{name}' was already registered in '{self._name}' registry!\"\n"
        "        self._obj_map[name] = obj\n"
        "    def register(self, obj=None):\n"
        "        if obj is None:\n"
        "            def deco(func_or_class):\n"
        "                self._do_register(func_or_class.__name__, func_or_class)\n"
        "                return func_or_class\n"
        "            return deco\n"
        "        self._do_register(obj.__name__, obj)\n"
        "    def get(self, name):\n"
        "        ret = self._obj_map.get(name)\n"
        "        if ret is None:\n"
        "            raise KeyError(f\"No object named '{name}' found in '{self._name}' registry!\")\n"
        "        return ret\n"
        "ARCH_REGISTRY = Registry('arch')\n"),
    "lbasicsr/archs/__init__.py": (
        "import importlib\n"
        "from copy import deepcopy\n"
        "from os import listdir, path as osp\n"
        "from lbasicsr.utils.registry import ARCH_REGISTRY\n"
        "__all__ = ['build_network']\n"
        "arch_folder = osp.dirname(osp.abspath(__file__))\n"
        "arch_filenames = sorted(osp.splitext(v)[0] for v in listdir(arch_folder) if v.endswith('_arch.py'))\n"
        "_arch_modules = [importlib.import_module(f'lbasicsr.archs.{file_name}') for file_name in arch_filenames]\n"
        "def build_network(opt):\n"
        "    opt = deepcopy(opt)\n"
        "    return ARCH_REGISTRY.get(opt.pop('type'))(**opt)\n"),
    "lbasicsr/archs/savsr_arch.py": "raise ImportError('the reference savsr_arch.py was imported instead of the overlay')\n",
    "lbasicsr/archs/edvr_arch.py": (
        "from lbasicsr.utils.registry import ARCH_REGISTRY\n"
        "@ARCH_REGISTRY.register()\n"
        "class EDVR:\n"
        "    pass\n"),
}


def test_overlay_serves_the_new_arch_to_the_reference_registry(tmp_path):
    import subprocess
    import sys
    ref = tmp_path / "reference"
    for rel, text in REFERENCE_STAND_IN.items():
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(text)
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from savsr_b200 import overlay; overlay.install(%r)\n"
            "import lbasicsr\n"
            "from lbasicsr.archs import build_network\n"
            "from lbasicsr.utils.registry import ARCH_REGISTRY\n"
            "net = build_network(dict(type='SAVSR', num_in_ch=3, num_feat=64, num_frame=7, slid_win=3, fusion_win=5, interval=0,"
            " w1_num_block=4, w2_num_block=2, n_resgroups=4, n_resblocks=8, center_frame_idx=None))\n"
            "import savsr_b200.engine\n"
            "assert type(net).__module__ == 'lbasicsr.archs.savsr_arch' and hasattr(net, 'plan_for'), type(net)\n"
            "assert ARCH_REGISTRY.get('EDVR').__module__ == 'lbasicsr.archs.edvr_arch'\n"
            "print('OVERLAY_OK', len(net.state_dict()))\n") % (ROOT, str(ref))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "OVERLAY_OK 791" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with the contract's keys, and
    --dump-outputs writes the output of its last timed window."""
    import json
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "cfg1_x2", "--steps", "1",
                          "--warmup", "0", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "hr_mpix_per_s" and line["unit"] == "HR Mpix/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["value"] == line["value"] and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "HR Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"] == "cfg1_x2"
    import bench
    assert line["config"] == bench.workload_config("cfg1_x2", 1)      # both arms print the same config object
    assert sorted(os.listdir(tmp_path)) == ["hr.npy"]
    y = np.load(tmp_path / "hr.npy")
    assert y.dtype == np.float32 and y.shape == (1, 3, 128, 128) and np.isfinite(y).all()


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: float32 .npy files within the 64 MB budget, a larger output cut to the same rows on every run, and a refusal
    when a single row does not fit."""
    import numpy as np
    import bench
    big = torch.arange(40 * 3 * 400 * 400, dtype=torch.float64).view(40, 3, 400, 400)      # 153.6 MB in float32
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), {"hr": big, "loss": torch.tensor([0.5])})
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["hr.npy", "loss.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= bench.DUMP_BYTES
    hr = np.load(tmp_path / "a" / "hr.npy")
    assert hr.dtype == np.float32 and hr.shape[1:] == (3, 400, 400) and 1 <= hr.shape[0] < 40
    rows = hr[:, 0, 0, 0].astype(np.int64) // (3 * 400 * 400)
    assert np.all(np.diff(rows) > 0) and np.array_equal(hr, big[torch.from_numpy(rows)].float().numpy())
    assert np.array_equal(hr, np.load(tmp_path / "b" / "hr.npy"))
    assert np.load(tmp_path / "a" / "loss.npy").tolist() == [0.5]
    with pytest.raises(ValueError, match="larger than"):
        bench.write_outputs(str(tmp_path / "c"), {"hr": torch.zeros(2, 3, 3000, 3000)})       # one row = 108 MB


def test_bench_our_arm_needs_a_gpu():
    """No CPU fallback: without CUDA our arm exits with an error instead of measuring something else."""
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
