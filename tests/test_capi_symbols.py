"""CPU: the C-ABI shared library loads and exports every symbol include/nngp_b200.h declares.
No compute call is made (there is no GPU here); nngp_create must fail loudly, not fall back."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "nngp_b200.h"


def declared_functions():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(nngp_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from nngp_b200 import _lib
    return _lib


def test_header_and_binding_agree(lib):
    funcs = declared_functions()
    assert len(funcs) >= 15
    assert sorted(lib.EXPORTS) == funcs


def test_library_exports_every_declared_symbol(lib):
    cdll = ctypes.CDLL(str(lib.LIB_PATH))
    for name in declared_functions():
        assert hasattr(cdll, name), f"{name} declared in include/nngp_b200.h but not exported"
    assert cdll.nngp_abi_version() == 7
    cdll.nngp_build_id.restype = ctypes.c_char_p
    from nngp_b200 import _build
    assert cdll.nngp_build_id().decode() == _build.source_hash() == lib.built_id()


def test_build_id_tracks_every_source_file(lib):
    """The staleness check is by content and covers the C++ encoder and the header too (an mtime / *.cu-only check
    would ship a stale binary for those)."""
    from nngp_b200 import _build
    names = {f.name for f in _build.source_files()}
    assert {"capi.cu", "encoder.cc", "gemm_nt.cuh", "nngp_b200.h", "build.sh"} <= names


def test_struct_layouts_match_header(lib):
    # nngp_config: int32, 3 doubles, 2 int32, int64, 2 int32 (56 bytes) + n_gpus, device_ids[8], latency_mode
    # ... + per_layer (int32, padded to 8) + sigma_w_layers[16] + sigma_b_layers[16]
    # ... + variance_slices, reserved0 (int32 each)
    assert ctypes.sizeof(lib.NngpConfig) == 104 + 2 * 16 * 8 + 8
    assert lib.NngpConfig.variance_slices.offset == 360
    assert lib.NngpConfig.n_gpus.offset == 56 and lib.NngpConfig.device_ids.offset == 60
    assert lib.NngpConfig.latency_mode.offset == 92 and lib.NngpConfig.per_layer.offset == 96
    assert lib.NngpConfig.sigma_w_layers.offset == 104 and lib.NngpConfig.sigma_b_layers.offset == 232
    assert ctypes.sizeof(lib.NngpStats) == 8 * 28
    assert lib.NngpStats.device_allocs.offset == 8 * 27            # ABI 7 appended it; earlier fields keep their offsets


def test_no_cpu_fallback_without_gpu(lib):
    """Creating a handle where no GPU is visible (CUDA_VISIBLE_DEVICES empty, in a child process) fails loudly."""
    import os
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from nngp_b200 import _lib\n"
            "try:\n    _lib.Handle()\nexcept Exception as e:\n    print('RAISED', e)\n") % str(ROOT / "nngp-src_b200")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.startswith("RAISED "), r.stdout
    msg = r.stdout[len("RAISED "):]
    assert "no CUDA device" in msg or "error" in msg.lower()


def test_no_kernel_uses_local_memory(lib):
    """Every kernel must be spill-free (STACK:0, LOCAL:0) and the DMMA kernels must fit 2 CTAs per SM."""
    import shutil
    import subprocess
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([tool, "--dump-resource-usage", str(lib.LIB_PATH)], capture_output=True, text=True).stdout
    funcs = re.findall(r"Function (\S+):\s*\n?\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    assert len(funcs) >= 15, out[:400]
    bad = [(f, st, lo) for f, _r, st, lo in funcs if int(st) or int(lo)]
    assert not bad, f"kernels using local memory: {bad}"
    regs = {f: int(r) for f, r, _s, _l in funcs}
    for f, r in regs.items():
        if "gemm_nt_kernel" in f or "trsm_fused_kernel" in f:
            assert r <= 128, (f, r)        # 2 CTAs x 256 threads x 128 registers = one SM's register file


def test_stage_release_carries_a_dependence_on_the_fragment_loads(lib):
    """Regression guard for the ring-stage release hazard (DESIGN.md 5.3): in every kernel built on mma_mainloop the
    consumer's mbarrier arrive (SASS ``SYNCS.ARRIVE.TRANS64.A1T0``) must take its address from an add whose input is
    ``seen & zero`` (a ``LOP3.LUT ... 0xc0``) -- i.e. the arrive cannot issue before the fragment LDS results have
    landed.  If a compiler or a refactor folds that away, the arrive is again free to overtake the loads."""
    import shutil
    import subprocess
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([tool, "-sass", str(lib.LIB_PATH)], capture_output=True, text=True).stdout
    # (sliced_gemm_kernel is not built on mma_mainloop: its operands are read by the tensor core itself, and the
    # stage release is a tcgen05.commit, ordered by the hardware)
    sass = "".join(part for part in re.split(r"(?=\n\s*Function : )", sass) if "sliced_gemm_kernel" not in part.split("\n", 2)[1])
    instrs = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+(.*?);", sass)]
    arrives = [i for i, t in enumerate(instrs) if "SYNCS.ARRIVE.TRANS64.A1T0" in t]
    nvcc = subprocess.run(["/usr/local/cuda/bin/nvcc", "--version"], capture_output=True, text=True).stdout.strip().splitlines()
    where = f" [compiler: {nvcc[-2] if len(nvcc) > 1 else nvcc}; the guard is tied to this ptxas' code generation]"
    assert len(arrives) >= 10, "expected the consumer releases of gemm_nt_kernel<0..3> and trsm_fused_kernel" + where
    for i in arrives:
        reg = re.search(r"\[(R\d+)\+", instrs[i]).group(1)
        add = next((j for j in range(i - 1, max(i - 16, 0), -1)
                    if re.search(r"IADD\w*(\.\w+)* %s," % reg, instrs[j])), None)
        assert add is not None, f"arrive address {reg} is not computed by an add: {instrs[max(i - 4, 0):i + 1]}" + where
        srcs = set(re.findall(r"R\d+", instrs[add].split(",", 1)[1]))
        masked = [j for j in range(add - 1, max(add - 60, 0), -1)
                  if "LOP3.LUT" in instrs[j] and "0xc0" in instrs[j]
                  and (re.search(r"LOP3\.LUT (?:P\d+, )?(R\d+|RZ),", instrs[j]) or [None, None])[1] in srcs]
        assert masked, f"no `seen & zero` feeding the arrive address: {instrs[max(add - 6, 0):i + 1]}" + where
