"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU, exports every
symbol include/*.h declares, the numpy/ctypes mirrors have the C sizes, and the product path
fails loudly (no CPU fallback) when no CUDA device is present."""
import ctypes as C
import os
import re

import pytest

import gigapaxos_b200
from gigapaxos_b200 import abi
from helpers import ROOT


def declared_functions():
    names = set()
    for h in ("gpx.h", "gpx_wire.h"):
        p = os.path.join(ROOT, "include", h)
        if not os.path.exists(p):
            continue
        src = open(p).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        for m in re.finditer(r"\b(gpx_[a-z0-9_]+)\s*\(", src):
            names.add(m.group(1))
    return sorted(names)


def test_library_exports_every_declared_symbol(cuda_lib):
    fns = declared_functions()
    assert len(fns) >= 25
    missing = [f for f in fns if not hasattr(cuda_lib.lib, f)]
    assert not missing, f"libgpx.so lacks {missing}"


def test_oracle_mirrors_the_data_path_symbols(oracle_lib):
    for f in ("engine_create", "create_groups", "propose", "handle_accepts", "handle_accept_replies",
              "handle_decisions", "round", "log_read", "dump_rows", "load_rows", "patch", "get_counters"):
        assert oracle_lib.has(f)


def test_struct_sizes_match_header():
    src = open(os.path.join(ROOT, "include", "gpx.h")).read()
    assert "GPX_ABI_VERSION %d" % abi.GPX_ABI_VERSION in src
    assert abi.request_dtype.itemsize == 32
    assert abi.accept_dtype.itemsize == 48
    assert abi.decision_dtype.itemsize == 32
    assert abi.reply_dtype.itemsize == 32
    assert abi.exec_dtype.itemsize == 24
    assert abi.seg_hdr_dtype.itemsize == 64
    assert abi.patch_dtype.itemsize == 32
    # compile-time check of the C side
    code = r"""
    #include "gpx.h"
    #include <stdio.h>
    int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(gpx_request_rec), sizeof(gpx_accept_rec),
      sizeof(gpx_decision_rec), sizeof(gpx_accept_reply_rec), sizeof(gpx_exec_rec), sizeof(gpx_log_seg_hdr),
      sizeof(gpx_row), sizeof(gpx_group_desc), sizeof(gpx_patch_rec), sizeof(gpx_config), sizeof(gpx_counters),
      sizeof(gpx_exec_sum), sizeof(gpx_round_io), sizeof(gpx_request_packed));}
    """
    import subprocess
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(code)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "t"),
                               os.path.join(d, "t.c")])
        out = subprocess.check_output([os.path.join(d, "t")]).decode().split()
    sizes = [int(x) for x in out]
    assert sizes[:9] == [32, 48, 32, 32, 24, 64, abi.row_dtype.itemsize, abi.group_desc_dtype.itemsize, 32]
    assert sizes[9] == C.sizeof(abi.Config) and sizes[10] == C.sizeof(abi.Counters)
    assert sizes[11] == abi.exec_sum_dtype.itemsize == 8 and sizes[12] == C.sizeof(abi.RoundIO)
    assert sizes[13] == abi.request_packed_dtype.itemsize == 16


def test_config_defaults_match_reference_defaults(cuda_lib, oracle_lib):
    for lib in (cuda_lib, oracle_lib):
        c = lib.config_defaults()
        assert c.abi_version == abi.GPX_ABI_VERSION
        assert (c.batching_enabled, c.max_batch_size, c.checkpoint_interval) == (1, 2000, 400)  # PaxosConfig.java:309,403,410
        assert (c.gc_majority_executed, c.log_meta_decisions, c.journaling_enabled) == (1, 1, 1)  # :882,:588,:240
        assert c.cpi_noise == 0.0 and c.log_backpressure == 0  # :746
        assert c.max_batch_bytes == 4 * 1024 * 1024
        assert list(c.lane_node)[:3] == [100, 101, 102]  # TESTPaxosConfig.java:100


def test_properties_parser(cuda_lib, tmp_path):
    p = tmp_path / "gigapaxos.properties"
    p.write_text("# comment\nAPPLICATION=edu.umass.cs.gigapaxos.examples.noop.NoopPaxosApp\n"
                 "active.100=127.0.0.1:2000\nactive.101=127.0.0.1:2001\nactive.102=127.0.0.1:2002\n"
                 "MAX_BATCH_SIZE = 123\nCHECKPOINT_INTERVAL=50\nBATCHING_ENABLED=false\nUNKNOWN_KEY=7\n"
                 "CPI_NOISE=0.25\nLOG_META_DECISIONS=false\n")
    cfg = abi.Config()
    rc = cuda_lib.fn("config_from_properties")(str(p).encode(), C.byref(cfg))
    assert rc == 0
    assert cfg.max_batch_size == 123 and cfg.checkpoint_interval == 50 and cfg.batching_enabled == 0
    assert cfg.cpi_noise == 0.25 and cfg.log_meta_decisions == 0 and cfg.gc_majority_executed == 1
    buf = C.create_string_buffer(1024)
    assert cuda_lib.fn("properties_actives")(buf, C.c_size_t(1024)) == 0
    assert buf.value.decode().splitlines() == ["100=127.0.0.1:2000", "101=127.0.0.1:2001", "102=127.0.0.1:2002"]
    assert cuda_lib.fn("config_from_properties")(b"/nonexistent/x.properties", C.byref(cfg)) == abi.GPX_EIO
    # the reference's own loopback config (its tests/loopback_1_group/gigapaxos.properties, stored verbatim) parses
    ref = os.path.join(ROOT, "tests", "golden", "loopback_1_group.gigapaxos.properties")
    assert cuda_lib.fn("config_from_properties")(ref.encode(), C.byref(cfg)) == 0
    assert cuda_lib.fn("properties_actives")(buf, C.c_size_t(1024)) == 0
    assert buf.value.decode().splitlines() == ["100=127.0.0.1:2000", "101=127.0.0.1:2001", "102=127.0.0.1:2002"]


def test_java_helpers_in_product_library(cuda_lib):
    h = cuda_lib.fn("java_string_hash")
    h.restype = C.c_int32
    h.argtypes = [C.c_char_p, C.c_size_t]
    for s in ["", "paxos0", "NoopPaxosApp42"]:
        assert h(s.encode(), len(s)) == abi.java_string_hash(s)
    g = cuda_lib.fn("get_cpi")
    g.restype = C.c_int32
    g.argtypes = [C.c_int32, C.c_double, C.c_int32]
    assert g(400, 0.0, 123) == 400
    assert g(400, 0.1, 123) == int(400 * 0.9 + (123 % 400) * 2 * 0.1)


def test_no_cpu_fallback(cuda_lib):
    """Without a CUDA device the product refuses to run instead of silently using a CPU path."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    with pytest.raises(gigapaxos_b200.GpxError) as ei:
        gigapaxos_b200.create_engine()
    assert ei.value.code == abi.GPX_ENOGPU


def test_product_never_references_oracle():
    """The product tree must not import, link or load anything under oracle/."""
    pkg = os.path.join(ROOT, "gigapaxos_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")) and f != "build.py":
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "gpxo_" not in src and "libgpx_oracle" not in src, f
