"""CPU: what the documents promise about the library's switches matches the source."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAPI = os.path.join(ROOT, "midas-journal-740_b200", "csrc", "cuberille_capi.cu")


def test_every_tuning_knob_is_documented_and_read_once():
    src = open(CAPI).read()
    knobs = re.findall(r'env_int\("(CUB_[A-Z0-9_]+)",\s*(-?\d+)', src)
    assert len(knobs) >= 10
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name, default in knobs:
        assert f"`{name}`" in doc, f"{name} is read by cub_create but missing from INTEGRATION.md"
    # the environment is read in cub_create only (VERDICT r1: no getenv on the hot path): env_int's own getenv is the one call
    assert src.count("getenv(") == 1
    create = src[src.index("int cub_create("):]
    create = create[:create.index("\n}\n")]
    for name, _ in knobs:
        assert name in create, f"{name} is not read in cub_create"


def test_every_switch_the_tests_and_tools_set_is_read_by_the_library():
    """a test that sets a variable the library no longer reads runs the same path twice and checks nothing"""
    src = open(CAPI).read()
    read = set(re.findall(r'env_int\("(CUB_[A-Z0-9_]+)"', src))
    api = set(re.findall(r"\bCUB_[A-Z0-9_]+\b", open(os.path.join(ROOT, "include", "cuberille_c.h")).read()))
    allowed = {"CUB_FORCE_BUILD"}  # read by __graft_entry__.build(), not by the library
    named = {}
    for top in ("tests", "tools"):
        for d, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                path = os.path.join(d, f)
                if path == os.path.abspath(__file__) or not f.endswith((".py", ".sh", ".md", ".cxx", ".txt")):
                    continue  # (this file names switches that must not exist)
                for name in re.findall(r"\bCUB_[A-Z0-9_]+\b", open(path, errors="replace").read()):
                    named.setdefault(name, os.path.relpath(path, ROOT))
    switches = {n: p for n, p in named.items() if n not in api}
    assert "CUB_FUSE" in switches and "CUB_K1_PACKED" in switches
    stale = {n: p for n, p in switches.items() if n not in read and n not in allowed}
    assert not stale, f"variables named under tests/ or tools/ that cuberille_capi.cu does not read: {stale}"


def test_fused_kernel_has_no_debug_switch_left():
    src = open(CAPI).read() + open(os.path.join(ROOT, "midas-journal-740_b200", "csrc", "k_fused.cuh")).read()
    assert "CUB_FUSE_DBG" not in src and "dbg" not in src
