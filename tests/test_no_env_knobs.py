"""The library computes the same thing whatever the environment of the process that loads or builds it (no GPU)."""
import importlib.util
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "damvsnet_b200", "csrc")


def test_native_sources_do_not_read_the_environment():
    readers = []
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(CSRC, name)) as f:
                for lineno, line in enumerate(f, 1):
                    if re.search(r"getenv\s*\(", line):
                        readers.append(f"{name}:{lineno}: {line.strip()}")
    assert not readers, "environment reads in the CUDA library:\n" + "\n".join(readers)


def _nvcc_flags():
    # a fresh module object, so that module-level code runs again under the current environment
    spec = importlib.util.spec_from_file_location("_damvs_build_probe", os.path.join(ROOT, "damvsnet_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return list(mod.NVCC_FLAGS)


def test_build_flags_do_not_depend_on_the_environment(monkeypatch):
    monkeypatch.delenv("DAMVS_TC_TRACE_BUILD", raising=False)
    plain = _nvcc_flags()
    monkeypatch.setenv("DAMVS_TC_TRACE_BUILD", "1")
    assert _nvcc_flags() == plain
