"""CPU: every build of the CUDA library compiles the same sources (csrc/Makefile for the shared library, rust/h2b200-sys/build.rs
for the static library of the Rust crate, and the list INTEGRATION.md gives); a file missing from one of them leaves symbols
unresolved in that build only."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def test_rust_build_and_makefile_compile_the_same_sources():
    make = re.search(r"^SRCS\s*:=\s*(.+)$", _read("halo2_scaffold_b200", "csrc", "Makefile"), re.M).group(1).split()
    rust = re.findall(r'"([a-z0-9_]+\.cu)"', re.search(r"let sources = \[(.*?)\];", _read("rust", "h2b200-sys", "build.rs"), re.S).group(1))
    assert sorted(make) == sorted(rust)
    doc = re.search(r"`\{([a-z0-9_,]+)\}\.cu`", _read("INTEGRATION.md")).group(1).split(",")
    assert sorted(make) == sorted(d + ".cu" for d in doc)
    on_disk = sorted(f for f in os.listdir(os.path.join(ROOT, "halo2_scaffold_b200", "csrc")) if f.endswith(".cu"))
    assert sorted(make) == on_disk
