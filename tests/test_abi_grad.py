"""Layout of the input-gradient descriptors (`usf_block_grad_desc`, `usf_stack_grad_desc`) in ctypes against gcc's."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_grad_structs_match_the_header_layout(tmp_path):
    gcc = shutil.which("gcc") or shutil.which("cc")
    if gcc is None:
        pytest.skip("no C compiler")
    from nf4ad_b200 import _lib
    structs = {"usf_block_grad_desc": (_lib.BlockGradDesc, ["G", "mlp"]),
               "usf_stack_grad_desc": (_lib.StackGradDesc, ["n_blocks", "blocks", "G_final"])}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "usflow_b200.h"', "int main(void) {"]
    for cname, (_, fields) in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for f in fields:
            lines.append(f'  printf("{cname} {f} %zu\\n", offsetof({cname}, {f}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    seen = {(p[0], p[1]): int(p[2]) for p in (line.split() for line in out.splitlines())}
    for cname, (ctype, fields) in structs.items():
        assert seen[(cname, "size")] == ctypes.sizeof(ctype), cname
        assert [f for f, _ in ctype._fields_] == fields, cname
        for f in fields:
            assert seen[(cname, f)] == getattr(ctype, f).offset, (cname, f)
