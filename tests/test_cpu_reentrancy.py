"""CPU tests of the library's threading contract (include/b200iop.h): every entry point may be called from any number of
threads at once.  Static storage in csrc is where that contract breaks, so every piece of it is either per thread,
immutable, atomic, a lock, or named below together with the lock that guards it.  And the kernel timing accepts every
name its header paragraph documents.  tests/test_concurrent_pipes_gpu.py runs the concurrent pipes themselves."""
import ctypes as C
import os
import re

import util

CSRC = os.path.join(util.ROOT, "ansel_b200", "csrc")

# namespace-scope g_* variables that are neither immutable, atomic, a lock nor per thread: what guards each one
GUARDED_GLOBALS = {
    "g_luts": "g_lut_mu (color.cu)",
    "g_stamp": "g_lut_mu (color.cu)",
    "g_timed": "g_timing_mu (runtime.cu)",
    "g_timed_gen": "g_timing_mu (runtime.cu)",
    "g_sm_count": "written once under b200_init's mutex, before g_ndev publishes it (runtime.cu)",
}
# storage that guards itself
SAFE = re.compile(r"\b(const|constexpr|thread_local)\b|std::(atomic|mutex|once_flag)\b")


def _code(txt: str) -> str:
    """the source without comments, string / character literals and B200_AMAZE_PROF-only blocks"""
    txt = re.sub(r"//[^\n]*|/\*.*?\*/", lambda m: "\n" * m.group(0).count("\n"), txt, flags=re.S)
    txt = re.sub(r'"(\\.|[^"\\\n])*"|\'(\\.|[^\'\\\n])*\'', '""', txt)
    out, skip, directive = [], [], False
    for line in txt.split("\n"):
        s = line.strip()
        if directive or s.startswith("#"):     # preprocessor lines, macro bodies with their continuation lines
            directive = s.endswith("\\")
            if re.match(r"#\s*if", s):
                skip.append(bool(re.match(r"#\s*ifdef\s+B200_AMAZE_PROF\b", s)) or bool(skip and skip[-1]))
            elif re.match(r"#\s*endif", s) and skip:
                skip.pop()
            out.append("")
        else:
            out.append("" if skip and skip[-1] else line)
    return "\n".join(out)


def _statements(code: str):
    """(text, scope) of every declaration-like statement; scope is 'namespace', 'class' or 'function'.  A brace opens a
    namespace (namespace, extern "C"), a class (struct / class / union / enum), an initializer (after `=` or a name) or
    a block (function bodies and everything inside them)."""
    stack, pending, out = [], "", []

    def scope():
        kinds = [k for k in stack if k != "init"]
        if "block" in kinds:
            return "function"
        return "class" if "class" in kinds else "namespace"

    for ch in code:
        if ch == "{":
            head = pending.strip()
            if re.search(r"\bnamespace\b|\bextern\s*\"\"\s*$", head):
                kind = "ns"
            elif re.search(r"\b(struct|class|union|enum)\b", head) and "=" not in head and "(" not in head:
                kind = "class"
            elif stack and stack[-1] == "init" or \
                    re.search(r"(=|\b(?!(else|do|try|const|override|noexcept)\b)[A-Za-z_]\w*|\])\s*$", head):
                kind = "init"
            else:
                kind = "block"
            stack.append(kind)
            if kind == "init":
                pending += ch
            else:
                pending = ""
        elif ch == "}":
            kind = stack.pop() if stack else "block"
            if kind == "init":
                pending += ch
            else:
                pending = ""
        elif ch == ";" and (not stack or stack[-1] != "init"):
            out.append((" ".join(pending.split()), scope()))
            pending = ""
        else:
            pending += ch
    return out


def test_static_state_is_per_thread_immutable_atomic_or_guarded():
    """Two pipes in two threads (the darkroom's preview and full pipe) run the same module at once: a function-local
    static or a namespace-scope g_* variable shared without a guard is a data race between them."""
    bad, seen = [], set()
    for fn in sorted(os.listdir(CSRC)):
        if not fn.endswith((".cu", ".cuh", ".h")):
            continue
        for text, scope in _statements(_code(open(os.path.join(CSRC, fn)).read())):
            if re.search(r"__(device|constant|shared)__", text) or SAFE.search(text):
                continue
            if scope == "function" and re.match(r"static\b", text):
                bad.append(f"{fn}: function-local static `{text}`")
            elif scope == "namespace" and not re.match(r"(using|typedef|template|struct|class|enum|union)\b", text):
                m = re.search(r"\b(g_\w+)\s*(\[|=|\{|$)", text)
                if m and "(" not in text[:m.start()]:
                    seen.add(m.group(1))
                    if m.group(1) not in GUARDED_GLOBALS:
                        bad.append(f"{fn}: namespace-scope `{text}` is shared by every thread and guarded by nothing")
    assert not bad, "\n".join(bad)
    assert seen == set(GUARDED_GLOBALS), f"stale allowlist entries: {sorted(set(GUARDED_GLOBALS) - seen)}"


def _timing_paragraph() -> str:
    hdr = open(os.path.join(util.ROOT, "include", "b200iop.h")).read()
    m = re.search(r"/\* Launch timing of .*?\*/", hdr, flags=re.S)
    assert m, "the timing paragraph of include/b200iop.h"
    return m.group(0)


def test_kernel_timing_accepts_every_documented_name(built):
    """b200_kernel_timing_read accepts every kernel its header paragraph quotes, and `nlm_kernel` (what bench.py
    reads).  With timing on and nothing launched, neither call touches CUDA: each returns 0 with count 0."""
    import ansel_b200 as ab
    L = ab.lib()
    names = re.findall(r"`(\w+_kernel)`", _timing_paragraph())
    assert names, "the timing paragraph quotes no kernel name"
    assert L.b200_kernel_timing(1) == 0
    try:
        for name in sorted(set(names) | {"nlm_kernel", "rcd_tiles_kernel"}):
            total, count = C.c_double(-1.0), C.c_int(-1)
            rc = L.b200_kernel_timing_read(name.encode(), C.byref(total), C.byref(count))
            assert rc == 0, f"{name}: {L.b200_last_error().decode()}"
            assert count.value == 0 and total.value == 0.0, name
        assert L.b200_kernel_timing_read(b"no_such_kernel", C.byref(C.c_double()), C.byref(C.c_int())) == ab.B200_ERR_ARG
    finally:
        assert L.b200_kernel_timing(0) == 0
