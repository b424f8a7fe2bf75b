"""The Python side's declarations of the C boundary against the C sources: the signature tables of r-pcc_b200/_lib.py
and oracle/__init__.py, the layout of the structures they mirror, and RPCC_EVAL_COLS.  ctypes checks nothing of this
by itself; a stale entry would pass arguments of the wrong width or read fields at the wrong offsets.  Needs neither
a GPU nor a built library."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rpcc_b200.h")

SCALARS = {"int": C.c_int, "float": C.c_float, "double": C.c_double, "size_t": C.c_size_t, "int64_t": C.c_int64,
           "uint64_t": C.c_uint64, "long long": C.c_longlong, "uint32_t": C.c_uint32}


def _source(path):
    """The file without comments and preprocessor directives (continuation lines included)."""
    s = open(path).read()
    s = re.sub(r"/\*.*?\*/", " ", s, flags=re.S)
    s = re.sub(r"//[^\n]*", " ", s)
    return re.sub(r"^[ \t]*#(?:[^\n]*\\\n)*[^\n]*", " ", s, flags=re.M)


def _ctype(decl, where):
    """ctypes type of a C type: every pointer is c_void_p except a string (const char*); void is None."""
    t = re.sub(r"\s*\*\s*", "*", " ".join(decl.split()))
    if t in ("const char*", "char*"):
        return C.c_char_p
    if "*" in t:
        return C.c_void_p
    if t == "void":
        return None
    t = re.sub(r"^const ", "", t)
    assert t in SCALARS, "%s: C type %r has no ctypes mapping" % (where, decl)
    return SCALARS[t]


def _prototypes(path, api, prefix, end):
    """name -> (restype, argtypes) of every `api <type> prefix_name(...)<end>` in the file, in its order."""
    out = {}
    for ret, name, params in re.findall(r"\b%s\s+([^;{}()]*?)\b(%s\w+)\s*\(([^)]*)\)\s*%s" % (api, prefix, end),
                                        _source(path)):
        args = []
        if params.strip() != "void":
            for p in params.split(","):
                m = re.fullmatch(r"\s*(.*?[\s*])(\w+)\s*", p)
                assert m, "%s: cannot parse parameter %r" % (name, p)
                args.append(_ctype(m.group(1), "%s(%s)" % (name, m.group(2))))
        assert name not in out, name
        out[name] = (_ctype(ret, name), tuple(args))
    return out


def _compare(declared, table, what):
    """Both directions: every declared function is in the table with exactly its types, and nothing else is."""
    assert len(declared) >= 20, "parsed only %d %s prototypes" % (len(declared), what)
    missing = sorted(set(declared) - set(table))
    extra = sorted(set(table) - set(declared))
    assert not missing, "%s functions missing from the table: %s" % (what, missing)
    assert not extra, "table entries with no %s function: %s" % (what, extra)

    def name(t):
        return None if t is None else t.__name__

    wrong = ["%s: table (%s, %s) vs C (%s, %s)" % (n, name(table[n][0]), [name(a) for a in table[n][1]],
                                                     name(declared[n][0]), [name(a) for a in declared[n][1]])
             for n in declared if (table[n][0], tuple(table[n][1])) != declared[n]]
    assert not wrong, "\n".join(wrong)
    assert list(table) == list(declared), "the table is not in the order of the %s source" % what


def test_rpcc_signature_table_matches_header():
    from rpcc_b200._lib import SIGNATURES
    _compare(_prototypes(HEADER, "RPCC_API", "rpcc_", ";"), SIGNATURES, "RPCC_API")


def test_oracle_signature_table_matches_definitions():
    import oracle
    _compare(_prototypes(os.path.join(ROOT, "oracle", "rpcc_oracle.c"), "ORC_API", "orc_", r"\{"), oracle.SIGNATURES,
             "ORC_API")


def _struct_fields(name):
    """[(field, ctypes type)] of `typedef struct name {...} name;` in the header; arrays as ctypes arrays."""
    body = re.search(r"typedef\s+struct\s+%s\s*\{(.*?)\}\s*%s\s*;" % (name, name), _source(HEADER), re.S)
    assert body, name
    fields = []
    for decl in body.group(1).split(";"):
        if not decl.strip():
            continue
        m = re.fullmatch(r"\s*(\w+(?:\s+\w+)?)\s+(.*?)\s*", decl, re.S)
        assert m, "%s: cannot parse %r" % (name, decl)
        base = _ctype(m.group(1), "%s.%s" % (name, m.group(2)))
        for d in m.group(2).split(","):
            dm = re.fullmatch(r"\s*(\w+)\s*(?:\[(\d+)\])?\s*", d)
            assert dm, "%s: cannot parse declarator %r" % (name, d)
            fields.append((dm.group(1), base * int(dm.group(2)) if dm.group(2) else base))
    return fields


def _same_type(a, b):
    if issubclass(a, C.Array) or issubclass(b, C.Array):
        return (issubclass(a, C.Array) and issubclass(b, C.Array) and a._length_ == b._length_
                and a._type_ is b._type_)
    return a is b


def test_struct_mirrors_declare_the_header_fields():
    """Same fields, same order, same types: a field added to the header and not to the mirror (or the reverse) fails
    here even where padding would hide it from the layout check."""
    import numpy as np
    from rpcc_b200._lib import RESULT_DTYPE, EncoderConfig
    want = _struct_fields("rpcc_encoder_config")
    got = list(EncoderConfig._fields_)
    assert [n for n, _ in got] == [n for n, _ in want], "EncoderConfig fields differ from rpcc_encoder_config"
    bad = [n for (n, a), (_, b) in zip(got, want) if not _same_type(a, b)]
    assert not bad, "EncoderConfig fields of the wrong type: %s" % bad
    want = _struct_fields("rpcc_frame_result")
    assert [n for n, _ in want] == list(RESULT_DTYPE.names), "RESULT_DTYPE fields differ from rpcc_frame_result"
    bad = [n for n, t in want if np.dtype(t) != RESULT_DTYPE.fields[n][0]]
    assert not bad, "RESULT_DTYPE fields of the wrong type: %s" % bad


def test_struct_mirrors_have_the_compiled_layout(tmp_path):
    """sizeof and every offsetof as the system C compiler lays the header's structures out."""
    from rpcc_b200._lib import RESULT_DTYPE, EncoderConfig
    cc = next((c for c in (os.environ.get("CC"), "cc", "gcc", "clang") if c and shutil.which(c)), None)
    if cc is None:
        pytest.skip("no C compiler")
    structs = {"rpcc_encoder_config": [n for n, _ in _struct_fields("rpcc_encoder_config")],
               "rpcc_frame_result": [n for n, _ in _struct_fields("rpcc_frame_result")]}
    lines = []
    for s, fields in structs.items():
        lines.append('printf("%s sizeof %%zu\\n", sizeof(%s));' % (s, s))
        lines += ['printf("%s %s %%zu\\n", offsetof(%s, %s));' % (s, f, s, f) for f in fields]
    src = tmp_path / "probe.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rpcc_b200.h"\nint main(void) {\n%s\nreturn 0;\n}\n'
                   % "\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    layout = {}
    for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines():
        s, f, v = line.split()
        layout[s, f] = int(v)
    got = {("rpcc_encoder_config", "sizeof"): C.sizeof(EncoderConfig),
           ("rpcc_frame_result", "sizeof"): RESULT_DTYPE.itemsize}
    got.update({("rpcc_encoder_config", f): getattr(EncoderConfig, f).offset for f, _ in EncoderConfig._fields_})
    got.update({("rpcc_frame_result", f): RESULT_DTYPE.fields[f][1] for f in RESULT_DTYPE.names})
    wrong = ["%s.%s: mirror %s, compiler %s" % (s, f, got.get((s, f)), layout.get((s, f)))
             for s, f in sorted(set(got) | set(layout)) if got.get((s, f)) != layout.get((s, f))]
    assert not wrong, "\n".join(wrong)


def test_eval_cols_matches_header():
    from rpcc_b200._lib import EVAL_COLS
    m = re.search(r"^#define\s+RPCC_EVAL_COLS\s+(\d+)\b", open(HEADER).read(), re.M)
    assert m and EVAL_COLS == int(m.group(1))
