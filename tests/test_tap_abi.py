"""CPU tests of the episode-tap entry point (dockauv_set_taps): bound in the ctypes table, its ring struct matches the
header, and it validates its arguments before touching a device."""
import ctypes as C


def test_set_taps_null_handle_is_refused():
    from gym_dockauv_b200 import _capi
    lib = _capi.load()
    ids = (C.c_int64 * 2)(0, 1)
    assert lib.dockauv_set_taps(None, ids, 2, 8, None) == -1
    assert b"null handle" in lib.dockauv_last_error()
    assert lib.dockauv_set_taps(None, None, 0, 0, None) == -1


def test_tap_buffer_struct_matches_header():
    import os
    import re
    from gym_dockauv_b200.params import TAP_FIELDS, DockauvTapBuffers
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "dockauv.h")).read()
    body = re.search(r"typedef struct DockauvTapBuffers \{(.*?)\} DockauvTapBuffers;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [n for decl in body.split(";") for n in re.findall(r"\*\s*(\w+)", decl)]
    assert tuple(names) == TAP_FIELDS
    assert C.sizeof(DockauvTapBuffers) == 8 * len(TAP_FIELDS)
