"""CPU: the Python mirror of tz_selfplay_data_t has the header's fields in the header's order, and its arrays are
exactly the struct's pointer fields."""
import os
import re

from takzero_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_fields():
    text = open(os.path.join(ROOT, "include", "takzero_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    body = re.search(r"typedef struct tz_selfplay_data_t \{(.*?)\} tz_selfplay_data_t;", text, flags=re.S).group(1)
    out = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if decl:
            out.append((decl.rsplit(" ", 1)[1], "*" in decl))
    return out


def test_selfplay_data_layout_matches_the_header():
    fields = header_fields()
    assert [name for name, _ in fields] == [name for name, _ in capi.SelfplayData._fields_]
    assert [name for name, ptr in fields if ptr] == list(capi.SELFPLAY_FIELDS)
    assert capi.STATUS_TARGETS_FULL == 1024
