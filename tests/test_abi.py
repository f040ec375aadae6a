"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol that
include/ruhvro_b200.h declares; schema parse / gate / Arrow-schema export work without a GPU;
the decode entry points fail loudly (never fall back) when no CUDA device is present."""
import ctypes
import json
import os
import random
import re

import pyarrow as pa
import pytest

import pyruhvro_b200 as pr
from oracle import pyoracle as po
from tests.golden import reference_datums as G
from tests.parity import expected_schema

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported():
    header = open(os.path.join(ROOT, "include", "ruhvro_b200.h")).read()
    names = set(re.findall(r"\b(rv_[a-z_0-9]+)\s*\(", header))
    assert len(names) >= 20
    lib = ctypes.CDLL(os.path.join(ROOT, "pyruhvro_b200", "libruhvro_b200.so"))
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing
    lib.rv_version.restype = ctypes.c_char_p
    assert b"sm_100a" in lib.rv_version()


def test_python_surface_matches_reference_module():
    import pyruhvro
    for name in ("deserialize_array", "deserialize_array_threaded", "serialize_record_batch",
                 "deserialize_array_threaded_spawn", "serialize_record_batch_spawn"):  # src/lib.rs:150-158
        assert callable(getattr(pyruhvro, name))


@pytest.mark.parametrize("seed", range(100))
def test_arrow_schema_matches_schema_translate(seed):
    sj = po.random_schema_json(random.Random(seed))
    s = pr.Schema(sj)
    assert s.is_supported
    assert s.arrow_schema.equals(expected_schema(sj), check_metadata=True)


def _walk_c_schema(addr):
    s = pr._ArrowSchema.from_address(addr)
    kids = []
    if s.n_children:
        arr = (ctypes.c_void_p * s.n_children).from_address(s.children)
        kids = [_walk_c_schema(arr[i]) for i in range(s.n_children)]
    return {"format": s.format.decode(), "name": (s.name or b"").decode(), "flags": s.flags, "children": kids}


def test_c_level_map_and_union_field_names():
    """pyarrow renames map children on import, so the names the reference produces
    (schema_translate.rs:66-75: entries/keys/values) are checked on the raw C structs."""
    sj = json.dumps({"type": "record", "name": "T", "fields": [
        {"name": "m", "type": {"type": "map", "values": ["null", "long"]}},
        {"name": "u", "type": ["null", "string", {"type": "enum", "name": "E", "namespace": "a.b", "symbols": ["X"]}]}]})
    s = pr.Schema(sj)
    cs = pr._ArrowSchema()
    assert pr.lib.rv_schema_export_arrow(s.handle, ctypes.addressof(cs)) == 0
    top = _walk_c_schema(ctypes.addressof(cs))
    m, u = top["children"]
    assert m["format"] == "+m" and m["flags"] == 0
    entries = m["children"][0]
    assert (entries["name"], entries["format"], entries["flags"]) == ("entries", "+s", 0)
    assert [(c["name"], c["format"], c["flags"]) for c in entries["children"]] == [("keys", "u", 0), ("values", "l", 2)]
    assert u["format"] == "+us:0,1,2" and u["flags"] == 2  # nullable because a null variant exists (:95-97)
    assert [c["name"] for c in u["children"]] == ["null", "varchar", "a.b.E"]  # enum variant: fullname (:127-131)
    pa.Schema._import_from_c(ctypes.addressof(cs))  # consumes/releases


def test_metadata_doc_and_aliases():
    sj = json.dumps({"type": "record", "name": "T", "namespace": "ns", "fields": [
        {"name": "r", "type": {"type": "record", "name": "R", "doc": "rdoc", "aliases": ["Old", "x.Y"], "fields": [
            {"name": "a", "type": "int", "doc": "adoc"}, {"name": "b", "type": "string"}]}},
        {"name": "e", "doc": "ignored", "type": {"type": "enum", "name": "E", "doc": "edoc", "symbols": ["A"]}}]})
    got = pr.Schema(sj).arrow_schema
    assert got.equals(expected_schema(sj), check_metadata=True)
    assert got.field("r").metadata == {b"avro::doc": b"rdoc", b"avro::aliases": b"[ns.Old,x.Y]"}
    assert got.field("r").type.field("a").metadata == {b"avro::doc": b"adoc"}
    assert got.field("e").metadata is None  # enum fields never carry metadata (schema_translate.rs:131)


@pytest.mark.parametrize("wide", ["bytes", {"type": "fixed", "name": "F", "size": 4}, {"type": "string", "logicalType": "uuid"},
                                  {"type": "int", "logicalType": "time-millis"}, {"type": "long", "logicalType": "time-micros"},
                                  {"type": "bytes", "logicalType": "decimal", "precision": 4, "scale": 2}])
def test_gate_is_wider_than_the_references_fast_path(wide, coracle):
    """These types make the reference leave its fast path (fast_decode.rs:16-17,59; both restatements agree) and its
    fallback cannot build them; the product decodes them (SURVEY.md 8(f) rank 3, tests/test_wide_types.py)."""
    sj = json.dumps({"type": "record", "name": "T", "fields": [{"name": "x", "type": wide}, {"name": "y", "type": "int"}]})
    assert not coracle.is_supported(sj) and not po.is_supported(po.parse_schema(sj))
    assert pr.Schema(sj).is_supported and po.is_supported(po.parse_schema(sj, wide=True))


@pytest.mark.parametrize("bad", [{"type": "fixed", "name": "D", "size": 12, "logicalType": "duration"},
                                 {"type": "long", "logicalType": "local-timestamp-micros"},
                                 {"type": "bytes", "logicalType": "decimal", "precision": 60, "scale": 2}])
def test_gate_still_rejects(bad):
    sj = json.dumps({"type": "record", "name": "T", "fields": [{"name": "x", "type": bad}, {"name": "y", "type": "int"}]})
    assert not pr.Schema(sj).is_supported


def test_gate_named_refs_and_non_records(coracle):
    sj = json.dumps({"type": "record", "name": "T", "fields": [
        {"name": "a", "type": {"type": "record", "name": "A", "fields": [{"name": "x", "type": "int"}]}}, {"name": "b", "type": "A"}]})
    assert not coracle.is_supported(sj)                   # Schema::Ref leaves the reference's fast path (fast_decode.rs:59)
    assert pr.Schema(sj).is_supported                     # here a reference decodes like the definition it names
    assert pr.Schema(sj).arrow_schema.field("b").type == pr.Schema(sj).arrow_schema.field("a").type
    rec = json.dumps({"type": "record", "name": "L", "fields": [{"name": "next", "type": ["null", "L"]}]})
    assert not pr.Schema(rec).is_supported                # a recursive type has no finite Arrow type
    assert not pr.Schema('"string"').is_supported
    assert not pr.Schema('{"type":"array","items":"int"}').is_supported


def test_unknown_logical_type_degrades_to_base():
    sj = '{"type":"record","name":"T","fields":[{"name":"x","type":{"type":"long","logicalType":"made-up"}}]}'
    s = pr.Schema(sj)
    assert s.is_supported and s.arrow_schema.field("x").type == pa.int64()


def test_schema_parse_errors_are_value_errors():
    for bad in ["{", '{"type":"record","name":"T"}', '{"type":"record","name":"T","fields":[{"name":"x","type":["int","int"]}]}',
                '{"type":"record","name":"T","fields":[{"name":"x","type":[["null","int"],"string"]}]}']:
        with pytest.raises(ValueError):
            pr.Schema(bad)


def _rec(field_json: str, name: str = "T") -> str:
    return '{"type":"record","name":"%s","fields":[%s]}' % (name, field_json)


@pytest.mark.parametrize("bad", [
    _rec('{"name":" x","type":"int"}'), _rec('{"name":"9x","type":"int"}'), _rec('{"name":"a-b","type":"int"}'), _rec('{"name":"","type":"int"}'),
    _rec('{"name":"a","type":"int"},{"name":"a","type":"long"}'),                       # Error::FieldNameDuplicate
    _rec('{"name":"a","type":"int"}', name="x y"), _rec('{"name":"a","type":"int"}', name="R."), _rec('{"name":"a","type":"int"}', name="9ns.R"),
    _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["A","A"]}}'),       # Error::EnumSymbolDuplicate
    _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["1A"]}}'), _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["A-B"]}}'),
    _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":[""]}}'),
])
def test_names_and_symbols_are_validated_like_apache_avro(bad):
    """Schema::parse_str (apache-avro 0.21, the reference's `parse_schema`, deserialize.rs:18-20) validates type names,
    record field names and enum symbols against the specification's pattern and rejects repeated field names and repeated
    enum symbols; the reference then raises ValueError before any decode.  So does the product."""
    with pytest.raises(ValueError):
        pr.Schema(bad)


def test_valid_names_still_parse_and_a_repeated_json_key_takes_the_last_value():
    s = pr.Schema(_rec('{"name":"_x9","type":{"type":"enum","name":"ns.sub.E","symbols":["A","_b","C9"]}}', name="a.b.T"))
    assert s.is_supported and s.arrow_schema.field("_x9").type == pa.utf8()
    assert pr.Schema(_rec('{"name":"a","type":"int"}', name=".T")).is_supported          # an empty namespace in front of the dot
    # serde_json's Map::insert: the later "logicalType" replaces the earlier one
    s = pr.Schema(_rec('{"name":"t","type":{"type":"long","logicalType":"long","logicalType":"timestamp-micros"}}'))
    assert s.arrow_schema.field("t").type == pa.timestamp("us")
    # an "aliases" array holding anything but strings is no aliases at all (collected into an Option), not an error
    s = pr.Schema('{"type":"record","name":"T","fields":[{"name":"r","type":{"type":"record","name":"R","aliases":["a",5],'
                  '"fields":[{"name":"x","type":"int"}]}}]}')
    assert s.is_supported and not (s.arrow_schema.field("r").metadata or {}).get(b"avro::aliases")


@pytest.mark.parametrize("attrs,fixed", [('"precision":4,"scale":"x"', False), ('"precision":2,"scale":3', False), ('', False),
                                         ('"precision":-2', True), ('"precision":2.0', False), ('"precision":0', True), ('"precision":"9"', False),
                                         ('"precision":4,"scale":-1', True)])
def test_invalid_decimal_metadata_falls_back_to_the_underlying_type(attrs, fixed):
    """apache-avro ignores an invalid decimal annotation with a warning ("Ignoring invalid decimal logical type") — the
    schema is then plain bytes / fixed; it neither fails nor guesses a scale.  Both restatements of the wider subset agree."""
    comma = "," if attrs else ""
    t = ('{"type":"fixed","name":"F","size":4,"logicalType":"decimal"%s%s}' if fixed else '{"type":"bytes","logicalType":"decimal"%s%s}') % (comma, attrs)
    sj = _rec('{"name":"d","type":%s}' % t)
    s = pr.Schema(sj)
    assert s.is_supported and s.arrow_schema.field("d").type == (pa.binary(4) if fixed else pa.binary())
    assert po.to_arrow_schema(po.parse_schema(sj, wide=True)).field("d").type == s.arrow_schema.field("d").type
    ok = pr.Schema(_rec('{"name":"d","type":{"type":"bytes","logicalType":"decimal","precision":9}}'))
    assert ok.arrow_schema.field("d").type == pa.decimal128(9, 0)                         # only "scale" may be absent


def test_union_duplicates_fixed_size_and_enum_default_follow_the_library():
    """UnionSchema::new only checks kinds that are not named (a record may repeat, two decimals on bytes may not); a fixed's size is a
    JSON number that is a non-negative integer; an enum's default is one of its symbols."""
    a = '{"type":"record","name":"A","fields":[{"name":"x","type":"int"}]}'
    assert pr.Schema(_rec('{"name":"a","type":%s},{"name":"u","type":["null","A","A"]}' % a)).is_supported
    for bad in [_rec('{"name":"u","type":[{"type":"bytes","logicalType":"decimal","precision":4},'
                     '{"type":"bytes","logicalType":"decimal","precision":9}]}'),
                _rec('{"name":"u","type":["int","int"]}'), _rec('{"name":"f","type":{"type":"fixed","name":"F","size":4.5}}'),
                _rec('{"name":"f","type":{"type":"fixed","name":"F","size":"4"}}'),
                _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["A","B"],"default":"C"}}'),
                _rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["A","B"],"default":5}}')]:
        with pytest.raises(ValueError):
            pr.Schema(bad)
    assert pr.Schema(_rec('{"name":"e","type":{"type":"enum","name":"E","symbols":["A","B"],"default":"B"}}')).is_supported
    assert pr.Schema(_rec('{"name":"u","type":["int",{"type":"int","logicalType":"date"}]}')).is_supported     # distinct kinds


def test_every_schema_literal_in_the_reference_tree_parses():
    """The stricter front-end must not turn away anything the reference itself uses: every `r#"{...}"#` schema in its Rust
    sources (stored with its file:line in tests/golden/reference_schema_literals.json) goes through rv_schema_parse."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_schema_literals.json")) as f:
        literals = json.load(f)
    for lit in literals:
        pr.Schema(lit["schema"])
    assert len(literals) >= 30


def test_documented_limits_are_errors_not_crashes():
    deep = "int"
    for _ in range(5):
        deep = {"type": "array", "items": deep}
    sj = json.dumps({"type": "record", "name": "T", "fields": [{"name": "x", "type": deep}]})
    s = pr.Schema(sj)
    assert not s.is_supported  # array nesting > 3: no plan


def test_decode_without_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ValueError) as e:
        pr.deserialize_array([bytes.fromhex(G.G2_HEX)], G.G2_SCHEMA)
    assert "CUDA" in str(e.value) or "pinned" in str(e.value)
    with pytest.raises(ValueError):
        import numpy as np
        data, off = po.pack_records([bytes.fromhex(G.G2_HEX)])
        pr.decode_packed(data, off, 1, G.G2_SCHEMA, 1)
    with pytest.raises(ValueError) as e:   # encode has no CPU path either
        pr.serialize_record_batch(pa.record_batch({"firstName": ["a"], "lastName": ["b"], "age": pa.array([1], pa.int32()),
                                                   "addresses": pa.array([[]], pa.list_(pa.struct([("street", pa.string()), ("city", pa.string()), ("zipCode", pa.string())]))),
                                                   "email": ["x"]}), G.G2_SCHEMA, 1)
    assert "CUDA" in str(e.value)


def test_encode_plan_errors_need_no_gpu():
    with pytest.raises(ValueError) as e:
        pr.serialize_record_batch(pa.record_batch({"x": [1]}), G.G2_SCHEMA, 1)
    assert "Arrow struct missing column 'firstName' required by Avro schema. Available columns: [\"x\"]" in str(e.value)
    with pytest.raises(TypeError):
        pr.serialize_record_batch(None, G.G2_SCHEMA, 1)


def test_arrow_array_ingest_view_is_zero_copy_and_rebased():
    """deserialize_arrow_array's host-side adapter (no GPU needed): payload is viewed, offsets widened to i64."""
    import numpy as np
    import pyarrow as pa
    recs = [b"ab", b"", b"cdef", b"g" * 40, b"hi"]
    for typ in (pa.binary(), pa.large_binary()):
        arr = pa.array(recs, type=typ)
        data, off, n = pr._packed_view(arr)
        assert n == 5 and off.dtype == np.int64 and off.tolist() == [0, 2, 2, 6, 46, 48]
        assert data.ctypes.data == arr.buffers()[2].address          # no copy of the payload
        sl = arr.slice(2, 2)
        data, off, n = pr._packed_view(sl)
        assert n == 2 and off.tolist() == [2, 6, 46] and bytes(data[off[0]:off[1]]) == b"cdef"
    ch = pa.chunked_array([pa.array(recs[:2], type=pa.binary()), pa.array(recs[2:], type=pa.binary())])
    data, off, n = pr._packed_view(ch)
    assert n == 5 and [bytes(data[off[i]:off[i + 1]]) for i in range(5)] == recs
    assert pr._packed_view(pa.array([], type=pa.binary()))[2] == 0
    with pytest.raises(ValueError):
        pr._packed_view(pa.array([b"a", None], type=pa.binary()))
    with pytest.raises(TypeError):
        pr._packed_view(pa.array([1, 2]))
    with pytest.raises(OverflowError):
        pr.deserialize_arrow_array(pa.array(recs, type=pa.binary()), "{}", -1)


def test_specialised_kernels_compile_for_sm100a_and_use_the_copy_engine(tmp_path, monkeypatch):
    """No GPU needed: NVRTC cross-compiles the schema-specialised kernel for sm_100a.  The cubin must hold the fused
    kernel and the Blackwell bulk-copy path: TMA load of the input window (UBLKCP.S.G + mbarrier SYNCS), TMA store of
    the staged strings (UBLKCP.G.S), and the look-back's relaxed gpu-scope status accesses."""
    import glob
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    monkeypatch.setenv("RV_JIT_CACHE", str(tmp_path))
    s = pr.Schema(G.G345_SCHEMA)
    s.precompile("sm_100a")
    assert "op_str<MODE" in s.walker_source and "struct Walker" in s.walker_source
    cubins = glob.glob(str(tmp_path / "*.cubin"))
    assert len(cubins) == 1
    sass = subprocess.run([cuobjdump, "-sass", cubins[0]], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in sass or "SM100" in sass.upper() or "EF_CUDA_SM100" in sass
    fn = {}
    cur = None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split(":")[1].strip()
            fn[cur] = []
        elif cur:
            fn[cur].append(line)
    assert "rvj_fused" in fn
    body = "\n".join(fn["rvj_fused"])
    assert "UBLKCP.S.G" in body and "SYNCS.ARRIVE.TRANS64" in body and "TRYWAIT" in body
    assert "UBLKCP.G.S" in body
    assert "LDG.E.64.STRONG.GPU" in body or "LD.E.64.STRONG.GPU" in body   # look-back status loads bypass L1


def test_list_packing_matches_binaryarray_from_vec():
    """`_native.pack` is the list[bytes] walk + gather of decode_list (pymod.cpp) into ordinary memory: values buffer +
    i64 offsets, exactly what BinaryArray::from_vec builds at ruhvro/src/deserialize.rs:90."""
    import numpy as np
    ext = pr._ext()
    rng = random.Random(3)
    for n in (0, 1, 2, 257, 5000):
        recs = [bytes(rng.randrange(256) for _ in range(rng.choice([0, 0, 1, 7, 64, 300]))) for _ in range(n)]
        data, offs = ext.pack(recs)
        want_data, want_off = po.pack_records(recs)
        assert np.array_equal(np.frombuffer(offs, dtype=np.int64), want_off)
        assert data == bytes(want_data)
    big = [bytes([i & 255]) * 1024 for i in range(20_000)]            # > 8 MiB: the multi-threaded gather
    data, offs = ext.pack(big)
    assert data == b"".join(big) and np.frombuffer(offs, dtype=np.int64)[-1] == len(data)
    skew = [b"x" * (12 << 20)] + [b"y"] * 1000 + [b""] * 10 + [b"z" * (3 << 20)]   # byte-balanced split, skewed sizes
    data, offs = ext.pack(skew)
    assert data == b"".join(skew)
    with pytest.raises(TypeError, match="element 1 is 'str', expected 'bytes'"):
        ext.pack([b"a", "b"])
    long = [bytes([i & 255]) * (i % 7) for i in range(200_000)]       # >= 2^16 elements: the multi-threaded header walk
    data, offs = ext.pack(long)
    assert data == b"".join(long)
    assert np.array_equal(np.frombuffer(offs, dtype=np.int64), np.concatenate([[0], np.cumsum([len(x) for x in long])]))
    long[150_000], long[70_001], long[199_999] = None, 7, "s"          # several threads fail: the lowest index is reported
    with pytest.raises(TypeError, match="element 70001 is 'int', expected 'bytes'"):
        ext.pack(long)
    with pytest.raises(TypeError):
        ext.pack((b"a",))                                              # a list, like PyO3's Vec<Bound<PyBytes>> extraction
    # PyBackedBytes (src/lib.rs:29-33) extracts from `bytes` (subclasses included) and from `bytearray`, nothing else
    class MyBytes(bytes):
        pass
    mixed = [bytearray(b"ab"), MyBytes(b"c"), bytearray(), b"de"]
    data, offs = ext.pack(mixed)
    assert data == b"abcde" and list(np.frombuffer(offs, dtype=np.int64)) == [0, 2, 3, 3, 5]
    many = [bytearray([i & 255]) * (i % 5) if i % 3 else bytes([i & 255]) * (i % 5) for i in range(150_000)]   # the threaded walk
    assert ext.pack(many)[0] == b"".join(bytes(x) for x in many)
    with pytest.raises(TypeError, match="element 0 is 'memoryview', expected 'bytes' or 'bytearray'"):
        ext.pack([memoryview(b"ab")])


def test_framed_entry_points_validate_before_touching_the_gpu():
    """Argument and container errors of the framed adapters are host-side: they surface without a CUDA device."""
    import numpy as np
    sj = '{"type":"record","name":"R","fields":[{"name":"x","type":"int"}]}'
    data, off = np.zeros(8, dtype=np.uint8), np.array([0, 8], dtype=np.int64)
    with pytest.raises(ValueError, match="header_bytes >= 5"):
        pr.decode_packed(data, off, 1, sj, 1, framing=pr.Framing(3, 1, -1))
    with pytest.raises(ValueError, match="out of range"):
        pr.decode_packed(data, off, 1, sj, 1, framing=pr.Framing(-1, 0, -1))
    with pytest.raises(ValueError, match="magic"):
        pr.deserialize_ocf(b"not an object container file", 1)
    header = b"Obj\x01" + po.zigzag_bytes(1) + po.zigzag_bytes(11) + b"avro.schema" + po.zigzag_bytes(len(sj)) + sj.encode() + po.zigzag_bytes(0)
    with pytest.raises(ValueError, match="sync"):
        pr.deserialize_ocf(header + bytes(8), 1)                                   # truncated sync marker
    sync = bytes(range(16))
    with pytest.raises(ValueError, match="truncated block"):
        pr.deserialize_ocf(header + sync + po.zigzag_bytes(3) + po.zigzag_bytes(100) + b"\x02", 1)
    with pytest.raises(ValueError, match="sync marker mismatch"):
        pr.deserialize_ocf(header + sync + po.zigzag_bytes(1) + po.zigzag_bytes(1) + b"\x02" + bytes(16), 1)
    codec = header[:-1].replace(po.zigzag_bytes(1), po.zigzag_bytes(2), 1) + po.zigzag_bytes(10) + b"avro.codec" + po.zigzag_bytes(7) + b"deflate" + po.zigzag_bytes(0)
    with pytest.raises(ValueError, match="codec"):
        pr.deserialize_ocf(codec + sync, 1)
