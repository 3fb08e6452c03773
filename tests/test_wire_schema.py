"""Wire schema pins: the 201-byte ParserSchema fixture and the reference descriptor."""
import json
import os

from oracle.schemas import ParserSchema, build_file_descriptor, parser_schema_from_dict


def test_parser_fixture1_wire_image(golden_dir):
    """library_integration_base_fixtures.py:27-43 serialised (map entries sorted by key)."""
    g = json.load(open(os.path.join(golden_dir, "parser_fixture1.json")))
    wire = parser_schema_from_dict(g["fields"]).SerializeToString(deterministic=True)
    assert wire.hex() == g["wire_hex"] and len(wire) == 201
    m = ParserSchema()
    m.ParseFromString(bytes.fromhex(g["wire_hex"]))
    assert m.EventID == 1 and list(m.variables) == ["john", "192.168.1.100"]
    assert dict(m.logFormatVariables) == g["fields"]["logFormatVariables"]
    assert m.receivedTimestamp == 1634567890 and m.parsedTimestamp == 1634567891


def test_restated_schema_equals_reference_descriptor(golden_dir):
    """Field names, numbers, types and labels of LogSchema/ParserSchema/DetectorSchema equal
    the descriptor embedded in the reference's container/fluentout/schemas_pb.rb:8 (stored in
    schemas_descriptor.json by scripts/make_golden.py)."""
    from google.protobuf import descriptor_pb2
    g = json.load(open(os.path.join(golden_dir, "schemas_descriptor.json")))
    ref = descriptor_pb2.FileDescriptorProto()
    ref.ParseFromString(bytes.fromhex(g["file_descriptor_hex"]))
    assert {"LogSchema", "ParserSchema", "DetectorSchema"} <= {m.name for m in ref.message_type}
    mine = build_file_descriptor()
    ref_msgs = {m.name: m for m in ref.message_type}
    for m in mine.message_type:
        r = ref_msgs[m.name]
        got = sorted((f.name, f.number, f.type, f.label, f.proto3_optional) for f in m.field)
        want = sorted((f.name, f.number, f.type, f.label, f.proto3_optional) for f in r.field)
        assert got == want, m.name
        for f in m.field:
            if f.type_name:
                rn = {n.name: n for n in r.nested_type}[f.type_name.split(".")[-1]]
                assert rn.options.map_entry
                assert [(x.name, x.number, x.type) for x in rn.field] == [("key", 1, 9), ("value", 2, 9)]
