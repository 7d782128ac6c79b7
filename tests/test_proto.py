"""The hand-written plan encoder/decoder must use the reference's field numbers."""
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proto_field_numbers.json")


def test_field_numbers_match_reference():
    """Every number the encoder uses, against the reference's .proto files as recorded by tools/proto_field_numbers.py."""
    with open(GOLDEN) as f:
        ref = json.load(f)
    from comet_b200 import proto as P
    expr, op, types, lit, part = (ref[k] for k in ("expr", "operator", "types", "literal", "partitioning"))
    for k, v in P.EXPR_FIELD.items():
        assert expr["Expr"][k] == v, k
    for k, v in P.AGG_FIELD.items():
        assert expr["AggExpr"][k] == v, k
    for k, v in P.OP_FIELD.items():
        assert op["Operator"][k] == v, k
    for k, v in P.DATA_TYPE_ID.items():
        assert types["DataTypeId"][k] == v, k
    for k, v in P.LITERAL_FIELD.items():
        assert lit["Literal"][k] == v, k
    assert expr["MathExpr"] == {"left": 1, "right": 2, "return_type": 4, "eval_mode": 5, "check_divide_overflow": 6}
    assert expr["Sum"] == {"child": 1, "datatype": 2, "eval_mode": 3}
    assert expr["Avg"] == {"child": 1, "datatype": 2, "sum_datatype": 3, "eval_mode": 4}
    assert expr["CheckOverflow"] == {"child": 1, "datatype": 2, "fail_on_error": 3}
    assert expr["BoundReference"] == {"index": 1, "datatype": 2}
    assert expr["AggExpr"]["filter"] == 89
    assert op["HashAggregate"]["grouping_exprs"] == 1 and op["HashAggregate"]["agg_exprs"] == 2 and op["HashAggregate"]["mode"] == 5
    assert op["Operator"]["children"] == 1 and op["Operator"]["plan_id"] == 2
    assert op["Scan"] == {"fields": 1, "source": 2}
    assert op["NativeScanCommon"]["required_schema"] == 1 and op["NativeScanCommon"]["projection_vector"] == 5
    assert op["NativeScan"] == {"common": 1, "file_partition": 2}
    assert op["AggregateMode"] == {"Partial": 0, "Final": 1, "PartialMerge": 2}
    assert expr["EvalMode"] == {"LEGACY": 0, "TRY": 1, "ANSI": 2}
    assert part["HashPartition"] == {"hash_expression": 1, "num_partitions": 2}
    assert types["DecimalInfo"] == {"precision": 1, "scale": 2}


def test_varint_and_literal_encoding_roundtrip_through_the_decoder():
    """Negative ints are 10-byte varints, decimals big-endian two's complement (planner.rs:544-548): the C++
    decoder must read back what the encoder wrote -- checked through generated kernel source."""
    from comet_b200 import native, proto as P
    sc = P.scan([P.DECIMAL(12, 2), P.INT32])
    pred = P.and_(P.gt(P.bound(0, P.DECIMAL(12, 2)), P.literal(-12345, P.DECIMAL(12, 2))), P.gt(P.bound(1, P.INT32), P.literal(-7, P.INT32)))
    plan = P.projection(P.filter_(sc, pred), [P.bound(1, P.INT32)])
    src = native.kernel_source(plan, 1)      # the predicates live in the count pass (kernel 1); pass 2 takes its keep bits
    assert "((cb::i32)-7)" in src
    assert str((-12345) & ((1 << 64) - 1)) + "ull" in src  # sign-extended low limb of the decimal literal
