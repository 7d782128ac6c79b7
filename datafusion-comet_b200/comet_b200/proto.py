"""Encoder for the reference's plan IR (prost/protobuf wire format).

This is the stand-in for the JVM side (`QueryPlanSerde.scala`, `operators.scala:1046-1900`) that
*produces* `spark.spark_operator.Operator` bytes: tests and bench.py build the same messages the
Spark plugin would send through `Native.createPlan` (`Native.scala:60-79`).  Field numbers are the
reference's (native/proto/src/proto/{operator,expr,literal,types,partitioning}.proto); the test
`tests/test_proto.py::test_field_numbers_match_reference` checks every number used here against
the numbers recorded from those files in tests/golden/proto_field_numbers.json.

No protoc / generated code: the wire format is five rules (varint, fixed64, length-delimited,
fixed32, tags), written out below.
"""
import struct

# ---- wire primitives ----------------------------------------------------------------------------
VARINT, FIXED64, LEN, FIXED32 = 0, 1, 2, 5


def _varint(n):
    if n < 0:
        n += 1 << 64
    out = bytearray()
    while True:
        b = n & 0x7F
        n >>= 7
        if n:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def _tag(field, wt):
    return _varint((field << 3) | wt)


def f_varint(field, v):
    return _tag(field, VARINT) + _varint(int(v))


def f_bool(field, v):
    return f_varint(field, 1 if v else 0)


def f_len(field, payload):
    payload = bytes(payload)
    return _tag(field, LEN) + _varint(len(payload)) + payload


def f_str(field, s):
    return f_len(field, s.encode() if isinstance(s, str) else s)


def f_double(field, v):
    return _tag(field, FIXED64) + struct.pack("<d", v)


def f_float(field, v):
    return _tag(field, FIXED32) + struct.pack("<f", v)


# ---- field-number tables (checked against the .proto files by tests/test_proto.py) --------------
DATA_TYPE_ID = dict(BOOL=0, INT8=1, INT16=2, INT32=3, INT64=4, FLOAT=5, DOUBLE=6, STRING=7, BYTES=8, TIMESTAMP=9,
                    DECIMAL=10, TIMESTAMP_NTZ=11, DATE=12, NULL=13)  # types.proto:43-66
EXPR_FIELD = dict(literal=2, bound=3, add=4, subtract=5, multiply=6, divide=7, cast=8, eq=9, neq=10, gt=11, gt_eq=12,
                  lt=13, lt_eq=14, is_null=15, is_not_null=16, **{"and": 17, "or": 18}, check_overflow=25,
                  caseWhen=38, **{"in": 39, "not": 40}, unary_minus=41, **{"if": 44}, unbound=51)  # expr.proto:30-109
AGG_FIELD = dict(count=2, sum=3, min=4, max=5, avg=6)  # expr.proto:143-176
OP_FIELD = dict(scan=100, projection=101, filter=102, sort=103, hash_agg=104, limit=105, shuffle_writer=106,
                native_scan=111, shuffle_scan=116)  # operator.proto:32-86
LITERAL_FIELD = dict(bool_val=1, byte_val=2, short_val=3, int_val=4, long_val=5, float_val=6, double_val=7,
                     string_val=8, bytes_val=9, decimal_val=10, datatype=12, is_null=13)  # literal.proto:26-47
LEGACY, TRY, ANSI = 0, 1, 2  # expr.proto:324 EvalMode
PARTIAL, FINAL, PARTIAL_MERGE = 0, 1, 2  # operator.proto AggregateMode


# ---- DataType (types.proto:43-114) ---------------------------------------------------------------
class DT:
    def __init__(self, name, precision=0, scale=0):
        self.name, self.precision, self.scale = name, precision, scale

    def encode(self):
        out = f_varint(1, DATA_TYPE_ID[self.name])
        if self.name == "DECIMAL":
            info = f_varint(1, self.precision) + f_varint(2, self.scale)  # DecimalInfo
            out += f_len(2, f_len(2, info))  # type_info { decimal = 2 }
        return out

    def __repr__(self):
        return f"DECIMAL({self.precision},{self.scale})" if self.name == "DECIMAL" else self.name


BOOL, INT8, INT16, INT32, INT64 = DT("BOOL"), DT("INT8"), DT("INT16"), DT("INT32"), DT("INT64")
FLOAT, DOUBLE, STRING, DATE, TIMESTAMP = DT("FLOAT"), DT("DOUBLE"), DT("STRING"), DT("DATE"), DT("TIMESTAMP")


def DECIMAL(p, s):
    return DT("DECIMAL", p, s)


# ---- Expr (expr.proto) ---------------------------------------------------------------------------
def _expr(kind, payload):
    return f_len(EXPR_FIELD[kind], payload)


def bound(index, dt):  # BoundReference expr.proto:375
    return _expr("bound", f_varint(1, index) + f_len(2, dt.encode()))


def unbound(name, dt):
    return _expr("unbound", f_str(1, name) + f_len(2, dt.encode()))


def literal(value, dt):
    """value=None -> typed NULL.  Decimal value = unscaled python int (sent as big-endian signed bytes)."""
    body = b""
    if value is None:
        body += f_bool(LITERAL_FIELD["is_null"], True)
    elif dt.name == "BOOL":
        body += f_bool(1, value)
    elif dt.name == "INT8":
        body += f_varint(2, value)
    elif dt.name == "INT16":
        body += f_varint(3, value)
    elif dt.name in ("INT32", "DATE"):
        body += f_varint(4, value)
    elif dt.name in ("INT64", "TIMESTAMP", "TIMESTAMP_NTZ"):
        body += f_varint(5, value)
    elif dt.name == "FLOAT":
        body += f_float(6, value)
    elif dt.name == "DOUBLE":
        body += f_double(7, value)
    elif dt.name == "STRING":
        body += f_str(8, value)
    elif dt.name == "DECIMAL":
        v = int(value)
        nbytes = max(1, (v.bit_length() + 8) // 8)
        body += f_len(10, v.to_bytes(nbytes, "big", signed=True))
    else:
        raise ValueError(dt)
    body += f_len(LITERAL_FIELD["datatype"], dt.encode())
    return _expr("literal", body)


def _math(kind, l, r, ret, eval_mode=LEGACY):  # MathExpr expr.proto:330
    return _expr(kind, f_len(1, l) + f_len(2, r) + f_len(4, ret.encode()) + f_varint(5, eval_mode))


def add(l, r, ret, eval_mode=LEGACY):
    return _math("add", l, r, ret, eval_mode)


def subtract(l, r, ret, eval_mode=LEGACY):
    return _math("subtract", l, r, ret, eval_mode)


def multiply(l, r, ret, eval_mode=LEGACY):
    return _math("multiply", l, r, ret, eval_mode)


def divide(l, r, ret, eval_mode=LEGACY):
    return _math("divide", l, r, ret, eval_mode)


def _binary(kind, l, r):  # BinaryExpr
    return _expr(kind, f_len(1, l) + f_len(2, r))


def eq(l, r):
    return _binary("eq", l, r)


def neq(l, r):
    return _binary("neq", l, r)


def gt(l, r):
    return _binary("gt", l, r)


def gt_eq(l, r):
    return _binary("gt_eq", l, r)


def lt(l, r):
    return _binary("lt", l, r)


def lt_eq(l, r):
    return _binary("lt_eq", l, r)


def and_(l, r):
    return _binary("and", l, r)


def or_(l, r):
    return _binary("or", l, r)


def not_(c):
    return _expr("not", f_len(1, c))


def is_null(c):
    return _expr("is_null", f_len(1, c))


def is_not_null(c):
    return _expr("is_not_null", f_len(1, c))


def cast(child, dt, eval_mode=LEGACY, timezone="UTC"):
    return _expr("cast", f_len(1, child) + f_len(2, dt.encode()) + f_str(3, timezone) + f_varint(4, eval_mode))


def check_overflow(child, dt, fail_on_error=False):
    return _expr("check_overflow", f_len(1, child) + f_len(2, dt.encode()) + f_bool(3, fail_on_error))


def unary_minus(child, fail_on_error=False):
    return _expr("unary_minus", f_len(1, child) + f_bool(2, fail_on_error))


def if_(c, t, f):
    return _expr("if", f_len(1, c) + f_len(2, t) + f_len(3, f))


def case_when(whens, thens, else_expr=None):  # CaseWhen expr.proto:473
    body = b"".join(f_len(2, w) for w in whens) + b"".join(f_len(3, t) for t in thens)
    if else_expr is not None:
        body += f_len(4, else_expr)
    return _expr("caseWhen", body)


def in_(value, lst, negated=False):
    return _expr("in", f_len(1, value) + b"".join(f_len(2, x) for x in lst) + f_bool(3, negated))


# ---- AggExpr (expr.proto:143-215) ----------------------------------------------------------------
def _agg(kind, payload, filter_expr=None):
    out = f_len(AGG_FIELD[kind], payload)
    if filter_expr is not None:
        out += f_len(89, filter_expr)
    return out


def agg_count(children, filter_expr=None):
    return _agg("count", b"".join(f_len(1, c) for c in children), filter_expr)


def agg_sum(child, dt, eval_mode=LEGACY, filter_expr=None):
    return _agg("sum", f_len(1, child) + f_len(2, dt.encode()) + f_varint(3, eval_mode), filter_expr)


def agg_min(child, dt, filter_expr=None):
    return _agg("min", f_len(1, child) + f_len(2, dt.encode()), filter_expr)


def agg_max(child, dt, filter_expr=None):
    return _agg("max", f_len(1, child) + f_len(2, dt.encode()), filter_expr)


def agg_avg(child, dt, sum_dt, eval_mode=LEGACY, filter_expr=None):
    return _agg("avg", f_len(1, child) + f_len(2, dt.encode()) + f_len(3, sum_dt.encode()) + f_varint(4, eval_mode),
                filter_expr)


# ---- Operator (operator.proto) -------------------------------------------------------------------
def _op(kind, payload, children=(), plan_id=0):
    out = b"".join(f_len(1, c) for c in children)
    out += f_varint(2, plan_id)
    out += f_len(OP_FIELD[kind], payload)
    return out


def scan(fields, source="scan", plan_id=0):  # Scan operator.proto:104
    return _op("scan", b"".join(f_len(1, dt.encode()) for dt in fields) + f_str(2, source), (), plan_id)


def shuffle_scan(fields, source="shuffle", plan_id=0):
    return _op("shuffle_scan", b"".join(f_len(1, dt.encode()) for dt in fields) + f_str(2, source), (), plan_id)


def projection(child, exprs, plan_id=0):  # operator.proto:633
    return _op("projection", b"".join(f_len(1, e) for e in exprs), (child,), plan_id)


def filter_(child, predicate, plan_id=0):  # operator.proto:637
    return _op("filter", f_len(1, predicate), (child,), plan_id)


def hash_agg(child, grouping, aggs, mode=PARTIAL, plan_id=0):  # operator.proto:647
    body = b"".join(f_len(1, g) for g in grouping) + b"".join(f_len(2, a) for a in aggs) + f_varint(5, mode)
    return _op("hash_agg", body, (child,), plan_id)


def hash_partitioning(exprs, num_partitions):  # partitioning.proto:38
    return f_len(1, b"".join(f_len(1, e) for e in exprs) + f_varint(2, num_partitions))


def shuffle_writer(child, partitioning, plan_id=0):  # operator.proto:688
    return _op("shuffle_writer", f_len(1, partitioning), (child,), plan_id)


def struct_field(name, dt, nullable=True):  # SparkStructField operator.proto:97
    return f_str(1, name) + f_len(2, dt.encode()) + f_bool(3, nullable)


def partitioned_file(path, start=0, length=0, file_size=0):  # SparkPartitionedFile
    return f_str(1, path) + f_varint(2, start) + f_varint(3, length) + f_varint(4, file_size)


def native_scan(required_schema, data_schema, files, projection_vector=None, data_filters=(), source="native_scan",
                plan_id=0):
    """NativeScan operator.proto:141-185.  required_schema/data_schema: list of (name, DT, nullable)."""
    common = b"".join(f_len(1, struct_field(*f)) for f in required_schema)
    common += b"".join(f_len(2, struct_field(*f)) for f in data_schema)
    common += b"".join(f_len(4, e) for e in data_filters)
    pv = projection_vector if projection_vector is not None else list(range(len(required_schema)))
    common += f_len(5, b"".join(_varint(int(i)) for i in pv))  # packed repeated int64
    common += f_str(6, "UTC") + f_str(12, source)
    common += b"".join(f_len(13, f[1].encode()) for f in required_schema)
    part = b"".join(f_len(1, partitioned_file(*f) if isinstance(f, tuple) else partitioned_file(f)) for f in files)
    return _op("native_scan", f_len(1, common) + f_len(2, part), (), plan_id)


def config_map(entries):  # config.proto ConfigMap { map<string,string> entries = 1 }
    out = b""
    for k, v in entries.items():
        out += f_len(1, f_str(1, k) + f_str(2, v))
    return out
