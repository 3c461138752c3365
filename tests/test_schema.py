"""The schema modules written by tools/gen_pb2.py against (a) the field tables of the reference's own .proto files
(tests/golden/schema.json) and (b) the reference's dtype table / unit-test goldens."""

import numpy as np
import pytest

from tensorflow.core.framework import tensor_pb2, tensor_shape_pb2, types_pb2
from tensorflow.core.example import example_pb2, feature_pb2
from tensorflow_serving.apis import classification_pb2, get_model_status_pb2, input_pb2, model_pb2, predict_pb2, regression_pb2
from tensorflow_serving.util import status_pb2

import golden_util

SCHEMA = golden_util.load("schema.json")

# reference tests/unit/min_tfs_client/types_test.py:7-23
TEST_TARGETS = [(np.float16, "DT_HALF", 19), (np.float32, "DT_FLOAT", 1), (np.float64, "DT_DOUBLE", 2), (np.int8, "DT_INT8", 6),
                (np.int16, "DT_INT16", 5), (np.int32, "DT_INT32", 3), (np.int64, "DT_INT64", 9), (np.uint8, "DT_UINT8", 4),
                (np.uint16, "DT_UINT16", 17), (np.uint32, "DT_UINT32", 22), (np.uint64, "DT_UINT64", 23), (np.complex64, "DT_COMPLEX64", 8),
                (np.complex128, "DT_COMPLEX128", 18), (np.str_, "DT_STRING", 7), (np.bool_, "DT_BOOL", 10)]


@pytest.mark.parametrize("np_type,name,enum", TEST_TARGETS)
def test_datatype_three_constructor_forms(np_type, name, enum):
    from min_tfs_client.types import DataType

    for arg in (np_type, name, enum):
        d = DataType(arg)
        assert d.numpy_dtype == np_type and d.tf_dtype == name and d.enum == enum
    assert getattr(types_pb2, name) == enum


def test_datatype_errors():
    from min_tfs_client.types import DataType

    with pytest.raises(ValueError):
        DataType(np.bytes_)
    with pytest.raises(ValueError):
        DataType(3.5)
    with pytest.raises(KeyError):
        DataType(14)
    with pytest.raises(KeyError):
        DataType("DT_QINT8")


_TYPE = {1: "double", 2: "float", 3: "int64", 4: "uint64", 5: "int32", 8: "bool", 9: "string", 12: "bytes", 13: "uint32"}


@pytest.mark.parametrize("path,message,cls", [
    ("tensorflow/core/framework/tensor.proto", "TensorProto", tensor_pb2.TensorProto),
    ("tensorflow/core/framework/tensor.proto", "VariantTensorDataProto", tensor_pb2.VariantTensorDataProto),
    ("tensorflow/core/framework/tensor_shape.proto", "TensorShapeProto", tensor_shape_pb2.TensorShapeProto),
    ("tensorflow_serving/apis/model.proto", "ModelSpec", model_pb2.ModelSpec),
    ("tensorflow_serving/apis/predict.proto", "PredictRequest", predict_pb2.PredictRequest),
    ("tensorflow_serving/apis/predict.proto", "PredictResponse", predict_pb2.PredictResponse),
    # the other RPCs of the client (requests.py:67-110)
    ("tensorflow/core/example/feature.proto", "Feature", feature_pb2.Feature),
    ("tensorflow/core/example/feature.proto", "Features", feature_pb2.Features),
    ("tensorflow/core/example/feature.proto", "FloatList", feature_pb2.FloatList),
    ("tensorflow/core/example/feature.proto", "Int64List", feature_pb2.Int64List),
    ("tensorflow/core/example/feature.proto", "BytesList", feature_pb2.BytesList),
    ("tensorflow/core/example/example.proto", "Example", example_pb2.Example),
    ("tensorflow_serving/apis/input.proto", "Input", input_pb2.Input),
    ("tensorflow_serving/apis/input.proto", "ExampleList", input_pb2.ExampleList),
    ("tensorflow_serving/apis/input.proto", "ExampleListWithContext", input_pb2.ExampleListWithContext),
    ("tensorflow_serving/apis/classification.proto", "ClassificationRequest", classification_pb2.ClassificationRequest),
    ("tensorflow_serving/apis/classification.proto", "ClassificationResponse", classification_pb2.ClassificationResponse),
    ("tensorflow_serving/apis/classification.proto", "Class", classification_pb2.Class),
    ("tensorflow_serving/apis/regression.proto", "RegressionRequest", regression_pb2.RegressionRequest),
    ("tensorflow_serving/apis/regression.proto", "RegressionResponse", regression_pb2.RegressionResponse),
    ("tensorflow_serving/apis/get_model_status.proto", "GetModelStatusRequest", get_model_status_pb2.GetModelStatusRequest),
    ("tensorflow_serving/apis/get_model_status.proto", "GetModelStatusResponse", get_model_status_pb2.GetModelStatusResponse),
    ("tensorflow_serving/apis/get_model_status.proto", "ModelVersionStatus", get_model_status_pb2.ModelVersionStatus),
    ("tensorflow_serving/util/status.proto", "StatusProto", status_pb2.StatusProto),
])
def test_fields_match_reference_proto(path, message, cls):
    want = SCHEMA["messages"][path][message]
    have = {f.name: f for f in cls.DESCRIPTOR.fields}
    assert set(want) == set(have), (sorted(want), sorted(have))
    for name, (num, typ, rep) in want.items():
        f = have[name]
        assert f.number == num, name
        if typ == "map":
            assert f.message_type.GetOptions().map_entry
            continue
        is_rep = f.is_repeated if hasattr(f, "is_repeated") else f.label == f.LABEL_REPEATED
        assert bool(is_rep) == rep, name
        if typ in _TYPE.values():
            assert _TYPE[f.type] == typ, name
        elif f.type == f.TYPE_ENUM:
            assert f.enum_type.name == typ.split(".")[-1]
        else:
            assert f.message_type.name == typ.split(".")[-1], name


def test_datatype_enum_matches_reference_proto():
    want = SCHEMA["DataType"]
    have = {v.name: v.number for v in types_pb2.DataType.DESCRIPTOR.values}
    assert want == have


def test_reference_text_format_golden():
    """reference tests/unit/min_tfs_client/tensors_test.py:66-83: float64[4] text-format golden, through protobuf."""
    from google.protobuf import text_format

    p = tensor_pb2.TensorProto(dtype=types_pb2.DT_DOUBLE, tensor_shape=tensor_shape_pb2.TensorShapeProto(dim=[tensor_shape_pb2.TensorShapeProto.Dim(size=4)]))
    p.double_val.extend([0.314, 0.159, 0.268, 0.358])
    txt = text_format.MessageToString(p)
    assert "dtype: DT_DOUBLE" in txt and "size: 4" in txt and txt.count("double_val") == 4
