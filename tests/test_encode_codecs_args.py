"""The Python wrappers of the device encoder check `encodings` (one codec per column, among the six the device takes) before
they call the library, so the checks hold without a device."""
import pytest


def test_encodings_are_checked_before_the_library_call():
    from oceanbase_b200 import capi, compaction
    cols = [(0, None, capi.OBJ_INT, False), (0, None, capi.OBJ_INT, False)]
    with pytest.raises(ValueError, match="2 values expected"):
        compaction.encode_columns(None, cols, 10, 5, encodings=[capi.ENC_AUTO])
    with pytest.raises(ValueError, match="not among"):
        compaction.encode_columns(None, cols, 10, 5, encodings=[capi.ENC_AUTO, capi.ENC_STRING_DIFF])
    with pytest.raises(ValueError, match="not among"):
        compaction.encode_merge_result(None, [-1, 0], [capi.OBJ_INT] * 2, 5, encodings=[capi.ENC_CS_AUTO, capi.ENC_RAW])
    assert list(compaction._encodings([capi.ENC_RAW, capi.ENC_AUTO], 2)) == [capi.ENC_RAW, capi.ENC_AUTO]
