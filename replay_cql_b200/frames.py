"""Frame adapters: pandas / pyarrow / (optionally) pyspark -> pandas and back.

The reference moves data between the JVM and Python with ``toPandas()`` over
Arrow (``replay/session_handler.py:47``; pattern ``replay/models/neuromf.py:332``).
pyspark/JVM do not exist in this image, so Spark frames are accepted only if
pyspark is importable; the adapter code for them is written to the documented
contract and is exercised nowhere here (DESIGN.md "out of scope").
"""
from __future__ import annotations

import collections.abc
from typing import Any, Iterable, Optional

import numpy as np
import pandas as pd

try:  # optional
    import pyarrow as pa
except Exception:  # pragma: no cover
    pa = None

try:  # optional, absent in this image
    from pyspark.sql import DataFrame as SparkDataFrame  # type: ignore
except Exception:
    SparkDataFrame = None


def is_spark(df: Any) -> bool:
    return SparkDataFrame is not None and isinstance(df, SparkDataFrame)


def to_pandas(df: Any) -> Optional[pd.DataFrame]:
    """Any supported frame -> pandas (no copy for pandas input)."""
    if df is None:
        return None
    if isinstance(df, pd.DataFrame):
        return df
    if pa is not None and isinstance(df, pa.Table):
        return df.to_pandas()
    if is_spark(df):  # pragma: no cover - needs a JVM
        return df.toPandas()
    raise ValueError(f"Wrong type {type(df)}")


def like_input(result: pd.DataFrame, template: Any) -> Any:
    """Return ``result`` in the flavour of ``template`` (Spark in -> Spark out)."""
    if is_spark(template):  # pragma: no cover - needs a JVM
        return template.sparkSession.createDataFrame(result)
    if pa is not None and isinstance(template, pa.Table):
        return pa.Table.from_pandas(result, preserve_index=False)
    return result


def get_ids(data: Any, column: str) -> pd.DataFrame:
    """Unique ids of ``column`` as a one-column frame (``base_rec.py:541-558`` semantics)."""
    if isinstance(data, pd.DataFrame) or (pa is not None and isinstance(data, pa.Table)) or is_spark(data):
        pdf = to_pandas(data)
        return pd.DataFrame({column: pd.unique(pdf[column])})
    if isinstance(data, collections.abc.Iterable):
        return pd.DataFrame({column: pd.unique(pd.Series(list(data)))})
    raise ValueError(f"Wrong type {type(data)}")


def timestamps_to_int64(col: Any) -> np.ndarray:
    """Timestamps (pandas Series or numpy array; datetime64 / numeric) -> int64 keys with the same order and the same
    ties.  The one place a non-integer timestamp becomes an integer key: every builder (host, device, one-call,
    chunked) sorts these keys.  Floats map element by element to an order-preserving bit key (-0.0 and +0.0 are one
    key; NaN raises), so a chunked column converts chunk by chunk."""
    if isinstance(col, pd.Series) and isinstance(col.dtype, pd.DatetimeTZDtype):
        col = col.dt.tz_convert("UTC").dt.tz_localize(None)
    if col.dtype == object:
        return pd.to_datetime(pd.Series(col)).to_numpy().astype("datetime64[ns]").astype(np.int64)
    arr = col.to_numpy() if isinstance(col, pd.Series) else np.asarray(col)
    if np.issubdtype(arr.dtype, np.datetime64):
        return arr.astype("datetime64[ns]").astype(np.int64)
    if np.issubdtype(arr.dtype, np.integer):
        return arr.astype(np.int64)
    if not np.issubdtype(arr.dtype, np.floating):
        raise ValueError(f"unsupported timestamp dtype {arr.dtype}")
    x = arr.astype(np.float64)
    if np.isnan(x).any():
        raise ValueError("timestamp column has a NaN")
    b = (x + 0.0).view(np.int64)                   # + 0.0: -0.0 -> +0.0
    return np.where(b >= 0, b, b ^ np.int64(0x7FFF_FFFF_FFFF_FFFF))
