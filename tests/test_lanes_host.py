"""Host logic of the execution lanes, on the oracle: per circuit step, a query ingests all its tables in one
grouped call and runs each incremental join as one join step; a single-table query makes a grouped call of one."""
import pytest

from oracle_backend import OracleBackend
from dbsp_b200.nexmark import NexmarkGenerator
from parity_util import build_query, feed


class RecordingBackend(OracleBackend):
    """Records the circuit's calls into the backend (not the single calls a grouped call is made of)."""

    def __init__(self):
        super().__init__()
        self.calls = []
        self.depth = 0

    def _rec(name):
        def method(self, *a, **k):
            if self.depth == 0:
                self.calls.append((name, len(a[0]) if name == "batches_from_tables" else 1))
            self.depth += 1
            try:
                return getattr(OracleBackend, name)(self, *a, **k)
            finally:
                self.depth -= 1
        return method

    batches_from_tables = _rec("batches_from_tables")
    batch_from_table = _rec("batch_from_table")
    batch_from_upload = _rec("batch_from_upload")
    join_step = _rec("join_step")
    join_delta_trace = _rec("join_delta_trace")


@pytest.mark.parametrize("query,tables,joins", [("q3", 2, 1), ("q4", 2, 1), ("q7", 1, 1)])
def test_one_grouped_ingest_and_one_join_step_per_join(query, tables, joins):
    be = RecordingBackend()
    c, h, out = build_query(be, query)
    gen = NexmarkGenerator()
    for s0 in range(0, 30_000, 10_000):
        feed(h, gen.tables(s0, 10_000))
        be.calls = []
        c.step()
        assert [k for name, k in be.calls if name == "batches_from_tables"] == [tables]
        assert sum(1 for name, _ in be.calls if name == "join_step") == joins
        for name in ("batch_from_table", "batch_from_upload", "join_delta_trace"):
            assert all(n != name for n, _ in be.calls), f"{query} still calls {name}"


def test_empty_table_is_not_ingested():
    """A table left unset for a step yields an empty batch without a library call."""
    be = RecordingBackend()
    c, h, out = build_query(be, "q3")
    t = NexmarkGenerator().tables(0, 10_000)
    h["auction"].set(t["auction"])
    be.calls = []
    c.step()
    assert [k for name, k in be.calls if name == "batches_from_tables"] == [1]
