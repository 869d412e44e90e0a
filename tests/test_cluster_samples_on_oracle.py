"""Per-sample clustering in the batched multi-sample pass on the CPU: the QIIME 2 actions at cluster_id = 0.995 write the
same files batched as in the per-sample loop, with tests/cluster_ref.c clustering each sample for the device, and the
rule that decides which runs may batch."""
import pytest

import cluster_ref as R
import cluster_samples_cases as S
from itsxpress_b200 import SeqSample
from itsxpress_b200 import q2_itsxpress as q2


class SampleClusterOracleContext(R.ClusterOracleContext):
    """ClusterOracleContext that, with sample ids set and per_sample, clusters every sample on its own with the
    reference (centroid rows in the batch's processing order, as on the device)."""

    def cluster(self, cluster_id, order=None, per_sample=False):
        if self._sample is None:
            return super().cluster(cluster_id, order)
        assert per_sample, "sample ids without per_sample are refused"
        self._note("cluster")
        nc, crow, strand, ed_, uor = S.per_sample_reference(self._seq, self._off, self._first, self._uid, self._sample,
                                                            cluster_id, order)
        self._cl = (crow, strand, ed_, uor)
        self._uid = crow[self._uid] if len(self._uid) else self._uid
        self._first = self._first[uor]
        return nc


@pytest.fixture()
def on_ref(oracle, monkeypatch):
    ctx = SampleClusterOracleContext(oracle)
    monkeypatch.setattr(SeqSample, "get_context", lambda: ctx)
    SeqSample.reset_sessions()
    yield ctx
    SeqSample.reset_sessions()


def test_q2_batches_equal_the_per_sample_loop_on_the_reference(on_ref, tmp_path, monkeypatch):
    S.check_q2_batches_equal_loop(on_ref, tmp_path, monkeypatch)


def test_can_batch(monkeypatch):
    monkeypatch.setattr(q2, "BATCH_READS", 4_000_000)
    monkeypatch.delenv("ITSX_CLUSTER", raising=False)
    monkeypatch.delenv("ITSX_STREAM", raising=False)
    assert q2._can_batch(0.995, False) and q2._can_batch(1.0, False)
    assert not q2._can_batch(0.995, True)
    monkeypatch.setenv("ITSX_CLUSTER", "vsearch")
    assert not q2._can_batch(0.995, False)
    assert q2._can_batch(1.0, False)                  # the exact path never shells out
    monkeypatch.delenv("ITSX_CLUSTER")
    monkeypatch.setenv("ITSX_STREAM", "1")            # streamed samples order cluster ties by first occurrence
    assert not q2._can_batch(0.995, False) and q2._can_batch(1.0, False)
    monkeypatch.setenv("ITSX_STREAM", "0")
    assert q2._can_batch(0.995, False)
    monkeypatch.setattr(q2, "BATCH_READS", 0)
    assert not q2._can_batch(0.995, False)
