"""Which selections run from sparse k-mer rows (distance.counts_sparse_for_selection): DNA at 10 <= k <= 12."""
from diverseseq_b200.distance import counts_sparse_for_selection


def test_sparse_rows_only_for_dna_at_k10_to_12():
    assert [k for k in range(1, 17) if counts_sparse_for_selection(k, 4)] == [10, 11, 12]
    assert not any(counts_sparse_for_selection(k, ns) for k in range(1, 17) for ns in (2, 3, 5, 20))
