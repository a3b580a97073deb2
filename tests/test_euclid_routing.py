"""Which rows the Euclidean matrix is formed from (DESIGN.md §5.11): sparse rows for DNA at 10 <= k <= 12, the
dense rows everywhere else (k = 9 measured faster dense on 4 Mbp genomes; other alphabets have no sparse path)."""
from diverseseq_b200.distance import counts_sparse_for_euclidean


def test_sparse_rows_for_dna_at_k_10_to_12_only():
    assert [k for k in range(1, 14) if counts_sparse_for_euclidean(k, 4)] == [10, 11, 12]
    assert not any(counts_sparse_for_euclidean(k, 20) for k in range(1, 14))
