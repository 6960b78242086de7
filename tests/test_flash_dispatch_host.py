"""Host logic: which decode steps the MX attention block sends to the K3 -> K4a -> K3 chain instead of K4b
(attention_ops.chain_is_faster).  No GPU needed."""


def test_small_decode_batches_on_long_rows_take_the_chain():
    from torchmx_b200 import attention_ops as ao
    fast = ao.chain_is_faster
    assert fast(1, 8, 1, 2048, False) and fast(1, 8, 1, 32768, False) and fast(1, 2, 1, 8448, False)
    assert fast(1, 8, 1, 8224, True) and fast(4, 2, 1, 32768, True)
    assert not fast(1, 8, 1, 1024, False) and not fast(1, 8, 1, 8192, True)   # rows K4b took before: unchanged
    assert fast(2, 8, 1, 32768, False) and fast(8, 2, 1, 4096, False)
    assert not fast(4, 8, 1, 32768, False) and not fast(32, 8, 1, 2048, False)  # enough CTAs for K4b
    assert not fast(1, 8, 2, 32768, True)                                    # not a decode step
    assert not fast(1, 8, 1, ao.MAX_KV + 32, False)                          # K4a cannot take the row: K4b it is
    assert ao.MAX_FLASH_KV == 131072
