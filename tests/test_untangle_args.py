"""CPU check of the untangling entry point hdgnn_set_predictions: it rejects bad arguments before any CUDA call, so it needs
no GPU.  The stateless entry points are checked in test_stateless_args.py."""


def test_set_predictions_validates_arguments_without_a_gpu():
    from hdgnn_b200 import _lib
    assert _lib.lib.hdgnn_set_predictions(None, None) == _lib.E_INVALID
    assert _lib.lib.hdgnn_infer_host(None, 1, None, None, None, None, None, None, None, None, None) == _lib.E_INVALID
