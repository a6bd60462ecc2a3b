"""CPU tests: the Spectral2DCNN backward entry points validate their arguments on the host (status codes without a
device): NULL pointers, unsupported shapes, empty batches and grids too large."""
import ctypes

from mod_extraction_b200 import _lib


def test_backward_entry_points_validate_before_touching_the_gpu():
    L = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    q = ctypes.cast(ctypes.addressof(buf) + 64, ctypes.c_void_p)
    r = ctypes.cast(ctypes.addressof(buf) + 128, ctypes.c_void_p)
    nul = ctypes.c_void_p(0)
    assert L.modfx_cnn_train_workspace_bytes(4, 64, 33, 1) > 0 and L.modfx_cnn_train_workspace_bytes(1, 1, 1, 1) == -1

    train = L.modfx_cnn_conv_pool_prelu_train_f32
    assert train(nul, q, r, p, 1, 2, 4, 64, 1, p, p, p, nul) == -1                 # NULL x
    assert train(p, p, r, p, 1, 2, 4, 64, 1, p, p, p, nul) == -1                   # x aliases y
    assert train(p, q, r, p, 1, 3, 4, 64, 1, p, p, p, nul) == -2                   # odd H
    assert train(p, q, r, p, 1, 2, 4, 64, 32, p, p, p, nul) == -2                  # dilation 32
    assert train(p, q, r, p, 1, 2, 4, 2, 2, p, p, p, nul) == -2                    # 2 channels, dilated
    assert train(p, q, r, p, 1, 2, 4, 16, 1, p, p, p, nul) == -2                   # 16 channels
    assert train(p, q, r, p, 0, 2, 4, 64, 1, p, p, p, nul) == 0                    # empty batch
    assert train(p, q, r, p, 70000, 2, 4, 64, 1, p, p, p, nul) == -1               # more examples than grid.z holds
    assert train(p, q, r, p, 1, 2 * 70000, 4, 64, 1, p, p, p, nul) == -1           # more rows than grid.y holds

    dgrad = L.modfx_cnn_conv_dgrad_tf32_f32
    assert dgrad(p, nul, 1, 2, 4, 1, p, nul) == -1
    assert dgrad(p, p, 1, 2, 4, 1, p, nul) == -1
    assert dgrad(p, q, 1, 2, 4, 17, p, nul) == -2
    assert dgrad(p, q, 0, 2, 4, 1, p, nul) == 0
    assert dgrad(p, q, 70000, 2, 4, 1, p, nul) == -1

    wgrad = L.modfx_cnn_conv_wgrad_tf32_f32
    assert wgrad(p, q, r, 1, 2, 4, 64, 1, nul, nul) == -1                          # NULL workspace
    assert wgrad(p, q, r, 0, 2, 4, 64, 1, p, nul) == -1                            # empty batch: no gradient to form
    assert wgrad(p, q, r, 1, 2, 4, 32, 1, p, nul) == -2
    assert wgrad(p, q, r, 1, 2, 4, 2, 4, p, nul) == -2
    assert wgrad(p, q, r, 1, 5, 4, 64, 1, p, nul) == -2

    pool = L.modfx_cnn_pool_prelu_bwd_f32
    assert pool(p, p, p, p, p, p, nul, 1, 2, 4, p, nul) == -1
    assert pool(p, p, p, p, p, p, p, 1, 3, 4, p, nul) == -1                        # odd H
    assert pool(p, p, p, p, p, p, p, 0, 2, 4, p, nul) == -1

    ln = L.modfx_cnn_layernorm_bwd_f32
    assert ln(p, p, nul, q, 1, 64, 2, 4, 1e-5, p, nul) == -1                       # NULL statistics
    assert ln(p, p, p, q, 1, 3, 2, 4, 1e-5, p, nul) == -2                          # 3 does not divide 256
    assert ln(p, p, p, q, 0, 64, 2, 4, 1e-5, p, nul) == 0
    assert ln(p, p, p, q, 70000, 64, 2, 4, 1e-5, p, nul) == -1

    head = L.modfx_cnn_head_bwd_f32
    assert head(p, p, p, p, p, p, nul, 1, 1, 4, 64, 1, p, p, nul) == -1
    assert head(p, p, p, p, p, p, p, 0, 1, 4, 64, 1, p, p, nul) == -1
    assert head(p, p, p, p, p, p, p, 1, 1, 4, 2048, 1, p, p, nul) == -2
    assert head(p, p, p, p, p, p, p, 70000, 1, 4, 64, 1, p, p, nul) == -1
