"""CPU: the Guided Grad-CAM entry points reject bad arguments before any CUDA call — lrpx_cam_expand_rows_f32 and the
cam_rows / cam_kw / cam_w fields of lrpx_tc_conv_args."""
import ctypes as C


def _input3_args(**kw):
    from lrpx import _lib, tc
    fake = 0x1000                      # never dereferenced: validation fails first
    a = _lib.TcConvArgs(n_img=1, h=16, w=16, cin=64, ncol=24, ksize=3, epilogue=tc.EPI_INPUT3, rule=3, cam_w=8)
    a.a = a.wt = a.out = a.x = a.cam_rows = a.cam_kw = fake
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_tc_conv_rejects_misplaced_cam_factor():
    from lrpx import _lib, tc
    lib = _lib.lib()
    for kw, msg in ((dict(rule=2), b"guided rule"), (dict(epilogue=tc.EPI_INPUT, ncol=16), b"INPUT3"),
                    (dict(cam_kw=None), b"cam_kw"), (dict(cam_w=0), b"cam_w"), (dict(cam_w=65), b"cam_w")):
        assert lib.lrpx_tc_conv(C.byref(_input3_args(**kw)), None) == -1, kw
        assert msg in lib.lrpx_last_error(), (kw, lib.lrpx_last_error())


def test_cam_expand_rows_rejects_bad_arguments():
    from lrpx import _lib
    lib = _lib.lib()
    p = C.c_void_p(0x1000)
    assert lib.lrpx_cam_expand_rows_f32(None, p, p, 1, 2, 2, 4, None) == -1
    assert lib.lrpx_cam_expand_rows_f32(p, p, p, 1, 0, 2, 4, None) == -1
    assert lib.lrpx_cam_expand_rows_f32(p, p, p, -1, 2, 2, 4, None) == -1
    assert b"bad argument" in lib.lrpx_last_error()
    assert lib.lrpx_cam_expand_rows_f32(p, p, p, 0, 2, 2, 4, None) == 0          # nothing to do: no launch
