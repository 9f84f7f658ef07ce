"""Hidden widths 65..128 (CPU side): the library accepts them for the forward in
the tensor-core math modes only, and everything that would train such a model
refuses before any kernel, device or run directory is touched."""
import ctypes as C

import pytest

FAKE = C.c_void_p(256)   # never dereferenced: the calls return before any launch


def _cfg(k, math):
    from pointvs_b200 import _cabi
    return _cabi.LayerConfig(k, 3, 0, 0, _cabi.MATH[math], 0, None, None)


def test_capability_bit_and_limits():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    assert lib.pvs_capabilities() & _cabi.CAP_FWD_WIDE_K
    assert (_cabi.MAX_K, _cabi.MAX_K_TC_FWD) == (64, 128)
    assert b'hidden width' in lib.pvs_status_string(2)


@pytest.mark.parametrize('k', [65, 96, 128])
@pytest.mark.parametrize('math', ['bf16x3', 'fp16x2', 'bf16'])
def test_layer_workspace_for_wide_tensor_core_layers(k, math):
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    cfg = _cfg(k, math)
    nbytes = lib.pvs_egnn_layer_workspace_bytes(1000, 20000, C.byref(cfg))
    # P, Q, M at pitch 128
    assert nbytes >= 3 * 1000 * 128 * 4
    narrow = lib.pvs_egnn_layer_workspace_bytes(1000, 20000,
                                                C.byref(_cfg(64, math)))
    assert nbytes > narrow > 0


def test_wide_width_refused_in_fp32_and_beyond_128():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    assert lib.pvs_egnn_layer_workspace_bytes(
        10, 10, C.byref(_cfg(96, 'fp32'))) == -1
    for math in ('bf16x3', 'fp16x2', 'bf16'):
        assert lib.pvs_egnn_layer_workspace_bytes(
            10, 10, C.byref(_cfg(129, math))) == -1
    g = _cabi.Graph(10, 10, None, None, None, None, None, 1)
    p = _cabi.LayerParams()
    for k, math in ((96, 'fp32'), (129, 'bf16x3')):
        rc = lib.pvs_egnn_layer_fwd(
            C.byref(g), C.byref(_cfg(k, math)), C.byref(p), None, None, None,
            None, None, None, None, None, None, C.c_int64(0), None)
        assert rc == 2, (k, math)


def test_training_calls_refuse_wide_layers_before_any_launch():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    g = _cabi.Graph(10, 10, FAKE, FAKE, None, FAKE, FAKE, 1, FAKE, FAKE, 1)
    p = _cabi.LayerParams()
    grads = _cabi.LayerGrads()
    cfg = _cfg(96, 'bf16x3')
    assert lib.pvs_egnn_layer_bwd_workspace_bytes(10, 10, C.byref(cfg)) == -1
    rc = lib.pvs_egnn_layer_bwd(
        C.byref(g), None, None, C.byref(cfg), C.byref(p), None, None, None,
        None, None, None, None, None, None, C.byref(grads), None, C.c_int64(0),
        None)
    assert rc == 2
    cfgs = (_cabi.LayerConfig * 2)(cfg, cfg)
    params = (_cabi.LayerParams * 2)()
    rc = lib.pvs_egnn_stack_fwd(C.byref(g), 2, cfgs, params, FAKE, FAKE, FAKE,
                                C.c_int64(1 << 30), None)
    assert rc == 2
    grads2 = (_cabi.LayerGrads * 2)()
    rc = lib.pvs_egnn_stack_bwd(
        C.byref(g), FAKE, FAKE, 2, cfgs, params, grads2, FAKE, FAKE, FAKE,
        C.c_int64(1 << 30), FAKE, FAKE, FAKE, FAKE, FAKE, C.c_int64(1 << 40),
        None)
    assert rc == 2


def _model_desc(k, math):
    from pointvs_b200 import _cabi
    cfgs = (_cabi.LayerConfig * 2)(_cfg(k, math), _cfg(k, math))
    params = (_cabi.LayerParams * 2)()
    heads = (_cabi.HeadLayer * 1)(_cabi.HeadLayer(FAKE, FAKE, k, 1, 0))
    desc = _cabi.ModelDesc(2, k, 13, 1, FAKE, FAKE, cfgs, params, heads)
    return desc, (cfgs, params, heads)


def test_fused_scoring_pass_accepts_wide_tensor_core_models_only():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    desc, _keep = _model_desc(96, 'bf16x3')
    assert lib.pvs_egnn_model_workspace_bytes(1000, 20000, 8,
                                              C.byref(desc)) > 0
    for k, math in ((96, 'fp32'), (129, 'bf16x3')):
        desc, _keep = _model_desc(k, math)
        assert lib.pvs_egnn_model_workspace_bytes(10, 10, 1,
                                                  C.byref(desc)) == -1
        g = _cabi.Graph(10, 10, FAKE, FAKE, None, FAKE, FAKE, 1, FAKE, FAKE, 1)
        rc = lib.pvs_egnn_model_fwd(
            C.byref(g), C.byref(desc), FAKE, 13, FAKE, FAKE, 1, FAKE, None,
            None, FAKE, C.c_int64(1 << 40), None)
        assert rc == 2, (k, math)


def test_train_cli_refuses_wide_channels_before_the_run_directory(tmp_path):
    from pointvs_b200 import train
    run = tmp_path / 'wide'
    with pytest.raises(NotImplementedError, match='hidden width 96'):
        train.main(['egnn', str(run), '--channels', '96'])
    assert not (run / 'cmd_args.yaml').exists()
    assert not run.exists()


def test_resume_training_refuses_a_wide_run(tmp_path):
    import yaml
    from pointvs_b200 import resume_training
    (tmp_path / 'checkpoints').mkdir()
    (tmp_path / 'checkpoints' / 'ckpt_epoch_1.pt').write_bytes(b'')
    (tmp_path / 'cmd_args.yaml').write_text(yaml.dump({'channels': 128}))
    (tmp_path / 'model_kwargs.yaml').write_text(yaml.dump({'k': 128}))
    with pytest.raises(NotImplementedError, match='hidden width 128'):
        resume_training.main([str(tmp_path)])


def test_train_model_and_backprop_refuse_a_wide_model(tmp_path):
    import torch
    import pointvs_b200 as pv
    model = pv.SartorrasEGNN(tmp_path, 0, 0, None, None, silent=True,
                             dim_input=13, dim_output=1, k=96, num_layers=2)
    with pytest.raises(NotImplementedError, match='hidden width 96'):
        model.train_model(None)
    with pytest.raises(NotImplementedError, match='hidden width 96'):
        model.backprop(torch.zeros(2), torch.zeros(2))
