"""The reference's mixed-precision mode (num_fp16_res / conv_clamp) on CUDA: fp16 activations through the FIR / bias_act kernels (SGV_F16
dispatch) and the library contraction, against the reference golden minted on CPU.
(Round 1 shipped this test opt-in because it had never run on a GPU; it is a normal member of the GPU suite now.)"""
import pytest
import torch

from conftest import load_golden, rel_err
from oracle import synthesis_ref as sr
from stylegan_v_b200.networks import Discriminator
from stylegan_v_b200.synthesis import SynthesisNetwork
from test_networks_cpu import _t

pytestmark = pytest.mark.gpu


def test_mixed_precision_cuda_vs_reference_golden(cuda):
    g, meta = load_golden('mixed_precision_g_tiny.npz')
    cfg = sr.SynthesisConfig(**meta['G'])
    net = SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, channel_base=cfg.channel_base, channel_max=cfg.channel_max,
                           motion_z_dim=cfg.motion_z_dim, motion_v_dim=cfg.motion_v_dim, time_enc_dim=cfg.time_enc_dim,
                           num_fp16_res=meta['num_fp16_res'], conv_clamp=meta['conv_clamp'])
    net.load_state_dict({k[2:]: _t(g[k]) for k in g.files if k.startswith('p:')})
    net = net.to(cuda).train()
    img = net(_t(g['ws']).to(cuda), _t(g['t']).to(cuda), motion_z=_t(g['motion_z']).to(cuda))
    assert img.dtype == torch.float32 and rel_err(img, _t(g['img_train'])) < 5e-3
    g, meta = load_golden('mixed_precision_d_tiny.npz')
    md = meta['D']
    D = Discriminator(c_dim=0, img_resolution=md['img_resolution'], channel_base=md['channel_base'], channel_max=md['channel_max'],
                      num_frames_per_video=md['num_frames_per_video'], max_num_frames=md['max_num_frames'], concat_res=md['concat_res'],
                      num_frames_div_factor=md['num_frames_div_factor'], mbstd_group_size=md['mbstd_group_size'], mapping_layers=md['mapping_layers'],
                      num_fp16_res=meta['num_fp16_res'], conv_clamp=meta['conv_clamp'])
    D.load_state_dict({k[2:]: _t(g[k]) for k in g.files if k.startswith('d:')})
    D = D.to(cuda).train()
    logits = D(_t(g['d_img']).to(cuda), torch.zeros(2, 0, device=cuda), _t(g['d_t']).to(cuda))['image_logits']
    assert rel_err(logits, _t(g['d_logits'])) < 5e-3
