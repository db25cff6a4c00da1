import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'multimodal-baselines_b200')); sys.path.insert(0, os.path.join(ROOT, 'tools'))
import torch, bench_mmb as bm, models, simplesif, utils
name = os.environ.get('SHAPE', 'mosi')
dev = torch.device('cuda')
S = bm.synth(name, dev)
Ad, Vd = S['dims']
torch.manual_seed(0)
model = models.AudioVisualGeneratorMultimodal(bm.D, Ad, Vd, norm='layer_norm', frozen_weights=False).to(dev)
word_fn = simplesif.make_word_log_prob_fn({'word_sim_metric': 'angular'}, None, S['table'], a=bm.A_SIF)
mk = {'text': S['text_m'], 'covarep': S['aud_m'], 'facet': S['vis_m']}
ds = utils.MMData(S['text'], S['aud'], S['vis'], mk, S['text_w'], dev)
lat = S['latents'].clone().requires_grad_(True)
opt = torch.optim.SGD([lat] + list(model.parameters()), lr=1e-7)
st = simplesif.GraphedStep({'dataset': 'mosi', 'unimodal': False}, model, lat, ds, opt, word_fn, dev)
perm = torch.randperm(S['N']).to(dev)
for i in range(4):
    st(perm[i * 64:(i + 1) * 64])
torch.cuda.synchronize()
print('done')
