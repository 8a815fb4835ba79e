import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from oct_segmentation_b200.model import OCTSegmentationModel
from oct_segmentation_b200.engine.network import CompiledNet
from oracle import synth
cfg = synth.MODEL_CONFIGS['FC_LC']
torch.manual_seed(0)
m = OCTSegmentationModel(arch=cfg['architecture'], encoder_name=cfg['encoder'], model_name=cfg['model_name'], in_channels=3, classes=cfg['classes'], encoder_weights=None)
def timeit(net):
    for _ in range(3): net.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): net.run()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 10
net = CompiledNet(m.model, 16, 896, 896, 'cuda', 'u8', 'u8_nchw', use_graph=True)
print('full graph', timeit(net))
b = net.builder
kinds = {'se': lambda n: n.endswith('.se'), 'dw': lambda n: 'depthwise' in n, 'expand': lambda n: 'expand' in n, 'project': lambda n: n.endswith('_project_conv'), 'head': lambda n: 'head' in n, 'stem': lambda n: 'stem' in n, 'decoder': lambda n: n.startswith('decoder')}
ops0 = list(b.ops)
for kname, pred in kinds.items():
    b.ops = [op for op, n in zip(ops0, b.op_names) if not pred(n)]
    net.graph = None
    print('without', kname, timeit(net))
