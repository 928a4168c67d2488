"""CPU probe behind the split-precision format of the tcgen05 convolutions (csrc/split_planes.cuh): SuperPoint's conv stack
evaluated with (a) exact fp64 products, (b) two fp16 planes / three products (hi, lo * 2^11), (c) three bf16 planes / six
products (round 1), activations stored as fp32 between layers; reports the dense-score error of each against (a), next to
the error of the plain fp32 reference graph, and the keypoint-set differences.  28 images of the bench stream: fp32
reference 1.0-2.0e-6, fp16x2 1.7-3.8e-6, bf16x3 2.1-3.0e-7, keypoint-set differences 0 everywhere.

  python tools/split_precision_probe.py FIRST_SEED LAST_SEED      (uses oracle/ = test infrastructure; not a product path)
"""
import sys, time, numpy as np, torch, torch.nn.functional as F
sys.path.insert(0, __import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))))
import oracle
from oracle import superpoint as osp
from imcui_b200.utils import synth
torch.set_num_threads(8)
ws = oracle.synthetic_weights("superpoint")
CONF = {"nms_radius": 3, "keypoint_threshold": 0.005, "max_keypoints": -1, "remove_borders": 4}

def split_f16(x):
    hi = x.half().float()
    lo = ((x - hi) * 2048.0).half().float() / 2048.0
    return hi, lo
def split_bf16(x):
    p0 = x.bfloat16().float(); r = x - p0; p1 = r.bfloat16().float(); p2 = (r - p1).bfloat16().float()
    return p0, p1, p2

def conv_mode(x, w, b, mode, pad):
    x = x.float(); w = w.float()
    if mode == 'exact':
        return F.conv2d(x.double(), w.double(), b.double(), padding=pad)
    if mode == 'f16x2':
        xh, xl = split_f16(x); wh, wl = split_f16(w)
        c = lambda a, bb: F.conv2d(a.double(), bb.double(), None, padding=pad)
        return c(xh, wh) + (c(xh, wl) + c(xl, wh)) + b.double().view(1,-1,1,1)
    if mode == 'bf16x3':
        a1,a2,a3 = split_bf16(x); b1,b2,b3 = split_bf16(w)
        c = lambda a, bb: F.conv2d(a.double(), bb.double(), None, padding=pad)
        return c(a1,b1) + (c(a1,b2)+c(a2,b1)) + (c(a1,b3)+c(a2,b2)+c(a3,b1)) + b.double().view(1,-1,1,1)

def sp_dense(img, mode):
    x = img
    def cv(x, name, relu=True, pad=1):
        y = conv_mode(x, ws[name+'.weight'], ws[name+'.bias'], mode, pad).float()   # activations stored as fp32
        return F.relu(y) if relu else y
    x = cv(x,'conv1a'); x = cv(x,'conv1b'); x = F.max_pool2d(x,2)
    x = cv(x,'conv2a'); x = cv(x,'conv2b'); x = F.max_pool2d(x,2)
    x = cv(x,'conv3a'); x = cv(x,'conv3b'); x = F.max_pool2d(x,2)
    x = cv(x,'conv4a'); x = cv(x,'conv4b')
    cPa = cv(x,'convPa'); logits = cv(cPa,'convPb',relu=False,pad=0)
    return osp.dense_scores(logits)

def kset(dense):
    nms = osp.simple_nms(dense, 3)
    k,_ = osp.select_keypoints(nms[0], CONF)
    k = k.numpy().astype(np.int64)
    return set((k[:,1]*100000+k[:,0]).tolist())

for seed in range(int(sys.argv[1]), int(sys.argv[2])):
    a,b,_ = synth.make_pair(seed)
    for im in (a,b):
        img = torch.from_numpy(im.astype(np.float64)/255.0).float()[None,None]
        t=time.time()
        ref32 = osp.dense_scores(osp.detector_logits(ws, osp.encoder(ws, img)))
        ex = sp_dense(img,'exact'); f16 = sp_dense(img,'f16x2'); b3 = sp_dense(img,'bf16x3')
        k32, kex, kf, kb = kset(ref32), kset(ex), kset(f16), kset(b3)
        print(f"seed {seed}: n={len(k32)} | err vs exact: fp32ref {float((ref32-ex).abs().max()):.2e} f16x2 {float((f16-ex).abs().max()):.2e} bf16x3 {float((b3-ex).abs().max()):.2e}"
              f" | kpt-set diff vs fp32ref: exact {len(k32^kex)} f16x2 {len(k32^kf)} bf16x3 {len(k32^kb)} | f16x2 vs exact {len(kex^kf)} ({time.time()-t:.0f}s)", flush=True)
