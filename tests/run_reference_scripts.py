#!/usr/bin/env python
"""Drive the reference's OWN scripts (unmodified byte copies in baseline/_ref: test.py:model_test, verify.py:model_validation) and
the train.py:69-75 loop body over the drop-in shim on the GPU, in a fresh interpreter:

    PYTHONPATH=<repo>/shim:<repo>:<repo>/baseline/_ref  python tests/run_reference_scripts.py scripts train
    PYTHONPATH=<repo>/shim:<repo>  python tests/run_reference_scripts.py train        (needs no reference files)

sys.path order is the one INTEGRATION.md section 1 prescribes, so the scripts' own `from models.user_model import UserModel`
(test.py:7, verify.py:5, train.py:9) binds to the B200 implementation while `configs.run_config`, `tool.*`, `test`, `verify`
are the reference's files.  Prints one JSON object; tests/test_gpu_reference_scripts.py compares it with the golden fixtures
(outputs of the same reference functions run with the reference's own modules on the CPU)."""
import json
import os
import queue
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.modules.setdefault('zstandard', types.ModuleType('zstandard'))     # tool/process_data.py:16 imports it; never called here

from models.user_model import UserModel  # shim -> news_recommendation_model_b200
import news_recommendation_model_b200 as nrm
from fixtures import case_batch, load_case, load_weights, stored


def scripts(out, dev):
    import test as ref_test                 # baseline/_ref/test.py      (not the stdlib package: the reference root precedes it)
    import verify as ref_verify             # baseline/_ref/verify.py
    ref_root = os.path.join(os.path.dirname(HERE), 'baseline', '_ref')
    assert os.path.abspath(ref_test.__file__).startswith(ref_root), ref_test.__file__
    assert os.path.abspath(ref_verify.__file__).startswith(ref_root), ref_verify.__file__
    assert ref_test.UserModel is nrm.UserModel and ref_verify.UserModel is nrm.UserModel
    out.update({'test_py': os.path.abspath(ref_test.__file__), 'verify_py': os.path.abspath(ref_verify.__file__)})

    # ---- test.py:31-74 and verify.py:19-43 on the ragged-candidate golden case, ensemble of the two shipped checkpoints
    case = load_case('case_eval_b8')
    b = case_batch(case)
    B = int(case['meta'][0])
    models = []
    for name in ('train', 'validation'):
        path = os.path.join(ref_root, 'ckpt', f'ckpt_ebnerd_large_{name}_final.pth')
        m = UserModel()
        m.load_state_dict(torch.load(path, map_location=dev), strict=False)          # test.py:159-160
        models.append(m)
    records = [[b.impression_id[i].numpy(), b.user_id[i].numpy(), b.x_history[i].numpy(), b.x_target[i].numpy(),
                b.x_global[i].numpy(), b.label[i].numpy(), b.label_id[i].numpy(), b.empty_num[i].numpy()] for i in range(B)]
    q, ids = ref_test.model_test(models, records, dev, queue.Queue(), [], batch_size=4)
    recs = []
    while not q.empty():
        recs.append(q.get())
    out['scores'], out['ids'] = [np.asarray(r[2]).tolist() for r in recs], ids
    q2, lines = queue.Queue(), {}
    for r in recs:
        q2.put(r)
    ref_test.get_string_of_prediction(q2, lines, queue.Queue())                      # test.py:118-132, unmodified
    out['submission_lines'] = [lines[i] for i in ids]
    auc, tpr = ref_verify.model_validation(models, records, dev, batch_size=4)
    out['auc'], out['tpr'] = float(auc), float(tpr)


def train(out, dev):
    # ---- the train.py:46-48, 69-75 loop body on the golden training case (torch.optim.Adam, as the script has it)
    tc = load_case('case_train_b16')
    tb = case_batch(tc)
    user_num = int(tc['meta'][3])
    model = UserModel(user_num)
    model.load_state_dict(load_weights('train'), strict=False)
    with torch.no_grad():
        model.delta.copy_(torch.from_numpy(tc['delta0']))
    model.to(dev)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    model.train()
    o = model(tb.x_history.to(dev), tb.x_target.to(dev), tb.x_global.to(dev))
    loss = model.loss(tb.user_id.to(dev), o, tb.label.to(dev))
    loss.backward()
    optimizer.step()
    optimizer.zero_grad()
    out['train_loss'] = float(loss.item())
    out['train_logits'] = o.detach().cpu().numpy().tolist()
    sd = model.state_dict()
    before = dict(load_weights('train'))
    before['delta'] = torch.from_numpy(tc['delta0'])
    out['after_err'] = {}
    for k in sd:
        if ('after/' + k) not in tc.files:
            continue
        ref = tc['after/' + k].astype(np.float64)
        err = float(np.abs(stored(tc, k, sd[k].detach().cpu().double().numpy()) - ref).max())
        moved = float(np.abs(ref - stored(tc, k, before[k].double().numpy())).max()) if k in before else 0.0
        out['after_err'][k] = [err, moved]
    model_ckpt = model.state_dict()
    model_ckpt.pop('delta')                                                         # train.py:95-96
    out['ckpt_keys'] = list(model_ckpt.keys())


def main():
    assert UserModel is nrm.UserModel
    dev = torch.device('cuda:0')
    out = {}
    for part in sys.argv[1:]:
        {'scripts': scripts, 'train': train}[part](out, dev)
    print('RESULT ' + json.dumps(out))


if __name__ == '__main__':
    main()
