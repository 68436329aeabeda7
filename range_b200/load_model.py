"""`load_model` - drop-in for range/load_model.py:16-51 (RANGE / RANGE+ only).

    from range_b200.load_model import load_model
    model = load_model(model_name='RANGE+', pretrained_path=ckpt, device='cuda', db_path=npz, beta=0.5)
    emb = model(locs)            # locs (N,2) float64 (lon, lat) degrees -> np.ndarray float64 (N, 1280)
"""
from argparse import Namespace

from .engine import check_retrieval_precision
from .range import LocationEncoder


def load_model(model_name='RANGE+', pretrained_path=None, device='cuda', **kwargs):
    """Same arguments and errors as the reference:
      * `pretrained_path is None` -> ValueError                         (load_model.py:31-32)
      * names containing 'RANGE' need `db_path`                         (load_model.py:33-35)
      * `beta` defaults to 0.5                                          (load_model.py:37-40)
    Extra, optional keywords (not in the reference): `chunk` (queries per pipelined chunk),
    `db_shard=(rank, world)` + `db_group` (torch.distributed group) for an M-sharded database (model(locs) is then a
    collective call: every rank passes its own queries; `db_merge='peer'|'reduce_scatter'`), `db_cache` (path of the
    prepared device layout: written on first use, validated against source and shard, read afterwards), `host_path`
    ('auto' | 'copy' | 'packed': how the float64 result reaches the host, range.py:_forward_host),
    `out_dtype` (np.float64 like the reference, or np.float32: half the device->host bytes), `retrieval_precision`
    ('fp16', the default: Q.K^T and P'.V on fp16 operands, 11 significant bits of every query, key, weight and value;
    or 'f16x3': every operand split into hi + lo fp16 and three tensor-core products per term, 22 significant bits at
    about three times the retrieval's tensor work and twice the device memory of the database's keys and values -
    for value vectors whose information sits below a large common offset, which fp16 rounds away; the location
    columns are the same in both), `pinned_limit` (bytes), `host_threads`, `devices` (several GPUs of this host for one
    model: an int n = the first n visible GPUs, 'all', or a list of indices / 'cuda:i' strings whose first entry is the
    primary device; None, the default, is `device` alone.  The database is prepared once on the primary and copied to the
    others; every call of 2 x 6144 rows or more splits its rows into contiguous slabs, one per device, each computed by
    the single-device code, and returns what it returns today - device-resident results on the primary.  A duplicate
    entry is a second replica on the same GPU, run after the first: a way to test the path on one GPU, with no speed-up.
    Not with `db_shard`: ValueError).
    """
    if pretrained_path is None:
        raise ValueError("Please provide the pretrained model path.")
    check_retrieval_precision(kwargs.get('retrieval_precision', 'fp16'))
    if 'RANGE' in model_name:
        assert 'db_path' in kwargs, "db_path is required for RANGE model."
        db_path = kwargs.get('db_path')
        beta = kwargs.get('beta') if 'beta' in kwargs else 0.5
    else:
        raise NotImplementedError(f"{model_name}: range_b200 implements the RANGE and RANGE+ encoders only")
    args = Namespace(location_model_name=model_name, pretrained_path=pretrained_path, device=device,
                     range_db=db_path, beta=beta)
    for k in ('chunk', 'db_shard', 'db_group', 'db_cache', 'db_merge', 'tail', 'taper', 'super_batch', 'host_path', 'out_dtype', 'pinned_limit',
              'host_threads', 'retrieval_precision', 'devices'):
        if k in kwargs:
            setattr(args, k, kwargs[k])
    model = LocationEncoder(args)
    model.eval()
    model.to(device)
    return model
