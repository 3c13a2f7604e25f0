"""CPU statement of the tile schedules of the persistent convolution kernels.

Both kernels cut the (n, H, W) output into tiles of 16 rows x 8 columns, numbered patch-major, then row-major.
  conv_pair_kernel (csrc/conv_pair.cu, fill_tiles + launch_pair): a CTA pair takes two consecutive tiles (2 pt, 2 pt + 1);
      npairs = min(ceil(tiles / 2), sms / 2) pairs walk the pair-tile list with a stride of npairs.  With an odd tile count
      the rank-1 CTA of the last pair-tile decodes tile number `tiles`, whose batch index is n: a phantom tile.
  conv_tail_swapped_kernel (csrc/conv_tail.cu, tail16_common + launch_tail): min(tiles, sms) CTAs walk the tile list with a
      stride of gridDim.x.  The stitching form leaves out the tile columns that lie inside the patch border.
What a CTA carries from one tile to the next (stage rings and their phases, the two TMEM accumulators, the walk of the
tile list, next-tile prefetches) only runs from a CTA's second tile on, and both accumulators are reused from the third.
"""
from collections import namedtuple

PATCH = (5, 128, 128)          # 640 tiles: 320 pair-tiles, 4-5 per pair, 320 % 74 = 24; 4-5 per tail CTA
RAGGED = (7, 104, 88)          # 7 x 7 x 11 = 539 tiles (odd), the last tile row half outside the patch
BATCH128 = (128, 32, 32)       # DSen2's training batch (supres_train.py): 1024 tiles, 7 per pair
BATCH64 = (64, 32, 32)         # the benchmark's batch-64 VDSen2 training step: 512 tiles, 4 per pair or tail CTA

# the geometries whose cases exist to run the loop-carried paths: at least 3 tiles on the busiest pair or CTA and a
# partial last round on a 148-SM B200; odd: the tile count is odd too
LOOPED = {PATCH: dict(odd=False), RAGGED: dict(odd=True), BATCH128: dict(odd=False), BATCH64: dict(odd=False)}

Schedule = namedtuple('Schedule', 'kernel shape tiles workers busiest partial tx0 tiles_x')


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


def pair_schedule(n, H, W, sms=None):
    """conv_pair_kernel: workers = CTA pairs, busiest = pair-tiles on the busiest pair."""
    sms = sm_count() if sms is None else sms
    tiles_x = _cdiv(W, 8)
    tiles = n * tiles_x * _cdiv(H, 16)
    pair_tiles = (tiles + 1) // 2
    pairs = min(pair_tiles, sms // 2)
    return Schedule('pair', (n, H, W), tiles, pairs, _cdiv(pair_tiles, pairs), pair_tiles % pairs != 0, 0, tiles_x)


def tail_schedule(n, H, W, border=None, sms=None):
    """conv_tail_swapped_kernel: workers = CTAs, busiest = tiles on the busiest CTA.  border: the stitching form."""
    sms = sm_count() if sms is None else sms
    tiles_x, tx0 = _cdiv(W, 8), 0
    if border is not None:
        tx0 = border // 8
        tiles_x = (W - border - 1) // 8 - tx0 + 1
    tiles = n * tiles_x * _cdiv(H, 16)
    ctas = min(tiles, sms)
    return Schedule('tail', (n, H, W), tiles, ctas, _cdiv(tiles, ctas), tiles % ctas != 0, tx0, tiles_x)


def report(s, label, err):
    unit = 'pair-tiles per pair' if s.kernel == 'pair' else 'tiles per CTA'
    print('%s (n, H, W) = %s: %d tiles%s over %d %s, busiest %d %s, last round %s%s; worst error %.3e' % (
        label, s.shape, s.tiles, ' (odd)' if s.tiles % 2 else '', s.workers, 'pairs' if s.kernel == 'pair' else 'CTAs',
        s.busiest, unit, 'partial' if s.partial else 'full', '' if s.tx0 == 0 else ', tile columns from %d' % s.tx0, err))


def check(s, label, err):
    """Print the schedule and the case's worst error; a case at one of the LOOPED geometries must reach what it is for."""
    report(s, label, err)
    claim = LOOPED.get(s.shape)
    if claim is None:
        return
    assert s.busiest >= 3, '%s: only %d tiles on the busiest %s' % (label, s.busiest, s.kernel)
    assert s.partial, '%s: the last round is full' % label
    if claim['odd']:
        assert s.tiles % 2 == 1, '%s: %d tiles, not odd' % (label, s.tiles)
