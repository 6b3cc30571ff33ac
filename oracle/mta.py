"""Oracle: MTA (MeanShift for Test-time Augmentation) mode seeking, fp32 on CPU.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py; parity unpinned).

Restates test.py:1310-1318 (gaussian_kernel, cdist), test.py:1391-1461 (solve_mta, returns the
mode [1,512]) and ood.py:751-820 (same solver, returns 100 * mode @ text).

Two deliberate, documented deviations from the reference text (SURVEY.md Appendix A.5 / C-1):
  * cdist clamps D^2 >= 0 before sqrt.  The reference takes sqrt of x.x - 2x.x + x.x, which for
    unit rows rounds to +-1e-7 on the diagonal and yields NaN for about half of the rows; where the
    NaN sorts is backend-dependent.  Clamping makes self-distance 0 sort first, as the reference's
    comment "exclude the distance to the point itself" (test.py:1406) intends.
  * k = max(int(0.3 * (V-1)), 1).  With V=2 the reference slices an empty range and averages
    nothing (NaN).
"""
import torch

LAMBDA_Y = 0.2      # test.py:1395
LAMBDA_Q = 4.0      # test.py:1396
MAX_ITER = 5        # test.py:1397
TEMPERATURE = 1.0   # test.py:1398
TH = 1e-6           # test.py:1421
K_FRAC = 0.3        # test.py:1405


def gaussian_kernel(mu, bandwidth, datapoints):
    # test.py:1310-1313
    dist = torch.norm(datapoints - mu, dim=-1, p=2)
    return torch.exp(-dist ** 2 / (2 * bandwidth ** 2))


def cdist(x1, x2):
    # test.py:1314-1318 (+ clamp, see module docstring)
    x1_square = torch.sum(x1 ** 2, dim=1, keepdim=True)
    x2_square = torch.sum(x2 ** 2, dim=1, keepdim=True)
    d2 = x1_square - 2 * torch.matmul(x1, x2.t()) + x2_square.t()
    return torch.sqrt(torch.clamp(d2, min=0.0))


@torch.no_grad()
def solve_mta(image_features, text_features, return_state=False, *, dtype=torch.float32, lambda_y=LAMBDA_Y,
              lambda_q=LAMBDA_Q, th=TH, temperature=TEMPERATURE, k_frac=K_FRAC, max_iter=MAX_ITER):
    """image_features [V,512] unit rows (row 0 = un-augmented view), text_features [512,C].
    Returns the unit mode [1,512] (test.py:1461).

    `dtype` is the arithmetic precision (float64 gives the reference the kernels' fp32 rounding is measured against);
    the keywords are the solver's constants (jcb_mta_params), defaulting to the reference's."""
    x = image_features.to(dtype)
    t = text_features.to(dtype)
    logits = x @ t * 100                                           # :1393
    V = x.shape[0]

    dist = cdist(x, x)                                             # :1403
    sorted_dist, _ = torch.sort(dist, dim=1)                       # :1404 jt.argsort -> (idx, values), ascending
    k = max(int(k_frac * (V - 1)), 1)                              # :1405 (+ max, see docstring)
    selected = sorted_dist[:, 1:k + 1] ** 2                        # :1406
    bandwidth = torch.sqrt(0.5 * selected.mean(dim=1))             # :1407-1408

    p = torch.softmax(logits / temperature, dim=1)
    affinity = p @ p.t()                                           # :1411

    y = torch.ones(V, dtype=dtype) / V                             # :1414
    mode = x[0]                                                    # :1417-1418
    it = 0
    while True:                                                    # :1424
        density = gaussian_kernel(mode, bandwidth, x)              # :1426
        i = 0
        while True:                                                # :1430
            i += 1
            old_y = y
            weighted_affinity = affinity * y.unsqueeze(0)          # :1433
            y = torch.softmax(1 / lambda_y * (density + lambda_q * weighted_affinity.sum(dim=1)), dim=-1)  # :1434
            if torch.norm(old_y - y) < th or i >= max_iter:        # :1436
                break
        i = 0
        while True:                                                # :1443
            i += 1
            old_mode = mode
            density = gaussian_kernel(mode, bandwidth, x)          # :1446
            w = density * y                                        # :1447
            mode = (w.unsqueeze(1) * x).sum(dim=0) / w.sum()       # :1448
            mode = mode / mode.norm(p=2, dim=-1)                   # :1449
            if torch.norm(old_mode - mode) < th or i >= max_iter:  # :1452
                break
        it += 1                                                    # :1455
        if it >= max_iter:
            break
    if return_state:
        return mode.unsqueeze(0), {"bandwidth": bandwidth, "affinity": affinity, "y": y, "logits": logits}
    return mode.unsqueeze(0)                                       # :1461


@torch.no_grad()
def solve_mta_logits(image_features, text_features):
    """ood.py:751-820 variant: returns 100 * mode @ text  ([1,C])."""
    mode = solve_mta(image_features, text_features)
    return mode @ text_features.to(torch.float32) * 100            # ood.py:819
