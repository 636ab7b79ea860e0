"""Device-side reference of the observation history (get_obs, flexibility_provision_env.py:370-403, quirk Q7) for
batches up to 2^20 envs, and the NaN-poisoned profile table of the row-clamp tests.

The reference keeps what every push wrote: `hist[H, N, na, 6]` fp64 on the device, push k of an env (0-based since its
last reset) in slot k mod H, and a push count per env.  Every push source is one rule -- the window of an env is its last
H pushes since its last reset, oldest first, zero-padded in front:
  * a step push (step(..., return_obs=True / "ring"): every stepped env);
  * a reset's own push (reset(return_obs="ring"): the reset envs; reset(return_obs=True): every env, through get_obs());
  * a generic pushing get_obs() (every env).
The pushed values are the mirror's current_obs() (fp64), so every device result is a copy of them: fp64, or the fp64
value rounded once to fp32.  From that state the reference produces, in chunks of CHUNK envs, the dense windows, the
expected env-minor ring (flex_kernels.cu, k_obsr_*), the live entries of the fp64 history ring and the push-count word."""
import numpy as np
import torch

CHUNK = 65536
SLOT = 32                                            # FP_HIST_SLOT: doubles per history-ring slot (<= 30 used)


class ObsRef:
    def __init__(self, n, na, H, device):
        self.n, self.na, self.H, self.device = n, na, H, torch.device(device)
        self.hist = torch.zeros(H, n, na, 6, dtype=torch.float64, device=self.device)
        self.cnt = torch.zeros(n, dtype=torch.int64, device=self.device)

    def _mask(self, mask):
        if mask is None:
            return None
        return torch.as_tensor(np.asarray(mask)).to(self.device).bool()

    def reset(self, mask=None):
        """The envs of `mask` (None: all) restart their history: zero padding in front again."""
        m = self._mask(mask)
        if m is None:
            self.cnt.zero_()
        else:
            self.cnt[m] = 0

    def push(self, cur, mask=None):
        """One push of `cur` [N, na, 6] (fp64, numpy or tensor) for the envs of `mask` (None: all)."""
        cur = torch.as_tensor(cur).to(self.device, torch.float64)
        m = self._mask(mask)
        idx = torch.arange(self.n, device=self.device) if m is None else torch.nonzero(m).view(-1)
        self.hist[self.cnt[idx] % self.H, idx] = cur[idx]
        self.cnt[idx] += 1

    def round_f32(self):
        """Every stored entry rounded to fp32 and widened: the fp64 history restored from the fp32 ring (k_hist_from_ring)."""
        self.hist.copy_(self.hist.float().double())

    def chunks(self):
        return [(lo, min(lo + CHUNK, self.n)) for lo in range(0, self.n, CHUNK)]

    def window(self, lo, hi, cur=None):
        """Dense windows [hi - lo, na, 6 H] fp64 of envs lo .. hi-1.  With `cur` ([N, na, 6]): the window a push of cur
        would return, without pushing it (get_obs(push=False))."""
        H = self.H
        cnt = self.cnt[lo:hi] + (0 if cur is None else 1)
        s = torch.arange(H, device=self.device)
        k = cnt[:, None] - H + s[None, :]                                 # push index of window entry s
        e = torch.arange(lo, hi, device=self.device)[:, None].expand(-1, H)
        w = self.hist[k.clamp(min=0) % H, e]                              # [n, H, na, 6]
        if cur is not None:
            c = torch.as_tensor(cur).to(self.device, torch.float64)[lo:hi]
            w = torch.where((k == cnt[:, None] - 1)[:, :, None, None], c[:, None], w)
        w = torch.where((k >= 0)[:, :, None, None], w, torch.zeros((), dtype=w.dtype, device=w.device))
        return w.permute(0, 2, 1, 3).reshape(hi - lo, self.na, H * 6)

    def ring(self, slot, lo, hi):
        """Expected env-minor ring columns lo .. hi-1, [H, na, 6, hi - lo] fp32: window entry s in slot (slot - H + 1 + s)
        mod H.  The pad columns n .. n_pad-1 of the whole ring are zero (checked by the caller)."""
        H = self.H
        w = self.window(lo, hi).view(hi - lo, self.na, H, 6).permute(2, 1, 3, 0)     # [H(s), na, 6, n]
        j = torch.arange(H, device=self.device)
        s = (j - slot - 1) % H                                            # window entry held by ring slot j
        return w[s].float()

    def history(self, lo, hi):
        """Expected fp64 history ring of envs lo .. hi-1 as the device holds it ([n, H * 32]) and the mask of its live
        entries: push k in slot k mod H, pad entries 30-31 of a slot zero, only k >= max(0, cnt - H)."""
        H, na = self.H, self.na
        out = torch.zeros(hi - lo, H, SLOT, dtype=torch.float64, device=self.device)
        out[:, :, :6 * na] = self.hist[:, lo:hi].permute(1, 0, 2, 3).reshape(hi - lo, H, 6 * na)
        cnt = self.cnt[lo:hi]
        sl = torch.arange(H, device=self.device)
        live = (sl[None, :] < cnt[:, None]) | (cnt[:, None] >= H)         # slot k mod H holds a push k >= cnt - H
        return out.view(hi - lo, H * SLOT), live.repeat_interleave(SLOT, dim=1)

    def count_word(self):
        """The push count as the record's history word holds it (low 32 bits)."""
        return self.cnt


def clamp_tables(profiles, s0):
    """Profiles cut to s0 + 131 rows, and the same table with every row after s0 + episode_limit + history (= s0 + 120, the
    last row of the slice of an episode that starts at s0) set to NaN.  The poisoned rows lie inside the table, so a
    reader that does not clamp reads NaN rather than past the end."""
    from flexgpu.profiles import Profiles
    T = s0 + 131
    P, Q, PV, price = (np.array(a[:T]) for a in (profiles.P, profiles.Q, profiles.PV, profiles.price))
    finite = Profiles(P.copy(), Q.copy(), PV.copy(), price.copy())
    for a in (P, Q, PV, price):
        a[s0 + 121:] = np.nan
    return finite, Profiles(P, Q, PV, price)
