"""Quadratic limb-darkening coefficient grids (Claret-style tables shipped with the reference as
triceratops/data/ldc_tess.csv and ldc_kepler.csv, loaded at marginal_likelihoods.py:21-37) and
the three look-ups the lnZ_* functions make into them.  The per-draw Python loops of the
reference (marginal_likelihoods.py:968-972, :1183-1187, :1913-1924, :2122-2137) are replaced by
vectorised look-ups that return the same values (nearest grid node with numpy.argmin's
first-occurrence tie rule).
"""
from pathlib import Path

import numpy as np
from pandas import read_csv

_DATA_DIR = Path(__file__).parent / "data"


def _first_occurrence_unique(values):
    """Distinct values ordered by where they first appear (argmin's tie order over the table)."""
    _, first = np.unique(values, return_index=True)
    return values[np.sort(first)]


class LdcGrid:
    def __init__(self, fname, col_u1, col_u2):
        df = read_csv(_DATA_DIR / fname)
        self.Zs = np.array(df.Z, dtype=float)
        self.Teffs = np.array(df.Teff, dtype=int)
        self.loggs = np.array(df.logg, dtype=float)
        self.u1s = np.array(df[col_u1], dtype=float)
        self.u2s = np.array(df[col_u2], dtype=float)
        self._nearest_cache = {}
        self._node_tables = {}
        self._uZ = _first_occurrence_unique(self.Zs)
        self._uT = _first_occurrence_unique(self.Teffs)
        self._ug = _first_occurrence_unique(self.loggs)

    def _unique_row(self, sel):
        idx = np.flatnonzero(sel)
        if idx.size != 1:
            # the reference's `.item()` raises the same way when the node is missing/duplicated
            raise ValueError("can only convert an array of size 1 to a Python scalar")
        return idx[0]

    # ---- target star: nearest node in (Z, Teff, logg)         marginal_likelihoods.py:90-98
    def nearest(self, Z, Teff, logg):
        key = (float(Z), float(Teff), float(logg))
        if key not in self._nearest_cache:      # (asked for by every scenario of a target)
            self._nearest_cache[key] = self._nearest(Z, Teff, logg)
        return self._nearest_cache[key]

    def _nearest(self, Z, Teff, logg):
        this_Z = self.Zs[np.argmin(np.abs(self.Zs - Z))]
        this_Teff = self.Teffs[np.argmin(np.abs(self.Teffs - Teff))]
        this_logg = self.loggs[np.argmin(np.abs(self.loggs - logg))]
        r = self._unique_row((self.Zs == this_Z) & (self.Teffs == this_Teff)
                             & (self.loggs == this_logg))
        return self.u1s[r].item(), self.u2s[r].item()

    def node_table(self, Z):
        """(sorted node codes Teff * 100 + round(logg * 10), u1, u2 in that order) of the grid
        slice at the target's Z -- at_Z_rounded()'s look-up table, for csrc/host_blocks.c."""
        key = float(Z)
        if key not in self._node_tables:
            at_Z = self.Zs == self.Zs[np.abs(self.Zs - Z).argmin()]
            T_at, g_at = self.Teffs[at_Z], self.loggs[at_Z]
            code_tab = T_at.astype(np.int64) * 100 + np.round(g_at * 10).astype(np.int64)
            order = np.argsort(code_tab, kind="stable")
            code_sorted = np.ascontiguousarray(code_tab[order])
            if np.any(np.diff(code_sorted) == 0):
                raise ValueError("can only convert an array of size 1 to a Python scalar")
            self._node_tables[key] = (code_sorted,
                                      np.ascontiguousarray(self.u1s[at_Z][order]),
                                      np.ascontiguousarray(self.u2s[at_Z][order]))
        return self._node_tables[key]

    def dense_table(self, Z):
        """(u1, u2) of node_table(Z) as two (27, 4) arrays indexed by ((Teff - 3500) / 250,
        (logg - 3.5) / 0.5), NaN where the grid has no node -- the layout the device sampler's
        kernel reads."""
        codes, u1, u2 = self.node_table(Z)
        it, ig = (codes // 100 - 3500) // 250, (codes % 100 - 35) // 5
        tab1, tab2 = np.full((27, 4), np.nan), np.full((27, 4), np.nan)
        tab1[it, ig], tab2[it, ig] = u1, u2
        return tab1, tab2

    # ---- bound companions: round onto the grid at the target's Z    :945-972 / :1160-1187
    def at_Z_rounded(self, Z, Teffs, loggs, Teff_cap):
        code_sorted, u1_at, u2_at = self.node_table(Z)
        rg = np.round(loggs / 0.5) * 0.5
        rg[rg < 3.5] = 3.5
        rg[rg > 5.0] = 5.0
        rT = np.round(Teffs / 250) * 250
        rT[rT < 3500] = 3500
        rT[rT > Teff_cap] = Teff_cap
        # every draw must hit exactly one node, as with the reference's .item()
        code = rT.astype(np.int64) * 100 + np.round(rg * 10).astype(np.int64)
        pos = np.searchsorted(code_sorted, code)
        pos[pos >= code_sorted.size] = code_sorted.size - 1
        hit = (code_sorted[pos] == code) & (rT == np.round(rT))
        if not np.all(hit):
            raise ValueError("can only convert an array of size 1 to a Python scalar")
        return u1_at[pos], u2_at[pos]

    # ---- background stars: nearest Teff, nearest logg, then nearest tabulated Z   :1913-1924
    def nearest_each(self, Teffs, loggs, Zs):
        Teffs = np.asarray(Teffs, dtype=float)
        loggs = np.asarray(loggs, dtype=float)
        Zs = np.asarray(Zs, dtype=float)
        n = Teffs.size
        tT = self._uT[np.argmin(np.abs(self._uT[None, :] - Teffs[:, None]), axis=1)] if n else \
            np.zeros(0, dtype=int)
        tg = self._ug[np.argmin(np.abs(self._ug[None, :] - loggs[:, None]), axis=1)] if n else \
            np.zeros(0)
        u1 = np.zeros(n)
        u2 = np.zeros(n)
        pair = tT.astype(np.int64) * 100 + np.round(tg * 10).astype(np.int64)
        for c in np.unique(pair):
            who = np.flatnonzero(pair == c)
            sel = np.flatnonzero((self.Teffs == tT[who[0]]) & (self.loggs == tg[who[0]]))
            Zs_here = self.Zs[sel]                      # table order, as these_Zs in the reference
            pick = np.argmin(np.abs(Zs_here[None, :] - Zs[who][:, None]), axis=1)
            for zval in np.unique(Zs_here[pick]):
                rows = sel[Zs_here == zval]
                if rows.size != 1:
                    raise ValueError("can only convert an array of size 1 to a Python scalar")
                m = Zs_here[pick] == zval
                u1[who[m]] = self.u1s[rows[0]]
                u2[who[m]] = self.u2s[rows[0]]
        return u1, u2


_grids = {}


def grid_for(mission):
    """TESS grid for mission == "TESS", Kepler grid otherwise (marginal_likelihoods.py:78-89)."""
    key = "TESS" if mission == "TESS" else "Kepler"
    if key not in _grids:
        _grids[key] = (LdcGrid("ldc_tess.csv", "aLSM", "bLSM") if key == "TESS"
                       else LdcGrid("ldc_kepler.csv", "a", "b"))
    return _grids[key]
