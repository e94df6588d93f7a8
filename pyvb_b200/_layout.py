"""Stat-buffer / globals layout -- mirrors pyvb::StatLayout (csrc/common.cuh) and include/pyvb_b200.h."""

NSCAL = 16
SC_SXX, SC_SUMV, SC_NE, SC_QLDZ, SC_LOGDETZ, SC_LATQLD, SC_NLAT, SC_PNMISS, SC_PLNV, SC_NROWS = range(10)

GL_QA, GL_QB, GL_TAU, GL_ELBO, GL_ELBO_W, GL_ELBO_MU, GL_ELBO_Z, GL_ELBO_X, GL_ELBO_BETA, GL_ELBO_ALPHA = range(10)
GL_RESID2 = 10
GL_NONPD = 11
GL_I8BAD = 12
GL_LNS = 13         # weighted data: 1/2 sum ln s_nd over the observed entries of positive weight (all rows, all ranks)
GL_I8FALL = 14
GL_ALPHA = 16
GL_ALQB = 80
GL_LEN = 144

# per-dimension noise block (noise="diagonal"): row k of the (ND_LEN, D) array
ND_TAU, ND_QB, ND_QA, ND_PSI_QA, ND_LGAM_QA, ND_A0, ND_B0, ND_LGAM_A0, ND_SXX, ND_R, ND_EX, ND_EB = range(12)
ND_LEN = 12

OP_MU, OP_BETA, OP_ALPHA, OP_ELBO = 1, 2, 4, 8
ALGO_AUTO, ALGO_GENERIC, ALGO_DMMA, ALGO_DMMA_K1, ALGO_F32 = 0, 1, 2, 3, 4
QMAX = 64


class StatLayout(object):
    def __init__(self, D, q):
        self.D, self.q = D, q
        self.P = P = q * (q + 1) // 2
        self.t1 = 0
        self.bst = self.t1 + D * P
        self.ast = self.bst + D * q
        self.cnt = self.ast + D * q
        self.colx = self.cnt + D
        self.S = self.colx + D
        self.zsum = self.S + P
        self.scal = self.zsum + q
        self.len = self.scal + NSCAL

    def views(self, stats):
        """Named views of a flat stats tensor/array."""
        D, q, P = self.D, self.q, self.P
        return {
            "T1": stats[self.t1:self.bst].reshape(D, P),
            "Bst": stats[self.bst:self.ast].reshape(D, q),
            "Ast": stats[self.ast:self.cnt].reshape(D, q),
            "cnt": stats[self.cnt:self.colx],
            "colx": stats[self.colx:self.S],
            "S": stats[self.S:self.zsum],
            "zsum": stats[self.zsum:self.scal],
            "scal": stats[self.scal:self.len],
        }
