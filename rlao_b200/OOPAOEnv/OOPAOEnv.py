"""Pyramid environment — mirror of MAIN_CODE/OOPAOEnv/OOPAOEnv.py `class OOPAO` (the environment drl4ao's test_int.sh /
test_po4ao.sh scripts build): the optical train and step of the Shack-Hartmann environment with a Pyramid WFS, a step that
also returns the WFS camera frame (OOPAOEnv.py:485-536: `obs, wfsf, reward, strehl, done, info`), and the science path of
OOPAOEnv.py:118-196,300-333,473-482: an NGS and an off-axis science source, science cameras looking at the PSF of either
(`atm*src*tel*cam`), and the short- / long-exposure PSF products of `render4plot`.

Differences kept on purpose: the Zernike basis is computed (the reference loads a file, manual_m2c.npy, that only fits its
21 x 21 DM); the interactive plot of `render` is not built; the Pyramid's focal-plane camera is not built."""
import math

import torch

from ..Detector import Detector
from ..Source import Source
from .OOPAOEnvRazor import OOPAO as _RazorOOPAO


class OOPAO(_RazorOOPAO):
    returns_frame = True          # step() is a 6-tuple: wrappers must not take the step apart and drop the frame

    def _load_param(self, args):
        param = super()._load_param(args)
        param.setdefault("fov", 1)                   # OOPAOEnv.py:126: Telescope(..., fov=1)
        if not param["fov"]:
            param["fov"] = 1
        return param

    def set_params(self, args=None, wfs_type="pyramid", modal_basis="zernike", gainCL=0.5, **kw):
        """OOPAOEnv.py:93-404."""
        super().set_params(args, wfs_type, modal_basis, gainCL, **kw)
        param, tel = self.param, self.tel
        # :128-143 the guide star (on axis, the WFS looks at it) and the science target
        self.ngs = self.source
        self.src = Source(optBand=param["opticalBand"], magnitude=param["magnitude"], coordinates=[1, 0])
        self.src.coordinates = list(param.get("science_coordinates", [0.4, 0]))                       # :304
        # :172-190 science detectors (full sampling, and binned 4 x 4 with read noise)
        self.cam = Detector(integrationTime=tel.samplingTime, photonNoise=True, readoutNoise=0, QE=1, psf_sampling=2, binning=1,
                            seed=self.wfs.cam.seed + 11)
        self.cam_binned = Detector(integrationTime=tel.samplingTime, photonNoise=True, readoutNoise=2, QE=0.8, psf_sampling=2,
                                   binning=4, seed=self.wfs.cam.seed + 12)
        # :300-309 instrument-path and WFS-path cameras on the PSF at 4 pixels per lambda/D
        self.src_cam = Detector(tel.resolution * 4, seed=self.wfs.cam.seed + 13)
        self.src_cam.psf_sampling, self.src_cam.integrationTime = 4, tel.samplingTime * 1
        self.ngs_cam = Detector(tel.resolution, seed=self.wfs.cam.seed + 14)
        self.ngs_cam.psf_sampling, self.ngs_cam.integrationTime = 4, tel.samplingTime
        if tel.fov < 2 * self.src.coordinates[0]:
            raise ValueError("the science target lies outside the telescope field of view: pass fov >= 2 * its zenith distance "
                             "in the parameter file (the reference builds Telescope(fov=1))")
        # :321-329 first screens of the episode, PSFs of both paths (the telescope ends up pointed at the science target,
        # as in the reference; both sources share band and magnitude, and every layer is at the ground)
        self.atm.generateNewPhaseScreen(seed=10)
        self.tel + self.atm
        self.tel.computePSF(4)
        self.atm * self.ngs * self.tel * self.ngs_cam
        self.atm * self.src * self.tel * self.src_cam
        self.SE_PSF = []
        self.LE_PSFs = []
        self.LE_PSF = torch.log10(self.tel.PSF)                                                       # :339
        self._le_sum, self._le_n = None, 0
        self.modal_CM = self.calib_CL.M
        self.display = False

    def step(self, i, action):
        """OOPAOEnv.py:485-536."""
        obs, reward, strehl, done, info = super().step(i, action)
        frame = self.wfs.cam.frame
        return obs, frame.clone(), reward, strehl, done, info

    def reset_envs(self, env_ids, seed):
        raise NotImplementedError("reset_envs is not available on the Pyramid environment: its science cameras integrate "
                                  "exposures across steps over the whole batch")

    def render4plot(self, current_i):
        """OOPAOEnv.py:473-482: short-exposure PSF of the current residual (log10) and, after the first 15 frames, its
        running mean over the frames rendered so far (the long-exposure product the plots show).  The mean is kept as a
        running sum on the device; `SE_PSF` holds the last frame only (the reference keeps every frame in a list)."""
        self.tel.computePSF(4)
        se = torch.log10(self.tel.PSF)
        if current_i > 15:
            self._le_sum = se.clone() if self._le_sum is None else self._le_sum + se
            self._le_n += 1
            self.SE_PSF = [se]
            self.LE_PSF = self._le_sum / self._le_n
        return self.LE_PSF, se

    def render(self, current_i, mode="rgb_array"):
        raise NotImplementedError("the interactive matplotlib display (OOPAOEnv.py:447-471) is not built; render4plot returns its data")
