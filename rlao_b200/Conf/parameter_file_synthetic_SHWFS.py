"""Parameter file for the synthetic 8 m Shack-Hartmann systems of BASELINE.json / SURVEY.md section 8(d), in
the format of the reference's parameter files (MAIN_CODE/Conf/parameter_fileRAZOR_SHWFS.py,
parameterFile_oopao_parser.py): `initializeParameterFile(args) -> param` dict.

`args` carries the atmosphere (r0, L0, fractionalR0, windSpeed, windDirection, altitude), nLoop and gainCL as
in the reference's YAML files, plus optional nSubaperture (default 20), nPixelPerSubap (6), diameter (8),
magnitude (8), opticalBand ('I'), nZernike (50), noise (False), is_geometric (False).
"""
import numpy as np

# drl4ao's 5-layer profile (MAIN_CODE/Conf/papyrus_config.yaml:13-15); shorter atmospheres use renormalised prefixes
PROFILE_FRACTIONAL_R0 = [0.45, 0.1, 0.1, 0.25, 0.1]
PROFILE_WIND_SPEED = [10, 12, 11, 15, 20]
PROFILE_WIND_DIRECTION = [0, 72, 144, 216, 288]


def layer_profile(n_layers):
    f = np.asarray(PROFILE_FRACTIONAL_R0[:n_layers], dtype=float)
    return dict(fractionalR0=list(f / f.sum()), windSpeed=PROFILE_WIND_SPEED[:n_layers],
                windDirection=PROFILE_WIND_DIRECTION[:n_layers], altitude=[0] * n_layers)


def initializeParameterFile(args):
    g = lambda k, d: getattr(args, k, d)
    param = dict()
    # atmosphere
    param["r0"], param["L0"] = g("r0", 0.13), g("L0", 25)
    param["fractionalR0"] = g("fractionalR0", [1])
    param["windSpeed"], param["windDirection"] = g("windSpeed", [10]), g("windDirection", [0])
    param["altitude"] = g("altitude", [0] * len(param["fractionalR0"]))
    # telescope
    param["diameter"] = g("diameter", 8)
    param["nSubaperture"] = g("nSubaperture", 20)
    param["nPixelPerSubap"] = g("nPixelPerSubap", 6)
    param["resolution"] = param["nSubaperture"] * param["nPixelPerSubap"]
    param["sizeSubaperture"] = param["diameter"] / param["nSubaperture"]
    param["samplingTime"] = g("samplingTime", 1 / 500)
    param["centralObstruction"] = 0
    param["fov"] = g("fov", 0)                                       # arcsec; the papyrus environment asks for 1 (OOPAOEnv.py:126)
    # guide star
    param["magnitude"], param["opticalBand"] = g("magnitude", 8), g("opticalBand", "I")
    # deformable mirror: Fried geometry, DeformableMirror(nSubap=nSubaperture) (OOPAO/DeformableMirror.py:286-305)
    param["nActuator"] = param["nSubaperture"] + 1
    param["mechanicalCoupling"] = 0.35
    param["isM4"] = False
    param["dm_geometry"] = "cartesian"
    for k in ("shiftX", "shiftY", "rotationAngle", "anamorphosisAngle", "radialScaling", "tangentialScaling"):
        param[k] = 0
    # wavefront sensor
    param["lightRatio"] = 0.5
    param["threshold_cog"] = 0.01
    param["shannon_sampling"] = False
    param["is_geometric"] = bool(g("is_geometric", False))           # geometric sensor (DESIGN.md section 2)
    noisy = bool(g("noise", False))
    param["cam_photonNoise"] = noisy
    param["cam_readoutNoise"] = 14 if noisy else 0                   # OOPAOEnvRazor.py:332-333
    if noisy:                                                        # OOPAOEnvRazor.py:243-250
        param.update(cam_sensor="CMOS", cam_FWC=10000, cam_bits=10, cam_QE=0.56, cam_darkCurrent=5)
    # Pyramid WFS (only read when the environment is built with wfs_type="pyramid"; Conf/parameterFile_oopao_parser.py:64-68)
    param["modulation"] = g("modulation", 3)
    param["n_pix_separation"] = 4
    param["lightThreshold"] = 0.1
    param["postProcessing"] = g("postProcessing", "slopesMaps_incidence_flux")
    # control
    param["nZernike"] = g("nZernike", 50)
    param["nMeasurements"] = 25
    param["nLoop"] = g("nLoop", 1000)
    param["gainCL"] = g("gainCL", 0.5)
    param["name"] = "SYNTH_8m_SH_%dx%d" % (param["nSubaperture"], param["nSubaperture"])
    return param
