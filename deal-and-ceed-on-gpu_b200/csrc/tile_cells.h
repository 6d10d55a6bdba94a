// Cells per tile (= cells per CTA pass) of the cell kernels, per degree.
#pragma once
namespace bp5 {
// cells per tile for each degree: fills the CTA's warps ((p+1)^2 threads per
// cell) while keeping >= 2-4 CTAs resident per SM.
template <int P> struct TileCells;
template <> struct TileCells<1> { static constexpr int value = 32; };
template <> struct TileCells<2> { static constexpr int value = 14; };
template <> struct TileCells<3> { static constexpr int value = 8; };
template <> struct TileCells<4> { static constexpr int value = 5; };
template <> struct TileCells<5> { static constexpr int value = 3; };
template <> struct TileCells<6> { static constexpr int value = 3; };
template <> struct TileCells<7> { static constexpr int value = 2; };
template <> struct TileCells<8> { static constexpr int value = 1; };

// the on-the-fly-geometry kernel keeps 12-15 work arrays per cell in shared memory: fewer cells per tile
// (round 2, deformed mesh, 27 M DoFs, vmult GDoF/s: p=4 5/3/2 cells 22.7/22.3/23.5; p=5 3/2/1 cells 14.2/18.2/16.0;
//  p=6 3/2/1 cells 13.0/18.2/20.9)
template <int P> struct OtfTileCells { static constexpr int value = TileCells<P>::value; };
template <> struct OtfTileCells<4> { static constexpr int value = 2; };
template <> struct OtfTileCells<5> { static constexpr int value = 2; };
template <> struct OtfTileCells<6> { static constexpr int value = 1; };
template <> struct OtfTileCells<7> { static constexpr int value = 1; };

// the general on-the-fly kernel (apply_otfg.cuh) stages the Jacobian of the tile's cells next to three work arrays
// (round 2, deformed mesh, 11-16 M DoFs, vmult GDoF/s Gauss / collocation + Helmholtz, profiles/r2_otf_general_tuning.log:
//  p=4 1/2/3 cells 16.3/15.7/15.7 and 18.8/17.8/17.6; p=5 1/2/3 cells 12.5/15.2/15.9 and 16.3/16.9/18.5;
//  p=6 1/2/3 cells 17.8/17.3/16.2 and 20.3/19.8/18.7)
template <int P> struct OtfgTileCells { static constexpr int value = OtfTileCells<P>::value; };
template <> struct OtfgTileCells<4> { static constexpr int value = 1; };
template <> struct OtfgTileCells<5> { static constexpr int value = 3; };
}  // namespace bp5
