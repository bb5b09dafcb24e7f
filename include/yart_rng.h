/* yart_rng.h -- the counter-based random-number CONTRACT shared by the CUDA path and the CPU
 * oracle (constants only; each side implements Philox4x32-10 itself).
 *
 * The reference draws from rand::thread_rng() (ChaCha12, OS-seeded, unreproducible; SURVEY.md
 * 7.3).  Here every draw site of the reference gets a fixed address in a Philox4x32-10 stream
 *
 *     key     = (seed & 0xffffffff, seed >> 32)
 *     counter = (pixel = y*width + x, sample, bounce, slot)
 *
 * One Philox call yields four u32 r0..r3 and from them two uniform doubles in [0,1):
 *     u0 = ((r0 | r1<<32) >> 11) * 2^-53        u1 = ((r2 | r3<<32) >> 11) * 2^-53
 * (53-bit resolution like rand's `gen::<f64>()`).  gen_range(a..b) is a + (b-a)*u.
 *
 * bounce 0 is the camera sample; bounce k>=1 is the k-th `world.hit` of the path
 * (ray_reflectance depth = max_depth-k+1, main.rs:537-588).
 */
#ifndef YART_RNG_H
#define YART_RNG_H

/* ---- bounce 0: camera sample (main.rs:690-698, camera.rs:82-94) ---- */
#define YART_SLOT_CAM_JITTER 0u    /* u0 = pixel jitter x (main.rs:693), u1 = jitter y (:695)       */
#define YART_SLOT_CAM_WL_TIME 1u   /* u0 = wavelength (color.rs:20-23), u1 = shutter time (cam:91)  */
#define YART_SLOT_CAM_LENS 2u      /* + i: i-th rejection iteration of random_in_unit_disk
                                      (camera.rs:25-33): p = (2*u0-1, 2*u1-1)                       */
#define YART_MAX_REJECT 64u        /* both sides give up after this many iterations and use 0       */

/* ---- bounce k >= 1 ---- */
#define YART_SLOT_MIX 0u           /* u0 = MixurePDF pick (<0.5 -> lights, pdf.rs:91-97),
                                      u1 = light index pick floor(u1*(len-1)) (hittable.rs:119)     */
#define YART_SLOT_DIR 1u           /* u0 = r1, u1 = r2 of random_cosine_direction (pdf.rs:15-25),
                                      random_to_sphere (sphere.rs:11-21) or the XZRect point
                                      (aarect.rs:164-171: u0 -> x, u1 -> z)                          */
#define YART_SLOT_DIELECTRIC 2u    /* u0 = reflect-vs-refract draw (material.rs:274)                */
#define YART_SLOT_RR 3u            /* u0 = Russian-roulette survival draw (only with YART_FLAG_RUSSIAN_ROULETTE;
                                      the reference has none)                                      */
#define YART_SLOT_NEE_PICK 4u      /* u0 = which light the next-event sample aims at, floor(u0*len)
                                      (only with YART_FLAG_NEXT_EVENT; the reference has none)      */
#define YART_SLOT_NEE_DIR 5u       /* u0 = r1, u1 = r2 of that light's random() for the sample      */
#define YART_NEE_BOUNCE_BASE 0x10000u /* the shadow ray of bounce k is a world.hit of its own: it draws
                                      its ConstantMedium free paths at bounce YART_NEE_BOUNCE_BASE + k,
                                      so they do not reuse (and correlate with) the path's draws at k */
#define YART_RR_FIRST_BOUNCE 4u    /* roulette is played from this bounce on ...                    */
#define YART_RR_MIN_SURVIVAL 0.05  /* ... with survival probability clamp(throughput, this, 1)      */
#define YART_SLOT_SPHERE 0x100u    /* + 2*i, +2*i+1: i-th rejection iteration of
                                      random_in_unit_sphere (material.rs:308-324):
                                      x = 2*u0-1, y = 2*u1-1 (slot 2i), z = 2*u0-1 (slot 2i+1)      */
#define YART_SLOT_MEDIUM 0x1000u   /* + world object index: u0 = free-path draw of that
                                      ConstantMedium inside world.hit (hittable.rs:276-293)         */

#define YART_PHILOX_M0 0xD2511F53u
#define YART_PHILOX_M1 0xCD9E8D57u
#define YART_PHILOX_W0 0x9E3779B9u
#define YART_PHILOX_W1 0xBB67AE85u

#endif
