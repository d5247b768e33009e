//! `strolle::Engine<P>` on B200s.
//!
//! The public surface of the reference crate (`/strolle/src/lib.rs:104-409`: `Engine`, `Camera`, `CameraMode`, `CameraViewport`, `Mesh`,
//! `MeshTriangle`, `Material`, `AlphaMode`, `Light`, `Instance`, `Image`, `ImageData`, `Sun`, `Params`), with every method forwarding
//! to the C ABI of `libstrolle_b200.so` (`strolle-b200-sys`).  What differs, and why:
//!
//! * `Engine::new` takes CUDA device ordinals instead of a `&wgpu::Device`; one ordinal = one GPU, several = the frame is partitioned
//!   into row strips across them (`st_multi_*`), or, with `create_camera_on`, each camera lives whole on one of them.
//!   `create_camera` / `update_camera` / `tick` lose their `device` / `queue` arguments.
//! * `render_camera` delivers the composed frame into a [`Frame`] (host pixels in the viewport's format) instead of recording into a
//!   wgpu command encoder — the CUDA kernels run on the engine's own stream.  A wgpu host uploads it with `Queue::write_texture`
//!   (what `bevy-strolle-b200` does); `render_camera_to_raw` composes straight into a caller-owned surface in device or host memory
//!   with a row pitch (e.g. a texture imported through CUDA external memory).
//! * `ImageData::Texture` (a live wgpu texture) cannot be sampled from CUDA.  Its dynamic case, a texture that the atlas copies at every
//!   tick, is `insert_dynamic_image_raw` over a CUDA address instead (device, managed or page-locked host memory, e.g. another camera's
//!   `render_camera_to_raw` target); a static texture is passed as `ImageData::Raw`.
//! * Misuse returns `Err(Error)` where the reference panics (`triangles.rs:44-53`, `camera_controllers.rs:21-25`); the infallible
//!   scene verbs log the error and carry on like the reference's `warn!` paths (`images.rs:71-79`).
use std::collections::HashMap;
use std::ffi::CStr;
use std::fmt::{self, Debug};
use std::hash::Hash;
use std::marker::PhantomData;
use std::os::raw::{c_int, c_void};

pub use glam;
use glam::{Affine3A, Mat4, UVec2, Vec2, Vec3, Vec4};
use strolle_b200_sys as sys;

/// Parameters used by Strolle to index textures, meshes etc. (`lib.rs:402-409`; `ImageTexture` has no CUDA meaning and is gone).
pub trait Params {
    type ImageHandle: Clone + Copy + Debug + Eq + Hash;
    type InstanceHandle: Clone + Copy + Debug + Eq + Hash;
    type LightHandle: Clone + Copy + Debug + Eq + Hash;
    type MaterialHandle: Clone + Copy + Debug + Eq + Hash;
    type MeshHandle: Clone + Copy + Debug + Eq + Hash;
}

#[derive(Clone, Debug)]
pub struct Error {
    pub code: i32,
    pub message: String,
}

impl fmt::Display for Error {
    fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result {
        write!(f, "strolle_b200 error {}: {}", self.code, self.message)
    }
}

impl std::error::Error for Error {}

fn check(code: c_int) -> Result<(), Error> {
    if code == sys::ST_OK {
        return Ok(());
    }
    let message = unsafe { CStr::from_ptr(sys::st_last_error()) }.to_string_lossy().into_owned();
    Err(Error { code, message })
}

fn soft(what: &str, code: c_int) {
    if let Err(err) = check(code) {
        log::warn!("{what}: {err}");
    }
}

// ---- scene types ------------------------------------------------------------------------------------------------------------------

/// `strolle::MeshTriangle` (`mesh_triangle.rs:7-45`)
#[derive(Clone, Debug, Default)]
pub struct MeshTriangle {
    positions: [Vec3; 3],
    normals: [Vec3; 3],
    uvs: [Vec2; 3],
    tangents: [Vec4; 3],
}

impl MeshTriangle {
    pub fn with_positions(mut self, positions: [impl Into<Vec3>; 3]) -> Self {
        self.positions = positions.map(Into::into);
        self
    }
    pub fn with_normals(mut self, normals: [impl Into<Vec3>; 3]) -> Self {
        self.normals = normals.map(Into::into);
        self
    }
    pub fn with_uvs(mut self, uvs: [impl Into<Vec2>; 3]) -> Self {
        self.uvs = uvs.map(Into::into);
        self
    }
    pub fn with_tangents(mut self, tangents: [impl Into<Vec4>; 3]) -> Self {
        self.tangents = tangents.map(Into::into);
        self
    }
    pub fn positions(&self) -> [Vec3; 3] {
        self.positions
    }
    pub fn normals(&self) -> [Vec3; 3] {
        self.normals
    }
    pub fn uvs(&self) -> [Vec2; 3] {
        self.uvs
    }
    fn to_ffi(&self) -> sys::st_mesh_triangle {
        sys::st_mesh_triangle {
            positions: self.positions.map(|v| v.to_array()),
            normals: self.normals.map(|v| v.to_array()),
            uvs: self.uvs.map(|v| v.to_array()),
            tangents: self.tangents.map(|v| v.to_array()),
        }
    }
}

/// `strolle::Mesh` (`mesh.rs:3-16`)
#[derive(Clone, Debug)]
pub struct Mesh {
    triangles: Vec<MeshTriangle>,
}

impl Mesh {
    pub fn new(triangles: Vec<MeshTriangle>) -> Self {
        Self { triangles }
    }
}

#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub enum AlphaMode {
    #[default]
    Opaque,
    Blend,
}

/// `strolle::Material` (`material.rs:8-23`)
#[derive(Clone, Debug)]
pub struct Material<P: Params> {
    pub base_color: Vec4,
    pub base_color_texture: Option<P::ImageHandle>,
    pub emissive: Vec4,
    pub emissive_texture: Option<P::ImageHandle>,
    pub perceptual_roughness: f32,
    pub metallic: f32,
    pub metallic_roughness_texture: Option<P::ImageHandle>,
    pub reflectance: f32,
    pub ior: f32,
    pub normal_map_texture: Option<P::ImageHandle>,
    pub alpha_mode: AlphaMode,
}

impl<P: Params> Default for Material<P> {
    fn default() -> Self {
        Self {
            base_color: Vec4::ONE,
            base_color_texture: None,
            emissive: Vec4::ZERO,
            emissive_texture: None,
            perceptual_roughness: 0.5,
            metallic: 0.0,
            metallic_roughness_texture: None,
            reflectance: 0.5,
            ior: 1.0,
            normal_map_texture: None,
            alpha_mode: AlphaMode::Opaque,
        }
    }
}

/// `strolle::Light` (`light.rs:6-22`)
#[derive(Clone, Debug)]
pub enum Light {
    Point { position: Vec3, radius: f32, color: Vec3, range: f32 },
    Spot { position: Vec3, radius: f32, color: Vec3, range: f32, direction: Vec3, angle: f32 },
}

impl Light {
    fn to_ffi(&self) -> sys::st_light {
        match *self {
            Light::Point { position, radius, color, range } => sys::st_light {
                kind: sys::ST_LIGHT_POINT,
                position: position.to_array(),
                radius,
                color: color.to_array(),
                range,
                direction: [0.0; 3],
                angle: 0.0,
            },
            Light::Spot { position, radius, color, range, direction, angle } => sys::st_light {
                kind: sys::ST_LIGHT_SPOT,
                position: position.to_array(),
                radius,
                color: color.to_array(),
                range,
                direction: direction.to_array(),
                angle,
            },
        }
    }
}

/// `strolle::Instance` (`instance.rs:6-31`)
#[derive(Debug)]
pub struct Instance<P: Params> {
    mesh_handle: P::MeshHandle,
    material_handle: P::MaterialHandle,
    transform: Affine3A,
}

impl<P: Params> Instance<P> {
    pub fn new(mesh_handle: P::MeshHandle, material_handle: P::MaterialHandle, transform: Affine3A) -> Self {
        Self { mesh_handle, material_handle, transform }
    }
}

/// `strolle::ImageData::Raw` (`image.rs:36-47`): tightly packed RGBA8 texels of an `Rgba8UnormSrgb` image
#[derive(Debug)]
pub enum ImageData {
    Raw { data: Vec<u8> },
}

/// `strolle::Image` (`image.rs:3-34`)
#[derive(Debug)]
pub struct Image {
    data: ImageData,
    size: UVec2,
}

impl Image {
    pub fn new(data: ImageData, size: UVec2) -> Self {
        Self { data, size }
    }
}

/// `strolle::Sun` (`sun.rs:1-14`)
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct Sun {
    pub azimuth: f32,
    pub altitude: f32,
}

impl Default for Sun {
    fn default() -> Self {
        Self { azimuth: 0.0, altitude: 0.35 }
    }
}

// ---- cameras ----------------------------------------------------------------------------------------------------------------------

/// `strolle::CameraMode` (`camera.rs:83-105`)
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum CameraMode {
    Image { denoise: bool },
    DiDiffuse { denoise: bool },
    DiSpecular { denoise: bool },
    GiDiffuse { denoise: bool },
    GiSpecular { denoise: bool },
    BvhHeatmap,
    Reference { depth: u8 },
}

impl Default for CameraMode {
    fn default() -> Self {
        Self::Image { denoise: true }
    }
}

/// The formats the engine composes into (`CameraViewport::format`, `camera.rs:170-185`).  `Rgba16Float` is the format of an HDR
/// Bevy view target (`ViewTarget::TEXTURE_FORMAT_HDR`), which is what the reference's Bevy plugin renders into.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum ViewportFormat {
    Rgba8UnormSrgb,
    Rgba16Float,
    Rgba32Float,
}

impl ViewportFormat {
    pub fn bytes_per_pixel(self) -> usize {
        match self {
            Self::Rgba8UnormSrgb => 4,
            Self::Rgba16Float => 8,
            Self::Rgba32Float => 16,
        }
    }
    fn to_ffi(self) -> c_int {
        match self {
            Self::Rgba8UnormSrgb => sys::ST_FORMAT_RGBA8_SRGB,
            Self::Rgba16Float => sys::ST_FORMAT_RGBA16F,
            Self::Rgba32Float => sys::ST_FORMAT_RGBA32F,
        }
    }
}

#[derive(Clone, Debug)]
pub struct CameraViewport {
    pub format: ViewportFormat,
    pub size: UVec2,
    pub position: UVec2,
}

impl Default for CameraViewport {
    fn default() -> Self {
        Self { format: ViewportFormat::Rgba8UnormSrgb, size: UVec2::new(512, 512), position: UVec2::ZERO }
    }
}

/// `strolle::Camera` (`camera.rs:8-14`)
#[derive(Clone, Debug, Default)]
pub struct Camera {
    pub mode: CameraMode,
    pub viewport: CameraViewport,
    pub transform: Mat4,
    pub projection: Mat4,
}

impl Camera {
    fn to_ffi(&self) -> sys::st_camera {
        let (mode, denoise, ref_depth) = match self.mode {
            CameraMode::Image { denoise } => (sys::ST_MODE_IMAGE, denoise, 0),
            CameraMode::DiDiffuse { denoise } => (sys::ST_MODE_DI_DIFFUSE, denoise, 0),
            CameraMode::DiSpecular { denoise } => (sys::ST_MODE_DI_SPECULAR, denoise, 0),
            CameraMode::GiDiffuse { denoise } => (sys::ST_MODE_GI_DIFFUSE, denoise, 0),
            CameraMode::GiSpecular { denoise } => (sys::ST_MODE_GI_SPECULAR, denoise, 0),
            CameraMode::BvhHeatmap => (sys::ST_MODE_BVH_HEATMAP, false, 0),
            CameraMode::Reference { depth } => (sys::ST_MODE_REFERENCE, false, depth as i32),
        };
        sys::st_camera {
            mode,
            denoise: denoise as i32,
            ref_depth,
            width: self.viewport.size.x,
            height: self.viewport.size.y,
            transform: self.transform.to_cols_array(),
            projection: self.projection.to_cols_array(),
        }
    }
}

#[derive(Clone, Copy, Debug, PartialEq, Eq, Hash)]
pub struct CameraHandle(sys::st_camera_handle);

/// Where [`Engine::create_camera_on`] puts a camera: whole on one device of the group (view parallelism), instead of split into row
/// strips across all of them.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum Placement {
    /// The device at this index of the list given to [`Engine::new`].
    Device(usize),
    /// The device with the fewest pixels of placed cameras, the lowest index on a tie; decided at creation only.
    Auto,
}

/// Host pixels of one composed frame, `viewport.size.x * viewport.size.y` texels of `format`, row-major.  Allocate once per camera
/// (page-locked memory makes the device-to-host copy asynchronous and full speed) and reuse.
#[derive(Debug)]
pub struct Frame {
    pub format: ViewportFormat,
    pub size: UVec2,
    pub pixels: Vec<u8>,
}

impl Frame {
    pub fn new(viewport: &CameraViewport) -> Self {
        let n = viewport.size.x as usize * viewport.size.y as usize * viewport.format.bytes_per_pixel();
        Self { format: viewport.format, size: viewport.size, pixels: vec![0; n] }
    }
}

// ---- engine -----------------------------------------------------------------------------------------------------------------------

/// Maps the host's own handle types (`P::*Handle`) to the opaque `u64` handles of the C ABI.
#[derive(Debug)]
struct Interner<H: Copy + Eq + Hash> {
    ids: HashMap<H, u64>,
    next: u64,
}

impl<H: Copy + Eq + Hash> Default for Interner<H> {
    fn default() -> Self {
        Self { ids: HashMap::new(), next: 1 }
    }
}

impl<H: Copy + Eq + Hash> Interner<H> {
    fn id(&mut self, handle: H) -> u64 {
        if let Some(id) = self.ids.get(&handle) {
            return *id;
        }
        let id = self.next;
        self.next += 1;
        self.ids.insert(handle, id);
        id
    }
    fn get(&self, handle: H) -> Option<u64> {
        self.ids.get(&handle).copied()
    }
    fn forget(&mut self, handle: H) -> Option<u64> {
        self.ids.remove(&handle)
    }
}

/// `strolle::Engine<P>` (`lib.rs:104-395`) over one or several B200s.
pub struct Engine<P: Params> {
    raw: *mut sys::st_multi,
    meshes: Interner<P::MeshHandle>,
    materials: Interner<P::MaterialHandle>,
    images: Interner<P::ImageHandle>,
    instances: Interner<P::InstanceHandle>,
    lights: Interner<P::LightHandle>,
    viewports: HashMap<CameraHandle, CameraViewport>,
    _params: PhantomData<P>,
}

// The C ABI is externally synchronised (single writer) like `ResMut<Engine>` in the host; the raw pointer is not aliased.
unsafe impl<P: Params> Send for Engine<P> {}
unsafe impl<P: Params> Sync for Engine<P> {}

impl<P: Params> Debug for Engine<P> {
    fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result {
        write!(f, "Engine({} device(s))", unsafe { sys::st_multi_size(self.raw) })
    }
}

impl<P: Params> Engine<P> {
    /// `Engine::new` (`lib.rs:132-158`).  `devices` = CUDA ordinals; more than one partitions every camera's frame into row strips.
    pub fn new(devices: &[i32]) -> Result<Self, Error> {
        log::info!("Initializing on CUDA device(s) {devices:?}");
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::st_multi_create(devices.as_ptr(), devices.len() as c_int, &mut raw) })?;
        // the 256x256 RGBA8 blue-noise tile the reference embeds as a PNG (`noise.rs:30-66`, strolle/assets/blue-noise.png)
        static BLUE_NOISE: &[u8] = include_bytes!("../../../strolle_b200/assets/blue_noise_256_rgba8.bin");
        check(unsafe { sys::st_multi_set_blue_noise(raw, BLUE_NOISE.as_ptr()) })?;
        Ok(Self {
            raw,
            meshes: Default::default(),
            materials: Default::default(),
            images: Default::default(),
            instances: Default::default(),
            lights: Default::default(),
            viewports: HashMap::new(),
            _params: PhantomData,
        })
    }

    /// Creates or updates a mesh (`lib.rs:161-164`).
    pub fn insert_mesh(&mut self, handle: P::MeshHandle, item: Mesh) {
        let id = self.meshes.id(handle);
        let tris: Vec<sys::st_mesh_triangle> = item.triangles.iter().map(MeshTriangle::to_ffi).collect();
        soft("insert_mesh", unsafe { sys::st_multi_insert_mesh(self.raw, id, tris.as_ptr(), tris.len()) });
    }

    /// Removes a mesh (`lib.rs:166-171`); instances that refer to it are not removed.
    pub fn remove_mesh(&mut self, handle: P::MeshHandle) {
        if let Some(id) = self.meshes.forget(handle) {
            soft("remove_mesh", unsafe { sys::st_multi_remove_mesh(self.raw, id) });
        }
    }

    /// Creates or updates a material (`lib.rs:174-181`).
    pub fn insert_material(&mut self, handle: P::MaterialHandle, item: Material<P>) {
        let id = self.materials.id(handle);
        let ffi = sys::st_material {
            base_color: item.base_color.to_array(),
            emissive: item.emissive.to_array(),
            perceptual_roughness: item.perceptual_roughness,
            metallic: item.metallic,
            reflectance: item.reflectance,
            ior: item.ior,
            alpha_blend: (item.alpha_mode == AlphaMode::Blend) as i32,
        };
        soft("insert_material", unsafe { sys::st_multi_insert_material(self.raw, id, &ffi) });
        let slots = [item.base_color_texture, item.emissive_texture, item.metallic_roughness_texture, item.normal_map_texture];
        let mut tex = sys::st_material_textures::default();
        let mut ids = [0u64; 4];
        for (k, slot) in slots.iter().enumerate() {
            if let Some(image) = slot {
                ids[k] = self.images.id(*image);
                tex.mask |= 1 << k;
            }
        }
        tex.base_color = ids[0];
        tex.emissive = ids[1];
        tex.metallic_roughness = ids[2];
        tex.normal_map = ids[3];
        soft("insert_material (textures)", unsafe { sys::st_multi_set_material_textures(self.raw, id, &tex) });
    }

    /// Returns whether given material exists (`lib.rs:184-186`).
    pub fn has_material(&self, handle: P::MaterialHandle) -> bool {
        match self.materials.get(handle) {
            Some(id) => unsafe { sys::st_multi_has_material(self.raw, id) != 0 },
            None => false,
        }
    }

    /// Removes a material (`lib.rs:192-195`).
    pub fn remove_material(&mut self, handle: P::MaterialHandle) {
        if let Some(id) = self.materials.forget(handle) {
            soft("remove_material", unsafe { sys::st_multi_remove_material(self.raw, id) });
        }
    }

    /// Creates or updates an image (`lib.rs:198-205`).
    pub fn insert_image(&mut self, handle: P::ImageHandle, image: Image) {
        let id = self.images.id(handle);
        let ImageData::Raw { data } = &image.data;
        let expected = image.size.x as usize * image.size.y as usize * 4;
        if data.len() != expected {
            log::warn!("insert_image: {} bytes given, {}x{} RGBA8 needs {expected}; image skipped", data.len(), image.size.x, image.size.y);
            return;
        }
        soft("insert_image", unsafe { sys::st_multi_insert_image(self.raw, id, data.as_ptr(), image.size.x, image.size.y) });
    }

    /// Creates or updates a dynamic image (`ImageData::Texture { is_dynamic: true }`, `images.rs:97-102`): its texels live in a
    /// caller-owned surface of `size.x * size.y` Rgba8UnormSrgb texels, rows `pitch_bytes` apart (0 = packed), which every
    /// [`Self::tick`] copies into the image's atlas rectangle before the tick's other work, and after the writes the engine itself queued
    /// to it.  A camera that renders into the surface with [`Self::render_camera_to_raw`] and [`ViewportFormat::Rgba8UnormSrgb`] is
    /// therefore seen by the other cameras one frame later, as in the reference.  [`Self::remove_image`], [`Self::insert_image`] or
    /// another call of this on the handle end the refresh; they return once the engine no longer reads the old surface.
    ///
    /// # Safety
    /// `src` must point to device memory every device of the group can reach, managed memory, or page-locked host memory, of at least
    /// `(size.y - 1) * pitch_bytes + size.x * 4` bytes, valid until the refresh ends.  Writes to it from other CUDA streams must be
    /// ordered before [`Self::tick`] by the caller.
    pub unsafe fn insert_dynamic_image_raw(&mut self, handle: P::ImageHandle, src: *const u8, pitch_bytes: usize, size: UVec2) -> Result<(), Error> {
        let id = self.images.id(handle);
        check(sys::st_multi_insert_dynamic_image(self.raw, id, src as *const c_void, pitch_bytes, size.x, size.y))
    }

    /// Removes an image (`lib.rs:211-214`).
    pub fn remove_image(&mut self, handle: P::ImageHandle) {
        if let Some(id) = self.images.forget(handle) {
            soft("remove_image", unsafe { sys::st_multi_remove_image(self.raw, id) });
        }
    }

    /// Creates or updates an instance (`lib.rs:217-223`).
    pub fn insert_instance(&mut self, handle: P::InstanceHandle, instance: Instance<P>) {
        let id = self.instances.id(handle);
        let mesh = self.meshes.id(instance.mesh_handle);
        let material = self.materials.id(instance.material_handle);
        let m = instance.transform.matrix3;
        let t = instance.transform.translation;
        let affine = [m.x_axis.x, m.x_axis.y, m.x_axis.z, m.y_axis.x, m.y_axis.y, m.y_axis.z, m.z_axis.x, m.z_axis.y, m.z_axis.z, t.x, t.y, t.z];
        soft("insert_instance", unsafe { sys::st_multi_insert_instance(self.raw, id, mesh, material, affine.as_ptr()) });
    }

    /// Removes an instance (`lib.rs:226-229`).
    pub fn remove_instance(&mut self, handle: P::InstanceHandle) {
        if let Some(id) = self.instances.forget(handle) {
            soft("remove_instance", unsafe { sys::st_multi_remove_instance(self.raw, id) });
        }
    }

    /// Creates or updates a light (`lib.rs:232-234`).
    pub fn insert_light(&mut self, handle: P::LightHandle, item: Light) {
        let id = self.lights.id(handle);
        soft("insert_light", unsafe { sys::st_multi_insert_light(self.raw, id, &item.to_ffi()) });
    }

    /// Removes a light (`lib.rs:237-239`).
    pub fn remove_light(&mut self, handle: P::LightHandle) {
        if let Some(id) = self.lights.forget(handle) {
            soft("remove_light", unsafe { sys::st_multi_remove_light(self.raw, id) });
        }
    }

    /// Updates sun's parameters (`lib.rs:242-245`).
    pub fn update_sun(&mut self, sun: Sun) {
        soft("update_sun", unsafe { sys::st_multi_update_sun(self.raw, sun.azimuth, sun.altitude) });
    }

    /// Creates a new camera (`lib.rs:252-259`): allocates its per-camera buffers on every device of the group.
    pub fn create_camera(&mut self, camera: Camera) -> Result<CameraHandle, Error> {
        let mut out = 0;
        check(unsafe { sys::st_multi_create_camera(self.raw, &camera.to_ffi(), &mut out) })?;
        let handle = CameraHandle(out);
        self.viewports.insert(handle, camera.viewport);
        Ok(handle)
    }

    /// Creates a camera that lives whole on one device of the group: its buffers exist there only, and it renders whole frames there
    /// with no exchange between devices.  Many small independent views (split screen, monitors, mirrors) spread this way across the
    /// devices and render concurrently through [`Self::render_cameras_to_raw`]; one large view is better split with [`Self::create_camera`].
    pub fn create_camera_on(&mut self, camera: Camera, placement: Placement) -> Result<CameraHandle, Error> {
        let rank = match placement {
            Placement::Device(index) => c_int::try_from(index).map_err(|_| Error { code: sys::ST_ERR_INVALID, message: "device index out of range".into() })?,
            Placement::Auto => sys::ST_PLACE_AUTO,
        };
        let mut out = 0;
        check(unsafe { sys::st_multi_create_camera_on(self.raw, &camera.to_ffi(), rank, &mut out) })?;
        let handle = CameraHandle(out);
        self.viewports.insert(handle, camera.viewport);
        Ok(handle)
    }

    /// Moves a camera made by [`Self::create_camera_on`], with all of its temporal state, to the device at `device` of the group; its
    /// next frame is the one it would have rendered where it was.  Waits for the camera's queued work first.
    pub fn move_camera(&mut self, handle: CameraHandle, device: usize) -> Result<(), Error> {
        let rank = c_int::try_from(device).map_err(|_| Error { code: sys::ST_ERR_INVALID, message: "device index out of range".into() })?;
        check(unsafe { sys::st_multi_move_camera(self.raw, handle.0, rank) })
    }

    /// Updates camera, changing its mode, position, size etc. (`lib.rs:262-273`).
    pub fn update_camera(&mut self, handle: CameraHandle, camera: Camera) -> Result<(), Error> {
        check(unsafe { sys::st_multi_update_camera(self.raw, handle.0, &camera.to_ffi()) })?;
        self.viewports.insert(handle, camera.viewport);
        Ok(())
    }

    /// Renders camera (`lib.rs:279-286`) and delivers the composed frame into `target`, whose format and size must be the
    /// viewport's.  Returns once the pixels are in `target`.
    pub fn render_camera(&self, handle: CameraHandle, target: &mut Frame) -> Result<(), Error> {
        let viewport = self.viewports.get(&handle).ok_or_else(|| Error { code: sys::ST_ERR_NOT_FOUND, message: "unknown camera".into() })?;
        if target.format != viewport.format || target.size != viewport.size {
            return Err(Error { code: sys::ST_ERR_INVALID, message: "target frame does not match the camera's viewport".into() });
        }
        check(unsafe { sys::st_multi_render_camera(self.raw, handle.0, target.pixels.as_mut_ptr().cast(), target.format.to_ffi()) })
    }

    /// Renders camera (`lib.rs:279-286`) into a caller-owned surface, as the reference's composition pass does into the view's
    /// texture at `viewport.position` (`LoadOp::Load`: only the viewport's `size.x * size.y` texels are written).
    ///
    /// `dst` is the address of the viewport's first texel inside the surface (the caller adds `position.y * pitch_bytes +
    /// position.x * format.bytes_per_pixel()`), `pitch_bytes` the distance between rows (0 = tightly packed).  The surface may be
    /// device memory (a device of the group or one it reaches by peer access, e.g. a Vulkan image imported as CUDA external memory)
    /// or host memory; device surfaces are written by the engine's kernels and the call returns once they are enqueued.
    ///
    /// # Safety
    /// `dst` must point to a surface of at least `(size.y - 1) * pitch_bytes + size.x * format.bytes_per_pixel()` bytes that stays
    /// valid, and is not otherwise accessed, until the engine's work is done.
    pub unsafe fn render_camera_to_raw(&self, handle: CameraHandle, dst: *mut c_void, pitch_bytes: usize, format: ViewportFormat) -> Result<(), Error> {
        check(sys::st_multi_render_camera_to(self.raw, handle.0, dst, pitch_bytes, format.to_ffi()))
    }

    /// Renders several cameras for this frame, each as [`Self::render_camera_to_raw`] with `dsts[i]` and `pitches[i]` would, bit for
    /// bit; cameras of one size and mode run as one launch per pass.  A null `dsts[i]` renders camera `i` without output; empty
    /// `dsts` / `pitches` mean no outputs / packed rows.  In a group of several devices the cameras must have been made by
    /// [`Self::create_camera_on`]: every device renders the listed cameras it holds, all devices at once, and a surface may be on any
    /// device the camera's device reaches.
    ///
    /// # Safety
    /// Every non-null `dsts[i]` must satisfy the requirements of [`Self::render_camera_to_raw`] for camera `handles[i]`.
    pub unsafe fn render_cameras_to_raw(&self, handles: &[CameraHandle], dsts: &[*mut c_void], pitches: &[usize], format: ViewportFormat) -> Result<(), Error> {
        if (!dsts.is_empty() && dsts.len() != handles.len()) || (!pitches.is_empty() && pitches.len() != handles.len()) {
            return Err(Error { code: sys::ST_ERR_INVALID, message: "one surface and one pitch per camera".into() });
        }
        let cameras: Vec<sys::st_camera_handle> = handles.iter().map(|h| h.0).collect();
        check(sys::st_multi_render_cameras(
            self.raw,
            cameras.as_ptr(),
            cameras.len() as c_int,
            if dsts.is_empty() { std::ptr::null() } else { dsts.as_ptr() },
            if pitches.is_empty() { std::ptr::null() } else { pitches.as_ptr() },
            format.to_ffi(),
        ))
    }

    /// Enqueues the camera's passes without reading the frame back (e.g. `CameraMode::Reference` accumulation frames).
    pub fn render_camera_offscreen(&self, handle: CameraHandle) -> Result<(), Error> {
        check(unsafe { sys::st_multi_render_camera(self.raw, handle.0, std::ptr::null_mut(), sys::ST_FORMAT_RGBA32F) })
    }

    /// Deletes a camera (`lib.rs:292-294`).
    pub fn delete_camera(&mut self, handle: CameraHandle) -> Result<(), Error> {
        self.viewports.remove(&handle);
        check(unsafe { sys::st_multi_delete_camera(self.raw, handle.0) })
    }

    /// Sends all changes to the GPUs and prepares them for the upcoming frame (`lib.rs:301-395`); call once per frame before
    /// [`Self::render_camera`].
    pub fn tick(&mut self) -> Result<(), Error> {
        check(unsafe { sys::st_multi_tick(self.raw) })
    }

    /// Engine options of the C ABI (`ST_OPT_*`), applied to every device.
    pub fn set_option(&mut self, option: i32, value: i32) -> Result<(), Error> {
        check(unsafe { sys::st_multi_set_option(self.raw, option, value) })
    }
}

impl<P: Params> Drop for Engine<P> {
    fn drop(&mut self) {
        unsafe { sys::st_multi_destroy(self.raw) };
    }
}
