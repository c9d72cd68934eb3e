/*=========================================================================
 * itkCuberilleImageToMeshFilter.h — drop-in replacement of the reference header
 *   Source/itkCuberilleImageToMeshFilter.h (+ .txx)
 * whose GenerateData() runs on a B200 through the C-ABI of include/cuberille_c.h.
 *
 * Same class name, template parameters, typedefs and public interface as the
 * reference (h:110-228): SetInput, Set/GetIsoSurfaceValue, Set/GetInterpolator,
 * GenerateTriangleFaces / ProjectVerticesToIsoSurface with On/Off, the three
 * projection knobs with their clamp ranges, ProjectVertexMaximumNumberOfSteps,
 * plus SavePixelAsCellData (BASELINE.json north star; the reference only has
 * commented SetCellData stubs, txx:314,321,330).  Update() / GetOutput() come from
 * itk::ImageToMeshFilter as in the reference.  Constructor defaults: txx:31-41.
 *
 * This header contains NO algorithm: GenerateData() hands the image buffer to
 * libcuberille_cuda.so (cub_set_volume / cub_run / cub_fetch) and fills the
 * itk::Mesh with what comes back, in the reference's point and cell order.
 * Link with -lcuberille_cuda.  C-ABI errors become itk::ExceptionObject through
 * itkExceptionMacro, like every other ITK filter failure the reference's driver
 * catches (Testing/CuberilleTest01.cxx:207-212).
 *
 * Differences from the reference, all documented in DESIGN.md §7:
 *  - TInterpolator must be itk::LinearInterpolateImageFunction<TInputImage>
 *    (the device kernel implements ITK's trilinear interpolation; another
 *    interpolator type raises an exception instead of being silently ignored);
 *  - an oriented image (non-identity direction) is handled with ITK's oriented-image
 *    arithmetic (cuberille_c.h, cub_set_volume); a buffered region that does not
 *    start at index 0 is passed on (cub_set_region_index);
 *  - an empty voxel slice between occupied ones, where the reference's lookup-plane
 *    rotation merges vertices of different planes (txx:155-161), is meshed by the
 *    intended rule and reported through itkWarningMacro (cub_last_warning);
 *  - a zero image gradient stops a vertex instead of dividing by zero (txx:452),
 *    out-of-image interpolation reads are clamped instead of undefined.
 *=========================================================================*/
#ifndef __itkCuberilleImageToMeshFilter_h
#define __itkCuberilleImageToMeshFilter_h

#include <chrono>
#include <cstdint>
#include <type_traits>
#include <vector>

#include "itkMacro.h"
#include "itkMesh.h"
#include "itkImageToMeshFilter.h"
#include "itkCellInterface.h"
#include "itkTriangleCell.h"
#include "itkQuadrilateralCell.h"
#include "itkLinearInterpolateImageFunction.h"
#include "itkVectorLinearInterpolateImageFunction.h"
#include "itkConstShapedNeighborhoodIterator.h"
#include "itkGradientImageFilter.h"
#include "itkNumericTraits.h"

#include "cuberille_c.h"

// The reference selects its alternative projection schemes at compile time (h:22-23, all 0 by default); defining one
// of them to 1 before including this header selects the same scheme here (cub_params.projection_method).
#ifndef USE_ADVANCED_PROJECTION
#define USE_ADVANCED_PROJECTION 0
#endif
#ifndef USE_LINESEARCH_PROJECTION
#define USE_LINESEARCH_PROJECTION 0
#endif

namespace itk
{

namespace cuberille_detail
{
template <typename T> struct PixelCode;
template <> struct PixelCode<unsigned char>  { static const int value = CUB_U8; };
template <> struct PixelCode<signed char>    { static const int value = CUB_I8; };
template <> struct PixelCode<char>           { static const int value = std::is_signed<char>::value ? CUB_I8 : CUB_U8; };
template <> struct PixelCode<unsigned short> { static const int value = CUB_U16; };
template <> struct PixelCode<short>          { static const int value = CUB_I16; };
template <> struct PixelCode<unsigned int>   { static const int value = CUB_U32; };
template <> struct PixelCode<int>            { static const int value = CUB_I32; };
template <> struct PixelCode<float>          { static const int value = CUB_F32; };
template <> struct PixelCode<double>         { static const int value = CUB_F64; };
}

template < class TInputImage, class TOutputMesh, class TInterpolator = itk::LinearInterpolateImageFunction<TInputImage> >
class ITK_EXPORT CuberilleImageToMeshFilter : public ImageToMeshFilter< TInputImage, TOutputMesh >
{
public:
  /** Standard "Self" typedef. */
  typedef CuberilleImageToMeshFilter                    Self;
  typedef ImageToMeshFilter< TInputImage, TOutputMesh > Superclass;
  typedef SmartPointer<Self>                            Pointer;
  typedef SmartPointer<const Self>                      ConstPointer;

  itkNewMacro(Self);
  itkTypeMacro(CuberilleImageToMeshFilter, ImageToMeshFilter);

  /** Same convenience typedefs as the reference (h:126-159). */
  typedef TOutputMesh                           OutputMeshType;
  typedef typename OutputMeshType::Pointer      OutputMeshPointer;
  typedef typename OutputMeshType::MeshTraits   OutputMeshTraits;
  typedef typename OutputMeshType::PointType    OutputPointType;
  typedef typename OutputMeshTraits::PixelType  OutputPixelType;
  typedef typename OutputMeshType::CellTraits   CellTraits;
  typedef typename OutputMeshType::PointsContainerPointer PointsContainerPointer;
  typedef typename OutputMeshType::PointsContainer        PointsContainer;
  typedef typename OutputMeshType::CellsContainerPointer  CellsContainerPointer;
  typedef typename OutputMeshType::CellsContainer         CellsContainer;
  typedef typename OutputMeshType::PointIdentifier        PointIdentifier;
  typedef typename OutputMeshType::CellIdentifier         CellIdentifier;
  typedef CellInterface<OutputPixelType, CellTraits>      CellInterfaceType;
  typedef TriangleCell<CellInterfaceType>                 TriangleCellType;
  typedef typename TriangleCellType::SelfAutoPointer      TriangleAutoPointer;
  typedef typename TriangleCellType::CellAutoPointer      TriangleCellAutoPointer;
  typedef QuadrilateralCell<CellInterfaceType>            QuadrilateralCellType;
  typedef typename QuadrilateralCellType::SelfAutoPointer QuadrilateralAutoPointer;
  typedef typename QuadrilateralCellType::CellAutoPointer QuadrilateralCellAutoPointer;

  typedef TInputImage                               InputImageType;
  typedef typename InputImageType::Pointer          InputImagePointer;
  typedef typename InputImageType::ConstPointer     InputImageConstPointer;
  typedef typename InputImageType::PixelType        InputPixelType;
  typedef typename InputImageType::SizeType         SizeType;
  typedef typename InputImageType::SpacingType      SpacingType;
  typedef typename InputImageType::SpacingValueType SpacingValueType;
  typedef typename InputImageType::IndexType        IndexType;
  typedef typename OutputMeshType::PointType        PointType;

  typedef TInterpolator                      InterpolatorType;
  typedef typename InterpolatorType::Pointer InterpolatorPointer;
  typedef typename InterpolatorType::OutputType InterpolatorOutputType;

  /** Other convenient typedefs of the reference (h:163-175).  The library evaluates the iterator's boundary
   * condition, the gradient filter and its interpolator on the device; the types are exported because user code
   * may name them. */
  typedef ConstShapedNeighborhoodIterator< InputImageType > InputImageIteratorType;
  typedef GradientImageFilter< InputImageType >             GradientFilterType;
  typedef typename GradientFilterType::Pointer              GradientFilterPointer;
  typedef typename GradientFilterType::OutputImageType      GradientImageType;
  typedef typename GradientImageType::Pointer               GradientImagePointer;
  typedef typename GradientFilterType::OutputPixelType      GradientPixelType;
  typedef itk::VectorLinearInterpolateImageFunction< GradientImageType > GradientInterpolatorType;
  typedef typename GradientInterpolatorType::Pointer        GradientInterpolatorPointer;

  /** Get/set the iso-surface value (h:180-181): pixels >= this value are inside (txx:139-141). */
  itkGetMacro( IsoSurfaceValue, InputPixelType );
  itkSetMacro( IsoSurfaceValue, InputPixelType );

  /** Accept the input image (h:184, txx:53-56). */
  virtual void SetInput( const InputImageType * inputImage )
    {
    this->ProcessObject::SetNthInput( 0, const_cast< InputImageType * >( inputImage ) );
    }

  /** Get/set interpolate function (h:187-188).  Kept for source compatibility; only its TYPE matters. */
  itkGetObjectMacro( Interpolator, InterpolatorType );
  itkSetObjectMacro( Interpolator, InterpolatorType );

  /** True = triangle faces, false = quadrilateral faces; default true (h:193-195). */
  itkGetMacro( GenerateTriangleFaces, bool );
  itkSetMacro( GenerateTriangleFaces, bool );
  itkBooleanMacro( GenerateTriangleFaces );

  /** Project the vertices onto the iso-surface; default true (h:199-201). */
  itkGetMacro( ProjectVerticesToIsoSurface, bool );
  itkSetMacro( ProjectVerticesToIsoSurface, bool );
  itkBooleanMacro( ProjectVerticesToIsoSurface );

  /** Store the generating voxel's pixel value as cell data of every cell; default false. */
  itkGetMacro( SavePixelAsCellData, bool );
  itkSetMacro( SavePixelAsCellData, bool );
  itkBooleanMacro( SavePixelAsCellData );

  /** Extension (default false): number the vertices in raster order of the lattice corners instead of the
      reference's creation order.  Same points and connectivity up to that renumbering, less GPU work. */
  itkGetMacro( RasterVertexOrder, bool );
  itkSetMacro( RasterVertexOrder, bool );
  itkBooleanMacro( RasterVertexOrder );

  /** Opt-in, off by default (no counterpart in the reference, which leaves the mesh open where the
   * surface meets the image border, h:55-57 / the TODO at txx:133): treat everything outside the image
   * as outside the surface, i.e. mesh the image as if it were padded with one outside layer. */
  itkGetMacro( ImageBorderFaces, bool );
  itkSetMacro( ImageBorderFaces, bool );
  itkBooleanMacro( ImageBorderFaces );

  /** Extension (off by default): mesh the voxels whose value lies in [lower, upper] instead of those >= the iso value
   * (cub_set_inside_range).  A label k of a label map is SetLabelValue( k ) = the range [k, k]; a range of several labels
   * gives the surface of their union.  The projection needs an iso-surface, so Update() throws while a range is set and
   * ProjectVerticesToIsoSurface is on (the constructor default). */
  void SetInsideRange( InputPixelType lower, InputPixelType upper )
    {
    if ( !m_InsideRangeOn || m_InsideRangeLower != lower || m_InsideRangeUpper != upper )
      {
      m_InsideRangeOn = true;
      m_InsideRangeLower = lower;
      m_InsideRangeUpper = upper;
      this->Modified();
      }
    }
  void SetLabelValue( InputPixelType label ) { this->SetInsideRange( label, label ); }
  void InsideRangeOff()
    {
    if ( m_InsideRangeOn )
      {
      m_InsideRangeOn = false;
      this->Modified();
      }
    }
  itkGetMacro( InsideRangeOn, bool );
  itkGetMacro( InsideRangeLower, InputPixelType );
  itkGetMacro( InsideRangeUpper, InputPixelType );

  /** Projection knobs with the reference's clamp ranges (h:209-228). */
  itkGetMacro( ProjectVertexSurfaceDistanceThreshold, double );
  itkSetClampMacro( ProjectVertexSurfaceDistanceThreshold, double, 0.0, NumericTraits<InputPixelType>::max() );
  itkGetMacro( ProjectVertexStepLength, double );
  itkSetClampMacro( ProjectVertexStepLength, double, 0.0, 100000.0 );
  itkGetMacro( ProjectVertexStepLengthRelaxationFactor, double );
  itkSetClampMacro( ProjectVertexStepLengthRelaxationFactor, double, 0.0, 1.0 );
  itkGetMacro( ProjectVertexMaximumNumberOfSteps, unsigned int );
  itkSetMacro( ProjectVertexMaximumNumberOfSteps, unsigned int );

  /** CUDA device ordinal used by this filter instance (default 0). */
  itkGetMacro( Device, int );
  itkSetMacro( Device, int );

  /** Which ProjectVertexToIsoSurface scheme runs: CUB_PROJECT_DEFAULT (txx:440-474), CUB_PROJECT_ADVANCED (txx:340-397)
   * or CUB_PROJECT_LINESEARCH (txx:398-438).  The default follows the reference's compile-time switches. */
  itkGetMacro( ProjectionMethod, int );
  itkSetMacro( ProjectionMethod, int );

  /** Page-lock the input image buffer while GenerateData() runs (cudaHostRegister), default off.  Speeds up the
   * host -> device copy of large images; registering costs time of its own. */
  itkGetMacro( PinInputBuffer, bool );
  itkSetMacro( PinInputBuffer, bool );
  itkBooleanMacro( PinInputBuffer );

  /** Where the time of the last GenerateData() went, in milliseconds (host clock): [0] host -> device copy of the
   * image, [1] the kernels (cub_run), [2] device -> host copy of the mesh, [3] filling the itk::Mesh (one heap cell
   * per face, as ITK requires, txx:310-329), [4] total. */
  const double * GetLastTimings() const { return m_LastTimings; }

protected:
  CuberilleImageToMeshFilter()
    {
    // txx:31-41
    this->SetNumberOfRequiredInputs(1);
    m_IsoSurfaceValue = NumericTraits< InputPixelType >::One;
    m_GenerateTriangleFaces = true;
    m_ProjectVerticesToIsoSurface = true;
    m_SavePixelAsCellData = false;
    m_RasterVertexOrder = false;
    m_ImageBorderFaces = false;
    m_InsideRangeOn = false;
    m_InsideRangeLower = NumericTraits< InputPixelType >::One;
    m_InsideRangeUpper = NumericTraits< InputPixelType >::One;
    m_ProjectVertexSurfaceDistanceThreshold = 0.5;
    m_ProjectVertexStepLength = -1.0;
    m_ProjectVertexStepLengthRelaxationFactor = 0.95;
    m_ProjectVertexMaximumNumberOfSteps = 50;
    m_Device = 0;
    m_Handle = 0;
    m_PinInputBuffer = false;
    m_ProjectionMethod = USE_ADVANCED_PROJECTION ? CUB_PROJECT_ADVANCED
                       : ( USE_LINESEARCH_PROJECTION ? CUB_PROJECT_LINESEARCH : CUB_PROJECT_DEFAULT );
    for ( int i = 0; i < 5; i++ ) { m_LastTimings[i] = 0.0; }
    for ( int i = 0; i < 3; i++ ) { m_Staging[i] = 0; m_StagingBytes[i] = 0; }
    }

  ~CuberilleImageToMeshFilter()
    {
    if ( m_Handle )
      {
      for ( int i = 0; i < 3; i++ ) { if ( m_Staging[i] ) { cub_host_free( m_Handle, m_Staging[i] ); } }
      cub_destroy( m_Handle );
      }
    }

  void PrintSelf( std::ostream& os, Indent indent ) const
    {
    // txx:501-520
    Superclass::PrintSelf( os, indent );
    os << indent << "IsoSurfaceValue: "
       << static_cast< typename NumericTraits<InputPixelType>::PrintType >( m_IsoSurfaceValue ) << std::endl;
    os << indent << "GenerateTriangleFaces: " << m_GenerateTriangleFaces << std::endl;
    os << indent << "ProjectVerticesToIsoSurface: " << m_ProjectVerticesToIsoSurface << std::endl;
    os << indent << "SavePixelAsCellData: " << m_SavePixelAsCellData << std::endl;
    os << indent << "InsideRange: " << m_InsideRangeOn << " ["
       << static_cast< typename NumericTraits<InputPixelType>::PrintType >( m_InsideRangeLower ) << ", "
       << static_cast< typename NumericTraits<InputPixelType>::PrintType >( m_InsideRangeUpper ) << "]" << std::endl;
    }

  virtual void GenerateOutputInformation() { } // do nothing (h:236)

  /** The hot path: txx:59-216, executed by libcuberille_cuda.so. */
  void GenerateData()
    {
    if ( !std::is_same< TInterpolator, LinearInterpolateImageFunction<TInputImage> >::value )
      {
      itkExceptionMacro( << "the CUDA cuberille path implements itk::LinearInterpolateImageFunction only" );
      }
    InputImageConstPointer image = Superclass::GetInput( 0 );
    typename OutputMeshType::Pointer mesh = Superclass::GetOutput();

    // image geometry (txx:75-79, 266-270)
    const typename InputImageType::RegionType region = image->GetBufferedRegion();
    uint64_t dims[3];
    int64_t regionIndex[3];
    double spacing[3], origin[3], direction[9];
    double maxSpacing = 0.0;
    for ( unsigned int i = 0; i < 3; i++ )
      {
      regionIndex[i] = static_cast<int64_t>( region.GetIndex()[i] );  // TransformIndexToPhysicalPoint sees it (txx:266)
      dims[i] = region.GetSize()[i];
      spacing[i] = image->GetSpacing()[i];
      origin[i] = image->GetOrigin()[i];
      for ( unsigned int j = 0; j < 3; j++ ) { direction[3*i + j] = image->GetDirection()[i][j]; }
      maxSpacing = ( spacing[i] > maxSpacing ) ? spacing[i] : maxSpacing;
      }
    // sticky default step length (txx:82-85)
    if ( m_ProjectVertexStepLength < 0.0 )
      {
      m_ProjectVertexStepLength = maxSpacing * 0.25;
      }

    if ( !m_Handle )
      {
      if ( cub_create( m_Device, 0, &m_Handle ) != CUB_OK )
        {
        m_Handle = 0;
        itkExceptionMacro( << "cub_create failed: no usable CUDA device " << m_Device << " (there is no CPU fallback)" );
        }
      }
    typedef std::chrono::steady_clock Clock;
    const Clock::time_point t0 = Clock::now();
    // an itk::Image buffer is pageable memory: the copy to the device then runs at a fraction of the PCIe rate.
    // Page-locking it for the duration of the run (cudaHostRegister) is worth it for large images only.
    const uint64_t imageBytes = dims[0] * dims[1] * dims[2] * sizeof( InputPixelType );
    const bool pinned = m_PinInputBuffer &&
      cub_host_register( m_Handle, const_cast<InputPixelType *>( image->GetBufferPointer() ), imageBytes ) == CUB_OK;
    this->Check( cub_set_volume( m_Handle, image->GetBufferPointer(),
                                 cuberille_detail::PixelCode<InputPixelType>::value,
                                 dims, spacing, origin, direction, CUB_MEM_HOST ) );
    this->Check( cub_set_region_index( m_Handle, regionIndex ) );
    if ( m_InsideRangeOn )
      {
      if ( m_ProjectVerticesToIsoSurface )
        {
        itkExceptionMacro( << "an inside range has no iso-surface to project the vertices onto: call "
                           "ProjectVerticesToIsoSurfaceOff() (projection is on by default)" );
        }
      this->Check( cub_set_inside_range( m_Handle, 1, static_cast<double>( m_InsideRangeLower ),
                                         static_cast<double>( m_InsideRangeUpper ) ) );
      }
    this->Check( cub_synchronize( m_Handle ) );
    const Clock::time_point t1 = Clock::now();
    cub_params params;
    cub_default_params( &params );
    params.iso_value = static_cast<double>( m_IsoSurfaceValue );
    params.generate_triangles = m_GenerateTriangleFaces ? 1 : 0;
    params.project_vertices = m_ProjectVerticesToIsoSurface ? 1 : 0;
    params.save_pixel_as_cell_data = m_SavePixelAsCellData ? 1 : 0;
    params.vertex_order = m_RasterVertexOrder ? CUB_ORDER_RASTER : CUB_ORDER_REFERENCE;
    params.image_border_faces = m_ImageBorderFaces ? 1u : 0u;
    params.surface_distance_threshold = m_ProjectVertexSurfaceDistanceThreshold;
    params.step_length = m_ProjectVertexStepLength;
    params.step_relaxation = m_ProjectVertexStepLengthRelaxationFactor;
    params.max_steps = m_ProjectVertexMaximumNumberOfSteps;
    params.projection_method = m_ProjectionMethod;

    // PointIdentifier is unsigned long (64 bits), but a mesh of one handle has fewer than 2^32 points (cub_count
    // refuses more): the ids travel as 32-bit values - half the bytes over PCIe - and are widened when the cells
    // are created below.
    uint64_t numberOfPoints = 0, numberOfCells = 0;
    this->Check( cub_run( m_Handle, &params, 4, &numberOfPoints, &numberOfCells ) );
    this->Check( cub_synchronize( m_Handle ) );
    const Clock::time_point t2 = Clock::now();
    const char * warning = cub_last_warning( m_Handle );
    if ( warning && warning[0] ) { itkWarningMacro( << warning ); }

    // the mesh comes back through page-locked staging buffers that the filter keeps from run to run (grow-only):
    // a fresh pageable std::vector costs more in page faults than the copy itself
    const unsigned int verticesPerCell = m_GenerateTriangleFaces ? 3 : 4;
    this->Stage( 0, 3 * numberOfPoints * sizeof( float ) );
    this->Stage( 1, verticesPerCell * numberOfCells * sizeof( uint32_t ) );
    this->Stage( 2, m_SavePixelAsCellData ? numberOfCells * sizeof( InputPixelType ) : 0 );
    const float * points = static_cast<const float *>( m_Staging[0] );
    const uint32_t * cells = static_cast<const uint32_t *>( m_Staging[1] );
    const InputPixelType * cellData = static_cast<const InputPixelType *>( m_Staging[2] );
    this->Check( cub_fetch( m_Handle, numberOfPoints ? static_cast<float *>( m_Staging[0] ) : 0, numberOfCells ? m_Staging[1] : 0,
                            ( m_SavePixelAsCellData && numberOfCells ) ? m_Staging[2] : 0, CUB_MEM_HOST ) );
    const Clock::time_point t3 = Clock::now();

    // mesh->GetPoints()->InsertElement( id, vertex )   (txx:275)
    mesh->GetPoints()->Reserve( numberOfPoints );
    for ( uint64_t id = 0; id < numberOfPoints; id++ )
      {
      PointType p;
      p[0] = points[3*id]; p[1] = points[3*id + 1]; p[2] = points[3*id + 2];
      mesh->GetPoints()->SetElement( static_cast<PointIdentifier>( id ), p );
      }
    // mesh->SetCell( id, cell )   (txx:310-329): one heap cell per face, as ITK meshes require
    for ( uint64_t id = 0; id < numberOfCells; id++ )
      {
      PointIdentifier ids[4];
      for ( unsigned int k = 0; k < verticesPerCell; k++ )
        {
        ids[k] = static_cast<PointIdentifier>( cells[verticesPerCell*id + k] );
        }
      if ( m_GenerateTriangleFaces )
        {
        TriangleCellAutoPointer tri;
        tri.TakeOwnership( new TriangleCellType );
        tri->SetPointIds( ids );
        mesh->SetCell( static_cast<CellIdentifier>( id ), tri );
        }
      else
        {
        QuadrilateralCellAutoPointer quad;
        quad.TakeOwnership( new QuadrilateralCellType );
        quad->SetPointIds( ids );
        mesh->SetCell( static_cast<CellIdentifier>( id ), quad );
        }
      if ( m_SavePixelAsCellData )
        {
        mesh->SetCellData( static_cast<CellIdentifier>( id ), static_cast<OutputPixelType>( cellData[id] ) );
        }
      }
    if ( pinned )
      {
      cub_host_unregister( m_Handle, const_cast<InputPixelType *>( image->GetBufferPointer() ) );
      }
    const Clock::time_point t4 = Clock::now();
    m_LastTimings[0] = std::chrono::duration<double, std::milli>( t1 - t0 ).count();
    m_LastTimings[1] = std::chrono::duration<double, std::milli>( t2 - t1 ).count();
    m_LastTimings[2] = std::chrono::duration<double, std::milli>( t3 - t2 ).count();
    m_LastTimings[3] = std::chrono::duration<double, std::milli>( t4 - t3 ).count();
    m_LastTimings[4] = std::chrono::duration<double, std::milli>( t4 - t0 ).count();
    }

private:
  CuberilleImageToMeshFilter(const Self&); //purposely not implemented
  void operator=(const Self&);             //purposely not implemented

  /** page-locked staging buffer i of at least `bytes` bytes (grow-only) */
  void Stage( int i, uint64_t bytes )
    {
    if ( bytes <= m_StagingBytes[i] ) { return; }
    if ( m_Staging[i] ) { this->Check( cub_host_free( m_Handle, m_Staging[i] ) ); m_Staging[i] = 0; m_StagingBytes[i] = 0; }
    const uint64_t want = bytes + bytes / 8;
    this->Check( cub_host_alloc( m_Handle, want, &m_Staging[i] ) );
    m_StagingBytes[i] = want;
    }

  void Check( int status )
    {
    if ( status != CUB_OK )
      {
      itkExceptionMacro( << "cuberille C-ABI error " << status << ": " << cub_last_error( m_Handle ) );
      }
    }

  InputPixelType      m_IsoSurfaceValue;
  InterpolatorPointer m_Interpolator;
  bool                m_GenerateTriangleFaces;
  bool                m_ProjectVerticesToIsoSurface;
  bool                m_SavePixelAsCellData;
  bool                m_RasterVertexOrder;
  bool                m_ImageBorderFaces;
  bool                m_InsideRangeOn;
  InputPixelType      m_InsideRangeLower;
  InputPixelType      m_InsideRangeUpper;
  double              m_ProjectVertexSurfaceDistanceThreshold;
  double              m_ProjectVertexStepLength;
  double              m_ProjectVertexStepLengthRelaxationFactor;
  unsigned int        m_ProjectVertexMaximumNumberOfSteps;
  int                 m_Device;
  cub_handle          m_Handle;
  bool                m_PinInputBuffer;
  int                 m_ProjectionMethod;
  double              m_LastTimings[5];
  void *              m_Staging[3];
  uint64_t            m_StagingBytes[3];
};

} // end namespace itk

#endif
